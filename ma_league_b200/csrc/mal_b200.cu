// libmal_b200.so -- C ABI (include/mal_b200.h) over the sm_100a kernels.  Host side: argument checks,
// workspace planning and launches only.  No allocation, no synchronisation, no CPU fallback.
#include <stdarg.h>
#include <string.h>
#include <utility>
#include "mal_common.cuh"
#include "replay.cuh"
#include "actsel.cuh"
#include "learner.cuh"
#include "gru_rec.cuh"
#include "tc_gemm.cuh"
#include "gru_rec_tc.cuh"
#include "agent_in_gemm.cuh"
#include "tc_reduce.cuh"
#include "autograd.cuh"
#include "per.cuh"
#include "td_lambda.cuh"

// ---------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
void mal_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
extern "C" const char *mal_last_error(void) { return g_err; }
extern "C" int mal_version(void) { return MAL_ABI_VERSION; }

// ---------------------------------------------------------------------------------------------
// launch accounting + opt-in per-kernel timing (CUDA events on the launching stream; bench.py's roofline leg)
// ---------------------------------------------------------------------------------------------
#define PROF_MAX 8192
static uint64_t g_launches = 0;
static bool g_prof_on = false;
static int g_prof_n = 0;
static cudaEvent_t g_prof_ev[PROF_MAX][2];
static const char *g_prof_name[PROF_MAX];
static bool g_prof_created = false;

struct ProfScope {
    int slot;
    cudaStream_t st;
    ProfScope(const char *name, cudaStream_t stream) : slot(-1), st(stream) {
        ++g_launches;
        if (g_prof_on && g_prof_n < PROF_MAX) {
            slot = g_prof_n++;
            g_prof_name[slot] = name;
            cudaEventRecord(g_prof_ev[slot][0], st);
        }
    }
    ~ProfScope() {
        if (slot >= 0) cudaEventRecord(g_prof_ev[slot][1], st);
    }
};

extern "C" uint64_t mal_launch_count(void) { return g_launches; }
// a replayed CUDA graph launches its captured kernels without passing through this library: the host layer reports them
extern "C" void mal_count_launches(uint64_t n) { g_launches += n; }

extern "C" int mal_profile_begin(void) {
    if (!g_prof_created) {
        for (int i = 0; i < PROF_MAX; ++i) {
            MAL_CUDA(cudaEventCreate(&g_prof_ev[i][0]));
            MAL_CUDA(cudaEventCreate(&g_prof_ev[i][1]));
        }
        g_prof_created = true;
    }
    g_prof_n = 0;
    g_prof_on = true;
    return 0;
}

// Synchronises, then writes one line per kernel name: "<name> <launches> <total_ms>\n".
extern "C" int mal_profile_end(char *out, int64_t out_len) {
    g_prof_on = false;
    MAL_REQUIRE(out && out_len > 0, "mal_profile_end: bad buffer");
    MAL_CUDA(cudaDeviceSynchronize());
    const char *names[256];
    int counts[256];
    double totals[256];
    int nn = 0;
    for (int i = 0; i < g_prof_n; ++i) {
        float ms = 0.f;
        MAL_CUDA(cudaEventElapsedTime(&ms, g_prof_ev[i][0], g_prof_ev[i][1]));
        int j = 0;
        for (; j < nn; ++j) if (strcmp(names[j], g_prof_name[i]) == 0) break;
        if (j == nn) { if (nn == 256) continue; names[nn] = g_prof_name[i]; counts[nn] = 0; totals[nn] = 0; ++nn; }
        counts[j] += 1; totals[j] += ms;
    }
    int64_t pos = 0;
    out[0] = 0;
    for (int j = 0; j < nn; ++j) {
        int w = snprintf(out + pos, (size_t)(out_len - pos), "%s %d %.6f\n", names[j], counts[j], totals[j]);
        if (w < 0 || pos + w >= out_len) break;
        pos += w;
    }
    g_prof_n = 0;
    return 0;
}

// Like mal_profile_end, but one line per LAUNCH in issue order: "<name> <start_us> <end_us>\n" relative to the first
// recorded launch (events on different streams share the device's clock): the overlapped timeline of a step.
extern "C" int mal_profile_end_timeline(char *out, int64_t out_len) {
    g_prof_on = false;
    MAL_REQUIRE(out && out_len > 0, "mal_profile_end_timeline: bad buffer");
    MAL_CUDA(cudaDeviceSynchronize());
    int64_t pos = 0;
    out[0] = 0;
    for (int i = 0; i < g_prof_n; ++i) {
        float t0 = 0.f, t1 = 0.f;
        MAL_CUDA(cudaEventElapsedTime(&t0, g_prof_ev[0][0], g_prof_ev[i][0]));
        MAL_CUDA(cudaEventElapsedTime(&t1, g_prof_ev[0][0], g_prof_ev[i][1]));
        int w = snprintf(out + pos, (size_t)(out_len - pos), "%s %.3f %.3f\n", g_prof_name[i], t0 * 1e3, t1 * 1e3);
        if (w < 0 || pos + w >= out_len) break;
        pos += w;
    }
    g_prof_n = 0;
    return 0;
}

extern "C" int64_t mal_agent_param_count(int32_t d_in, int32_t n_actions) { return agent_layout(d_in, n_actions).total; }
extern "C" int64_t mal_agent_param_count_kind(int32_t kind, int32_t d_in, int32_t n_actions) { return agent_layout(d_in, n_actions, kind).total; }
extern "C" int64_t mal_mixer_param_count(int32_t mixer, int32_t S, int32_t N, int32_t E, int32_t HE) {
    return mixer_layout(mixer, S, N, E, HE).total;
}

// Per-device state is indexed by the device ordinal (a thread may drive several GPUs one after the other).
#define MAL_MAX_DEV 64
// Opt `kernel` into `bytes` of dynamic shared memory on the CURRENT device.  `cache` is the call site's per-device
// high-water mark (static, zero-initialised; a benign race sets the attribute twice).
template <typename K>
static int ensure_dyn_smem(K kernel, size_t bytes, size_t *cache) {
    int dev = 0;
    MAL_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= MAL_MAX_DEV) {
        MAL_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
        return 0;
    }
    if (bytes > cache[dev]) {
        MAL_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
        cache[dev] = bytes;
    }
    return 0;
}

// The L1 / shared-memory split of an SM is fixed while CTAs are resident: a kernel that is happy with the small default
// carve-out keeps every big-shared-memory kernel (the tcgen05 GEMMs of the side streams: 104+ KB per CTA) off its SMs until
// it has drained.  The recurrences ask for the largest carve-out so that the hypernet / gradient GEMMs can move in beside them.
template <typename K>
static int ensure_max_carveout(K kernel, bool *cache, bool want = true) {   // cache[dev]: the preference currently set on this device
    int dev = 0;
    MAL_CUDA(cudaGetDevice(&dev));
    const bool cached = dev >= 0 && dev < MAL_MAX_DEV;
    if (cached && cache[dev] == want) return 0;
    MAL_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                  want ? (int)cudaSharedmemCarveoutMaxShared : (int)cudaSharedmemCarveoutDefault));
    if (cached) cache[dev] = want;
    return 0;
}
// bit 0 / 1: the forward / backward recurrence prefers the largest shared-memory carve-out (the side-stream GEMMs can then be
// resident beside it); bit 2: the small kernels of the step too.  5v5 / B = 32, ms per step: 0 -> 0.3235, 1 -> 0.3225,
// 2 -> 0.3111, 3 -> 0.3130, 7 -> 0.3152: the gain is the mixer's backward chain moving in beside the BPTT instead of queueing
// behind it; beside the forward recurrence the hypernet GEMMs already find free SMs (its CTAs pile up on the SMs that
// k_agent_in_tc vacates first) and co-residence only slows the chains down.
static thread_local int g_rec_carveout = 2;

// kernel-flavour counters (tests assert which variant the launch heuristics picked): see mal_stat()
static uint64_t g_stat_tc2 = 0, g_stat_tc1 = 0, g_stat_reduce_tc = 0, g_stat_reduce_tc_swap = 0, g_stat_reduce_ffma = 0,
                g_stat_agent_in_fused = 0;

static int device_sm_count(int *sms, int *threads_per_sm) {
    static thread_local int c_dev = -1, c_sms = 0, c_tps = 0;
    int dev = 0;
    MAL_CUDA(cudaGetDevice(&dev));
    if (dev != c_dev) {
        MAL_CUDA(cudaDeviceGetAttribute(&c_sms, cudaDevAttrMultiProcessorCount, dev));
        MAL_CUDA(cudaDeviceGetAttribute(&c_tps, cudaDevAttrMaxThreadsPerMultiProcessor, dev));
        c_dev = dev;
    }
    *sms = c_sms;
    *threads_per_sm = c_tps;
    return 0;
}

// ---------------------------------------------------------------------------------------------
// side streams: independent kernel chains of one learner step run concurrently (the recurrences are latency-bound
// and leave most SMs idle).  Fork/join with events only, so the pattern is also capturable into a CUDA graph.
// ---------------------------------------------------------------------------------------------
struct SideStreams {
    bool ready = false;
    cudaStream_t s[2];
    cudaEvent_t fork_ev[4], join_ev[2];
    cudaEvent_t aux_fork_ev, aux_join_ev;   // forward: the weight transposes on s[1], beside the hypernet GEMMs on s[0]
    // k_gru_fwd9 balanced mode: hand-over flags of split chains (zero between launches).  MAL_FLAG_SLOTS sets, handed out
    // round-robin per launch (a captured launch keeps its set), so that two learners driven by one thread on two streams do
    // not share flags when their recurrences overlap on the device
    int *chain_flags = nullptr;
    unsigned flag_slot = 0;
};
#define MAL_CHAIN_FLAGS 1024
#define MAL_FLAG_SLOTS 16
static thread_local SideStreams g_side[MAL_MAX_DEV];   // one set per (thread, device)
// mal_set_option switches are PER CALLING THREAD (like the side streams): two learners driven by two threads of one
// process do not see each other's settings
static thread_local int g_overlap = 1;
static thread_local int g_pdl = 1;              // programmatic dependent launch on the main kernel chain (prologues overlap the predecessor's tail)
static thread_local bool g_defer_stats = false;   // set by mal_learner_step around its forward half
static thread_local bool g_next_pdl = false;      // the next launch_linear / launch_reduce call may start under its stream predecessor
static thread_local bool g_in_step = false;       // inside mal_learner_step: the stream predecessors of backward / update are ours

// Launch with (pdl = true) the programmatic-serialization attribute: the kernel may be scheduled before its stream
// predecessor has finished and must call pdl_wait() before it touches anything but step constants.
template <typename... KArgs, typename... Args>
static void launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl, Args &&...args) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = (pdl && g_pdl && g_overlap) ? 1 : 0;
    cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);   // errors surface through MAL_LAUNCH_CHECK
}

static int side_streams(SideStreams **out) {
    int dev = 0;
    MAL_CUDA(cudaGetDevice(&dev));
    MAL_REQUIRE(dev >= 0 && dev < MAL_MAX_DEV, "device ordinal %d out of range", dev);
    SideStreams &ss = g_side[dev];
    if (!ss.ready) {
        for (int i = 0; i < 2; ++i) MAL_CUDA(cudaStreamCreateWithFlags(&ss.s[i], cudaStreamNonBlocking));
        for (int i = 0; i < 4; ++i) MAL_CUDA(cudaEventCreateWithFlags(&ss.fork_ev[i], cudaEventDisableTiming));
        for (int i = 0; i < 2; ++i) MAL_CUDA(cudaEventCreateWithFlags(&ss.join_ev[i], cudaEventDisableTiming));
        MAL_CUDA(cudaEventCreateWithFlags(&ss.aux_fork_ev, cudaEventDisableTiming));
        MAL_CUDA(cudaEventCreateWithFlags(&ss.aux_join_ev, cudaEventDisableTiming));
        MAL_CUDA(cudaMalloc(&ss.chain_flags, MAL_FLAG_SLOTS * MAL_CHAIN_FLAGS * sizeof(int)));
        MAL_CUDA(cudaMemset(ss.chain_flags, 0, MAL_FLAG_SLOTS * MAL_CHAIN_FLAGS * sizeof(int)));
        ss.ready = true;
    }
    *out = &ss;
    return 0;
}
// `side` starts after everything enqueued on `main` so far
static int fork_to(cudaStream_t main, cudaStream_t side, cudaEvent_t ev) {
    if (side == main) return 0;
    MAL_CUDA(cudaEventRecord(ev, main));
    MAL_CUDA(cudaStreamWaitEvent(side, ev, 0));
    return 0;
}
// `main` continues after everything enqueued on `side` so far
static int join_from(cudaStream_t main, cudaStream_t side, cudaEvent_t ev) {
    if (side == main) return 0;
    MAL_CUDA(cudaEventRecord(ev, side));
    MAL_CUDA(cudaStreamWaitEvent(main, ev, 0));
    return 0;
}

// ---------------------------------------------------------------------------------------------
// replay
// ---------------------------------------------------------------------------------------------
extern "C" int mal_record_copy(void *dst, int64_t dst_stride, const int64_t *dst_ids, const void *src,
                               int64_t src_stride, const int64_t *src_ids, int32_t n, int64_t bytes, void *stream) {
    if (n <= 0 || bytes <= 0) return 0;
    MAL_REQUIRE(dst && src, "mal_record_copy: null buffer");
    MAL_REQUIRE((bytes % 16) == 0 && (dst_stride % 16) == 0 && (src_stride % 16) == 0 &&
                    (((uintptr_t)dst | (uintptr_t)src) & 15) == 0,
                "mal_record_copy: records must be 16-byte aligned multiples of 16 bytes");
    int sms, tps;
    if (device_sm_count(&sms, &tps)) return 2;
    RecordCopyArgs a;
    a.dst = (uint8_t *)dst; a.src = (const uint8_t *)src;
    a.dst_stride = dst_stride; a.src_stride = src_stride;
    a.dst_ids = dst_ids; a.src_ids = src_ids;
    a.n = n; a.bytes = bytes;
    a.tiles_per_rec = (int32_t)ceil_div64(bytes, RC_TILE);
    a.n_tiles = (int64_t)a.tiles_per_rec * n;
    const size_t smem = (size_t)RC_STAGES * RC_TILE;
    static size_t attr[MAL_MAX_DEV];
    if (int rc = ensure_dyn_smem(k_record_copy_tma, smem, attr)) return rc;
    int64_t grid = a.n_tiles < (int64_t)sms * 3 ? a.n_tiles : (int64_t)sms * 3;   // 3 x 64 KB rings per SM
    { ProfScope _ps("k_record_copy_tma", (cudaStream_t)stream); k_record_copy_tma<<<(unsigned)grid, 32, smem, (cudaStream_t)stream>>>(a); }
    MAL_LAUNCH_CHECK("k_record_copy_tma");
    return 0;
}

extern "C" int mal_wire_layout(int32_t TT, int32_t N, int32_t OBS, int32_t S, mal_wire_layout_t *out) {
    MAL_REQUIRE(out && TT > 0 && N > 0 && OBS > 0 && S > 0, "mal_wire_layout: bad arguments");
    int64_t o = 0;
    auto take = [&](int64_t bytes) { int64_t r = o; o += align_up64(bytes, 16); return r; };
    out->off_state = take((int64_t)TT * S * 4);
    out->off_obs = take((int64_t)TT * N * OBS * 4);
    out->off_reward = take((int64_t)TT * 4);
    out->off_avail = take((int64_t)TT * N * 4);
    out->off_actions = take((int64_t)TT * N);
    out->off_flags = take(TT);
    out->record_bytes = align_up64(o, 128);
    return 0;
}

static int launch_wire(const mal_batch_t *b, void *wire, const mal_wire_layout_t *wl, int32_t *status, bool pack, void *stream) {
    MAL_REQUIRE(b && wire && wl, "mal_wire: null argument");
    MAL_REQUIRE(b->B >= 1 && b->TT >= 1 && b->N >= 1 && b->A >= 1 && b->A <= 32 && b->OBS >= 1 && b->S >= 1, "mal_wire: bad dims (n_actions <= 32)");
    MAL_REQUIRE((reinterpret_cast<uintptr_t>(wire) & 15) == 0 && (wl->record_bytes & 15) == 0, "mal_wire: the wire buffer must be 16-byte aligned");
    WireArgs a;
    a.B = b->B; a.TT = b->TT; a.N = b->N; a.A = b->A; a.OBS = b->OBS; a.S = b->S;
    a.obs = b->obs; a.onehot = b->onehot; a.actions = b->actions; a.avail = b->avail; a.state = b->state;
    a.reward = b->reward; a.terminated = b->terminated; a.filled = b->filled;
    a.wire = (uint8_t *)wire; a.record_bytes = wl->record_bytes; a.off_state = wl->off_state; a.off_obs = wl->off_obs;
    a.off_reward = wl->off_reward; a.off_actions = wl->off_actions; a.off_avail = wl->off_avail; a.off_flags = wl->off_flags;
    a.status = status;
    int sms, tps;
    if (device_sm_count(&sms, &tps)) return 2;
    int64_t grid = ceil_div64((int64_t)b->B * b->TT, 8); if (grid > (int64_t)sms * 8) grid = (int64_t)sms * 8;
    cudaStream_t st = (cudaStream_t)stream;
    if (pack) { ProfScope _ps("k_wire_pack", st); k_wire<true><<<(unsigned)grid, 256, 0, st>>>(a); }
    else { ProfScope _ps("k_wire_unpack", st); k_wire<false><<<(unsigned)grid, 256, 0, st>>>(a); }
    MAL_LAUNCH_CHECK("k_wire");
    return 0;
}
extern "C" int mal_wire_pack(const mal_batch_t *batch, void *wire, const mal_wire_layout_t *layout, int32_t *status, void *stream) {
    return launch_wire(batch, wire, layout, status, true, stream);
}
extern "C" int mal_wire_unpack(const mal_batch_t *batch, const void *wire, const mal_wire_layout_t *layout, void *stream) {
    return launch_wire(batch, const_cast<void *>(wire), layout, nullptr, false, stream);
}

extern "C" int mal_max_t_filled(const int64_t *filled, int64_t sb, int64_t st, int32_t B, int32_t TT, int32_t *out,
                                void *stream) {
    MAL_REQUIRE(filled && out && B > 0 && TT > 0, "mal_max_t_filled: bad arguments");
    { ProfScope _ps("k_max_t_filled", (cudaStream_t)stream); k_max_t_filled<<<1, 256, 0, (cudaStream_t)stream>>>(filled, sb, st, B, TT, out); }
    MAL_LAUNCH_CHECK("k_max_t_filled");
    return 0;
}

// ---------------------------------------------------------------------------------------------
// act-select
// ---------------------------------------------------------------------------------------------
static int fill_select(const mal_select_t *sel, int rows, int N, int A, SelectArgs *s) {
    MAL_REQUIRE(sel->avail && sel->actions && sel->greedy, "select: avail/actions/greedy must be set");
    MAL_REQUIRE(sel->rng_mode == 0 || sel->rng_mode == 1, "select: rng_mode must be 0 (injected) or 1 (philox)");
    if (sel->rng_mode == 0) MAL_REQUIRE(sel->u && sel->e, "select: rng_mode 0 needs u and e");
    int sms, tps;
    if (device_sm_count(&sms, &tps)) return 2;
    s->avail = sel->avail; s->avail_sb = sel->avail_sb; s->N = N; s->epsilon = sel->epsilon; s->rng_mode = sel->rng_mode;
    s->u = sel->u; s->e = sel->e; s->seed = sel->seed;
    s->actions = sel->actions; s->greedy = sel->greedy; s->status = sel->status;
    // torch's calc_execution_policy (ATen/native/cuda/DistributionTemplates.h): block 256, grid capped at
    // SMs * (maxThreadsPerSM / 256); each op advances the generator by ((numel-1)/(256*grid*4)+1)*4.
    const uint64_t cap = (uint64_t)sms * (uint64_t)(tps / 256);
    uint64_t n_u = (uint64_t)rows, n_e = (uint64_t)rows * (uint64_t)A;
    uint64_t g_u = (n_u + 255) / 256; if (g_u > cap) g_u = cap;
    uint64_t g_e = (n_e + 255) / 256; if (g_e > cap) g_e = cap;
    s->grid_u = (uint32_t)g_u; s->grid_e = (uint32_t)g_e;
    s->offset_u = sel->offset;
    s->offset_e = sel->offset + ((n_u - 1) / (256 * g_u * 4) + 1) * 4;
    return 0;
}

// total generator advance (in 32-bit outputs) of one select over rows x A, for the caller to apply to torch's generator
extern "C" int mal_select_philox_advance(int32_t rows, int32_t n_actions, uint64_t *advance) {
    MAL_REQUIRE(rows > 0 && n_actions > 0 && advance, "mal_select_philox_advance: bad arguments");
    int sms, tps;
    if (device_sm_count(&sms, &tps)) return 2;
    const uint64_t cap = (uint64_t)sms * (uint64_t)(tps / 256);
    uint64_t n_u = (uint64_t)rows, n_e = (uint64_t)rows * (uint64_t)n_actions;
    uint64_t g_u = (n_u + 255) / 256; if (g_u > cap) g_u = cap;
    uint64_t g_e = (n_e + 255) / 256; if (g_e > cap) g_e = cap;
    *advance = ((n_u - 1) / (256 * g_u * 4) + 1) * 4 + ((n_e - 1) / (256 * g_e * 4) + 1) * 4;
    return 0;
}

extern "C" int mal_eps_greedy_select(const float *q, int64_t q_ld, int32_t rows, int32_t n_agents, int32_t n_actions,
                                     const mal_select_t *sel, void *stream) {
    MAL_REQUIRE(q && sel && rows > 0 && n_agents > 0, "mal_eps_greedy_select: bad arguments");
    MAL_REQUIRE(n_actions >= 1 && n_actions <= MAL_MAX_ACTIONS, "n_actions must be in [1, %d]", MAL_MAX_ACTIONS);
    SelectArgs s;
    if (int rc = fill_select(sel, rows, n_agents, n_actions, &s)) return rc;
    const int warps_per_block = AS_THREADS / 32;
    { ProfScope _ps("k_eps_greedy_select", (cudaStream_t)stream); k_eps_greedy_select<<<(rows + warps_per_block - 1) / warps_per_block, AS_THREADS, 0, (cudaStream_t)stream>>>(
        q, q_ld, rows, n_actions, s); }
    MAL_LAUNCH_CHECK("k_eps_greedy_select");
    return 0;
}

static thread_local int g_actsel_lat = 1;    // 1: mma.sync latency kernel for rollout-sized launches; 0: lanes-along-k register kernel
// POOL: the per-match-policy instances; `ctas` is then the schedule's upper bound (CTAs past its used count exit at once)
// and the variant is chosen on that grid by the same rule
template <bool POOL>
static int launch_agent_step(AgentStepArgs &a, cudaStream_t stream, int ctas) {
    const int Kin = a.in.last_end();
    const size_t smem = sizeof(float) * (size_t)(AS_ROWS * (Kin + 1) + AS_ROWS * HID * 3 + AS_ROWS * 2 * G3 + AS_ROWS * 32);
    MAL_REQUIRE(smem <= 200 * 1024 && Kin <= 32 * AS_FC1_MAXK, "mal_agent_step: input width %d too large (max %d)", Kin,
                32 * AS_FC1_MAXK);
    int sms, tps;
    if (device_sm_count(&sms, &tps)) return 2;
    const char *name = POOL ? "k_agent_step_pool" : "k_agent_step";
    if (ctas <= sms && a.kind == MAL_AGENT_RNN && g_actsel_lat) {   // rollouts: latency is what counts
        const size_t smem_l = sizeof(float) * (size_t)(AS_ROWS * (((Kin + 7) & ~7) + 4) + AS_ROWS * 68 * 3 + AS_ROWS * 2 * G3 + AS_ROWS * 32);
        static size_t attr[MAL_MAX_DEV];
        if (smem_l > 48 * 1024) if (int rc = ensure_dyn_smem(k_agent_step_lat<POOL>, smem_l, attr)) return rc;
        ProfScope _ps(name, stream);
        k_agent_step_lat<POOL><<<ctas, AL_THREADS, smem_l, stream>>>(a);
    } else if (ctas <= 2 * sms && a.kind == MAL_AGENT_RNN) {   // all weights prefetched into registers
        static size_t attr[MAL_MAX_DEV];
        if (smem > 48 * 1024) if (int rc = ensure_dyn_smem(k_agent_step<POOL>, smem, attr)) return rc;
        ProfScope _ps(name, stream);
        k_agent_step<POOL><<<ctas, AS_THREADS, smem, stream>>>(a);
    } else {
        static size_t attr[MAL_MAX_DEV];
        if (smem > 48 * 1024) if (int rc = ensure_dyn_smem(k_agent_step_stream<POOL>, smem, attr)) return rc;
        ProfScope _ps(name, stream);
        k_agent_step_stream<POOL><<<ctas, AS_THREADS, smem, stream>>>(a);
    }
    MAL_LAUNCH_CHECK(name);
    return 0;
}
static int launch_agent_step(AgentStepArgs &a, cudaStream_t stream) {
    return launch_agent_step<false>(a, stream, (a.rows + AS_ROWS - 1) / AS_ROWS);
}

// dense_input of mal_agent_step / mal_dqn_step: bit 0 = the caller assembled the input (obs_dim columns, nothing to
// gather); otherwise bits 1..2 are the MAL_IN_* switches of the fused input assembly
static int step_input(int32_t dense_input, AgentStepArgs *a) {
    MAL_REQUIRE((dense_input & ~7) == 0 && !((dense_input & 1) && (dense_input >> 1)),
                "dense_input %d: bit 0 (dense) or the agent-input bits 1..2, nothing else", dense_input);
    a->dense = dense_input & 1;
    if (a->dense) { a->in.obs = a->in.d_in = a->OBS; a->in.last = a->in.id = 0; }
    else a->in = agent_input(a->OBS, a->A, a->N, dense_input >> 1);
    return 0;
}

static int agent_step_args(const char *what, const float *agent, int32_t rows, int32_t n_agents, int32_t obs_dim,
                           int32_t n_actions, int32_t dense_input, const float *obs, int64_t obs_sb, const float *last_onehot,
                           int64_t onehot_sb, const float *h_in, float *h_out, float *q, AgentStepArgs *ap) {
    MAL_REQUIRE(agent && obs && h_out && q && rows > 0, "%s: bad arguments", what);
    MAL_REQUIRE(n_actions >= 1 && n_actions <= MAL_MAX_ACTIONS, "n_actions must be in [1, %d]", MAL_MAX_ACTIONS);
    MAL_REQUIRE(n_agents >= 1 && obs_dim >= 1, "%s: bad dims", what);
    AgentStepArgs &a = *ap;
    memset(&a, 0, sizeof(a));
    a.params = agent; a.rows = rows; a.N = n_agents; a.OBS = obs_dim; a.A = n_actions;
    if (int rc = step_input(dense_input, &a)) return rc;
    a.obs = obs; a.obs_sb = obs_sb; a.onehot = a.in.last > 0 ? last_onehot : nullptr; a.onehot_sb = onehot_sb;
    a.h_in = h_in; a.h_out = h_out; a.q = q;
    return 0;
}

extern "C" int mal_agent_step(const float *agent, int32_t rows, int32_t n_agents, int32_t obs_dim, int32_t n_actions,
                              int32_t dense_input, const float *obs, int64_t obs_sb, const float *last_onehot,
                              int64_t onehot_sb, const float *h_in, float *h_out, float *q, const mal_select_t *sel,
                              void *stream) {
    AgentStepArgs a;
    if (int rc = agent_step_args("mal_agent_step", agent, rows, n_agents, obs_dim, n_actions, dense_input, obs, obs_sb,
                                 last_onehot, onehot_sb, h_in, h_out, q, &a)) return rc;
    a.do_select = sel ? 1 : 0;
    if (sel) if (int rc = fill_select(sel, rows, n_agents, n_actions, &a.sel)) return rc;
    return launch_agent_step(a, (cudaStream_t)stream);
}

// DQNAgentNetwork.forward (dqn_agent.py:34-37: q = fc2(relu(fc1(inputs))), no hidden state) through BasicMAC's input
// assembly, with the optional epsilon-greedy tail; same argument meaning as mal_agent_step.
extern "C" int mal_dqn_step(const float *agent, int32_t rows, int32_t n_agents, int32_t obs_dim, int32_t n_actions,
                            int32_t dense_input, const float *obs, int64_t obs_sb, const float *last_onehot,
                            int64_t onehot_sb, float *q, const mal_select_t *sel, void *stream) {
    MAL_REQUIRE(agent && obs && q && rows > 0, "mal_dqn_step: bad arguments");
    MAL_REQUIRE(n_actions >= 1 && n_actions <= MAL_MAX_ACTIONS, "n_actions must be in [1, %d]", MAL_MAX_ACTIONS);
    MAL_REQUIRE(n_agents >= 1 && obs_dim >= 1, "mal_dqn_step: bad dims");
    AgentStepArgs a;
    memset(&a, 0, sizeof(a));
    a.params = agent; a.kind = MAL_AGENT_DQN; a.rows = rows; a.N = n_agents; a.OBS = obs_dim; a.A = n_actions;
    if (int rc = step_input(dense_input, &a)) return rc;
    a.obs = obs; a.obs_sb = obs_sb; a.onehot = a.in.last > 0 ? last_onehot : nullptr; a.onehot_sb = onehot_sb;
    a.h_in = nullptr; a.h_out = nullptr; a.q = q; a.do_select = sel ? 1 : 0;
    if (sel) if (int rc = fill_select(sel, rows, n_agents, n_actions, &a.sel)) return rc;
    return launch_agent_step(a, (cudaStream_t)stream);
}

static int rollout_args(const char *what, const float *agent, int32_t bs, int32_t n_agents, int32_t obs_dim,
                        int32_t n_actions, const mal_rollout_io_t *io, const float *h_in, float *h_out, float *q,
                        const mal_select_t *sel, AgentStepArgs *ap) {
    MAL_REQUIRE(agent && io && sel && h_out && q && bs > 0, "%s: bad arguments", what);
    MAL_REQUIRE(n_actions >= 1 && n_actions <= MAL_MAX_ACTIONS, "n_actions must be in [1, %d]", MAL_MAX_ACTIONS);
    MAL_REQUIRE(n_agents >= 1 && obs_dim >= 1 && io->state_dim >= 1, "%s: bad dims", what);
    MAL_REQUIRE(io->env_state && io->env_avail && io->env_obs && io->state_t && io->avail_t && io->obs_t && io->filled_t &&
                    io->actions_t && io->onehot_t, "%s: environment / batch pointers missing", what);
    MAL_REQUIRE(!io->prev_reward || (io->prev_done && io->reward_tm1 && io->term_tm1), "%s: previous-step fields missing", what);
    MAL_REQUIRE((io->agent_input & ~3) == 0, "%s: unknown agent_input bits %d", what, io->agent_input);
    AgentStepArgs &a = *ap;
    memset(&a, 0, sizeof(a));
    const int rows = bs * n_agents;
    a.params = agent; a.rows = rows; a.N = n_agents; a.OBS = obs_dim; a.A = n_actions; a.dense = 0;
    a.in = agent_input(obs_dim, n_actions, n_agents, io->agent_input);
    a.obs = io->env_obs; a.obs_sb = io->env_obs_sb; a.onehot = io->onehot_tm1; a.onehot_sb = io->onehot_tm1_sb;
    a.h_in = h_in; a.h_out = h_out; a.q = q; a.do_select = 1;
    RolloutIO &r = a.io;
    r.enabled = 1; r.S = io->state_dim;
    r.env_state = io->env_state; r.env_state_sb = io->env_state_sb; r.alive = io->alive;
    r.prev_reward = io->prev_reward; r.prev_done = io->prev_done;
    r.state_t = io->state_t; r.state_sb = io->state_sb; r.avail_t = io->avail_t; r.avail_sb = io->avail_sb;
    r.obs_t = io->obs_t; r.obs_sb = io->obs_sb; r.filled_t = (long long *)io->filled_t; r.filled_sb = io->filled_sb;
    r.actions_t = (long long *)io->actions_t; r.actions_sb = io->actions_sb; r.onehot_t = io->onehot_t; r.onehot_sb = io->onehot_sb;
    r.reward_tm1 = io->reward_tm1; r.reward_sb = io->reward_sb; r.term_tm1 = io->term_tm1; r.term_sb = io->term_sb;
    return 0;
}
// the selector of a rollout step reads the environment's avail rows of `io`
static int rollout_select(const mal_select_t *sel, const mal_rollout_io_t *io, AgentStepArgs *a) {
    mal_select_t s2 = *sel;
    s2.avail = io->env_avail; s2.avail_sb = io->env_avail_sb;
    return fill_select(&s2, a->rows, a->N, a->A, &a->sel);
}

extern "C" int mal_rollout_step(const float *agent, int32_t bs, int32_t n_agents, int32_t obs_dim, int32_t n_actions,
                                const mal_rollout_io_t *io, const float *h_in, float *h_out, float *q, const mal_select_t *sel,
                                void *stream) {
    AgentStepArgs a;
    if (int rc = rollout_args("mal_rollout_step", agent, bs, n_agents, obs_dim, n_actions, io, h_in, h_out, q, sel, &a)) return rc;
    if (int rc = rollout_select(sel, io, &a)) return rc;
    return launch_agent_step(a, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------------
// per-match policies (actsel.cuh: k_policy_schedule and the POOL instances of the step kernels)
// ---------------------------------------------------------------------------------------------
static int check_pool_shape(const char *what, int32_t bs, int32_t n_agents, int32_t n_policies) {
    MAL_REQUIRE(bs >= 1 && n_agents >= 1, "%s: bs and n_agents must be >= 1", what);
    MAL_REQUIRE((int64_t)bs * n_agents <= (1 << 30), "%s: bs * n_agents = %lld rows is too many", what, (long long)bs * n_agents);
    MAL_REQUIRE(n_policies >= 1 && n_policies <= MAL_MAX_POLICIES, "%s: n_policies must be in [1, %d], got %d", what,
                MAL_MAX_POLICIES, n_policies);
    return 0;
}
// upper bound of the used CTAs: sum over policies of ceil(rows_p / 8) <= ceil(rows / 8) + (non-empty policies - 1)
static int64_t pool_grid(int32_t rows, int32_t bs, int32_t n_policies) {
    return ceil_div64(rows, AS_ROWS) + (n_policies < bs ? n_policies : bs) - 1;
}

extern "C" int64_t mal_policy_schedule_bytes(int32_t bs, int32_t n_agents, int32_t n_policies) {
    if (check_pool_shape("mal_policy_schedule_bytes", bs, n_agents, n_policies)) return -1;
    return (int64_t)sizeof(int32_t) * (PS_HDR + pool_grid(bs * n_agents, bs, n_policies) * PS_ENT);
}

extern "C" int mal_policy_schedule(const int32_t *match_policy, int32_t bs, int32_t n_agents, int32_t n_policies,
                                   void *schedule, int32_t *status, void *stream) {
    if (int rc = check_pool_shape("mal_policy_schedule", bs, n_agents, n_policies)) return rc;
    MAL_REQUIRE(match_policy && schedule, "mal_policy_schedule: null argument");
    MAL_REQUIRE(((uintptr_t)schedule & 15) == 0, "mal_policy_schedule: the schedule buffer must be 16-byte aligned");
    { ProfScope _ps("k_policy_schedule", (cudaStream_t)stream);
      k_policy_schedule<<<1, PS_THREADS, 0, (cudaStream_t)stream>>>(match_policy, bs, n_agents, n_policies, (int32_t *)schedule, status); }
    MAL_LAUNCH_CHECK("k_policy_schedule");
    return 0;
}

static int pool_args(const char *what, const float *table, int64_t table_ld, int32_t n_policies, const void *schedule,
                     AgentStepArgs *a) {
    if (int rc = check_pool_shape(what, a->rows / a->N, a->N, n_policies)) return rc;
    MAL_REQUIRE(table && schedule, "%s: null table or schedule", what);
    MAL_REQUIRE(a->rows % a->N == 0, "%s: rows %d is not a multiple of n_agents %d", what, a->rows, a->N);
    MAL_REQUIRE(((uintptr_t)schedule & 15) == 0, "%s: the schedule buffer must be 16-byte aligned", what);
    const int64_t P = agent_layout(a->in.d_in, a->A).total;
    MAL_REQUIRE(table_ld >= P, "%s: table_ld %lld is smaller than the agent's %lld parameters", what, (long long)table_ld,
                (long long)P);
    a->sched = (const int32_t *)schedule; a->table_ld = table_ld; a->n_policies = n_policies;
    return 0;
}

extern "C" int mal_agent_step_pool(const float *table, int64_t table_ld, int32_t n_policies, const void *schedule,
                                   int32_t rows, int32_t n_agents, int32_t obs_dim, int32_t n_actions, int32_t dense_input,
                                   const float *obs, int64_t obs_sb, const float *last_onehot, int64_t onehot_sb,
                                   const float *h_in, float *h_out, float *q, const mal_select_t *sel, void *stream) {
    AgentStepArgs a;
    if (int rc = agent_step_args("mal_agent_step_pool", table, rows, n_agents, obs_dim, n_actions, dense_input, obs, obs_sb,
                                 last_onehot, onehot_sb, h_in, h_out, q, &a)) return rc;
    if (int rc = pool_args("mal_agent_step_pool", table, table_ld, n_policies, schedule, &a)) return rc;
    a.do_select = sel ? 1 : 0;
    if (sel) if (int rc = fill_select(sel, rows, n_agents, n_actions, &a.sel)) return rc;
    return launch_agent_step<true>(a, (cudaStream_t)stream, (int)pool_grid(rows, rows / n_agents, n_policies));
}

extern "C" int mal_rollout_step_pool(const float *table, int64_t table_ld, int32_t n_policies, const void *schedule,
                                     int32_t bs, int32_t n_agents, int32_t obs_dim, int32_t n_actions,
                                     const mal_rollout_io_t *io, const float *h_in, float *h_out, float *q,
                                     const mal_select_t *sel, void *stream) {
    AgentStepArgs a;
    if (int rc = rollout_args("mal_rollout_step_pool", table, bs, n_agents, obs_dim, n_actions, io, h_in, h_out, q, sel, &a))
        return rc;
    if (int rc = pool_args("mal_rollout_step_pool", table, table_ld, n_policies, schedule, &a)) return rc;
    if (int rc = rollout_select(sel, io, &a)) return rc;
    return launch_agent_step<true>(a, (cudaStream_t)stream, (int)pool_grid(a.rows, bs, n_policies));
}

// ---------------------------------------------------------------------------------------------
// learner: planning
// ---------------------------------------------------------------------------------------------
struct Dims {
    int B, TT, T, N, A, OBS, S, R, E, HE, d_in, mixer, two, kind;
    AgentInput in;                  // fc1 input layout (d_in = in.d_in)
    int64_t M1, BT;
    int ld1, ld2;
};

static int get_dims(const mal_batch_t *b, const mal_learner_cfg_t *c, Dims *d) {
    MAL_REQUIRE(b && c, "null batch/cfg");
    MAL_REQUIRE(b->B >= 1 && b->TT >= 2 && b->N >= 1 && b->OBS >= 1 && b->S >= 1, "bad batch dims (need TT >= 2)");
    MAL_REQUIRE(b->A >= 1 && b->A <= MAL_MAX_ACTIONS, "n_actions must be in [1, %d]", MAL_MAX_ACTIONS);
    MAL_REQUIRE(b->N <= MAL_MAX_ACTIONS, "n_agents must be <= %d", MAL_MAX_ACTIONS);
    MAL_REQUIRE(c->mixer == MAL_MIXER_VDN || c->mixer == MAL_MIXER_QMIX2 || c->mixer == MAL_MIXER_QMIX1 ||
                c->mixer == MAL_MIXER_NONE, "Mixer %d not recognised.", c->mixer);
    MAL_REQUIRE(!b->weight.ptr || !c->unnormalized,
                "importance weights (prioritized replay) are not supported in unnormalized (data-parallel) mode");
    MAL_REQUIRE(c->returns == MAL_RETURNS_ONE_STEP || c->returns == MAL_RETURNS_TD_LAMBDA, "returns %d not recognised",
                c->returns);
    MAL_REQUIRE(c->td_lambda >= 0.0f && c->td_lambda <= 1.0f, "td_lambda must be a number in [0, 1]");   // false for NaN
    d->B = b->B; d->TT = b->TT; d->T = b->TT - 1; d->N = b->N; d->A = b->A; d->OBS = b->OBS; d->S = b->S;
    MAL_REQUIRE(c->agent_kind == MAL_AGENT_RNN || c->agent_kind == MAL_AGENT_DQN, "agent kind %d not recognised", c->agent_kind);
    d->kind = c->agent_kind;
    MAL_REQUIRE((c->agent_input & ~3) == 0, "agent_input %d: only MAL_IN_NO_LAST_ACTION | MAL_IN_NO_AGENT_ID", c->agent_input);
    d->in = agent_input(b->OBS, b->A, b->N, c->agent_input);
    d->R = b->B * b->N; d->d_in = d->in.d_in; d->mixer = c->mixer;
    d->E = c->embed; d->HE = c->hyper_embed; d->two = (c->mixer == MAL_MIXER_QMIX2);
    if (mixer_has_hypernet(c->mixer)) {
        MAL_REQUIRE(d->E >= 1 && d->E <= MAL_MAX_EMBED, "mixing_embed_dim must be in [1, %d]", MAL_MAX_EMBED);
        if (d->two) MAL_REQUIRE(d->HE >= 1, "hypernet_embed must be >= 1");
    } else { d->E = 0; d->HE = 0; }
    d->M1 = (int64_t)d->TT * d->R;
    d->BT = (int64_t)d->B * d->T;
    MAL_REQUIRE(d->M1 < ((int64_t)1 << 31), "batch too large: (T+1)*B*N must be < 2^31 (row indices are 32-bit in the kernels)");
    d->ld1 = !mixer_has_hypernet(d->mixer) ? 0 : (d->two ? 2 * d->HE + 2 * d->E : 2 * d->E);
    d->ld2 = !mixer_has_hypernet(d->mixer) ? 0 : d->E * d->N + d->E;
    return 0;
}

// split an M-row reduction into chunks: chunks * (128 x 64 output tiles) = at most one CTA per SM for the tensor-core
// reduction (which the 64 x 64-tile FFMA kernel then over-subscribes by < 2x); >= 128 rows per chunk, <= 256 chunks
static void chunking(int64_t M, int tiles, int sms, int *n_chunks, int64_t *rows_per_chunk) {
    int64_t nc = sms / (tiles > 0 ? tiles : 1);
    if (nc > 256) nc = 256;
    if (nc > ceil_div64(M, 128)) nc = ceil_div64(M, 128);
    if (nc < 1) nc = 1;
    int64_t rpc = align_up64(ceil_div64(M, nc), RED_MR);
    nc = ceil_div64(M, rpc);
    *n_chunks = (int)nc;
    *rows_per_chunk = rpc;
}

// offsets (in floats) inside the partials scratch; every reduction launch (one per loader kind) gets its own
// chunking so that each launch fills the machine
struct PartLayout {
    int nc_a; int64_t rpc_a;        // dense agent reductions (W_ih, W_hh x2) over M1 rows
    int nc_f1; int64_t rpc_f1;      // fc1 (agent-input loader) over M1 rows
    int nc_f2; int64_t rpc_f2;      // fc2 (one-hot dY) over T*R rows
    int nc_m2; int64_t rpc_m2;      // mixer layer-2 problems over BT rows
    int nc_m1; int64_t rpc_m1;      // mixer layer-1 block over BT rows
    int nblk_mix;
    int nblk_norm;
    int64_t wih_w, wih_b, whha_w, whha_b, whhb_w, whhb_b, fc1_w, fc1_b, fc2_w, fc2_b;
    int64_t m_l2a_w, m_l2a_b, m_l2b_w, m_l2b_b, m_l1_w, m_l1_b;   // mixer: layer-2 (w1b, wfb), layer-1 block
    int64_t mix_stats, mix_v2, mix_v2_sum, norm;
    int64_t total;
};

// narrow outputs with a wide inner dimension (fc1 at d_in > 64) are reduced in the transposed orientation (k_reduce_tc SWAP)
static bool red_swapped(int Nout, int K) { return Nout <= RT_KT && K > RT_KT; }
static int tiles_of(int Nout, int K) {   // 128 x 64 output tiles of the tensor-core reduction
    if (red_swapped(Nout, K)) return ((K + RT_NT - 1) / RT_NT) * ((Nout + RT_KT - 1) / RT_KT);
    return ((Nout + RT_NT - 1) / RT_NT) * ((K + RT_KT - 1) / RT_KT);
}

static PartLayout part_layout(const Dims &d, int sms) {
    PartLayout p;
    memset(&p, 0, sizeof(p));
    // dense agent reductions: the fused k_reduce_gru handles a whole row chunk on one CTA -> one chunk per SM once every
    // chunk is long (>= 1024 rows), half as many below that (fewer partials for k_grad_reduce to gather at B = 32)
    chunking(d.M1, d.M1 >= (int64_t)sms * 1024 ? 1 : 2, sms, &p.nc_a, &p.rpc_a);
    // fc1: k_reduce_fc1 covers the full input width (<= 256 columns) on one CTA per chunk -> one chunk per SM
    chunking(d.M1, d.d_in <= 256 ? 1 : tiles_of(HID, d.d_in), sms, &p.nc_f1, &p.rpc_f1);
    {   // k_fc2_grad: one partial per CTA, 8 warps x >= 32 rows each; the kernel is HBM-bound on the h rows, so large batches
        // fill every SM with as many CTAs as their [8][A*64+32]-float accumulators allow (<= 4)
        const int64_t smem = (int64_t)sizeof(float) * 8 * ((int64_t)d.A * HID + 32);
        int64_t per_sm = (200 * 1024) / smem; if (per_sm > 4) per_sm = 4; if (per_sm < 1) per_sm = 1;
        int64_t nb = ceil_div64((int64_t)d.T * d.R, 256);
        if (nb > sms * per_sm) nb = sms * per_sm;
        if (nb < 1) nb = 1;
        p.nc_f2 = (int)nb; p.rpc_f2 = 0;
    }
    const int K2 = d.two ? d.HE : d.S;
    if (d.mixer == MAL_MIXER_QMIX2) {
        chunking(d.BT, tiles_of(d.E * d.N, K2) + tiles_of(d.E, K2), sms, &p.nc_m2, &p.rpc_m2);
        chunking(d.BT, tiles_of(d.ld1, d.S), sms, &p.nc_m1, &p.rpc_m1);
    } else if (d.mixer == MAL_MIXER_QMIX1) {   // all three problems share the state loader -> one launch
        chunking(d.BT, tiles_of(d.E * d.N, K2) + tiles_of(d.E, K2) + tiles_of(d.ld1, d.S), sms, &p.nc_m2, &p.rpc_m2);
        p.nc_m1 = p.nc_m2; p.rpc_m1 = p.rpc_m2;
    }
    int64_t nm = ceil_div64(d.BT, 8); if (nm > (int64_t)sms * 4) nm = (int64_t)sms * 4; if (nm < 1) nm = 1;
    p.nblk_mix = (int)nm;
    const int64_t P = agent_layout(d.d_in, d.A, d.kind).total + mixer_layout(d.mixer, d.S, d.N, d.E, d.HE).total;
    p.nblk_norm = (int)ceil_div64(P, GRED_EPB);
    int64_t o = 0;
    auto take = [&](int64_t n) { int64_t r = o; o += align_up64(n, 64); return r; };
    p.wih_w = take((int64_t)p.nc_a * G3 * HID);   p.wih_b = take((int64_t)p.nc_a * G3);
    p.whha_w = take((int64_t)p.nc_a * 128 * HID); p.whha_b = take((int64_t)p.nc_a * 128);
    p.whhb_w = take((int64_t)p.nc_a * 64 * HID);  p.whhb_b = take((int64_t)p.nc_a * 64);
    p.fc1_w = take((int64_t)p.nc_f1 * HID * d.d_in); p.fc1_b = take((int64_t)p.nc_f1 * HID);
    p.fc2_w = take((int64_t)p.nc_f2 * d.A * HID);    p.fc2_b = take((int64_t)p.nc_f2 * d.A);
    if (mixer_has_hypernet(d.mixer)) {
        p.m_l2a_w = take((int64_t)p.nc_m2 * d.E * d.N * K2); p.m_l2a_b = take((int64_t)p.nc_m2 * d.E * d.N);
        p.m_l2b_w = take((int64_t)p.nc_m2 * d.E * K2);       p.m_l2b_b = take((int64_t)p.nc_m2 * d.E);
        p.m_l1_w = take((int64_t)p.nc_m1 * d.ld1 * d.S);     p.m_l1_b = take((int64_t)p.nc_m1 * d.ld1);
        p.mix_v2 = take((int64_t)p.nblk_mix * (d.E + 1));
        p.mix_v2_sum = take(d.E + 1);
    }
    p.mix_stats = take((int64_t)p.nblk_mix * MIX_NSTAT);
    p.norm = take(p.nblk_norm);
    p.total = o;
    return p;
}

extern "C" int mal_learner_plan(const mal_batch_t *batch, const mal_learner_cfg_t *cfg, mal_plan_t *plan) {
    Dims d;
    if (int rc = get_dims(batch, cfg, &d)) return rc;
    MAL_REQUIRE(plan, "null plan");
    int sms, tps;
    if (device_sm_count(&sms, &tps)) { sms = 148; }   // planning also works without a device (CPU-side tests)
    memset(plan, 0, sizeof(*plan));
    int64_t o = 0;
    auto take = [&](int64_t n_elems, int64_t elem) { int64_t r = o; o += align_up64(n_elems * elem, 256); return r; };
    plan->n_agent_params = agent_layout(d.d_in, d.A, d.kind).total;
    plan->n_mixer_params = mixer_layout(d.mixer, d.S, d.N, d.E, d.HE).total;
    plan->scalars = take(64, 4);
    plan->x_on = take(d.M1 * HID, 4);   plan->x_tg = take(d.M1 * HID, 4);
    plan->gi_on = take(d.M1 * G3, 4);   plan->gi_tg = take(d.M1 * G3, 4);
    plan->h_on = take(d.M1 * HID, 4);   plan->h_tg = take(d.M1 * HID, 4);
    plan->gates = take(d.M1 * 4 * HID, 4);
    const int64_t nq = cfg->save_q ? (int64_t)d.B * d.TT * d.N * d.A : 0;
    plan->mac_out = take(nq, 4);        plan->target_mac_out = take(nq, 4);
    plan->chosen = take(d.BT * d.N, 4); plan->target_max = take(d.BT * d.N, 4);
    plan->argmax = take(d.BT * d.N, 4);
    plan->mask = take(d.BT, 4);
    plan->y1_on = take(d.BT * d.ld1, 4); plan->y1_tg = take(d.BT * d.ld1, 4);
    plan->a2_on = take(d.BT * d.ld2, 4); plan->a2_tg = take(d.BT * d.ld2, 4);
    const int64_t nq_tot = d.mixer == MAL_MIXER_NONE ? d.BT * d.N : d.BT;   // IQL: one TD error per agent
    plan->q_tot = take(nq_tot, 4); plan->target_q_tot = take(nq_tot, 4);
    plan->targets = take(nq_tot, 4); plan->td = take(nq_tot, 4);
    plan->d_a2 = take(d.BT * d.ld2, 4); plan->d_y1 = take(d.BT * d.ld1, 4);
    plan->d_chosen = take(d.BT * d.N, 4);
    plan->d_g = take(d.M1 * 4 * HID, 4);
    plan->d_x = take(d.M1 * HID, 4);
    plan->dh_head = take(d.M1 * HID, 4);
    PartLayout pl = part_layout(d, sms);
    plan->partials_bytes = pl.total * 4;
    plan->partials = take(pl.total, 4);
    plan->w_t = take((int64_t)HID * G3 + (d.mixer == MAL_MIXER_QMIX2 ? (int64_t)d.HE * (d.E * d.N + d.E) : 0), 4);
    plan->total_bytes = o;
    return 0;
}

// ---------------------------------------------------------------------------------------------
// learner: launches
// ---------------------------------------------------------------------------------------------
static BatchView make_view(const mal_batch_t *b, const Dims &d) {
    BatchView v;
    v.B = d.B; v.TT = d.TT; v.T = d.T; v.N = d.N; v.A = d.A; v.OBS = d.OBS; v.S = d.S; v.R = d.R;
    v.obs = b->obs; v.onehot = b->onehot; v.state = b->state; v.actions = b->actions;
    v.in = d.in;
    return v;
}

static thread_local int g_use_tc = 1;   // tcgen05 3xTF32 panel GEMM (0: fp32 FFMA panel GEMM)
static thread_local int g_tc_dbg = 0;
// k_gru_fwd9 may run a chain count between 2 and 3 per SM as 2 * SMs equal workers (GruFwdArgs.bal_D): 87 -> 66 us alone at
// 5v5 / B = 32.  Every worker is then on the critical path, so GEMMs that move in beside it (the mixer hypernets) cost more
// than the balance gains (0.322 vs 0.313 ms per step): 1 (default) balances only when nothing runs beside the forward
// recurrence (VDN, no mixer), 2 always, 0 never.
static thread_local int g_gru_balance = 1;
static thread_local int g_gru_balance_pdl = 0;
static thread_local int g_gru_variant = 9;     // recurrences: 9 = 64-thread CTAs, time loop unrolled over the ring slots; 7 = the same before the trimming; 8 = one chain per 128-thread CTA
static thread_local int g_reduce_mn = 3;       // k_reduce_tc operands MN-major straight from the loads (0: round-1 transposition into K-major tiles)
static thread_local int g_reduce_tc = 1;       // weight-gradient reductions on tcgen05 (k_reduce_tc); 0: fp32 FFMA k_reduce_group
static thread_local int g_time_chunks = 1;     // 2: time-chunked forward (input projection of the 2nd half beside the recurrence of the 1st): measured 0.406 vs 0.400 ms at B=32, off by default
static thread_local int g_fuse_agent_in = 1;   // fc1 + W_ih in one tcgen05 kernel (k_agent_in_tc); 0: two grouped GEMM launches
static thread_local int g_tc_pipelined = 1;   // software-pipelined k_linear_tc2 (0: the one-tile-at-a-time k_linear_tc)
static thread_local int g_rec_tc = 1;         // tensor-core recurrence k_gru_fwd_tc: 0 off, 1 when both nets have >= REC_TC_MIN_ROWS chains, 2 whenever R % 32 == 0
#define REC_TC_MIN_ROWS 8192                  // chains (both nets) from which a 128-chain MMA tile per SM beats one FFMA CTA per chain
static thread_local int g_rec_tc_bwd = 0;     // tensor-core BPTT k_gru_bwd_tc beside k_gru_fwd_tc (A operand in tensor memory): correct, but measured slower than k_gru_bwd9 (4.16 vs 3.08 ms at 20v20); 1: on
static uint64_t g_stat_rec_tc = 0, g_stat_rec_tc_bwd = 0, g_stat_reduce_fc1 = 0, g_stat_gru_balanced = 0;
static thread_local int g_fc1_fused = 1;      // fc1 weight gradient over the full input width on one CTA per row chunk (k_reduce_fc1); 0: 128-column tiles of k_reduce_tc3

// Launch counters per kernel flavour since process start (tests check which variant the heuristics picked).
extern "C" uint64_t mal_stat(const char *name) {
    if (!name) return 0;
    if (strcmp(name, "linear_tc2") == 0) return g_stat_tc2;
    if (strcmp(name, "linear_tc") == 0) return g_stat_tc1;
    if (strcmp(name, "reduce_tc") == 0) return g_stat_reduce_tc;
    if (strcmp(name, "reduce_tc_swap") == 0) return g_stat_reduce_tc_swap;
    if (strcmp(name, "reduce_ffma") == 0) return g_stat_reduce_ffma;
    if (strcmp(name, "agent_in_fused") == 0) return g_stat_agent_in_fused;
    if (strcmp(name, "rec_tc") == 0) return g_stat_rec_tc;
    if (strcmp(name, "rec_tc_bwd") == 0) return g_stat_rec_tc_bwd;
    if (strcmp(name, "reduce_fc1") == 0) return g_stat_reduce_fc1;
    if (strcmp(name, "gru_balanced") == 0) return g_stat_gru_balanced;
    return 0;
}
extern "C" int mal_set_option(const char *name, int value) {
    MAL_REQUIRE(name, "mal_set_option: null name");
    if (strcmp(name, "tensor_cores") == 0) { g_use_tc = value ? 1 : 0; return 0; }
    if (strcmp(name, "tc_dbg") == 0) { g_tc_dbg = value; return 0; }
    if (strcmp(name, "gru_variant") == 0) { g_gru_variant = (value == 7 || value == 8) ? value : 9; return 0; }
    if (strcmp(name, "reduce_mn") == 0) { g_reduce_mn = value < 0 ? 0 : (value > 3 ? 3 : value); return 0; }   // 0 K-major transposition, 1 MN-major from registers, 2 MN-major cp.async pipeline, 3 the same with 512 threads
    if (strcmp(name, "reduce_tc") == 0) { g_reduce_tc = value < 0 ? 0 : (value > 2 ? 2 : value); return 0; }   // 0 off, 1 heuristic, 2 always
    if (strcmp(name, "time_chunks") == 0) { g_time_chunks = value; return 0; }
    if (strcmp(name, "gru_balance") == 0) { g_gru_balance = value; return 0; }
    if (strcmp(name, "rec_carveout") == 0) { g_rec_carveout = value; return 0; }
    if (strcmp(name, "gru_balance_pdl") == 0) { g_gru_balance_pdl = value; return 0; }
    if (strcmp(name, "fuse_agent_in") == 0) { g_fuse_agent_in = value ? 1 : 0; return 0; }
    if (strcmp(name, "tc_pipelined") == 0) { g_tc_pipelined = value < 0 ? 0 : (value > 2 ? 2 : value); return 0; }   // 0 off, 1 heuristic, 2 always
    if (strcmp(name, "overlap") == 0) { g_overlap = value ? 1 : 0; return 0; }
    if (strcmp(name, "actsel_lat") == 0) { g_actsel_lat = value ? 1 : 0; return 0; }
    if (strcmp(name, "pdl") == 0) { g_pdl = value ? 1 : 0; return 0; }
    if (strcmp(name, "rec_tc") == 0) { g_rec_tc = value < 0 ? 0 : (value > 2 ? 2 : value); return 0; }   // 0 off, 1 heuristic, 2 always
    if (strcmp(name, "rec_tc_bwd") == 0) { g_rec_tc_bwd = value ? 1 : 0; return 0; }
    if (strcmp(name, "fc1_fused") == 0) { g_fc1_fused = value ? 1 : 0; return 0; }
    mal_set_error("mal_set_option: unknown option %s", name);
    return 1;
}

template <int AK, int EK>
static int launch_tc_inst(const LinGroup &g, dim3 grid, cudaStream_t st, const char *tag, bool pdl) {
    static size_t attr[MAL_MAX_DEV];
    if (int rc = ensure_dyn_smem(k_linear_tc<AK, EK>, TC_SMEM_BYTES, attr)) return rc;
    ++g_stat_tc1;
    { ProfScope _ps(tag, st); launch_k(k_linear_tc<AK, EK>, grid, dim3(TC_THREADS), TC_SMEM_BYTES, st, pdl, g); }
    MAL_LAUNCH_CHECK("k_linear_tc");
    return 0;
}

template <int AK, int EK>
static int launch_tc2_inst(const LinGroup &g, dim3 grid, cudaStream_t st, const char *tag, bool pdl) {
    static size_t attr[MAL_MAX_DEV];
    if (int rc = ensure_dyn_smem(k_linear_tc2<AK, EK>, TC2_SMEM_BYTES, attr)) return rc;
    ++g_stat_tc2;
    { ProfScope _ps(tag, st); launch_k(k_linear_tc2<AK, EK>, grid, dim3(TC2_THREADS), TC2_SMEM_BYTES, st, pdl, g); }
    MAL_LAUNCH_CHECK("k_linear_tc2");
    return 0;
}

static bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

static int launch_linear_tc(const LinGroup &g0, int64_t maxM, cudaStream_t st, const char *tag) {
    int sms, tps;
    if (device_sm_count(&sms, &tps)) return 2;
    // split wide outputs into independent <= TC_NMAX-wide problems (each keeps its W slice resident in smem)
    LinGroup g;
    g.bv = g0.bv;
    g.n = 0;
    g.dbg = g_tc_dbg;
    int pieces_total = 0;
    for (int i = 0; i < g0.n; ++i) pieces_total += (g0.p[i].Nout + TC_NMAX - 1) / TC_NMAX;
    const bool split = pieces_total <= LIN_MAX_PROBS;
    for (int i = 0; i < g0.n; ++i) {
        const LinProb &p = g0.p[i];
        const int np = split ? (p.Nout + TC_NMAX - 1) / TC_NMAX : 1;
        const int w = split ? ((((p.Nout + np - 1) / np) + 15) & ~15) : p.Nout;
        for (int j = 0; j < np; ++j) {
            LinProb q = p;
            const int n_off = j * w;
            q.Nout = (p.Nout - n_off) < w ? (p.Nout - n_off) : w;
            q.W = p.w_trans ? p.W + n_off : p.W + (int64_t)n_off * p.ldw;
            if (p.bias) q.bias = p.bias + n_off;
            if (p.aux) q.aux = p.aux + n_off;
            q.Y = p.Y + n_off;
            g.p[g.n++] = q;
        }
    }
    // kernel flavour: vectorised loaders need 16-byte aligned rows
    bool dense = true, state = true;
    int ek = -1;
    for (int i = 0; i < g.n; ++i) {
        const LinProb &p = g.p[i];
        dense = dense && p.a_kind == A_DENSE && (p.lda & 3) == 0 && (p.K & 3) == 0 && aligned16(p.A);
        state = state && p.a_kind == A_STATE && (p.K & 3) == 0 && (g.bv.state.sb & 3) == 0 && (g.bv.state.st & 3) == 0 &&
                aligned16(g.bv.state.ptr);
        const int e = (p.epi == EPI_BIAS || p.epi == EPI_RELU) ? TCE_BIAS_ACT : (p.epi == EPI_MASKPOS ? TCE_MASKPOS : TCE_FC1);
        MAL_REQUIRE(ek < 0 || ek == e, "launch_linear_tc: mixed epilogue kinds in one group");
        ek = e;
    }
    const int64_t tiles = ceil_div64(maxM, TC_M);
    const int ak = dense ? TCA_VEC_DENSE : (state ? TCA_VEC_STATE : TCA_GENERIC);
    // float4 loads over the obs part of the fc1 input rows (TCE_BIAS_ACT: an input without the agent-id block)
    bool agent_vec = (ek == TCE_FC1 || ek == TCE_BIAS_ACT) && maxM < (1 << 24);
    for (int i = 0; i < g.n; ++i)
        agent_vec = agent_vec && g.p[i].a_kind == A_AGENT_IN && (g.bv.OBS & 3) == 0 && (g.bv.obs.sb & 3) == 0 &&
            (g.bv.obs.st & 3) == 0 && aligned16(g.bv.obs.ptr);
    // the warp-specialised pipeline (one 208 KB CTA per SM) pays off once every SM has a long run of tile-steps; small
    // launches (B = 32 league matchups) keep the lighter kernel, two CTAs per SM, which also co-runs across streams
    int64_t steps_total = 0;
    for (int i = 0; i < g.n; ++i) steps_total += ceil_div64(g.p[i].M, TC_M) * ceil_div64(g.p[i].K, TC_KC);
    const bool long_run = g_tc_pipelined == 2 || steps_total >= (int64_t)16 * sms;
    if (split && g_tc_pipelined && long_run && maxM < (1 << 24)) {
        // software-pipelined kernel: one persistent CTA per SM (208 KB of smem, 512 TMEM columns), never a second wave
        int64_t per1 = sms / g.n; if (per1 < 1) per1 = 1;
        dim3 grid1((unsigned)(tiles < per1 ? tiles : per1), g.n);
        if (ak == TCA_VEC_DENSE && ek == TCE_BIAS_ACT) return launch_tc2_inst<TCA_VEC_DENSE, TCE_BIAS_ACT>(g, grid1, st, tag, g_next_pdl);
        if (ak == TCA_VEC_DENSE && ek == TCE_MASKPOS) return launch_tc2_inst<TCA_VEC_DENSE, TCE_MASKPOS>(g, grid1, st, tag, g_next_pdl);
        if (ak == TCA_VEC_STATE && ek == TCE_BIAS_ACT) return launch_tc2_inst<TCA_VEC_STATE, TCE_BIAS_ACT>(g, grid1, st, tag, g_next_pdl);
        if (agent_vec) return ek == TCE_FC1 ? launch_tc2_inst<TCA_AGENT, TCE_FC1>(g, grid1, st, tag, g_next_pdl)
                                            : launch_tc2_inst<TCA_AGENT, TCE_BIAS_ACT>(g, grid1, st, tag, g_next_pdl);
        if (ek == TCE_FC1) return launch_tc2_inst<TCA_GENERIC, TCE_FC1>(g, grid1, st, tag, g_next_pdl);
        if (ek == TCE_MASKPOS) return launch_tc2_inst<TCA_GENERIC, TCE_MASKPOS>(g, grid1, st, tag, g_next_pdl);
        return launch_tc2_inst<TCA_GENERIC, TCE_BIAS_ACT>(g, grid1, st, tag, g_next_pdl);
    }
    int64_t per = ceil_div64((int64_t)2 * sms, g.n); if (per < 1) per = 1;     // persistent: ~two CTAs per SM in total
    dim3 grid((unsigned)(tiles < per ? tiles : per), g.n);
    if (ak == TCA_VEC_DENSE && ek == TCE_BIAS_ACT) return launch_tc_inst<TCA_VEC_DENSE, TCE_BIAS_ACT>(g, grid, st, tag, g_next_pdl);
    if (ak == TCA_VEC_DENSE && ek == TCE_MASKPOS) return launch_tc_inst<TCA_VEC_DENSE, TCE_MASKPOS>(g, grid, st, tag, g_next_pdl);
    if (ak == TCA_VEC_STATE && ek == TCE_BIAS_ACT) return launch_tc_inst<TCA_VEC_STATE, TCE_BIAS_ACT>(g, grid, st, tag, g_next_pdl);
    // (no TCA_AGENT instance with the plain epilogue here: at the two-CTA register cap it spills; the generic loader serves)
    if (agent_vec && ek == TCE_FC1) return launch_tc_inst<TCA_AGENT, TCE_FC1>(g, grid, st, tag, g_next_pdl);
    if (ek == TCE_FC1) return launch_tc_inst<TCA_GENERIC, TCE_FC1>(g, grid, st, tag, g_next_pdl);
    if (ek == TCE_MASKPOS) return launch_tc_inst<TCA_GENERIC, TCE_MASKPOS>(g, grid, st, tag, g_next_pdl);
    return launch_tc_inst<TCA_GENERIC, TCE_BIAS_ACT>(g, grid, st, tag, g_next_pdl);
}

static int launch_linear(LinGroup &g, int64_t maxM, int maxK, cudaStream_t st, const char *tag) {
    if (g_use_tc) return launch_linear_tc(g, maxM, st, tag);
    const int nkc = (maxK + LIN_KC - 1) / LIN_KC;
    const size_t smem = sizeof(float) * ((size_t)LIN_TM * (nkc * LIN_KC + 4) + (size_t)LIN_TN * LIN_LDW);
    MAL_REQUIRE(smem <= 220 * 1024, "inner dimension %d too large for the panel GEMM", maxK);
    static size_t attr[MAL_MAX_DEV];
    if (int rc = ensure_dyn_smem(k_linear_group, smem, attr)) return rc;
    dim3 grid((unsigned)ceil_div64(maxM, LIN_TM), g.n);
    { ProfScope _ps(tag, st); k_linear_group<<<grid, 256, smem, st>>>(g); }
    MAL_LAUNCH_CHECK("k_linear_group");
    return 0;
}

static LinProb lin(int64_t M, int K, int Nout, int a_kind, int shift, const float *A, int64_t lda, const float *W,
                   int64_t ldw, int w_trans, const float *bias, int epi, const float *aux, int64_t ld_aux, float *Y,
                   int64_t ldy) {
    LinProb p;
    p.M = (int)M; p.K = K; p.Nout = Nout; p.a_kind = a_kind; p.shift = shift; p.A = A; p.lda = lda;
    p.W = W; p.ldw = ldw; p.w_trans = w_trans; p.bias = bias; p.epi = epi; p.aux = aux; p.ld_aux = ld_aux;
    p.Y = Y; p.ldy = ldy;
    return p;
}

static int launch_gru_fwd(const GruFwdArgs &a_in, int nets, int sms, int *chain_flags, bool alone, cudaStream_t st, bool pdl) {
    if (g_gru_variant == 9) { static bool cv[MAL_MAX_DEV]; if (int rc = ensure_max_carveout(k_gru_fwd9<0>, cv, (g_rec_carveout & 1) != 0)) return rc; }
    ProfScope _ps("k_gru_fwd", st);
    GruFwdArgs a = a_in;
    const int chains = nets * a.R, workers = 2 * sms;
    // Two-warp CTAs: up to two chains per SM every warp has a sub-partition to itself (~560 cycles per step); a third chain
    // on an SM puts two warps on two of its sub-partitions (~850, and the whole launch waits for those SMs).  In that window
    // the chains x TT steps are dealt out to 2 * SMs workers of equal length instead (a chain then changes workers once).
    if (g_gru_variant == 9 && (g_gru_balance == 2 || (g_gru_balance == 1 && alone)) && chain_flags && a.t0 == 0 && a.t1 == a.TT && a.TT >= 32 && chains > workers &&
        chains <= 3 * sms && chains <= MAL_CHAIN_FLAGS) {
        a.bal_chains = chains;
        a.bal_D = (int)ceil_div64((int64_t)chains * a.TT, workers);
        a.chain_flags = chain_flags;
        ++g_stat_gru_balanced;
        // NOT as a programmatic dependent launch: the workers must find all SMs free.  Launched early they are packed three
        // and four deep onto the SMs that the predecessor (k_agent_in_tc: one CTA per SM, ragged last round) vacates first,
        // and the point of the balance -- two workers per SM -- is lost (graph replay: 0.322 vs 0.313 ms per step)
        launch_k(k_gru_fwd9<0>, dim3(workers, 1), dim3(HID), 0, st, pdl && g_gru_balance_pdl, a);
        return 0;
    }
    if (g_gru_variant == 7) launch_k(k_gru_fwd7<0>, dim3(a.R, nets), dim3(HID), 0, st, pdl, a);      // one batch row per CTA
    else if (g_gru_variant == 9) launch_k(k_gru_fwd9<0>, dim3(a.R, nets), dim3(HID), 0, st, pdl, a);
    else launch_k(k_gru_fwd8<0>, dim3(a.R, nets), dim3(128), 0, st, pdl, a);
    return 0;
}
// fc1 + W_ih in one tcgen05 kernel (k_agent_in_tc)
static bool fused_in_selected(const Dims &d, const BatchView &bv) {
    return d.kind != MAL_AGENT_DQN && g_use_tc && g_fuse_agent_in && d.M1 < (1 << 24) && (bv.OBS & 3) == 0 && (bv.obs.sb & 3) == 0 &&
           (bv.obs.st & 3) == 0 && aligned16(bv.obs.ptr);
}
// Tensor-core recurrences (k_gru_fwd_tc / k_gru_bwd_tc; gi and the saved gates then use their tiled layouts).  The forward
// and the backward call must agree: both evaluate this on the same dims with the calling thread's option value.
static bool rec_tc_selected(const Dims &d, const BatchView &bv) {
    return fused_in_selected(d, bv) && (d.R % 32) == 0 && (g_rec_tc == 2 || (g_rec_tc == 1 && 2 * (int64_t)d.R >= REC_TC_MIN_ROWS));
}
static int rec_tc_groups(int G, int nets, int sms) {   // 32-chain groups per tile: fewest waves of CTAs, ties -> the smaller tile
    int best_g = 4; int64_t best_w = -1;
    for (int g = 1; g <= 4; ++g) {
        const int64_t w = ceil_div64(ceil_div64(G, g) * nets, sms);
        if (best_w < 0 || w < best_w) { best_w = w; best_g = g; }
    }
    return best_g;
}
static int launch_gru_bwd_tc(const GruBwdArgs &a, int sms, cudaStream_t st, bool pdl) {
    static size_t attr[MAL_MAX_DEV];
    if (int rc = ensure_dyn_smem(k_gru_bwd_tc, (size_t)GB_SMEM_BYTES, attr)) return rc;
    const int G = a.R / 32;
    GruBwdTcArgs ta;
    ta.g = a; ta.groups_per_tile = rec_tc_groups(G, 1, sms);
    ++g_stat_rec_tc_bwd;
    ProfScope _ps("k_gru_bwd", st);
    launch_k(k_gru_bwd_tc, dim3((unsigned)ceil_div64(G, ta.groups_per_tile)), dim3(GT_THREADS), (size_t)GB_SMEM_BYTES, st, pdl, ta);
    return 0;
}
// Tensor-core forward recurrence: tiles of g 32-chain groups (g <= 4), g chosen for the fewest waves of CTAs over the SMs
// (ties: the smaller tile -- fewer idle MMA rows, the per-step time of a tile does not depend on g).
static int launch_gru_fwd_tc(const GruFwdArgs &a, int nets, int sms, cudaStream_t st, bool pdl) {
    static size_t attr[MAL_MAX_DEV];
    if (int rc = ensure_dyn_smem(k_gru_fwd_tc, (size_t)GT_SMEM_BYTES, attr)) return rc;
    const int G = a.R / 32;
    const int best_g = rec_tc_groups(G, nets, sms);
    GruFwdTcArgs ta;
    ta.g = a; ta.groups_per_tile = best_g; ta.gates_tiled = g_rec_tc_bwd;
    ++g_stat_rec_tc;
    ProfScope _ps("k_gru_fwd", st);
    launch_k(k_gru_fwd_tc, dim3((unsigned)ceil_div64(G, best_g), nets), dim3(GT_THREADS), (size_t)GT_SMEM_BYTES, st, pdl, ta);
    return 0;
}
static int launch_gru_bwd(const GruBwdArgs &a, cudaStream_t st, bool pdl) {
    // (up to ~32 chains per SM: 10v10 / B = 128 gains 1.711 -> 1.671 ms per step; with many more waves of chains the smaller L1 costs
    // the kernel more than the co-residence gains -- 20v20 / B = 1024: k_gru_bwd 3.09 -> 3.15 ms, step unchanged)
    if (g_gru_variant == 9) { static bool cv[MAL_MAX_DEV]; if (int rc = ensure_max_carveout(k_gru_bwd9, cv, (g_rec_carveout & 2) && a.R <= 32 * 148)) return rc; }
    ProfScope _ps("k_gru_bwd", st);
    if (g_gru_variant == 7) launch_k(k_gru_bwd7, dim3(a.R), dim3(HID), 0, st, pdl, a);
    else if (g_gru_variant == 9) launch_k(k_gru_bwd9, dim3(a.R), dim3(HID), 0, st, pdl, a);
    else launch_k(k_gru_bwd8, dim3(a.R), dim3(128), 0, st, pdl, a);
    return 0;
}

extern "C" int mal_learner_forward(const mal_batch_t *batch, const mal_learner_cfg_t *cfg, const mal_plan_t *plan,
                                   const float *agent, const float *target_agent, const float *mixer,
                                   const float *target_mixer, void *workspace, void *stream) {
    Dims d;
    if (int rc = get_dims(batch, cfg, &d)) return rc;
    MAL_REQUIRE(plan && workspace && agent && target_agent, "mal_learner_forward: null argument");
    MAL_REQUIRE(!mixer_has_hypernet(d.mixer) || (mixer && target_mixer), "mal_learner_forward: mixer parameters missing");
    MAL_REQUIRE(d.M1 * 4 * HID < (int64_t)1 << 40, "problem too large");
    MAL_REQUIRE(d.M1 < 2147483647LL && d.BT < 2147483647LL, "row count overflows int32");
    int sms, tps;
    if (device_sm_count(&sms, &tps)) return 2;
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t *ws = (uint8_t *)workspace;
    auto F = [&](int64_t off) { return reinterpret_cast<float *>(ws + off); };
    const AgentLayout AL = agent_layout(d.d_in, d.A, d.kind);
    const bool dqn = d.kind == MAL_AGENT_DQN;       // feed-forward agent: h := x = relu(fc1(.)), no gi / recurrence
    const MixerLayout ML = mixer_layout(d.mixer, d.S, d.N, d.E, d.HE);
    const BatchView bv = make_view(batch, d);
    float *scalars = F(plan->scalars);
    const PartLayout pl = part_layout(d, sms);
    float *parts = F(plan->partials);
    const float *ap[2] = {agent, target_agent};
    const float *mp[2] = {mixer, target_mixer};
    float *x[2] = {F(plan->x_on), F(plan->x_tg)}, *gi[2] = {F(plan->gi_on), F(plan->gi_tg)};
    float *hh[2] = {F(plan->h_on), F(plan->h_tg)};
    float *y1[2] = {F(plan->y1_on), F(plan->y1_tg)}, *a2[2] = {F(plan->a2_on), F(plan->a2_tg)};

    SideStreams *ss;
    if (side_streams(&ss)) return 2;
    cudaStream_t sm = g_overlap ? ss->s[0] : st;    // mixer hypernets only depend on the state: run beside the agent path

    // x = relu(fc1([obs | last action | agent id])) and gi = W_ih x + b_ih for every (t,b,n), both nets
    //                                                  basic_controller.py:80-92, drqn_agent.py:30-31, GRUCell input half
    const bool fused_in = fused_in_selected(d, bv);
    // time-chunked forward: the recurrence over the first half of the timesteps runs while the input projection of the
    // second half is still being computed on a side stream (the recurrence is latency-bound and leaves the tensor
    // cores and most issue slots idle)
    const int t_split = (fused_in && g_time_chunks > 1 && g_overlap && d.TT >= 32) ? d.TT / 2 : d.TT;
    // tensor-core recurrence (k_gru_fwd_tc) for large row counts: gi then leaves k_agent_in_tc in the tiled layout
    const bool rec_tc = rec_tc_selected(d, bv);
    if (fused_in) {
        const size_t ai_smem = ai_smem_bytes(d.in.last_end());
        const bool default_in = d.in.last == d.A && d.in.id;
        static size_t attr[MAL_MAX_DEV], attr_g[MAL_MAX_DEV];
        if (int rc = default_in ? ensure_dyn_smem(k_agent_in_tc<true>, ai_smem, attr) : ensure_dyn_smem(k_agent_in_tc<false>, ai_smem, attr_g)) return rc;
        ++g_stat_agent_in_fused;
        auto launch_in = [&](int tb, int te, cudaStream_t s_) -> int {
            AgentInArgs a;
            for (int net = 0; net < 2; ++net) { a.params[net] = ap[net]; a.x[net] = x[net]; a.gi[net] = gi[net]; }
            a.M1 = d.M1; a.d_in = d.d_in; a.n_actions = d.A; a.bv = bv; a.gi_tiled = rec_tc ? 1 : 0;
            a.m_begin = (int64_t)tb * d.R; a.m_end = (int64_t)te * d.R;
            const int64_t tiles = ceil_div64(a.m_end - a.m_begin, TC_M);
            int64_t per = sms / 2; if (per < 1) per = 1;
            dim3 grid((unsigned)(tiles < per ? tiles : per), 2);
            {
                ProfScope _ps("k_agent_in_tc", s_);
                if (default_in) k_agent_in_tc<true><<<grid, AI_THREADS, ai_smem, s_>>>(a);
                else k_agent_in_tc<false><<<grid, AI_THREADS, ai_smem, s_>>>(a);
            }
            MAL_LAUNCH_CHECK("k_agent_in_tc");
            return 0;
        };
        if (int rc = launch_in(0, t_split, st)) return rc;
        if (t_split < d.TT) {
            if (fork_to(st, ss->s[1], ss->fork_ev[1])) return 2;      // starts once the first half's projection is done
            if (int rc = launch_in(t_split, d.TT, ss->s[1])) return rc;
        }
    } else {
    {
        LinGroup g; g.n = 2; g.bv = bv;
        for (int net = 0; net < 2; ++net)
            g.p[net] = lin(d.M1, d.in.last_end(), HID, A_AGENT_IN, 0, nullptr, 0, ap[net] + AL.fc1_w, d.d_in, 0, ap[net] + AL.fc1_b,
                           d.in.id ? EPI_FC1 : EPI_RELU, nullptr, 0, dqn ? hh[net] : x[net], HID);   // DQN: the "hidden state" IS relu(fc1)
        if (int rc = launch_linear(g, d.M1, d.in.last_end(), st, "k_linear_group:fc1")) return rc;
    }
    // gi = W_ih x + b_ih
    if (!dqn) {
        LinGroup g; g.n = 2; g.bv = bv;
        for (int net = 0; net < 2; ++net)
            g.p[net] = lin(d.M1, HID, G3, A_DENSE, 0, x[net], HID, ap[net] + AL.w_ih, HID, 0, ap[net] + AL.b_ih,
                           EPI_BIAS, nullptr, 0, gi[net], G3);
        if (int rc = launch_linear(g, d.M1, HID, st, "k_linear_group:w_ih")) return rc;
    }
    }
    // the mixer hypernet GEMMs start here, beside the (latency-bound) recurrence, not beside the agent-input GEMMs
    // they would compete with for shared memory and tensor cores
    if (fork_to(st, sm, ss->fork_ev[0])) return 2;
    // transposed weight copies for the backward GEMMs (d x = d gi . W_ih, mixer d h = d a . W_2): the tensor-core
    // kernels stage W row-wise with float4 loads; a transposed read would be element-wise.  Off the critical path, and on
    // the OTHER side stream: ahead of the hypernet GEMMs it held them back by its ~10 us, which put mixer_l2 behind the
    // Q head once the balanced recurrence had shortened the main chain.
    // When the forward recurrence may run balanced (nothing else beside it: VDN) the transposes start AFTER it: a dozen
    // CTAs that hold SMs (or just their default carve-out) when the 2 x SMs workers are placed push a third worker onto
    // some SMs, and the whole balanced schedule then runs at the three-per-SM pace (graph replay: 0.300 vs 0.285 ms).
    // No mixer (IQL) has nothing beside the recurrence either.
    cudaStream_t sx = g_overlap ? ss->s[1] : st;
    const bool rec_alone = !mixer_has_hypernet(d.mixer);
    auto launch_transposes = [&]() -> int {
        if (fork_to(st, sx, ss->aux_fork_ev)) return 2;
        TransArgs ta;
        memset(&ta, 0, sizeof(ta));
        float *wt = F(plan->w_t);
        ta.in[0] = agent + (dqn ? AL.fc1_w : AL.w_ih); ta.out[0] = wt; ta.rows[0] = dqn ? 1 : G3; ta.cols[0] = dqn ? 1 : HID; ta.n = 1;
        if (d.mixer == MAL_MIXER_QMIX2) {
            ta.in[1] = mixer + ML.w1b_w; ta.out[1] = wt + (int64_t)HID * G3; ta.rows[1] = d.E * d.N; ta.cols[1] = d.HE;
            ta.in[2] = mixer + ML.wfb_w; ta.out[2] = ta.out[1] + (int64_t)d.HE * d.E * d.N; ta.rows[2] = d.E; ta.cols[2] = d.HE;
            ta.n = 3;
        }
        int max_tiles = 0;
        for (int i = 0; i < ta.n; ++i) {
            const int tl = ((ta.rows[i] + 31) / 32) * ((ta.cols[i] + 31) / 32);
            if (tl > max_tiles) max_tiles = tl;
        }
        if (g_rec_carveout & 4) { static bool cv[MAL_MAX_DEV]; if (int rc = ensure_max_carveout(k_transpose_w, cv)) return rc; }
        { ProfScope _ps("k_transpose_w", sx); k_transpose_w<<<dim3(max_tiles, ta.n), dim3(32, 8), 0, sx>>>(ta); }
        MAL_LAUNCH_CHECK("k_transpose_w");
        return 0;
    };
    if (!rec_alone || dqn) { if (int rc = launch_transposes()) return rc; }
    // the recurrence (online + target concurrently)                         q_learner.py:46-51, 58-62
    if (!dqn) {
        GruFwdArgs a;
        for (int net = 0; net < 2; ++net) { a.params[net] = ap[net]; a.gi[net] = gi[net]; a.hout[net] = hh[net]; }
        a.gates = F(plan->gates); a.TT = d.TT; a.R = d.R; a.d_in = d.d_in; a.n_actions = d.A;
        a.t0 = 0; a.t1 = t_split;
        if (rec_tc ? launch_gru_fwd_tc(a, 2, sms, st, t_split == d.TT) : launch_gru_fwd(a, 2, sms, ss->chain_flags + (size_t)(ss->flag_slot++ % MAL_FLAG_SLOTS) * MAL_CHAIN_FLAGS, rec_alone, st, fused_in && t_split == d.TT)) return 2;   // stream predecessor: k_agent_in_tc
        MAL_LAUNCH_CHECK("k_gru_fwd");
        if (t_split < d.TT) {
            if (join_from(st, ss->s[1], ss->join_ev[1])) return 2;    // second half of gi is ready
            a.t0 = t_split; a.t1 = d.TT;
            if (rec_tc ? launch_gru_fwd_tc(a, 2, sms, st, false) : launch_gru_fwd(a, 2, sms, nullptr, rec_alone, st, false)) return 2;
            MAL_LAUNCH_CHECK("k_gru_fwd");
        }
    }
    // q, chosen-action gather, masked double-Q target max                   q_learner.py:52-78
    {
        HeadArgs a;
        for (int net = 0; net < 2; ++net) { a.params[net] = ap[net]; a.hout[net] = hh[net]; }
        a.B = d.B; a.TT = d.TT; a.N = d.N; a.A = d.A; a.R = d.R; a.d_in = d.d_in; a.double_q = cfg->double_q; a.kind = d.kind;
        a.actions = batch->actions; a.avail = batch->avail;
        a.mac_out = cfg->save_q ? F(plan->mac_out) : nullptr;
        a.target_mac_out = cfg->save_q ? F(plan->target_mac_out) : nullptr;
        a.chosen = F(plan->chosen); a.target_max = F(plan->target_max);
        a.argmax = reinterpret_cast<int *>(ws + plan->argmax);
        const size_t smem = qh_smem_bytes(d.A);
        const int64_t qh_tiles = ceil_div64(d.M1, 64), qh_slots = 3 * (int64_t)sms;      // balanced: every CTA walks the same
        const int64_t qh_grid = ceil_div64(qh_tiles, ceil_div64(qh_tiles, qh_slots));    // number of tiles (+-1), in one wave
        static size_t attr[MAL_MAX_DEV];
        if (int rc = ensure_dyn_smem(k_q_head, smem, attr)) return rc;
        if (g_rec_carveout & 4) { static bool cv[MAL_MAX_DEV]; if (int rc = ensure_max_carveout(k_q_head, cv)) return rc; }
        { ProfScope _ps("k_q_head", st); launch_k(k_q_head, dim3((unsigned)qh_grid), dim3(128), smem, st, true, a); }   // predecessor: k_gru_fwd7
        MAL_LAUNCH_CHECK("k_q_head");
    }
    if (rec_alone && !dqn) { if (int rc = launch_transposes()) return rc; }   // beside the mixing kernel; the backward reads them
    // mixer hypernetworks                                                   qmix.py:41-59
    if (d.mixer == MAL_MIXER_QMIX2) {
        LinGroup g; g.n = 8; g.bv = bv;
        for (int net = 0; net < 2; ++net) {
            const float *P = mp[net];
            g.p[net * 4 + 0] = lin(d.BT, d.S, d.HE, A_STATE, net, nullptr, 0, P + ML.w1a_w, d.S, 0, P + ML.w1a_b, EPI_RELU, nullptr, 0, y1[net], d.ld1);
            g.p[net * 4 + 1] = lin(d.BT, d.S, d.HE, A_STATE, net, nullptr, 0, P + ML.wfa_w, d.S, 0, P + ML.wfa_b, EPI_RELU, nullptr, 0, y1[net] + d.HE, d.ld1);
            g.p[net * 4 + 2] = lin(d.BT, d.S, d.E, A_STATE, net, nullptr, 0, P + ML.b1_w, d.S, 0, P + ML.b1_b, EPI_BIAS, nullptr, 0, y1[net] + 2 * d.HE, d.ld1);
            g.p[net * 4 + 3] = lin(d.BT, d.S, d.E, A_STATE, net, nullptr, 0, P + ML.v0_w, d.S, 0, P + ML.v0_b, EPI_RELU, nullptr, 0, y1[net] + 2 * d.HE + d.E, d.ld1);
        }
        if (int rc = launch_linear(g, d.BT, d.S, sm, "k_linear_group:mixer_l1")) return rc;
        LinGroup h; h.n = 4; h.bv = bv;
        for (int net = 0; net < 2; ++net) {
            const float *P = mp[net];
            h.p[net * 2 + 0] = lin(d.BT, d.HE, d.E * d.N, A_DENSE, 0, y1[net], d.ld1, P + ML.w1b_w, d.HE, 0, P + ML.w1b_b, EPI_BIAS, nullptr, 0, a2[net], d.ld2);
            h.p[net * 2 + 1] = lin(d.BT, d.HE, d.E, A_DENSE, 0, y1[net] + d.HE, d.ld1, P + ML.wfb_w, d.HE, 0, P + ML.wfb_b, EPI_BIAS, nullptr, 0, a2[net] + d.E * d.N, d.ld2);
        }
        if (int rc = launch_linear(h, d.BT, d.HE, sm, "k_linear_group:mixer_l2")) return rc;
    } else if (d.mixer == MAL_MIXER_QMIX1) {
        LinGroup g; g.n = 8; g.bv = bv;
        for (int net = 0; net < 2; ++net) {
            const float *P = mp[net];
            g.p[net * 4 + 0] = lin(d.BT, d.S, d.E * d.N, A_STATE, net, nullptr, 0, P + ML.w1b_w, d.S, 0, P + ML.w1b_b, EPI_BIAS, nullptr, 0, a2[net], d.ld2);
            g.p[net * 4 + 1] = lin(d.BT, d.S, d.E, A_STATE, net, nullptr, 0, P + ML.wfb_w, d.S, 0, P + ML.wfb_b, EPI_BIAS, nullptr, 0, a2[net] + d.E * d.N, d.ld2);
            g.p[net * 4 + 2] = lin(d.BT, d.S, d.E, A_STATE, net, nullptr, 0, P + ML.b1_w, d.S, 0, P + ML.b1_b, EPI_BIAS, nullptr, 0, y1[net], d.ld1);
            g.p[net * 4 + 3] = lin(d.BT, d.S, d.E, A_STATE, net, nullptr, 0, P + ML.v0_w, d.S, 0, P + ML.v0_b, EPI_RELU, nullptr, 0, y1[net] + d.E, d.ld1);
        }
        if (int rc = launch_linear(g, d.BT, d.S, sm, "k_linear_group:mixer_l1")) return rc;
    }
    if (join_from(st, sm, ss->join_ev[0])) return 2;
    if (join_from(st, sx, ss->aux_join_ev)) return 2;
    // mixing + TD error + masked loss + element-wise mixer backward          q_learner.py:81-98
    {
        MixArgs a;
        memset(&a, 0, sizeof(a));
        a.mixer = d.mixer; a.B = d.B; a.T = d.T; a.N = d.N; a.E = d.E; a.HE = d.HE; a.S = d.S;
        a.R = d.R; a.A = d.A; a.d_in = d.d_in; a.agent = agent; a.kind = d.kind;
        a.relu_src = dqn ? hh[0] : nullptr;          // DQN: the head seed is d x: masked by relu'(x) right here
        for (int net = 0; net < 2; ++net) { a.y1[net] = y1[net]; a.a2[net] = a2[net]; a.mparams[net] = mp[net]; }
        a.chosen = F(plan->chosen); a.target_max = F(plan->target_max); a.mask = F(plan->mask);
        a.reward = batch->reward; a.terminated = batch->terminated; a.filled = batch->filled; a.actions = batch->actions;
        a.gamma = cfg->gamma; a.dh_head = F(plan->dh_head);
        a.q_tot = F(plan->q_tot); a.target_q_tot = F(plan->target_q_tot); a.targets = F(plan->targets); a.td = F(plan->td);
        a.d_a2 = F(plan->d_a2); a.d_y1 = F(plan->d_y1); a.d_chosen = F(plan->d_chosen);
        a.part_stats = parts + pl.mix_stats; a.part_v2 = parts + pl.mix_v2;
        a.weight = batch->weight;
        if (cfg->returns == MAL_RETURNS_TD_LAMBDA) {
            // TD(lambda): target rows, then the per-episode reverse recursion, then the step over the given targets
            if (g_rec_carveout & 4) { static bool cv[MAL_MAX_DEV]; if (int rc = ensure_max_carveout(k_mix_tq, cv)) return rc; }
            { ProfScope _ps("k_mix_tq", st); launch_k(k_mix_tq, dim3(pl.nblk_mix), dim3(256), 0, st, true, a); }
            MAL_LAUNCH_CHECK("k_mix_tq");
            TdLambdaArgs tl;
            tl.tq = a.target_q_tot; tl.targets = a.targets;
            tl.reward = batch->reward; tl.terminated = batch->terminated; tl.filled = batch->filled;
            tl.B = d.B; tl.T = d.T; tl.Q = d.mixer == MAL_MIXER_NONE ? d.N : 1;
            tl.lg = (double)cfg->td_lambda * (double)cfg->gamma;
            tl.xg = (1.0 - (double)cfg->td_lambda) * (double)cfg->gamma;
            const int64_t n_ep = (int64_t)tl.B * tl.Q;
            { ProfScope _ps("k_td_lambda", st); launch_k(k_td_lambda, dim3((unsigned)ceil_div64(n_ep, TDL_WARPS)), dim3(32 * TDL_WARPS), 0, st, true, tl); }
            MAL_LAUNCH_CHECK("k_td_lambda");
            if (batch->weight.ptr) {
                if (g_rec_carveout & 4) { static bool cv[MAL_MAX_DEV]; if (int rc = ensure_max_carveout(k_mix_td_lambda<true>, cv)) return rc; }
                { ProfScope _ps("k_mix_td_lambda_w", st); launch_k(k_mix_td_lambda<true>, dim3(pl.nblk_mix), dim3(256), 0, st, true, a); }
            } else {
                if (g_rec_carveout & 4) { static bool cv[MAL_MAX_DEV]; if (int rc = ensure_max_carveout(k_mix_td_lambda<false>, cv)) return rc; }
                { ProfScope _ps("k_mix_td_lambda", st); launch_k(k_mix_td_lambda<false>, dim3(pl.nblk_mix), dim3(256), 0, st, true, a); }
            }
        } else if (batch->weight.ptr) {              // prioritized replay: importance-weighted loss and seeds
            if (g_rec_carveout & 4) { static bool cv[MAL_MAX_DEV]; if (int rc = ensure_max_carveout(k_mix_td<true>, cv)) return rc; }
            { ProfScope _ps("k_mix_td_w", st); launch_k(k_mix_td<true>, dim3(pl.nblk_mix), dim3(256), 0, st, true, a); }
        } else {
            if (g_rec_carveout & 4) { static bool cv[MAL_MAX_DEV]; if (int rc = ensure_max_carveout(k_mix_td<false>, cv)) return rc; }
            { ProfScope _ps("k_mix_td", st); launch_k(k_mix_td<false>, dim3(pl.nblk_mix), dim3(256), 0, st, true, a); }   // stream predecessor: k_q_head
        }
        MAL_LAUNCH_CHECK("k_mix_td");
        // nothing before the gradient gather reads the scalars: inside mal_learner_step the finalize runs on the side
        // stream (the backward joins that stream before k_grad_reduce) and leaves the critical path
        cudaStream_t sf = (g_defer_stats && g_overlap) ? ss->s[0] : st;
        if (fork_to(st, sf, ss->fork_ev[3])) return 2;
        { ProfScope _ps("k_stats_finalize", sf); k_stats_finalize<<<1 + (mixer_has_hypernet(d.mixer) ? (d.E + 1 + 7) / 8 : 0), 256, 0, sf>>>(
                                                       parts + pl.mix_stats, pl.nblk_mix, d.N, scalars, parts + pl.mix_v2,
                                                       d.E + 1, parts + pl.mix_v2_sum); }
        MAL_LAUNCH_CHECK("k_stats_finalize");
    }
    return 0;
}

// Y = epi(A W^T + bias) on dense row-major operands through the same kernels the learner uses (unit tests).
extern "C" int mal_debug_linear(int32_t M, int32_t K, int32_t Nout, const float *A, int64_t lda, const float *W,
                                int64_t ldw, int32_t w_trans, const float *bias, int32_t epi, const float *aux,
                                int64_t ld_aux, float *Y, int64_t ldy, int32_t use_tc, void *stream) {
    MAL_REQUIRE(A && W && Y && M > 0 && K > 0 && Nout > 0, "mal_debug_linear: bad arguments");
    MAL_REQUIRE(epi == EPI_BIAS || epi == EPI_RELU || epi == EPI_MASKPOS, "mal_debug_linear: unsupported epilogue");
    LinGroup g;
    memset(&g, 0, sizeof(g));
    g.n = 1;
    g.p[0] = lin(M, K, Nout, A_DENSE, 0, A, lda, W, ldw, w_trans, bias, epi, aux, ld_aux, Y, ldy);
    // use_tc: 0 fp32 FFMA panel GEMM, 1 tcgen05 kernel picked by the launch heuristic, 2 force the pipelined kernel,
    //         3 force the one-tile-at-a-time kernel
    const int saved = g_use_tc, saved_p = g_tc_pipelined;
    g_use_tc = use_tc ? 1 : 0;
    if (use_tc == 2) g_tc_pipelined = 2;
    if (use_tc == 3) g_tc_pipelined = 0;
    int rc = launch_linear(g, M, K, (cudaStream_t)stream, use_tc ? "k_linear_tc:debug" : "k_linear_group:debug");
    g_use_tc = saved;
    g_tc_pipelined = saved_p;
    return rc;
}

extern "C" int mal_mixer_forward(int32_t mixer, int32_t B, int32_t T, int32_t N, int32_t S, int32_t E, int32_t HE,
                                 const float *params, const float *agent_qs, const float *states, int64_t state_sb,
                                 int64_t state_st, float *scratch, float *q_tot, void *stream) {
    MAL_REQUIRE(agent_qs && q_tot && B > 0 && T > 0 && N > 0 && N <= MAL_MAX_ACTIONS, "mal_mixer_forward: bad arguments");
    MAL_REQUIRE(mixer == MAL_MIXER_VDN || mixer == MAL_MIXER_QMIX2 || mixer == MAL_MIXER_QMIX1, "Mixer %d not recognised.", mixer);
    int sms, tps;
    if (device_sm_count(&sms, &tps)) return 2;
    cudaStream_t st = (cudaStream_t)stream;
    MixArgs a;
    memset(&a, 0, sizeof(a));
    a.mixer = mixer; a.B = B; a.T = T; a.N = N; a.E = E; a.HE = HE; a.S = S;
    a.chosen = agent_qs; a.q_tot = q_tot;
    const int64_t BT = (int64_t)B * T;
    if (mixer_has_hypernet(mixer)) {
        MAL_REQUIRE(params && states && scratch && S > 0, "mal_mixer_forward: params/states/scratch missing");
        MAL_REQUIRE(E >= 1 && E <= MAL_MAX_EMBED, "mixing_embed_dim must be in [1, %d]", MAL_MAX_EMBED);
        const MixerLayout ML = mixer_layout(mixer, S, N, E, HE);
        const int two = mixer == MAL_MIXER_QMIX2;
        const int ld1 = two ? 2 * HE + 2 * E : 2 * E, ld2 = E * N + E;
        float *y1 = scratch, *a2 = scratch + BT * ld1;   // scratch: BT * (ld1 + ld2) floats
        BatchView bv;
        memset(&bv, 0, sizeof(bv));
        bv.B = B; bv.T = T; bv.TT = T; bv.N = N; bv.S = S; bv.R = B * N;
        bv.state.ptr = states; bv.state.sb = state_sb; bv.state.st = state_st;
        LinGroup g; g.bv = bv;
        if (two) {
            g.n = 4;
            g.p[0] = lin(BT, S, HE, A_STATE, 0, nullptr, 0, params + ML.w1a_w, S, 0, params + ML.w1a_b, EPI_RELU, nullptr, 0, y1, ld1);
            g.p[1] = lin(BT, S, HE, A_STATE, 0, nullptr, 0, params + ML.wfa_w, S, 0, params + ML.wfa_b, EPI_RELU, nullptr, 0, y1 + HE, ld1);
            g.p[2] = lin(BT, S, E, A_STATE, 0, nullptr, 0, params + ML.b1_w, S, 0, params + ML.b1_b, EPI_BIAS, nullptr, 0, y1 + 2 * HE, ld1);
            g.p[3] = lin(BT, S, E, A_STATE, 0, nullptr, 0, params + ML.v0_w, S, 0, params + ML.v0_b, EPI_RELU, nullptr, 0, y1 + 2 * HE + E, ld1);
            if (int rc = launch_linear(g, BT, S, st, "k_linear_group:mixer_fwd_l1")) return rc;
            LinGroup h; h.bv = bv; h.n = 2;
            h.p[0] = lin(BT, HE, E * N, A_DENSE, 0, y1, ld1, params + ML.w1b_w, HE, 0, params + ML.w1b_b, EPI_BIAS, nullptr, 0, a2, ld2);
            h.p[1] = lin(BT, HE, E, A_DENSE, 0, y1 + HE, ld1, params + ML.wfb_w, HE, 0, params + ML.wfb_b, EPI_BIAS, nullptr, 0, a2 + E * N, ld2);
            if (int rc = launch_linear(h, BT, HE, st, "k_linear_group:mixer_fwd_l2")) return rc;
        } else {
            g.n = 4;
            g.p[0] = lin(BT, S, E * N, A_STATE, 0, nullptr, 0, params + ML.w1b_w, S, 0, params + ML.w1b_b, EPI_BIAS, nullptr, 0, a2, ld2);
            g.p[1] = lin(BT, S, E, A_STATE, 0, nullptr, 0, params + ML.wfb_w, S, 0, params + ML.wfb_b, EPI_BIAS, nullptr, 0, a2 + E * N, ld2);
            g.p[2] = lin(BT, S, E, A_STATE, 0, nullptr, 0, params + ML.b1_w, S, 0, params + ML.b1_b, EPI_BIAS, nullptr, 0, y1, ld1);
            g.p[3] = lin(BT, S, E, A_STATE, 0, nullptr, 0, params + ML.v0_w, S, 0, params + ML.v0_b, EPI_RELU, nullptr, 0, y1 + E, ld1);
            if (int rc = launch_linear(g, BT, S, st, "k_linear_group:mixer_fwd_l1")) return rc;
        }
        a.y1[0] = y1; a.a2[0] = a2; a.mparams[0] = params;
    }
    int64_t grid = ceil_div64(BT, 8); if (grid > (int64_t)sms * 4) grid = (int64_t)sms * 4;
    { ProfScope _ps("k_mix_fwd", st); k_mix_fwd<<<(unsigned)grid, 256, 0, st>>>(a); }
    MAL_LAUNCH_CHECK("k_mix_fwd");
    return 0;
}

static RedProb red(int64_t M, int K, int Nout, const float *dY, int64_t ldy, int a_kind, int shift, const float *A,
                   int64_t lda, float *partW, float *partB, int n_chunks, int64_t rpc) {
    RedProb p;
    p.M0 = 0; p.M = M; p.K = K; p.Nout = Nout; p.dY = dY; p.ldy = ldy; p.dy_kind = 0; p.a_kind = a_kind; p.shift = shift;
    p.A = A; p.lda = lda; p.partW = partW; p.partB = partB; p.n_chunks = n_chunks; p.rows_per_chunk = rpc;
    p.tile0 = 0; p.n_ktiles = (K + 63) / 64;
    return p;
}

template <int AK, int DK>
static int launch_reduce_inst(RedGroup &g, cudaStream_t st, const char *tag, const char *tag_tc) {
    // the tensor-core kernel pays a per-CTA setup and two barriers per 32-row block: it wins once a CTA has a long run
    // of blocks (>= 512 rows per chunk); short reductions (B = 32 mixer / fc1 problems) stay on the FFMA kernel
    int64_t min_rpc = 1 << 30;
    for (int i = 0; i < g.n; ++i) if (g.p[i].rows_per_chunk < min_rpc) min_rpc = g.p[i].rows_per_chunk;
    const bool tc = g_use_tc && DK == 0 && (g_reduce_tc == 2 || (g_reduce_tc == 1 && min_rpc >= 512));
    bool swap = tc;
    for (int i = 0; i < g.n; ++i) swap = swap && red_swapped(g.p[i].Nout, g.p[i].K);
    int tiles = 0, maxc = 0;
    for (int i = 0; i < g.n; ++i) {
        g.p[i].tile0 = tiles;
        if (swap) tiles += ((g.p[i].K + RT_NT - 1) / RT_NT) * ((g.p[i].Nout + RT_KT - 1) / RT_KT);
        else tiles += ((g.p[i].Nout + (tc ? RT_NT : 64) - 1) / (tc ? RT_NT : 64)) * g.p[i].n_ktiles;
        if (g.p[i].n_chunks > maxc) maxc = g.p[i].n_chunks;
    }
    dim3 grid(maxc, tiles);
    if (tc) {
        static size_t attr0[MAL_MAX_DEV], attr1[MAL_MAX_DEV], attr2[MAL_MAX_DEV], attr3[MAL_MAX_DEV], attr4[MAL_MAX_DEV], attr5[MAL_MAX_DEV];
        if (int rc = ensure_dyn_smem(k_reduce_tc<AK, 0, 0>, RT_SMEM_BYTES, attr0)) return rc;
        if (int rc = ensure_dyn_smem(k_reduce_tc<AK, 1, 0>, RT_SMEM_BYTES, attr1)) return rc;
        if (int rc = ensure_dyn_smem(k_reduce_tc<AK, 0, 1>, RT_SMEM_BYTES, attr2)) return rc;
        if (int rc = ensure_dyn_smem(k_reduce_tc<AK, 1, 1>, RT_SMEM_BYTES, attr3)) return rc;
        if (int rc = ensure_dyn_smem(k_reduce_tc<AK, 0, 2>, RT_SMEM_BYTES_PIPE, attr4)) return rc;
        if (int rc = ensure_dyn_smem(k_reduce_tc<AK, 1, 2>, RT_SMEM_BYTES_PIPE, attr5)) return rc;
        if (swap) ++g_stat_reduce_tc_swap; else ++g_stat_reduce_tc;
        ProfScope _ps(tag_tc, st);
        if (g_reduce_mn == 3) {     // 512-thread MN-major cp.async pipeline
            static size_t attr6[MAL_MAX_DEV], attr7[MAL_MAX_DEV];
            if (int rc = ensure_dyn_smem(k_reduce_tc3<AK, 0>, RT_SMEM_BYTES_PIPE, attr6)) return rc;
            if (int rc = ensure_dyn_smem(k_reduce_tc3<AK, 1>, RT_SMEM_BYTES_PIPE, attr7)) return rc;
            if (swap) launch_k(k_reduce_tc3<AK, 1>, grid, dim3(RT3_THREADS), RT_SMEM_BYTES_PIPE, st, g_next_pdl, g);
            else launch_k(k_reduce_tc3<AK, 0>, grid, dim3(RT3_THREADS), RT_SMEM_BYTES_PIPE, st, g_next_pdl, g);
        } else if (g_reduce_mn == 2) {     // MN-major operands fed by a four-stage cp.async pipeline
            if (swap) launch_k(k_reduce_tc<AK, 1, 2>, grid, dim3(256), RT_SMEM_BYTES_PIPE, st, g_next_pdl, g);
            else launch_k(k_reduce_tc<AK, 0, 2>, grid, dim3(256), RT_SMEM_BYTES_PIPE, st, g_next_pdl, g);
        } else if (g_reduce_mn) {   // MN-major operands staged from registers (one block prefetched)
            if (swap) launch_k(k_reduce_tc<AK, 1, 1>, grid, dim3(256), RT_SMEM_BYTES, st, g_next_pdl, g);
            else launch_k(k_reduce_tc<AK, 0, 1>, grid, dim3(256), RT_SMEM_BYTES, st, g_next_pdl, g);
        } else if (swap) launch_k(k_reduce_tc<AK, 1, 0>, grid, dim3(256), RT_SMEM_BYTES, st, g_next_pdl, g);
        else launch_k(k_reduce_tc<AK, 0, 0>, grid, dim3(256), RT_SMEM_BYTES, st, g_next_pdl, g);
        MAL_LAUNCH_CHECK("k_reduce_tc");
        return 0;
    }
    ++g_stat_reduce_ffma;
    if (g_rec_carveout & 4) { static bool cv[MAL_MAX_DEV]; if (int rc = ensure_max_carveout((k_reduce_group<AK, DK>), cv)) return rc; }
    { ProfScope _ps(tag, st); launch_k(k_reduce_group<AK, DK>, grid, dim3(256), 0, st, g_next_pdl, g); }
    MAL_LAUNCH_CHECK("k_reduce_group");
    return 0;
}

// one launch per (A loader, dY kind) so that every kernel instance is straight-line code
static int launch_reduce(RedGroup &g, cudaStream_t st, const char *tag) {
    const int kinds[4][2] = {{A_DENSE, 0}, {A_STATE, 0}, {A_AGENT_IN, 0}, {A_DENSE, 1}};
    for (int q = 0; q < 4; ++q) {
        RedGroup h;
        h.bv = g.bv;
        h.n = 0;
        for (int i = 0; i < g.n; ++i)
            if (g.p[i].a_kind == kinds[q][0] && g.p[i].dy_kind == kinds[q][1]) h.p[h.n++] = g.p[i];
        if (h.n == 0) continue;
        int rc = 0;
        const bool agent = strstr(tag, "agent") != nullptr;
        if (q == 0) rc = launch_reduce_inst<A_DENSE, 0>(h, st, agent ? "k_reduce_group:agent_dense" : "k_reduce_group:mixer_dense",
                                                        agent ? "k_reduce_tc:agent_dense" : "k_reduce_tc:mixer_dense");
        else if (q == 1) rc = launch_reduce_inst<A_STATE, 0>(h, st, "k_reduce_group:mixer_state", "k_reduce_tc:mixer_state");
        else if (q == 2) rc = launch_reduce_inst<A_AGENT_IN, 0>(h, st, "k_reduce_group:agent_fc1", "k_reduce_tc:agent_fc1");
        else rc = launch_reduce_inst<A_DENSE, 1>(h, st, "k_reduce_group:agent_fc2", "k_reduce_group:agent_fc2");
        if (rc) return rc;
    }
    for (int i = 0; i < g.n; ++i)
        MAL_REQUIRE((g.p[i].dy_kind == 0) || g.p[i].a_kind == A_DENSE, "launch_reduce: unsupported loader combination");
    return 0;
}

// QMIX hypernet backward from the element-wise seeds d_a2 / d_y1: for two-layer hypernets the layer-2 input gradients
//   d h1 = (d a1 . W_1.2) * (h1 > 0),  d hf = (d af . W_f.2) * (hf > 0)   (written into the h1 | hf columns of d_y1),
// then the layer-2 and layer-1 weight-gradient split reductions into per-chunk partials.  Shared by the learner's backward and
// mal_mixer_backward.  wt1 / wtf: hyper_w_1.2.weight / hyper_w_final.2.weight as GEMM operands W(n,k) (LinProb's w_trans).
struct HyperBwd {
    int mixer, two, N, E, HE, S, ld1, ld2;
    int64_t BT;
    const float *d_a2; float *d_y1; const float *y1;
    const float *wt1, *wtf; int64_t ldw1, ldwf; int w_trans;
    float *l2a_w, *l2a_b, *l2b_w, *l2b_b, *l1_w, *l1_b;
    int nc_m2, nc_m1; int64_t rpc_m2, rpc_m1;
};
static void hyper_bwd_dims(const Dims &d, HyperBwd *h) {
    h->mixer = d.mixer; h->two = d.two; h->N = d.N; h->E = d.E; h->HE = d.HE; h->S = d.S; h->ld1 = d.ld1; h->ld2 = d.ld2;
    h->BT = d.BT;
}
static int launch_hyper_bwd(const HyperBwd &h, const BatchView &bv, cudaStream_t s1) {
    if (h.mixer == MAL_MIXER_QMIX2) {
        LinGroup g; g.n = 2; g.bv = bv;   // d h1 = (d a1 . W12) * (h1 > 0) ; d hf = (d af . Wf2) * (hf > 0)
        g.p[0] = lin(h.BT, h.E * h.N, h.HE, A_DENSE, 0, h.d_a2, h.ld2, h.wt1, h.ldw1, h.w_trans, nullptr, EPI_MASKPOS, h.y1, h.ld1, h.d_y1, h.ld1);
        g.p[1] = lin(h.BT, h.E, h.HE, A_DENSE, 0, h.d_a2 + h.E * h.N, h.ld2, h.wtf, h.ldwf, h.w_trans, nullptr, EPI_MASKPOS, h.y1 + h.HE, h.ld1, h.d_y1 + h.HE, h.ld1);
        if (int rc = launch_linear(g, h.BT, h.E * h.N, s1, "k_linear_group:mixer_bwd_dh")) return rc;
        RedGroup r; r.n = 3; r.bv = bv;
        r.p[0] = red(h.BT, h.HE, h.E * h.N, h.d_a2, h.ld2, A_DENSE, 0, h.y1, h.ld1, h.l2a_w, h.l2a_b, h.nc_m2, h.rpc_m2);
        r.p[1] = red(h.BT, h.HE, h.E, h.d_a2 + h.E * h.N, h.ld2, A_DENSE, 0, h.y1 + h.HE, h.ld1, h.l2b_w, h.l2b_b, h.nc_m2, h.rpc_m2);
        r.p[2] = red(h.BT, h.S, h.ld1, h.d_y1, h.ld1, A_STATE, 0, nullptr, 0, h.l1_w, h.l1_b, h.nc_m1, h.rpc_m1);
        if (int rc = launch_reduce(r, s1, "k_reduce_group:mixer")) return rc;
    } else if (h.mixer == MAL_MIXER_QMIX1) {
        RedGroup r; r.n = 3; r.bv = bv;
        r.p[0] = red(h.BT, h.S, h.E * h.N, h.d_a2, h.ld2, A_STATE, 0, nullptr, 0, h.l2a_w, h.l2a_b, h.nc_m2, h.rpc_m2);
        r.p[1] = red(h.BT, h.S, h.E, h.d_a2 + h.E * h.N, h.ld2, A_STATE, 0, nullptr, 0, h.l2b_w, h.l2b_b, h.nc_m2, h.rpc_m2);
        r.p[2] = red(h.BT, h.S, h.ld1, h.d_y1, h.ld1, A_STATE, 0, nullptr, 0, h.l1_w, h.l1_b, h.nc_m1, h.rpc_m1);
        if (int rc = launch_reduce(r, s1, "k_reduce_group:mixer")) return rc;
    }
    return 0;
}

extern "C" int mal_learner_backward(const mal_batch_t *batch, const mal_learner_cfg_t *cfg, const mal_plan_t *plan,
                                    const float *agent, const float *mixer, void *workspace, float *grad, void *stream) {
    Dims d;
    if (int rc = get_dims(batch, cfg, &d)) return rc;
    MAL_REQUIRE(plan && workspace && agent && grad, "mal_learner_backward: null argument");
    MAL_REQUIRE(!mixer_has_hypernet(d.mixer) || mixer, "mal_learner_backward: mixer parameters missing");
    int sms, tps;
    if (device_sm_count(&sms, &tps)) return 2;
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t *ws = (uint8_t *)workspace;
    auto F = [&](int64_t off) { return reinterpret_cast<float *>(ws + off); };
    const AgentLayout AL = agent_layout(d.d_in, d.A, d.kind);
    const bool dqn = d.kind == MAL_AGENT_DQN;
    const MixerLayout ML = mixer_layout(d.mixer, d.S, d.N, d.E, d.HE);
    const BatchView bv = make_view(batch, d);
    const PartLayout pl = part_layout(d, sms);
    float *parts = F(plan->partials);
    float *d_g = F(plan->d_g), *d_x = F(plan->d_x), *d_a2 = F(plan->d_a2), *d_y1 = F(plan->d_y1);
    float *y1 = F(plan->y1_on);

    SideStreams *ss;
    if (side_streams(&ss)) return 2;
    cudaStream_t s1 = g_overlap ? ss->s[0] : st, s2 = g_overlap ? ss->s[1] : st;
    if (fork_to(st, s1, ss->fork_ev[0])) return 2;
    if (fork_to(st, s2, ss->fork_ev[1])) return 2;

    // ---- side stream 1: mixer hypernet backward (independent of the agent BPTT)
    if (mixer_has_hypernet(d.mixer)) {
        HyperBwd h;
        hyper_bwd_dims(d, &h);
        h.d_a2 = d_a2; h.d_y1 = d_y1; h.y1 = y1;
        h.wt1 = F(plan->w_t) + (int64_t)HID * G3; h.wtf = h.wt1 + (int64_t)d.HE * d.E * d.N;   // transposed by the forward call
        h.ldw1 = d.E * d.N; h.ldwf = d.E; h.w_trans = 0;
        h.l2a_w = parts + pl.m_l2a_w; h.l2a_b = parts + pl.m_l2a_b; h.l2b_w = parts + pl.m_l2b_w; h.l2b_b = parts + pl.m_l2b_b;
        h.l1_w = parts + pl.m_l1_w; h.l1_b = parts + pl.m_l1_b;
        h.nc_m2 = pl.nc_m2; h.rpc_m2 = pl.rpc_m2; h.nc_m1 = pl.nc_m1; h.rpc_m1 = pl.rpc_m1;
        if (int rc = launch_hyper_bwd(h, bv, s1)) return rc;
    }
    const bool frozen = cfg->freeze_agent != 0;   // multi_agent_controller.py:74-76: the agent gets no gradient at all
    // ---- side stream 2: fc2 gradients only need d_chosen and h (both forward products)
    if (!frozen) {
        Fc2GradArgs a;
        a.d_chosen = F(plan->d_chosen); a.actions = batch->actions; a.hout = F(plan->h_on);
        a.partW = parts + pl.fc2_w; a.partB = parts + pl.fc2_b;
        a.T = d.T; a.N = d.N; a.A = d.A; a.R = d.R; a.rows = (int64_t)d.T * d.R;
        const size_t smem = sizeof(float) * 8 * ((size_t)d.A * HID + 32);
        static size_t attr[MAL_MAX_DEV];
        if (int rc = ensure_dyn_smem(k_fc2_grad, smem, attr)) return rc;
        if (g_rec_carveout & 4) { static bool cv[MAL_MAX_DEV]; if (int rc = ensure_max_carveout(k_fc2_grad, cv)) return rc; }
        { ProfScope _ps("k_fc2_grad", s2); k_fc2_grad<<<pl.nc_f2, 256, smem, s2>>>(a); }
        MAL_LAUNCH_CHECK("k_fc2_grad");
    }

    // ---- main stream: BPTT recurrence
    if (!frozen && !dqn) {
        GruBwdArgs a;
        a.params = agent; a.hout = F(plan->h_on); a.gates = F(plan->gates); a.dh_head = F(plan->dh_head);
        a.d_g = d_g; a.TT = d.TT; a.R = d.R; a.d_in = d.d_in; a.n_actions = d.A;
        if ((rec_tc_selected(d, bv) && g_rec_tc_bwd) ? launch_gru_bwd_tc(a, sms, st, g_in_step) : launch_gru_bwd(a, st, g_in_step)) return 2;        // inside a step the stream predecessor is k_mix_td
        MAL_LAUNCH_CHECK("k_gru_bwd");
    }
    // ---- side stream 2 (after the recurrence): W_ih / W_hh gradients, beside  d x = (d gi . W_ih) * (x > 0)  + fc1 grads
    if (fork_to(st, s2, ss->fork_ev[2])) return 2;
    const bool fused_gru_red = g_use_tc && g_reduce_tc && g_reduce_mn >= 3 && (g_reduce_tc == 2 || pl.rpc_a >= 256);
    if (!frozen && !dqn && fused_gru_red) {
        // W_ih, W_hh, b_ih, b_hh gradients: one [x | h_{t-1}]^T . d_g split-M GEMM per row chunk
        ReduceGruArgs ra;
        ra.x = F(plan->x_on); ra.hout = F(plan->h_on); ra.d_g = d_g;
        ra.wih_w = parts + pl.wih_w; ra.wih_b = parts + pl.wih_b;
        ra.whha_w = parts + pl.whha_w; ra.whha_b = parts + pl.whha_b;
        ra.whhb_w = parts + pl.whhb_w; ra.whhb_b = parts + pl.whhb_b;
        ra.M1 = d.M1; ra.rows_per_chunk = pl.rpc_a; ra.n_chunks = pl.nc_a; ra.R = d.R;
        static size_t attr[MAL_MAX_DEV];
        if (int rc = ensure_dyn_smem(k_reduce_gru, RG_SMEM_BYTES, attr)) return rc;
        ++g_stat_reduce_tc;
        { ProfScope _ps("k_reduce_gru", s2); launch_k(k_reduce_gru, dim3(pl.nc_a), dim3(RT3_THREADS), RG_SMEM_BYTES, s2, false, ra); }
        MAL_LAUNCH_CHECK("k_reduce_gru");
    }
    if (!frozen && !dqn && !fused_gru_red) {
        RedGroup r; r.n = 3; r.bv = bv;
        r.p[0] = red(d.M1, HID, G3, d_g, 4 * HID, A_DENSE, 0, F(plan->x_on), HID, parts + pl.wih_w, parts + pl.wih_b, pl.nc_a, pl.rpc_a);
        // W_hh: rows pair with h_{t-1} = hout shifted by R rows (zero for t == 0)
        r.p[1] = red(d.M1, HID, 128, d_g, 4 * HID, A_DENSE, d.R, F(plan->h_on), HID, parts + pl.whha_w, parts + pl.whha_b, pl.nc_a, pl.rpc_a);
        r.p[2] = red(d.M1, HID, 64, d_g + 3 * HID, 4 * HID, A_DENSE, d.R, F(plan->h_on), HID, parts + pl.whhb_w, parts + pl.whhb_b, pl.nc_a, pl.rpc_a);
        if (int rc = launch_reduce(r, s2, "k_reduce_group:agent")) return rc;
    }
    if (!frozen && dqn) {
        // feed-forward agent: d x (masked by relu' in k_mix_td) is the head seed of the rows t < T; fc1 gradients from it
        RedGroup r; r.n = 1; r.bv = bv;
        r.p[0] = red((int64_t)d.T * d.R, d.d_in, HID, F(plan->dh_head), HID, A_AGENT_IN, 0, nullptr, 0, parts + pl.fc1_w, parts + pl.fc1_b, pl.nc_f1, pl.rpc_f1);
        if (int rc = launch_reduce(r, st, "k_reduce_group:agent")) return rc;
    }
    if (!frozen && !dqn) {
        LinGroup g; g.n = 1; g.bv = bv;
        g.p[0] = lin(d.M1, G3, HID, A_DENSE, 0, d_g, 4 * HID, F(plan->w_t), G3, 0, nullptr, EPI_MASKPOS, F(plan->x_on), HID, d_x, HID);   // W_ih^T from the forward call
        g_next_pdl = true;                       // stream predecessor: k_gru_bwd7 (W_ih staging flies under its last timesteps)
        int rc = launch_linear(g, d.M1, G3, st, "k_linear_group:dx");
        g_next_pdl = false;
        if (rc) return rc;
        // inputs wider than one 128-column tile (20v20: d_in = 214): one CTA per row chunk over the full width instead of one
        // k_reduce_tc3 CTA per 128-column tile (4.02 -> 2.53 ms at 20v20 / B = 1024); a single tile (10v10) is a wash (144 vs 138 us)
        const bool fused_fc1 = g_use_tc && g_reduce_tc && g_reduce_mn >= 3 && g_fc1_fused && d.d_in <= 256 && d.M1 < 2147483647LL &&
                               (g_reduce_tc == 2 || (pl.rpc_f1 >= 256 && d.d_in > 128));
        if (fused_fc1) {
            ReduceFc1Args fa;
            fa.d_x = d_x; fa.partW = parts + pl.fc1_w; fa.partB = parts + pl.fc1_b;
            fa.M = d.M1; fa.rows_per_chunk = pl.rpc_f1; fa.n_chunks = pl.nc_f1; fa.d_in = d.d_in; fa.bv = bv;
            static size_t attr[MAL_MAX_DEV];
            if (int rc2 = ensure_dyn_smem(k_reduce_fc1, RF_SMEM_BYTES, attr)) return rc2;
            ++g_stat_reduce_fc1;
            { ProfScope _ps("k_reduce_tc:agent_fc1", st); launch_k(k_reduce_fc1, dim3(pl.nc_f1), dim3(RT3_THREADS), RF_SMEM_BYTES, st, g_use_tc != 0, fa); }   // stream predecessor: the dx GEMM
            MAL_LAUNCH_CHECK("k_reduce_fc1");
        } else {
            RedGroup r; r.n = 1; r.bv = bv;
            r.p[0] = red(d.M1, d.d_in, HID, d_x, HID, A_AGENT_IN, 0, nullptr, 0, parts + pl.fc1_w, parts + pl.fc1_b, pl.nc_f1, pl.rpc_f1);
            g_next_pdl = g_use_tc != 0;              // stream predecessor: the dx GEMM (the tcgen05 kernels trigger at their last tile)
            rc = launch_reduce(r, st, "k_reduce_group:agent");
            g_next_pdl = false;
            if (rc) return rc;
        }
    }
    if (join_from(st, s1, ss->join_ev[0])) return 2;
    if (join_from(st, s2, ss->join_ev[1])) return 2;
    // ---- gather partials into the flat gradient (state_dict order) + sum of squares
    {
        GradReduceArgs a;
        memset(&a, 0, sizeof(a));
        int n = 0;
        auto seg = [&](int64_t off, int64_t count, const float *part, int n_chunks, int64_t stride) {
            a.s[n].grad_off = off; a.s[n].count = (int)count; a.s[n].part = part; a.s[n].n_chunks = n_chunks;
            a.s[n].chunk_stride = stride; ++n;
        };
        seg(AL.fc1_w, (int64_t)HID * d.d_in, parts + pl.fc1_w, pl.nc_f1, (int64_t)HID * d.d_in);
        seg(AL.fc1_b, HID, parts + pl.fc1_b, pl.nc_f1, HID);
        if (!dqn) {
            seg(AL.w_ih, (int64_t)G3 * HID, parts + pl.wih_w, pl.nc_a, (int64_t)G3 * HID);
            seg(AL.w_hh, 128 * HID, parts + pl.whha_w, pl.nc_a, 128 * HID);
            seg(AL.w_hh + 128 * HID, 64 * HID, parts + pl.whhb_w, pl.nc_a, 64 * HID);
            seg(AL.b_ih, G3, parts + pl.wih_b, pl.nc_a, G3);
            seg(AL.b_hh, 128, parts + pl.whha_b, pl.nc_a, 128);
            seg(AL.b_hh + 128, 64, parts + pl.whhb_b, pl.nc_a, 64);
        }
        seg(AL.fc2_w, (int64_t)d.A * HID, parts + pl.fc2_w, pl.nc_f2, (int64_t)d.A * HID);
        seg(AL.fc2_b, d.A, parts + pl.fc2_b, pl.nc_f2, d.A);
        const int64_t o = AL.total;
        if (mixer_has_hypernet(d.mixer)) {
            const int K2 = d.two ? d.HE : d.S;
            const int64_t l1w = (int64_t)d.ld1 * d.S;
            const int b1row = d.two ? 2 * d.HE : 0;
            if (d.two) {
                seg(o + ML.w1a_w, (int64_t)d.HE * d.S, parts + pl.m_l1_w, pl.nc_m1, l1w);
                seg(o + ML.w1a_b, d.HE, parts + pl.m_l1_b, pl.nc_m1, d.ld1);
            }
            seg(o + ML.w1b_w, (int64_t)d.E * d.N * K2, parts + pl.m_l2a_w, pl.nc_m2, (int64_t)d.E * d.N * K2);
            seg(o + ML.w1b_b, d.E * d.N, parts + pl.m_l2a_b, pl.nc_m2, d.E * d.N);
            if (d.two) {
                seg(o + ML.wfa_w, (int64_t)d.HE * d.S, parts + pl.m_l1_w + (int64_t)d.HE * d.S, pl.nc_m1, l1w);
                seg(o + ML.wfa_b, d.HE, parts + pl.m_l1_b + d.HE, pl.nc_m1, d.ld1);
            }
            seg(o + ML.wfb_w, (int64_t)d.E * K2, parts + pl.m_l2b_w, pl.nc_m2, (int64_t)d.E * K2);
            seg(o + ML.wfb_b, d.E, parts + pl.m_l2b_b, pl.nc_m2, d.E);
            seg(o + ML.b1_w, (int64_t)d.E * d.S, parts + pl.m_l1_w + (int64_t)b1row * d.S, pl.nc_m1, l1w);
            seg(o + ML.b1_b, d.E, parts + pl.m_l1_b + b1row, pl.nc_m1, d.ld1);
            seg(o + ML.v0_w, (int64_t)d.E * d.S, parts + pl.m_l1_w + (int64_t)(b1row + d.E) * d.S, pl.nc_m1, l1w);
            seg(o + ML.v0_b, d.E, parts + pl.m_l1_b + b1row + d.E, pl.nc_m1, d.ld1);
            seg(o + ML.v2_w, d.E, parts + pl.mix_v2_sum, 1, d.E + 1);
            seg(o + ML.v2_b, 1, parts + pl.mix_v2_sum + d.E, 1, d.E + 1);
        }
        a.n = n;
        a.total = AL.total + ML.total;
        a.grad = grad;
        a.norm_part = parts + pl.norm;
        a.scalars = F(plan->scalars);
        a.unnormalized = cfg->unnormalized ? 1 : 0;
        a.n_frozen = frozen ? AL.total : 0;
        { ProfScope _ps("k_grad_reduce", st); launch_k(k_grad_reduce, dim3(pl.nblk_norm), dim3(256), 0, st, true, a); }   // stream predecessor: the fc1 reduction
        MAL_LAUNCH_CHECK("k_grad_reduce");
    }
    return 0;
}

// ---------------------------------------------------------------------------------------------
// autograd backward of the stand-alone module calls (one agent step, one QMixer.forward)
// ---------------------------------------------------------------------------------------------
// Chunk counts of the row reductions are a fixed function of the shapes (planned for a 148-SM B200), so that the workspace
// size queries need no device and a gradient does not depend on the GPU it was computed on.
#define MAL_BWD_SMS 148

struct AgentBwdPlan {
    AgentInput in;
    int dense, ldi, nc;
    int64_t rpc;
    int64_t xin, x1, hp, hn, dq, d_g, d_x;                                            // bytes
    int64_t fc1_w, fc1_b, wih_w, wih_b, whha_w, whha_b, whhb_w, whhb_b, fc2_w, fc2_b, norm;   // floats inside `parts`
    int64_t parts, total;                                                             // bytes
};

static int agent_bwd_plan(int32_t kind, int32_t rows, int32_t N, int32_t OBS, int32_t A, int32_t dense_input, AgentBwdPlan *p) {
    MAL_REQUIRE(kind == MAL_AGENT_RNN || kind == MAL_AGENT_DQN, "agent kind %d not recognised", kind);
    MAL_REQUIRE(rows > 0 && N >= 1 && OBS >= 1, "mal_agent_step_backward: bad dims");
    MAL_REQUIRE(A >= 1 && A <= MAL_MAX_ACTIONS, "n_actions must be in [1, %d]", MAL_MAX_ACTIONS);
    MAL_REQUIRE((dense_input & ~7) == 0 && !((dense_input & 1) && (dense_input >> 1)),
                "dense_input %d: bit 0 (dense) or the agent-input bits 1..2, nothing else", dense_input);
    memset(p, 0, sizeof(*p));
    p->dense = dense_input & 1;
    if (p->dense) { p->in.obs = p->in.d_in = OBS; p->in.last = p->in.id = 0; }
    else p->in = agent_input(OBS, A, N, dense_input >> 1);
    MAL_REQUIRE(agent_bwd_smem(p->in.d_in) <= 200 * 1024, "mal_agent_step_backward: input width %d too large", p->in.d_in);
    const bool rnn = kind == MAL_AGENT_RNN;
    const int d_in = p->in.d_in;
    p->ldi = (int)align_up64(d_in, 4);
    int64_t o = 0;
    auto take = [&](int64_t n_floats) { int64_t r = o; o += align_up64(n_floats * 4, 256); return r; };
    p->xin = take(p->dense ? 0 : (int64_t)rows * p->ldi);
    p->x1 = take((int64_t)rows * HID);
    p->hp = take(rnn ? (int64_t)rows * HID : 0);
    p->hn = take(rnn ? (int64_t)rows * HID : 0);
    p->dq = take((int64_t)rows * A);
    p->d_g = take(rnn ? (int64_t)rows * 4 * HID : 0);
    p->d_x = take((int64_t)rows * HID);
    int tiles = tiles_of(HID, d_in) + tiles_of(A, HID);
    if (rnn) tiles += tiles_of(G3, HID) + tiles_of(128, HID) + tiles_of(64, HID);
    chunking(rows, tiles, MAL_BWD_SMS, &p->nc, &p->rpc);
    int64_t q = 0;
    auto part = [&](int64_t n) { int64_t r = q; q += align_up64(n, 64); return r; };
    p->fc1_w = part((int64_t)p->nc * HID * d_in); p->fc1_b = part((int64_t)p->nc * HID);
    if (rnn) {
        p->wih_w = part((int64_t)p->nc * G3 * HID);   p->wih_b = part((int64_t)p->nc * G3);
        p->whha_w = part((int64_t)p->nc * 128 * HID); p->whha_b = part((int64_t)p->nc * 128);
        p->whhb_w = part((int64_t)p->nc * 64 * HID);  p->whhb_b = part((int64_t)p->nc * 64);
    }
    p->fc2_w = part((int64_t)p->nc * A * HID); p->fc2_b = part((int64_t)p->nc * A);
    p->norm = part(ceil_div64(agent_layout(d_in, A, kind).total, GRED_EPB));
    p->parts = take(q);
    p->total = o;
    return 0;
}

extern "C" int64_t mal_agent_step_backward_workspace(int32_t agent_kind, int32_t rows, int32_t n_agents, int32_t obs_dim,
                                                     int32_t n_actions, int32_t dense_input) {
    AgentBwdPlan p;
    if (agent_bwd_plan(agent_kind, rows, n_agents, obs_dim, n_actions, dense_input, &p)) return -1;
    return p.total;
}

extern "C" int mal_agent_step_backward(int32_t agent_kind, const float *agent, int32_t rows, int32_t n_agents, int32_t obs_dim,
                                       int32_t n_actions, int32_t dense_input, const float *obs, int64_t obs_sb,
                                       const float *last_onehot, int64_t onehot_sb, const float *h_in, const float *d_q,
                                       const float *d_h_out, float *d_h_in, float *d_agent, void *workspace, void *stream) {
    AgentBwdPlan p;
    if (int rc = agent_bwd_plan(agent_kind, rows, n_agents, obs_dim, n_actions, dense_input, &p)) return rc;
    MAL_REQUIRE(agent && obs && workspace, "mal_agent_step_backward: agent, obs and workspace are required");
    const bool rnn = agent_kind == MAL_AGENT_RNN;
    MAL_REQUIRE(rnn || (!h_in && !d_h_out && !d_h_in), "mal_agent_step_backward: the feed-forward agent has no hidden state");
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t *ws = (uint8_t *)workspace;
    auto F = [&](int64_t off) { return reinterpret_cast<float *>(ws + off); };
    AgentBwdArgs a;
    memset(&a, 0, sizeof(a));
    a.params = agent; a.kind = agent_kind; a.rows = rows; a.N = n_agents; a.OBS = obs_dim; a.A = n_actions; a.dense = p.dense;
    a.in = p.in; a.obs = obs; a.obs_sb = obs_sb; a.onehot = p.in.last > 0 ? last_onehot : nullptr; a.onehot_sb = onehot_sb;
    a.h_in = h_in; a.d_q = d_q; a.d_h_out = d_h_out;
    a.xin = p.dense ? nullptr : F(p.xin); a.ldi = p.ldi;
    a.x1 = F(p.x1); a.hp = rnn ? F(p.hp) : nullptr; a.hn = rnn ? F(p.hn) : nullptr; a.dq = F(p.dq);
    a.d_g = rnn ? F(p.d_g) : nullptr; a.d_x = F(p.d_x); a.d_h_in = d_h_in;
    const size_t smem = agent_bwd_smem(p.in.d_in);
    static size_t attr[MAL_MAX_DEV];
    if (smem > 48 * 1024) if (int rc = ensure_dyn_smem(k_agent_step_bwd, smem, attr)) return rc;
    { ProfScope _ps("k_agent_step_bwd", st); k_agent_step_bwd<<<(unsigned)ceil_div64(rows, ABR_ROWS), ABR_THREADS, smem, st>>>(a); }
    MAL_LAUNCH_CHECK("k_agent_step_bwd");
    if (!d_agent) return 0;                      // frozen agent: only d h_in

    // weight gradients: row reductions of the learner (one launch, dense loaders), then the fixed-order gather
    const int d_in = p.in.d_in;
    const AgentLayout AL = agent_layout(d_in, n_actions, agent_kind);
    float *parts = F(p.parts);
    const float *xin = p.dense ? obs : F(p.xin);
    const int64_t ldx = p.dense ? obs_sb : p.ldi;
    const float *hp = h_in ? h_in : F(p.hp);
    BatchView bv;
    memset(&bv, 0, sizeof(bv));
    RedGroup r; r.n = 0; r.bv = bv;
    r.p[r.n++] = red(rows, d_in, HID, F(p.d_x), HID, A_DENSE, 0, xin, ldx, parts + p.fc1_w, parts + p.fc1_b, p.nc, p.rpc);
    if (rnn) {
        const float *dg = F(p.d_g);
        r.p[r.n++] = red(rows, HID, G3, dg, 4 * HID, A_DENSE, 0, F(p.x1), HID, parts + p.wih_w, parts + p.wih_b, p.nc, p.rpc);
        r.p[r.n++] = red(rows, HID, 128, dg, 4 * HID, A_DENSE, 0, hp, HID, parts + p.whha_w, parts + p.whha_b, p.nc, p.rpc);
        r.p[r.n++] = red(rows, HID, 64, dg + 3 * HID, 4 * HID, A_DENSE, 0, hp, HID, parts + p.whhb_w, parts + p.whhb_b, p.nc, p.rpc);
    }
    r.p[r.n++] = red(rows, HID, n_actions, F(p.dq), n_actions, A_DENSE, 0, rnn ? F(p.hn) : F(p.x1), HID, parts + p.fc2_w,
                     parts + p.fc2_b, p.nc, p.rpc);
    if (int rc = launch_reduce(r, st, "k_reduce_group:agent_step_bwd")) return rc;
    GradReduceArgs g;
    memset(&g, 0, sizeof(g));
    int n = 0;
    auto seg = [&](int64_t off, int64_t count, const float *part, int64_t stride) {
        g.s[n].grad_off = off; g.s[n].count = (int)count; g.s[n].part = part; g.s[n].n_chunks = p.nc; g.s[n].chunk_stride = stride; ++n;
    };
    seg(AL.fc1_w, (int64_t)HID * d_in, parts + p.fc1_w, (int64_t)HID * d_in);
    seg(AL.fc1_b, HID, parts + p.fc1_b, HID);
    if (rnn) {
        seg(AL.w_ih, (int64_t)G3 * HID, parts + p.wih_w, (int64_t)G3 * HID);
        seg(AL.w_hh, 128 * HID, parts + p.whha_w, 128 * HID);
        seg(AL.w_hh + 128 * HID, 64 * HID, parts + p.whhb_w, 64 * HID);
        seg(AL.b_ih, G3, parts + p.wih_b, G3);
        seg(AL.b_hh, 128, parts + p.whha_b, 128);
        seg(AL.b_hh + 128, 64, parts + p.whhb_b, 64);
    }
    seg(AL.fc2_w, (int64_t)n_actions * HID, parts + p.fc2_w, (int64_t)n_actions * HID);
    seg(AL.fc2_b, n_actions, parts + p.fc2_b, n_actions);
    g.n = n; g.total = AL.total; g.grad = d_agent; g.norm_part = parts + p.norm; g.scalars = nullptr; g.unnormalized = 1;
    { ProfScope _ps("k_grad_reduce", st); launch_k(k_grad_reduce, dim3((unsigned)ceil_div64(AL.total, GRED_EPB)), dim3(256), 0, st, false, g); }
    MAL_LAUNCH_CHECK("k_grad_reduce");
    return 0;
}

struct MixerBwdPlan {
    int two, ld1, ld2, nblk, nc_m2, nc_m1;
    int64_t rpc_m2, rpc_m1;
    int64_t d_a2, d_y1, parts, total;                                         // bytes
    int64_t l2a_w, l2a_b, l2b_w, l2b_b, l1_w, l1_b, v2, norm;                 // floats inside `parts`
};

static int mixer_bwd_plan(int32_t mixer, int32_t B, int32_t T, int32_t N, int32_t S, int32_t E, int32_t HE, MixerBwdPlan *p) {
    MAL_REQUIRE(mixer_has_hypernet(mixer), "mal_mixer_backward: mixer %d has no kernel backward (VDN: d q_tot broadcast over agents)", mixer);
    MAL_REQUIRE(B > 0 && T > 0 && N > 0 && N <= MAL_MAX_ACTIONS && S > 0, "mal_mixer_backward: bad dims");
    MAL_REQUIRE(E >= 1 && E <= MAL_MAX_EMBED, "mixing_embed_dim must be in [1, %d]", MAL_MAX_EMBED);
    MAL_REQUIRE(mixer != MAL_MIXER_QMIX2 || HE >= 1, "hypernet_embed must be >= 1");
    memset(p, 0, sizeof(*p));
    const int64_t BT = (int64_t)B * T;
    p->two = mixer == MAL_MIXER_QMIX2;
    p->ld1 = p->two ? 2 * HE + 2 * E : 2 * E;
    p->ld2 = E * N + E;
    const int K2 = p->two ? HE : S;
    if (p->two) {   // the learner's chunking (part_layout)
        chunking(BT, tiles_of(E * N, K2) + tiles_of(E, K2), MAL_BWD_SMS, &p->nc_m2, &p->rpc_m2);
        chunking(BT, tiles_of(p->ld1, S), MAL_BWD_SMS, &p->nc_m1, &p->rpc_m1);
    } else {
        chunking(BT, tiles_of(E * N, K2) + tiles_of(E, K2) + tiles_of(p->ld1, S), MAL_BWD_SMS, &p->nc_m2, &p->rpc_m2);
        p->nc_m1 = p->nc_m2; p->rpc_m1 = p->rpc_m2;
    }
    int64_t nb = ceil_div64(BT, 8); if (nb > MAL_BWD_SMS * 4) nb = MAL_BWD_SMS * 4;
    p->nblk = (int)nb;
    int64_t o = 0;
    auto take = [&](int64_t n_floats) { int64_t r = o; o += align_up64(n_floats * 4, 256); return r; };
    p->d_a2 = take(BT * p->ld2);
    p->d_y1 = take(BT * p->ld1);
    int64_t q = 0;
    auto part = [&](int64_t n) { int64_t r = q; q += align_up64(n, 64); return r; };
    p->l2a_w = part((int64_t)p->nc_m2 * E * N * K2); p->l2a_b = part((int64_t)p->nc_m2 * E * N);
    p->l2b_w = part((int64_t)p->nc_m2 * E * K2);     p->l2b_b = part((int64_t)p->nc_m2 * E);
    p->l1_w = part((int64_t)p->nc_m1 * p->ld1 * S);  p->l1_b = part((int64_t)p->nc_m1 * p->ld1);
    p->v2 = part((int64_t)p->nblk * (E + 1));
    p->norm = part(ceil_div64(mixer_layout(mixer, S, N, E, HE).total, GRED_EPB));
    p->parts = take(q);
    p->total = o;
    return 0;
}

extern "C" int64_t mal_mixer_backward_workspace(int32_t mixer, int32_t B, int32_t T, int32_t N, int32_t S, int32_t E, int32_t HE) {
    MixerBwdPlan p;
    if (mixer_bwd_plan(mixer, B, T, N, S, E, HE, &p)) return -1;
    return p.total;
}

extern "C" int mal_mixer_backward(int32_t mixer, int32_t B, int32_t T, int32_t N, int32_t S, int32_t E, int32_t HE,
                                  const float *params, const float *agent_qs, const float *states, int64_t state_sb,
                                  int64_t state_st, const float *scratch, const float *d_q_tot, float *d_agent_qs,
                                  float *d_params, void *workspace, void *stream) {
    MixerBwdPlan p;
    if (int rc = mixer_bwd_plan(mixer, B, T, N, S, E, HE, &p)) return rc;
    MAL_REQUIRE(params && agent_qs && states && scratch && d_q_tot && d_agent_qs && d_params && workspace,
                "mal_mixer_backward: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t *ws = (uint8_t *)workspace;
    auto F = [&](int64_t off) { return reinterpret_cast<float *>(ws + off); };
    const int64_t BT = (int64_t)B * T;
    const MixerLayout ML = mixer_layout(mixer, S, N, E, HE);
    const float *y1 = scratch, *a2 = scratch + BT * p.ld1;      // mal_mixer_forward's scratch layout
    float *d_a2 = F(p.d_a2), *d_y1 = F(p.d_y1), *parts = F(p.parts);
    MixBwdArgs m;
    m.mixer = mixer; m.B = B; m.T = T; m.N = N; m.E = E; m.HE = HE; m.S = S;
    m.params = params; m.agent_qs = agent_qs; m.y1 = y1; m.a2 = a2; m.d_q_tot = d_q_tot;
    m.d_agent_qs = d_agent_qs; m.d_a2 = d_a2; m.d_y1 = d_y1; m.part_v2 = parts + p.v2;
    { ProfScope _ps("k_mix_bwd", st); k_mix_bwd<<<p.nblk, 256, 0, st>>>(m); }
    MAL_LAUNCH_CHECK("k_mix_bwd");
    BatchView bv;
    memset(&bv, 0, sizeof(bv));
    bv.B = B; bv.T = T; bv.TT = T; bv.N = N; bv.S = S; bv.R = B * N;
    bv.state.ptr = states; bv.state.sb = state_sb; bv.state.st = state_st;
    HyperBwd h;
    h.mixer = mixer; h.two = p.two; h.N = N; h.E = E; h.HE = HE; h.S = S; h.ld1 = p.ld1; h.ld2 = p.ld2; h.BT = BT;
    h.d_a2 = d_a2; h.d_y1 = d_y1; h.y1 = y1;
    h.wt1 = params + ML.w1b_w; h.wtf = params + ML.wfb_w; h.ldw1 = HE; h.ldwf = HE; h.w_trans = 1;   // W(n,k) = W_2[k, n]
    h.l2a_w = parts + p.l2a_w; h.l2a_b = parts + p.l2a_b; h.l2b_w = parts + p.l2b_w; h.l2b_b = parts + p.l2b_b;
    h.l1_w = parts + p.l1_w; h.l1_b = parts + p.l1_b;
    h.nc_m2 = p.nc_m2; h.rpc_m2 = p.rpc_m2; h.nc_m1 = p.nc_m1; h.rpc_m1 = p.rpc_m1;
    if (int rc = launch_hyper_bwd(h, bv, st)) return rc;
    GradReduceArgs g;
    memset(&g, 0, sizeof(g));
    int n = 0;
    auto seg = [&](int64_t off, int64_t count, const float *part, int n_chunks, int64_t stride) {
        g.s[n].grad_off = off; g.s[n].count = (int)count; g.s[n].part = part; g.s[n].n_chunks = n_chunks; g.s[n].chunk_stride = stride; ++n;
    };
    const int K2 = p.two ? HE : S;
    const int64_t l1w = (int64_t)p.ld1 * S;
    const int b1row = p.two ? 2 * HE : 0;
    const float *pl1w = parts + p.l1_w, *pl1b = parts + p.l1_b;
    if (p.two) {
        seg(ML.w1a_w, (int64_t)HE * S, pl1w, p.nc_m1, l1w);
        seg(ML.w1a_b, HE, pl1b, p.nc_m1, p.ld1);
    }
    seg(ML.w1b_w, (int64_t)E * N * K2, parts + p.l2a_w, p.nc_m2, (int64_t)E * N * K2);
    seg(ML.w1b_b, E * N, parts + p.l2a_b, p.nc_m2, E * N);
    if (p.two) {
        seg(ML.wfa_w, (int64_t)HE * S, pl1w + (int64_t)HE * S, p.nc_m1, l1w);
        seg(ML.wfa_b, HE, pl1b + HE, p.nc_m1, p.ld1);
    }
    seg(ML.wfb_w, (int64_t)E * K2, parts + p.l2b_w, p.nc_m2, (int64_t)E * K2);
    seg(ML.wfb_b, E, parts + p.l2b_b, p.nc_m2, E);
    seg(ML.b1_w, (int64_t)E * S, pl1w + (int64_t)b1row * S, p.nc_m1, l1w);
    seg(ML.b1_b, E, pl1b + b1row, p.nc_m1, p.ld1);
    seg(ML.v0_w, (int64_t)E * S, pl1w + (int64_t)(b1row + E) * S, p.nc_m1, l1w);
    seg(ML.v0_b, E, pl1b + b1row + E, p.nc_m1, p.ld1);
    seg(ML.v2_w, E, parts + p.v2, p.nblk, E + 1);
    seg(ML.v2_b, 1, parts + p.v2 + E, p.nblk, E + 1);
    g.n = n; g.total = ML.total; g.grad = d_params; g.norm_part = parts + p.norm; g.scalars = nullptr; g.unnormalized = 1;
    { ProfScope _ps("k_grad_reduce", st); launch_k(k_grad_reduce, dim3((unsigned)ceil_div64(ML.total, GRED_EPB)), dim3(256), 0, st, false, g); }
    MAL_LAUNCH_CHECK("k_grad_reduce");
    return 0;
}

static int launch_clip_rmsprop(float *agent, int64_t n_agent, float *mixer, int64_t n_mixer, float *grad,
                               float *sq, const float *norm_part, int n_part, float lr, float alpha, float eps,
                               float clip, float *scalars, const float *denominator, int64_t n_frozen, cudaStream_t st, bool pdl = false) {
    const int64_t P = n_agent + n_mixer;
    { ProfScope _ps("k_clip_rmsprop", st); launch_k(k_clip_rmsprop, dim3((unsigned)ceil_div64(P, 256)), dim3(256), 0, st, pdl, agent, n_agent, mixer, n_mixer, grad, sq, norm_part,
                                                                n_part, lr, alpha, eps, clip, scalars, denominator, n_frozen); }
    MAL_LAUNCH_CHECK("k_clip_rmsprop");
    return 0;
}

extern "C" int mal_clip_rmsprop(float *agent, int64_t n_agent, float *mixer, int64_t n_mixer, float *grad,
                                float *square_avg, float lr, float alpha, float eps, float clip, float *scalars,
                                float *scratch, const float *denominator, int64_t n_frozen, void *stream) {
    MAL_REQUIRE(agent && grad && square_avg && scalars && scratch && n_agent > 0 && n_mixer >= 0,
                "mal_clip_rmsprop: bad arguments (scratch needs ceil(P/256) floats)");
    MAL_REQUIRE(n_frozen >= 0 && n_frozen <= n_agent + n_mixer, "mal_clip_rmsprop: n_frozen out of range");
    MAL_REQUIRE(n_mixer == 0 || mixer, "mal_clip_rmsprop: mixer buffer missing");
    const int64_t P = n_agent + n_mixer;
    const int nb = (int)ceil_div64(P, 256);
    { ProfScope _ps("k_sumsq", (cudaStream_t)stream); k_sumsq<<<nb, 256, 0, (cudaStream_t)stream>>>(grad, P, scratch, denominator, n_frozen); }
    MAL_LAUNCH_CHECK("k_sumsq");
    return launch_clip_rmsprop(agent, n_agent, mixer, n_mixer, grad, square_avg, scratch, nb, lr, alpha, eps, clip,
                               scalars, denominator, n_frozen, (cudaStream_t)stream);
}

extern "C" int mal_peer_allreduce_clip_rmsprop(const void *const *peer_bufs, int32_t world, float *agent, int64_t n_agent,
                                               float *mixer, int64_t n_mixer, float *grad_out, float *tail_out, int32_t tail,
                                               float *square_avg, float lr, float alpha, float eps, float clip,
                                               float *scalars, float *scratch, int64_t n_frozen, void *stream) {
    MAL_REQUIRE(n_frozen >= 0 && n_frozen <= n_agent + n_mixer, "mal_peer_allreduce_clip_rmsprop: n_frozen out of range");
    MAL_REQUIRE(peer_bufs && world >= 1 && world <= PEER_MAX, "mal_peer_allreduce_clip_rmsprop: world size must be in [1, %d]", PEER_MAX);
    MAL_REQUIRE(agent && grad_out && tail_out && square_avg && scalars && scratch && n_agent > 0 && n_mixer >= 0 && tail >= 5 && tail <= 32,
                "mal_peer_allreduce_clip_rmsprop: bad arguments (scratch needs ceil(P/256) floats, tail >= 5)");
    PeerBufs pb;
    memset(&pb, 0, sizeof(pb));
    pb.world = world;
    for (int r = 0; r < world; ++r) {
        MAL_REQUIRE(peer_bufs[r], "mal_peer_allreduce_clip_rmsprop: null peer buffer");
        pb.p[r] = reinterpret_cast<const float *>(peer_bufs[r]);
    }
    const int64_t P = n_agent + n_mixer;
    const int nb = (int)ceil_div64(P, 256);
    cudaStream_t st = (cudaStream_t)stream;
    { ProfScope _ps("k_peer_allreduce_grad", st); k_peer_allreduce_grad<<<nb, 256, 0, st>>>(pb, P, tail, grad_out, tail_out, scratch, n_frozen); }
    MAL_LAUNCH_CHECK("k_peer_allreduce_grad");
    return launch_clip_rmsprop(agent, n_agent, mixer, n_mixer, grad_out, square_avg, scratch, nb, lr, alpha, eps, clip,
                               scalars, nullptr, n_frozen, st);
}

extern "C" int mal_learner_step(const mal_batch_t *batch, const mal_learner_cfg_t *cfg, const mal_plan_t *plan,
                                float *agent, const float *target_agent, float *mixer, const float *target_mixer,
                                void *workspace, float *grad, float *square_avg, void *stream) {
    MAL_REQUIRE(square_avg, "mal_learner_step: square_avg missing");
    MAL_REQUIRE(!cfg || !cfg->unnormalized, "mal_learner_step: unnormalized (data-parallel) mode needs the split calls");
    g_defer_stats = true;
    const int rc_f = mal_learner_forward(batch, cfg, plan, agent, target_agent, mixer, target_mixer, workspace, stream);
    g_defer_stats = false;
    if (rc_f) return rc_f;
    g_in_step = true;
    const int rc_b = mal_learner_backward(batch, cfg, plan, agent, mixer, workspace, grad, stream);
    g_in_step = false;
    if (rc_b) return rc_b;
    Dims d;
    if (int rc = get_dims(batch, cfg, &d)) return rc;
    int sms, tps;
    if (device_sm_count(&sms, &tps)) return 2;
    const PartLayout pl = part_layout(d, sms);
    uint8_t *ws = (uint8_t *)workspace;
    float *parts = reinterpret_cast<float *>(ws + plan->partials);
    float *scalars = reinterpret_cast<float *>(ws + plan->scalars);
    return launch_clip_rmsprop(agent, plan->n_agent_params, mixer, plan->n_mixer_params, grad, square_avg,
                               parts + pl.norm, pl.nblk_norm, cfg->lr, cfg->alpha, cfg->eps, cfg->clip, scalars,
                               nullptr, cfg->freeze_agent ? plan->n_agent_params : 0, (cudaStream_t)stream, true);   // stream predecessor: k_grad_reduce
}

extern "C" int mal_copy_f32(float *dst, const float *src, int64_t n, void *stream) {
    if (n <= 0) return 0;
    MAL_REQUIRE(dst && src, "mal_copy_f32: null buffer");
    int64_t grid = ceil_div64(n, 1024); if (grid > 1184) grid = 1184; if (grid < 1) grid = 1;
    { ProfScope _ps("k_copy_f32", (cudaStream_t)stream); k_copy_f32<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(dst, src, n); }
    MAL_LAUNCH_CHECK("k_copy_f32");
    return 0;
}

// ---------------------------------------------------------------------------------------------
// prioritized episode replay
// ---------------------------------------------------------------------------------------------
static bool finite_nonneg(float v) { return v >= 0.0f && v <= 3.402823466e38f; }   // false for NaN and +inf too

extern "C" int mal_per_sample_check(int64_t n, int32_t B, float beta) {
    MAL_REQUIRE(n >= 1, "mal_per_sample: the buffer holds no episode (n = %lld)", (long long)n);
    MAL_REQUIRE(B >= 1, "mal_per_sample: batch size %d must be >= 1", B);
    MAL_REQUIRE(finite_nonneg(beta), "mal_per_sample: beta must be finite and >= 0");
    return 0;
}

extern "C" int mal_per_sample(const float *priorities, int64_t n, int32_t B, float beta, const float *u, uint64_t seed,
                              uint64_t offset, int64_t *ids, float *weights, uint64_t *advance, void *stream) {
    if (int rc = mal_per_sample_check(n, B, beta)) return rc;
    MAL_REQUIRE(priorities && ids && weights, "mal_per_sample: null argument");
    MAL_REQUIRE((reinterpret_cast<uintptr_t>(priorities) & 15) == 0, "mal_per_sample: priorities must be 16-byte aligned");
    PerSampleArgs a;
    a.p = priorities; a.n = n; a.per = align_up64(ceil_div64(n, PER_THREADS), 4); a.B = B; a.beta = beta;
    a.u = u; a.seed = seed; a.offset = offset; a.ids = ids; a.w = weights; a.grid = 1;
    if (!u) {                                    // th.rand(B)'s grid and generator advance on this device
        int sms, tps;
        if (device_sm_count(&sms, &tps)) return 2;
        const uint64_t cap = (uint64_t)sms * (uint64_t)(tps / 256);
        uint64_t g = ((uint64_t)B + 255) / 256; if (g > cap) g = cap;
        a.grid = (uint32_t)g;
        if (advance) *advance = (((uint64_t)B - 1) / (256 * g * 4) + 1) * 4;
    } else if (advance) {
        *advance = 0;
    }
    { ProfScope _ps("k_per_sample", (cudaStream_t)stream); k_per_sample<<<1, PER_THREADS, 0, (cudaStream_t)stream>>>(a); }
    MAL_LAUNCH_CHECK("k_per_sample");
    return 0;
}

extern "C" int mal_per_update_check(int32_t B, int32_t T, int32_t n_q, float alpha, float eps) {
    MAL_REQUIRE(B >= 1, "mal_per_update: batch size %d must be >= 1", B);
    MAL_REQUIRE(T >= 1 && n_q >= 1 && n_q <= MAL_MAX_ACTIONS, "mal_per_update: bad shape (T = %d, n_q = %d)", T, n_q);
    MAL_REQUIRE(finite_nonneg(alpha), "mal_per_update: alpha must be finite and >= 0");
    MAL_REQUIRE(finite_nonneg(eps), "mal_per_update: eps must be finite and >= 0");
    return 0;
}

extern "C" int mal_per_update(const float *td, const float *mask, int32_t B, int32_t T, int32_t n_q, const int64_t *ids,
                              float alpha, float eps, float *priorities, int64_t capacity, float *max_priority,
                              void *stream) {
    if (int rc = mal_per_update_check(B, T, n_q, alpha, eps)) return rc;
    MAL_REQUIRE(td && mask && ids && priorities && max_priority && capacity >= 1, "mal_per_update: null argument");
    PerUpdateArgs a;
    a.td = td; a.mask = mask; a.B = B; a.T = T; a.nq = n_q; a.ids = ids; a.capacity = capacity;
    a.alpha = alpha; a.eps = eps; a.priorities = priorities; a.max_priority = max_priority;
    { ProfScope _ps("k_per_update", (cudaStream_t)stream); k_per_update<<<(unsigned)ceil_div64(B, 8), 256, 0, (cudaStream_t)stream>>>(a); }
    MAL_LAUNCH_CHECK("k_per_update");
    return 0;
}
