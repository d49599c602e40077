// K9: fused single-timestep agent forward + epsilon-greedy action selection.
//
// Reference: BasicMAC.select_actions / forward / _build_inputs (marl/controllers/basic_controller.py:29-54,80-92),
// DRQNAgentNetwork.forward (marl/modules/agents/drqn_agent.py:29-35) and EpsilonGreedyActionSelector.select
// (marl/components/action_selectors.py:44-62) -- ~25 ATen launches per env step in the reference, ONE here.
//
// Layout: a CTA owns AS_ROWS (= 8) agent rows; every weight row is streamed once per CTA straight from
// L2 with lanes along k (coalesced), the 8 per-row partial dot products are folded with a 9-shuffle
// multi-value butterfly, gate math and the argmax/selection run warp-per-row.
#pragma once
#include "mal_common.cuh"

#define AS_ROWS 8
#define AS_THREADS 256
#define AS_WARPS (AS_THREADS / 32)

// ---------------------------------------------------------------------------------------------
// Philox4x32-10, counter layout identical to curand_init(seed, subsequence, offset) as used by
// ATen/native/cuda/DistributionTemplates.h (distribution_elementwise_grid_stride_kernel).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}

// The uniform in (0,1] that torch's grid-stride distribution kernel hands to element `li` of a tensor of
// `numel` elements when the generator state is (seed, offset): thread idx = li % (256*grid), the (li / (256*grid))-th
// 32-bit output of that thread's stream.
__device__ __forceinline__ float torch_philox_uniform(uint64_t seed, uint64_t offset, uint32_t grid, uint64_t li) {
    const uint64_t span = 256ull * grid;
    const uint64_t idx = li % span, q = li / span;
    const uint64_t ctr = offset / 4 + q / 4;
    uint4 c = make_uint4((uint32_t)ctr, (uint32_t)(ctr >> 32), (uint32_t)idx, (uint32_t)(idx >> 32));
    uint4 o = philox4x32_10(c, make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const uint32_t comp = (uint32_t)(q & 3);
    uint32_t x = comp == 0 ? o.x : comp == 1 ? o.y : comp == 2 ? o.z : o.w;
    return x * 2.3283064365386963e-10f + (2.3283064365386963e-10f / 2.0f);   // _curand_uniform
}
__device__ __forceinline__ float torch_uniform01(float r) { return r == 1.0f ? 0.0f : r; }   // uniform_kernel
__device__ __forceinline__ float torch_exponential1(float r) {                                 // transformation::exponential
    const float eps_half = 1.1920928955078125e-07f / 2.0f;
    float lg = (r >= 1.0f - eps_half) ? -eps_half : logf(r);
    return -1.0f * lg;
}

// Rollout-step fusion (steppers/episode_stepper.py:110-142,177-186): besides selecting actions the launch also performs
// the EpisodeBatch.update calls around select_actions -- the environment's pre-transition data of step t, the previous
// step's reward / terminated, and the selected actions + their one-hot -- straight into the episode records.
struct RolloutIO {
    int enabled;
    int S;
    const float *env_state; int64_t env_state_sb;     // [bs,S]
    const uint8_t *alive;                              // [bs] or NULL: matches that have ended select on a dummy avail row
    const float *prev_reward; const uint8_t *prev_done;   // [bs] outcome of step t-1, NULL at t = 0
    float *state_t; int64_t state_sb;                 // episode batch fields at time index t: &field[0, t], batch strides in elements
    int32_t *avail_t; int64_t avail_sb;
    float *obs_t; int64_t obs_sb;
    long long *filled_t; int64_t filled_sb;
    long long *actions_t; int64_t actions_sb;
    float *onehot_t; int64_t onehot_sb;
    float *reward_tm1; int64_t reward_sb;             // &reward[0, t-1]
    uint8_t *term_tm1; int64_t term_sb;
};

struct SelectArgs {
    const int32_t *avail;
    int64_t avail_sb;
    int32_t N;
    float epsilon;
    int32_t rng_mode;
    const float *u, *e;
    uint64_t seed, offset_u, offset_e;
    uint32_t grid_u, grid_e;
    int64_t *actions, *greedy;
    int32_t *status;
};

// The draws of one lane for row `row`: ev = Exp(1) variate of (row, lane) (1 for lane >= A), uu = the row's uniform.
__device__ __forceinline__ void select_draws(const SelectArgs &s, int row, int A, int lane, float &ev, float &uu) {
    const bool valid = lane < A;
    if (s.rng_mode == 0) {
        ev = valid ? s.e[(int64_t)row * A + lane] : 1.0f;
        uu = s.u[row];
    } else {
        ev = valid ? torch_exponential1(torch_philox_uniform(s.seed, s.offset_e, s.grid_e, (uint64_t)row * A + lane)) : 1.0f;
        uu = torch_uniform01(torch_philox_uniform(s.seed, s.offset_u, s.grid_u, (uint64_t)row));
    }
}
__device__ __forceinline__ int select_avail(const SelectArgs &s, int row, int A, int lane) {
    const int b = row / s.N, n = row - b * s.N;
    return lane < A ? s.avail[(int64_t)b * s.avail_sb + (int64_t)n * A + lane] : 0;
}

// One warp selects for one row.  qv = this lane's Q-value (lane < A), av = its avail flag, (ev, uu) its draws.  With `io`
// the avail row, the chosen action and its one-hot also go into the episode batch at time index t.
__device__ __forceinline__ void select_core(const SelectArgs &s, int row, int A, int lane, float qv, int av, float ev, float uu,
                                            const RolloutIO *io) {
    const bool valid = lane < A;
    const int b = row / s.N, n = row - b * s.N;
    if (io && valid) io->avail_t[(int64_t)b * io->avail_sb + (int64_t)n * A + lane] = av;
    if (io && io->alive && !io->alive[b]) av = (lane == 0) ? 1 : 0;       // an ended match: any valid row (its data is cleared later)
    // greedy branch: masked_q[avail == 0] = -inf ; max(dim=2)[1]
    float gv = (valid && av != 0) ? qv : -INFINITY;
    int gi = lane;
    warp_argmax(gv, gi);
    // random branch: Categorical(avail.float()).sample() == argmax(p / Exp(1))
    const float avf = (float)av;
    const float tot = warp_sum(avf);
    float rv = valid ? (avf / tot) / ev : -INFINITY;
    int ri = lane;
    warp_argmax(rv, ri);
    int act = 0;
    if (lane == 0) {
        const long long pick_random = (uu < s.epsilon) ? 1 : 0;
        act = (int)(pick_random * ri + (1 - pick_random) * gi);
        s.actions[row] = act;
        s.greedy[row] = 1 - pick_random;
        if (!(tot > 0.0f) && s.status) atomicExch(s.status, 1);
    }
    if (io) {
        act = __shfl_sync(0xffffffffu, act, 0);
        if (lane == 0) io->actions_t[(int64_t)b * io->actions_sb + n] = act;
        if (valid) io->onehot_t[(int64_t)b * io->onehot_sb + (int64_t)n * A + lane] = (lane == act) ? 1.0f : 0.0f;   // OneHot, transforms.py:16-19
    }
}
__device__ __forceinline__ void select_row(const SelectArgs &s, int row, int A, int lane, float qv, const RolloutIO *io = nullptr) {
    float ev, uu;
    select_draws(s, row, A, lane, ev, uu);
    select_core(s, row, A, lane, qv, select_avail(s, row, A, lane), ev, uu, io);
}

// ---------------------------------------------------------------------------------------------
// Per-match policies (league rollouts / cross-play): one launch steps B matches that each play their own entry of a
// [K, table_ld] table of flat agent buffers.  k_policy_schedule buckets the matches by policy once per assignment and
// writes a work list; CTA c of a pooled step kernel (template parameter POOL) then runs entry c: the policy whose
// parameters it reads and up to AS_ROWS agent rows of matches that play it.  Every row keeps its ORIGINAL index for
// inputs, hidden state, outputs, avail rows and Philox draws, so a pooled step computes for each match exactly what the
// plain step computes over the whole batch with that match's parameters.
//
// Schedule buffer (int32, internal to the library; mal_policy_schedule_bytes sizes it):
//   header [PS_HDR]:      used CTAs, rows (bs * N), n_agents, n_policies, 0...
//   entries [PS_ENT] each: row[0..7] (-1: padding, always at the end), policy, 0...
// ---------------------------------------------------------------------------------------------
#define PS_HDR 16
#define PS_ENT 16
#define PS_THREADS 1024
static_assert(MAL_MAX_POLICIES <= PS_THREADS, "k_policy_schedule scans one policy per thread");

// the row of local slot r of this CTA: r0 + r, or the work list's entry (padding and anything outside [0, rows) -> rows,
// which every `row < rows` test of the step kernels skips)
template <bool POOL>
__device__ __forceinline__ int cta_row(int r0, const int32_t *rl, int r, int rows) {
    if constexpr (POOL) {
        const int v = __ldg(rl + r);
        return (v >= 0 && v < rows) ? v : rows;
    } else {
        return r0 + r;
    }
}
// two consecutive parameters: one 8-byte load in the plain kernels (flat_params() is 16-byte aligned); a pooled table row
// starts at policy * table_ld floats, which need not be even
template <bool POOL>
__device__ __forceinline__ float2 ldg_f2(const float2 *p) {
    if constexpr (POOL) {
        const float *f = reinterpret_cast<const float *>(p);
        return make_float2(__ldg(f), __ldg(f + 1));
    } else {
        return __ldg(p);
    }
}
// Pooled CTA set-up: false when the CTA has nothing to do (past the used count, a schedule built for another shape, or a
// policy outside the table), else P = this CTA's table row and rl = its row list.  Called before any barrier.
__device__ __forceinline__ bool pool_cta(const float *&P, const int32_t *&rl, const float *table, int64_t table_ld,
                                         int n_policies, const int32_t *sched, int rows, int N) {
    const int4 h = __ldg(reinterpret_cast<const int4 *>(sched));
    if ((int)blockIdx.x >= h.x || h.y != rows || h.z != N || h.w != n_policies) return false;
    rl = sched + PS_HDR + (int64_t)blockIdx.x * PS_ENT;
    const int p = __ldg(rl + AS_ROWS);
    if (p < 0 || p >= n_policies) return false;
    P = table + (int64_t)p * table_ld;
    return true;
}

// One CTA: match_policy[bs] -> work list.  A stable counting sort by policy: bucket p's rows are those of its matches in
// match order (each match's N rows consecutive), cut into CTAs of AS_ROWS.  sum over p of ceil(rows_p / 8) is at most
// ceil(rows / 8) + min(K, bs) - 1, the grid the pooled launch uses.  An id outside [0, K) sets *status and its match's
// rows are left out of the list.
__global__ void __launch_bounds__(PS_THREADS) k_policy_schedule(const int32_t *mp, int bs, int N, int K, int32_t *sched,
                                                                 int32_t *status) {
    __shared__ int cnt[MAL_MAX_POLICIES], end[MAL_MAX_POLICIES], run[MAL_MAX_POLICIES];
    __shared__ int wsum[PS_THREADS / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int p = tid; p < K; p += PS_THREADS) { cnt[p] = 0; run[p] = 0; }
    __syncthreads();
    for (int b = tid; b < bs; b += PS_THREADS) {
        const int p = mp[b];
        if (p >= 0 && p < K) atomicAdd(&cnt[p], 1);
        else if (status) atomicExch(status, 1);
    }
    __syncthreads();
    // inclusive scan of the CTAs per policy (K <= PS_THREADS: one bucket per thread)
    int c = tid < K ? (cnt[tid] * N + AS_ROWS - 1) / AS_ROWS : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, c, o); if (lane >= o) c += v; }
    if (lane == 31) wsum[warp] = c;
    __syncthreads();
    if (warp == 0) {
        int s = wsum[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += v; }
        wsum[lane] = s;
    }
    __syncthreads();
    if (warp > 0) c += wsum[warp - 1];
    if (tid < K) end[tid] = c;
    const int used = wsum[PS_THREADS / 32 - 1];
    if (tid == 0) {
        sched[0] = used; sched[1] = bs * N; sched[2] = N; sched[3] = K;
        for (int i = 4; i < PS_HDR; ++i) sched[i] = 0;
    }
    __syncthreads();
    // every used entry: its policy (the first bucket whose CTA range ends after it) and padding rows
    for (int e = tid; e < used; e += PS_THREADS) {
        int lo = 0, hi = K - 1;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (end[mid] > e) hi = mid; else lo = mid + 1; }
        int32_t *ent = sched + PS_HDR + (int64_t)e * PS_ENT;
        for (int r = 0; r < AS_ROWS; ++r) ent[r] = -1;
        ent[AS_ROWS] = lo;
        for (int r = AS_ROWS + 1; r < PS_ENT; ++r) ent[r] = 0;
    }
    __syncthreads();
    // one warp places the matches in order: the rank of a match in its bucket = matches of that policy before it
    if (warp == 0) {
        for (int b0 = 0; b0 < bs; b0 += 32) {
            const int b = b0 + lane;
            const int p = b < bs ? mp[b] : -1;
            const bool ok = p >= 0 && p < K;
            const unsigned same = __match_any_sync(0xffffffffu, ok ? p : -1);
            const int base = ok ? run[p] : 0;
            __syncwarp();
            if (ok) {
                const int rank = base + __popc(same & ((1u << lane) - 1));
                if ((same & ((1u << lane) - 1)) == 0) run[p] = base + __popc(same);
                const int e0 = p > 0 ? end[p - 1] : 0;                  // bucket p's first entry
                for (int n = 0; n < N; ++n) {
                    const int pos = rank * N + n;                        // row slot within the bucket
                    sched[PS_HDR + (int64_t)(e0 + pos / AS_ROWS) * PS_ENT + pos % AS_ROWS] = b * N + n;
                }
            }
            __syncwarp();
        }
    }
}

// Per-match part of the fused rollout step (rows of this CTA; the row with n == 0 acts for its match):
// state / filled at t, reward / terminated at t-1.
template <bool POOL = false>
__device__ __forceinline__ void rollout_match_fields(const RolloutIO &io, int r0, int rows, int N, int tid, int nthreads,
                                                     const int32_t *rl = nullptr) {
    for (int r = 0; r < AS_ROWS; ++r) {
        const int row = cta_row<POOL>(r0, rl, r, rows);
        if (row >= rows) { if (POOL) continue; break; }
        const int b = row / N;
        if (row - b * N != 0) continue;
        for (int k = tid; k < io.S; k += nthreads) io.state_t[(int64_t)b * io.state_sb + k] = io.env_state[(int64_t)b * io.env_state_sb + k];
        if (tid == 0) {
            io.filled_t[(int64_t)b * io.filled_sb] = 1;
            if (io.prev_reward) {
                io.reward_tm1[(int64_t)b * io.reward_sb] = io.prev_reward[b];
                io.term_tm1[(int64_t)b * io.term_sb] = io.prev_done[b] ? 1 : 0;
            }
        }
    }
}

__global__ void __launch_bounds__(AS_THREADS) k_eps_greedy_select(const float *q, int64_t q_ld, int rows, int A,
                                                                  SelectArgs s) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= rows) return;
    float qv = lane < A ? q[(int64_t)warp * q_ld + lane] : 0.0f;
    select_row(s, warp, A, lane, qv);
}

// fold 8 per-lane partials across the warp: afterwards lane L holds the full sum of value index (L >> 2).
__device__ __forceinline__ float warp_fold8(const float (&v)[8], int lane) {
    const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4;
    float w[4], u[2];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        float send = b4 ? v[q] : v[q + 4];
        float keep = b4 ? v[q + 4] : v[q];
        w[q] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        float send = b3 ? w[q] : w[q + 2];
        float keep = b3 ? w[q + 2] : w[q];
        u[q] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
    float send = b2 ? u[0] : u[1];
    float keep = b2 ? u[1] : u[0];
    float s = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    return s;
}

struct AgentStepArgs {
    const float *params;
    int kind;                                   // MAL_AGENT_RNN | MAL_AGENT_DQN (feed-forward: no hidden state; stream kernel only)
    int rows, N, OBS, A;
    int dense;                                  // 1: obs is the full [rows, d_in] agent input (row stride obs_sb)
    AgentInput in;                              // fc1 input columns of the fused input assembly (dense: last = id = 0)
    const float *obs; int64_t obs_sb;
    const float *onehot; int64_t onehot_sb;     // NULL at t == 0
    const float *h_in;                          // NULL -> zeros
    float *h_out, *q;
    int do_select;
    SelectArgs sel;
    RolloutIO io;
    // pooled instances only (POOL = true): params is the [n_policies, table_ld] table, sched the work list
    const int32_t *sched; int64_t table_ld; int n_policies;
};

// Latency plan: a CTA needs every weight exactly once, and nothing but the inputs depends on anything, so ALL
// global loads (inputs, 48 GRU weight rows per warp, fc1 / fc2 rows, biases) are issued back to back at kernel entry
// into registers; the phases below then only touch registers and shared memory.
#define AS_FC1_MAXK 7    // ceil(224 / 32): obs+action columns handled per lane
template <bool POOL>
__global__ void __launch_bounds__(AS_THREADS, 1) k_agent_step(AgentStepArgs a) {
    extern __shared__ float as_smem[];
    const AgentLayout L = agent_layout(a.dense ? a.OBS : a.OBS + a.in.last + a.in.id, a.A);
    const int Kin = a.dense ? a.OBS : a.OBS + a.in.last;   // [obs | last action]: the agent-id block is a bias gather
    const int ldin = Kin + 1;
    float *in_s = as_smem;                       // [8][ldin]
    float *x_s = in_s + AS_ROWS * ldin;          // [8][64]
    float *h_s = x_s + AS_ROWS * HID;            // [8][64]
    float *g_s = h_s + AS_ROWS * HID;            // [8][384]  W_ih x | W_hh h (no biases)
    float *hn_s = g_s + AS_ROWS * 2 * G3;        // [8][64]
    float *q_s = hn_s + AS_ROWS * HID;           // [8][32]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int r0 = blockIdx.x * AS_ROWS;
    const float *P = a.params;
    const int32_t *rl = nullptr;
    if constexpr (POOL) { if (!pool_cta(P, rl, a.params, a.table_ld, a.n_policies, a.sched, a.rows, a.N)) return; }

    // ---- issue every global load up front ---------------------------------------------------------------------
    float2 wg[2 * G3 / AS_WARPS];                // GRU rows warp, warp+8, ... of [W_ih ; W_hh]   (48 x float2)
#pragma unroll
    for (int i = 0; i < 2 * G3 / AS_WARPS; ++i) {
        const int jj = warp + AS_WARPS * i;
        const bool hh = jj >= G3;
        const int j = hh ? jj - G3 : jj;
        wg[i] = ldg_f2<POOL>(reinterpret_cast<const float2 *>(P + (hh ? L.w_hh : L.w_ih) + (int64_t)j * HID) + lane);
    }
    float w1[HID / AS_WARPS][AS_FC1_MAXK];       // fc1 rows warp, warp+8, ...; columns lane, lane+32, ...
    float b1x[HID / AS_WARPS];                   // fc1 bias + agent-id column, for the row this lane finalises
#pragma unroll
    for (int i = 0; i < HID / AS_WARPS; ++i) {
        const int j = warp + AS_WARPS * i;
        const float *w = P + L.fc1_w + (int64_t)j * L.d_in;
#pragma unroll
        for (int c = 0; c < AS_FC1_MAXK; ++c) w1[i][c] = (lane + 32 * c < Kin) ? __ldg(w + lane + 32 * c) : 0.0f;
        const int row = cta_row<POOL>(r0, rl, lane >> 2, a.rows);
        const int n = row < a.rows ? row % a.N : 0;
        b1x[i] = __ldg(P + L.fc1_b + j) + (a.in.id ? __ldg(w + Kin + n) : 0.0f);
    }
    float2 w2[MAL_MAX_ACTIONS / AS_WARPS];
    float b2[MAL_MAX_ACTIONS / AS_WARPS];
#pragma unroll
    for (int i = 0; i < MAL_MAX_ACTIONS / AS_WARPS; ++i) {
        const int j = warp + AS_WARPS * i;
        w2[i] = make_float2(0.f, 0.f);
        b2[i] = 0.0f;
        if (j < a.A) {
            w2[i] = ldg_f2<POOL>(reinterpret_cast<const float2 *>(P + L.fc2_w + (int64_t)j * HID) + lane);
            b2[i] = __ldg(P + L.fc2_b + j);
        }
    }
    // gate biases of the hidden unit this thread combines (items tid and tid+256 share i = tid & 63)
    const int gi_ = tid & 63;
    const float bir = __ldg(P + L.b_ih + gi_) + __ldg(P + L.b_hh + gi_);
    const float biz = __ldg(P + L.b_ih + HID + gi_) + __ldg(P + L.b_hh + HID + gi_);
    const float bin = __ldg(P + L.b_ih + 2 * HID + gi_), bhn = __ldg(P + L.b_hh + 2 * HID + gi_);

    // ---- stage inputs (obs | last action one-hot) and previous hidden state
    for (int idx = tid; idx < AS_ROWS * Kin; idx += AS_THREADS) {
        int r = idx / Kin, k = idx - r * Kin, row = cta_row<POOL>(r0, rl, r, a.rows);
        float v = 0.0f;
        if (row < a.rows) {
            const int b = row / a.N, n = row - b * a.N;
            if (a.dense) v = a.obs[(int64_t)row * a.obs_sb + k];
            else if (k < a.OBS) {
                v = a.obs[(int64_t)b * a.obs_sb + (int64_t)n * a.OBS + k];
                if (a.io.enabled) a.io.obs_t[(int64_t)b * a.io.obs_sb + (int64_t)n * a.OBS + k] = v;   // pre-transition update of step t
            }
            else if (a.onehot) v = a.onehot[(int64_t)b * a.onehot_sb + (int64_t)n * a.A + (k - a.OBS)];
        }
        in_s[r * ldin + k] = v;
    }
    if (a.io.enabled) rollout_match_fields<POOL>(a.io, r0, a.rows, a.N, tid, AS_THREADS, rl);
    for (int idx = tid; idx < AS_ROWS * HID; idx += AS_THREADS) {
        int r = idx >> 6, row = cta_row<POOL>(r0, rl, r, a.rows);
        h_s[idx] = (a.h_in && row < a.rows) ? a.h_in[(int64_t)row * HID + (idx & 63)] : 0.0f;
    }
    __syncthreads();

    // ---- fc1 + relu (agent-id one-hot column folded in as a bias gather)
#pragma unroll
    for (int i = 0; i < HID / AS_WARPS; ++i) {
        const int j = warp + AS_WARPS * i;
        float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
        for (int c = 0; c < AS_FC1_MAXK; ++c) {
            const int k = lane + 32 * c;
            if (k < Kin) {
#pragma unroll
                for (int r = 0; r < 8; ++r) acc[r] = fmaf(w1[i][c], in_s[r * ldin + k], acc[r]);
            }
        }
        float s = warp_fold8(acc, lane);
        if ((lane & 3) == 0) x_s[(lane >> 2) * HID + j] = fmaxf(s + b1x[i], 0.0f);
    }
    __syncthreads();

    // ---- W_ih x  and  W_hh h   (384 weight rows of 64, already in registers)
    {
        float xv[8][2], hv[8][2];
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            xv[r][0] = x_s[r * HID + 2 * lane]; xv[r][1] = x_s[r * HID + 2 * lane + 1];
            hv[r][0] = h_s[r * HID + 2 * lane]; hv[r][1] = h_s[r * HID + 2 * lane + 1];
        }
#pragma unroll
        for (int i = 0; i < 2 * G3 / AS_WARPS; ++i) {
            const int jj = warp + AS_WARPS * i;
            const bool hh = jj >= G3;          // compile-time per i after unrolling only if warp-independent; cheap anyway
            float acc[8];
#pragma unroll
            for (int r = 0; r < 8; ++r)
                acc[r] = hh ? fmaf(wg[i].y, hv[r][1], wg[i].x * hv[r][0]) : fmaf(wg[i].y, xv[r][1], wg[i].x * xv[r][0]);
            float s = warp_fold8(acc, lane);
            if ((lane & 3) == 0) g_s[(lane >> 2) * 2 * G3 + jj] = s;
        }
    }
    __syncthreads();

    // ---- gate math: r,z,n ; h' = n + z (h - n)
    for (int idx = tid; idx < AS_ROWS * HID; idx += AS_THREADS) {
        int r = idx >> 6, i = idx & 63, row = cta_row<POOL>(r0, rl, r, a.rows);
        const float *g = g_s + r * 2 * G3;
        float rr = sigmoidf_acc(g[i] + g[G3 + i] + bir);
        float zz = sigmoidf_acc(g[HID + i] + g[G3 + HID + i] + biz);
        float nn = tanhf(g[2 * HID + i] + bin + rr * (g[G3 + 2 * HID + i] + bhn));
        float hp = h_s[idx];
        float hn = nn + zz * (hp - nn);
        hn_s[idx] = hn;
        if (row < a.rows) a.h_out[(int64_t)row * HID + i] = hn;
    }
    __syncthreads();

    // ---- fc2
    {
        float hv[8][2];
#pragma unroll
        for (int r = 0; r < 8; ++r) { hv[r][0] = hn_s[r * HID + 2 * lane]; hv[r][1] = hn_s[r * HID + 2 * lane + 1]; }
#pragma unroll
        for (int i = 0; i < MAL_MAX_ACTIONS / AS_WARPS; ++i) {
            const int j = warp + AS_WARPS * i;
            if (j < a.A) {      // warp-uniform
                float acc[8];
#pragma unroll
                for (int r = 0; r < 8; ++r) acc[r] = fmaf(w2[i].y, hv[r][1], w2[i].x * hv[r][0]);
                float s = warp_fold8(acc, lane);
                if ((lane & 3) == 0) {
                    int r = lane >> 2, row = cta_row<POOL>(r0, rl, r, a.rows);
                    s += b2[i];
                    q_s[r * 32 + j] = s;
                    if (row < a.rows) a.q[(int64_t)row * a.A + j] = s;
                }
            }
        }
    }
    if (!a.do_select) return;
    __syncthreads();
    // ---- epsilon-greedy selection: one warp per row
    {
        int row = cta_row<POOL>(r0, rl, warp, a.rows);
        if (row < a.rows) select_row(a.sel, row, a.A, lane, lane < a.A ? q_s[warp * 32 + lane] : 0.0f, a.io.enabled ? &a.io : nullptr);
    }
}

// =============================================================================================
// Latency variant for rollouts (a handful of CTAs, typically ONE: batch_size_run = 1 -> 5 agent rows).
// The three projections of the step are [outputs x K] x [K x 8 rows] products with every weight used exactly once per
// CTA, so the weights go STRAIGHT from L2 into the A fragments of warp-level tensor-core MMAs (mma.sync m16n8k8, tf32
// inputs split hi + lo and applied three times -- hi*hi + lo*hi + hi*lo, fp32 accumulate -- i.e. fp32-level accuracy),
// the 8 agent rows of the CTA are the N dimension, and nothing is reduced across lanes (the lanes-along-k layout of
// k_agent_step spends most of its 20 us in shuffle folds).  16 warps:
//   warps 0-3   fc1: one 16-output tile each over the whole input width (loads issued 8 k-steps ahead)
//   warps 4-15  the twelve 16-row tiles of W_hh h (independent of fc1: runs beside it), then, after the barrier, the
//               twelve tiles of W_ih x; both tiles' weights are requested at kernel entry
//   all         gate math (one (row, unit) pair per thread), then warps 0-1: fc2, then one warp per row: selection
// =============================================================================================
#define AL_THREADS 512
__device__ __forceinline__ void mma_m16n8k8_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t tf32_hi(float x) { uint32_t r; asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x)); return r; }
// d += A_tile . B for one k-step: av = the lane's four A elements (fp32), (bv0, bv1) its two B elements
__device__ __forceinline__ void mma3(float (&d)[4], const float (&av)[4], float bv0, float bv1) {
    uint32_t ah[4], al[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) { ah[i] = tf32_hi(av[i]); al[i] = tf32_hi(av[i] - __uint_as_float(ah[i])); }
    const uint32_t bh0 = tf32_hi(bv0), bh1 = tf32_hi(bv1);
    const uint32_t bl0 = tf32_hi(bv0 - __uint_as_float(bh0)), bl1 = tf32_hi(bv1 - __uint_as_float(bh1));
    mma_m16n8k8_tf32(d, al, bh0, bh1);      // small terms first
    mma_m16n8k8_tf32(d, ah, bl0, bl1);
    mma_m16n8k8_tf32(d, ah, bh0, bh1);
}
// A fragment of k-step ks of the 16-row tile starting at row j0 of a row-major [M x K] weight matrix (zero padded)
__device__ __forceinline__ void load_a_frag(float (&av)[4], const float *W, int64_t ldw, int M, int K, int j0, int ks, int g, int tig) {
    const int r0 = j0 + g, r1 = j0 + g + 8, c0 = 8 * ks + tig, c1 = c0 + 4;
    av[0] = (r0 < M && c0 < K) ? __ldg(W + (int64_t)r0 * ldw + c0) : 0.0f;
    av[1] = (r1 < M && c0 < K) ? __ldg(W + (int64_t)r1 * ldw + c0) : 0.0f;
    av[2] = (r0 < M && c1 < K) ? __ldg(W + (int64_t)r0 * ldw + c1) : 0.0f;
    av[3] = (r1 < M && c1 < K) ? __ldg(W + (int64_t)r1 * ldw + c1) : 0.0f;
}

template <bool POOL>
__global__ void __launch_bounds__(AL_THREADS, 1) k_agent_step_lat(AgentStepArgs a) {
    extern __shared__ float as_smem[];
    const AgentLayout L = agent_layout(a.dense ? a.OBS : a.OBS + a.in.last + a.in.id, a.A);
    const int Kin = a.dense ? a.OBS : a.OBS + a.in.last;   // [obs | last action]: the agent-id block is a bias gather
    const int ldin = ((Kin + 7) & ~7) + 4;       // zero-padded to whole k-steps; +4: the 8 rows of a B fragment hit different banks
    float *in_s = as_smem;                       // [8][ldin]
    float *x_s = in_s + AS_ROWS * ldin;          // [8][68]
    float *h_s = x_s + AS_ROWS * 68;             // [8][68]
    float *g_s = h_s + AS_ROWS * 68;             // [8][384]  W_ih x | W_hh h (no biases)
    float *hn_s = g_s + AS_ROWS * 2 * G3;        // [8][68]
    float *q_s = hn_s + AS_ROWS * 68;            // [8][32]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, tig = lane & 3;
    const int r0 = blockIdx.x * AS_ROWS;
    const float *P = a.params;
    const int32_t *rl = nullptr;
    if constexpr (POOL) { if (!pool_cta(P, rl, a.params, a.table_ld, a.n_policies, a.sched, a.rows, a.N)) return; }

    // ---- EVERY global operand of the step is requested here, before the first barrier, so that the kernel pays one
    //      memory round trip: weights of this warp's tiles, biases, the selector's avail flags and draws
    float whh[8][4], wih[8][4];                  // warps 4-15: GRU tile gt; warps 0-3: wih = first 8 k-steps of fc1, whh (warps 0-1) = fc2
    const int gt = warp - 4;                     // GRU tile of warps 4..15: rows 16 gt .. 16 gt + 15 of W_ih and of W_hh
    const int nks1 = (Kin + 7) >> 3;
    float fb[4] = {0.f, 0.f, 0.f, 0.f};          // warps 0-3: fc1 bias + agent-id column of this lane's four outputs; later fc2 bias (2)
    float f2b[2] = {0.f, 0.f};
    if (warp >= 4) {
#pragma unroll
        for (int ks = 0; ks < 8; ++ks) load_a_frag(whh[ks], P + L.w_hh, HID, G3, HID, 16 * gt, ks, g, tig);
#pragma unroll
        for (int ks = 0; ks < 8; ++ks) load_a_frag(wih[ks], P + L.w_ih, HID, G3, HID, 16 * gt, ks, g, tig);
    } else {
#pragma unroll
        for (int q = 0; q < 8; ++q)
            if (q < nks1) load_a_frag(wih[q], P + L.fc1_w, L.d_in, HID, Kin, 16 * warp, q, g, tig);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int j = 16 * warp + g + 8 * (i >> 1), row = cta_row<POOL>(r0, rl, 2 * tig + (i & 1), a.rows);
            const int n = row < a.rows ? row % a.N : 0;
            fb[i] = __ldg(P + L.fc1_b + j) + (a.in.id ? __ldg(P + L.fc1_w + (int64_t)j * L.d_in + Kin + n) : 0.0f);
        }
        if (warp < 2) {
#pragma unroll
            for (int ks = 0; ks < 8; ++ks) load_a_frag(whh[ks], P + L.fc2_w, HID, a.A, HID, 16 * warp, ks, g, tig);
#pragma unroll
            for (int i = 0; i < 2; ++i) { const int j = 16 * warp + g + 8 * i; f2b[i] = j < a.A ? __ldg(P + L.fc2_b + j) : 0.0f; }
        }
    }
    float bir, biz, bin, bhn;                    // gate biases of this thread's (row, unit) pair
    {
        const int i = tid & 63;
        bir = __ldg(P + L.b_ih + i) + __ldg(P + L.b_hh + i);
        biz = __ldg(P + L.b_ih + HID + i) + __ldg(P + L.b_hh + HID + i);
        bin = __ldg(P + L.b_ih + 2 * HID + i); bhn = __ldg(P + L.b_hh + 2 * HID + i);
    }
    int sel_av = 0;                              // selector operands of this CTA's row `warp` (warps 0-7)
    float sel_ev = 1.0f, sel_uu = 1.0f;
    if (a.do_select && warp < AS_ROWS && cta_row<POOL>(r0, rl, warp, a.rows) < a.rows) {
        sel_av = select_avail(a.sel, cta_row<POOL>(r0, rl, warp, a.rows), a.A, lane);
        select_draws(a.sel, cta_row<POOL>(r0, rl, warp, a.rows), a.A, lane, sel_ev, sel_uu);     // Philox rounds run under the load latency
    }
    // ---- stage inputs (obs | last action one-hot, zero padded) and the previous hidden state
    for (int idx = tid; idx < AS_ROWS * ldin; idx += AL_THREADS) {
        const int r = idx / ldin, k = idx - r * ldin, row = cta_row<POOL>(r0, rl, r, a.rows);
        float v = 0.0f;
        if (row < a.rows && k < Kin) {
            const int b = row / a.N, n = row - b * a.N;
            if (a.dense) v = a.obs[(int64_t)row * a.obs_sb + k];
            else if (k < a.OBS) {
                v = a.obs[(int64_t)b * a.obs_sb + (int64_t)n * a.OBS + k];
                if (a.io.enabled) a.io.obs_t[(int64_t)b * a.io.obs_sb + (int64_t)n * a.OBS + k] = v;   // pre-transition update of step t
            }
            else if (a.onehot) v = a.onehot[(int64_t)b * a.onehot_sb + (int64_t)n * a.A + (k - a.OBS)];
        }
        in_s[idx] = v;
    }
    if (a.io.enabled) rollout_match_fields<POOL>(a.io, r0, a.rows, a.N, tid, AL_THREADS, rl);
    for (int idx = tid; idx < AS_ROWS * HID; idx += AL_THREADS) {
        const int r = idx >> 6, row = cta_row<POOL>(r0, rl, r, a.rows);
        h_s[r * 68 + (idx & 63)] = (a.h_in && row < a.rows) ? a.h_in[(int64_t)row * HID + (idx & 63)] : 0.0f;
    }
    __syncthreads();

    if (warp < 4) {
        // ---- fc1 + relu: outputs 16 warp .. 16 warp + 15, all 8 rows; the agent-id one-hot column is a bias gather
        float d[4] = {0.f, 0.f, 0.f, 0.f};
        const float *W1 = P + L.fc1_w;
        for (int k0 = 0; k0 < nks1; k0 += 8) {
            float av[8][4];
            if (k0 + 8 < nks1) {                 // wider inputs (10v10 / 20v20): the next eight k-steps fly under these MMAs
#pragma unroll
                for (int q = 0; q < 8; ++q)
                    if (k0 + 8 + q < nks1) load_a_frag(av[q], W1, L.d_in, HID, Kin, 16 * warp, k0 + 8 + q, g, tig);
            }
#pragma unroll
            for (int q = 0; q < 8; ++q)
                if (k0 + q < nks1) mma3(d, wih[q], in_s[g * ldin + 8 * (k0 + q) + tig], in_s[g * ldin + 8 * (k0 + q) + tig + 4]);
#pragma unroll
            for (int q = 0; q < 8; ++q)
#pragma unroll
                for (int c = 0; c < 4; ++c) wih[q][c] = av[q][c];
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {            // d[i]: output j = 16 warp + g + 8 (i >> 1), row r = 2 tig + (i & 1)
            const int j = 16 * warp + g + 8 * (i >> 1), r = 2 * tig + (i & 1);
            x_s[r * 68 + j] = fmaxf(d[i] + fb[i], 0.0f);
        }
    } else {
        // ---- W_hh h for this warp's 16 gate rows (does not depend on fc1)
        float d[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int ks = 0; ks < 8; ++ks) mma3(d, whh[ks], h_s[g * 68 + 8 * ks + tig], h_s[g * 68 + 8 * ks + tig + 4]);
#pragma unroll
        for (int i = 0; i < 4; ++i) g_s[(2 * tig + (i & 1)) * 2 * G3 + G3 + 16 * gt + g + 8 * (i >> 1)] = d[i];
    }
    __syncthreads();
    if (warp >= 4) {
        // ---- W_ih x
        float d[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int ks = 0; ks < 8; ++ks) mma3(d, wih[ks], x_s[g * 68 + 8 * ks + tig], x_s[g * 68 + 8 * ks + tig + 4]);
#pragma unroll
        for (int i = 0; i < 4; ++i) g_s[(2 * tig + (i & 1)) * 2 * G3 + 16 * gt + g + 8 * (i >> 1)] = d[i];
    }
    __syncthreads();

    // ---- gate math: r,z,n ; h' = n + z (h - n): one (row, unit) pair per thread
    {
        const int r = tid >> 6, i = tid & 63, row = cta_row<POOL>(r0, rl, r, a.rows);
        const float *gg = g_s + r * 2 * G3;
        const float rr = sigmoidf_acc(gg[i] + gg[G3 + i] + bir);
        const float zz = sigmoidf_acc(gg[HID + i] + gg[G3 + HID + i] + biz);
        const float nn = tanhf(gg[2 * HID + i] + bin + rr * (gg[G3 + 2 * HID + i] + bhn));
        const float hp = h_s[r * 68 + i];
        const float hn = nn + zz * (hp - nn);
        hn_s[r * 68 + i] = hn;
        if (row < a.rows) a.h_out[(int64_t)row * HID + i] = hn;
    }
    __syncthreads();

    // ---- fc2
    if (warp < 2 && 16 * warp < a.A) {
        float d[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int ks = 0; ks < 8; ++ks) mma3(d, whh[ks], hn_s[g * 68 + 8 * ks + tig], hn_s[g * 68 + 8 * ks + tig + 4]);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int j = 16 * warp + g + 8 * (i >> 1), r = 2 * tig + (i & 1), row = cta_row<POOL>(r0, rl, r, a.rows);
            if (j < a.A) {
                const float s = d[i] + f2b[i >> 1];
                q_s[r * 32 + j] = s;
                if (row < a.rows) a.q[(int64_t)row * a.A + j] = s;
            }
        }
    }
    if (!a.do_select) return;
    __syncthreads();
    // ---- epsilon-greedy selection: one warp per row
    if (warp < AS_ROWS) {
        const int row = cta_row<POOL>(r0, rl, warp, a.rows);
        if (row < a.rows) select_core(a.sel, row, a.A, lane, lane < a.A ? q_s[warp * 32 + lane] : 0.0f, sel_av, sel_ev, sel_uu,
                                      a.io.enabled ? &a.io : nullptr);
    }
}

// Throughput variant for large row counts (many CTAs per SM): weight rows are streamed from L2 as they are used
// instead of being parked in 255 registers per thread.
template <bool POOL>
__global__ void __launch_bounds__(AS_THREADS) k_agent_step_stream(AgentStepArgs a) {
    extern __shared__ float as_smem[];
    const AgentLayout L = agent_layout(a.dense ? a.OBS : a.OBS + a.in.last + a.in.id, a.A, a.kind);
    const bool rnn = a.kind == MAL_AGENT_RNN;
    const int Kin = a.dense ? a.OBS : a.OBS + a.in.last;   // [obs | last action]: the agent-id block is a bias gather
    const int ldin = Kin + 1;
    float *in_s = as_smem;                       // [8][ldin]
    float *x_s = in_s + AS_ROWS * ldin;          // [8][64]
    float *h_s = x_s + AS_ROWS * HID;            // [8][64]
    float *g_s = h_s + AS_ROWS * HID;            // [8][384]  gi | gh
    float *hn_s = g_s + AS_ROWS * 2 * G3;        // [8][64]
    float *q_s = hn_s + AS_ROWS * HID;           // [8][32]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int r0 = blockIdx.x * AS_ROWS;
    const float *P = a.params;
    const int32_t *rl = nullptr;
    if constexpr (POOL) { if (!pool_cta(P, rl, a.params, a.table_ld, a.n_policies, a.sched, a.rows, a.N)) return; }

    // ---- stage inputs (obs | last action one-hot) and previous hidden state
    for (int idx = tid; idx < AS_ROWS * Kin; idx += AS_THREADS) {
        int r = idx / Kin, k = idx - r * Kin, row = cta_row<POOL>(r0, rl, r, a.rows);
        float v = 0.0f;
        if (row < a.rows) {
            const int b = row / a.N, n = row - b * a.N;
            if (a.dense) v = a.obs[(int64_t)row * a.obs_sb + k];
            else if (k < a.OBS) {
                v = a.obs[(int64_t)b * a.obs_sb + (int64_t)n * a.OBS + k];
                if (a.io.enabled) a.io.obs_t[(int64_t)b * a.io.obs_sb + (int64_t)n * a.OBS + k] = v;   // pre-transition update of step t
            }
            else if (a.onehot) v = a.onehot[(int64_t)b * a.onehot_sb + (int64_t)n * a.A + (k - a.OBS)];
        }
        in_s[r * ldin + k] = v;
    }
    if (a.io.enabled) rollout_match_fields<POOL>(a.io, r0, a.rows, a.N, tid, AS_THREADS, rl);
    for (int idx = tid; idx < AS_ROWS * HID; idx += AS_THREADS) {
        int r = idx >> 6, row = cta_row<POOL>(r0, rl, r, a.rows);
        h_s[idx] = (rnn && a.h_in && row < a.rows) ? a.h_in[(int64_t)row * HID + (idx & 63)] : 0.0f;
    }
    __syncthreads();

    // ---- fc1 + relu (agent-id one-hot column folded in as a bias gather)
    for (int j = warp; j < HID; j += AS_WARPS) {
        const float *w = P + L.fc1_w + (int64_t)j * L.d_in;
        float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        for (int k = lane; k < Kin; k += 32) {
            float wv = __ldg(w + k);
#pragma unroll
            for (int r = 0; r < 8; ++r) acc[r] = fmaf(wv, in_s[r * ldin + k], acc[r]);
        }
        float s = warp_fold8(acc, lane);
        if ((lane & 3) == 0) {
            int r = lane >> 2, row = cta_row<POOL>(r0, rl, r, a.rows);
            int n = row < a.rows ? row % a.N : 0;
            s += __ldg(P + L.fc1_b + j) + (a.in.id ? __ldg(w + Kin + n) : 0.0f);
            x_s[r * HID + j] = fmaxf(s, 0.0f);
        }
    }
    __syncthreads();

    // ---- gi = W_ih x + b_ih ; gh = W_hh h + b_hh   (384 weight rows of 64)
    if (rnn) {
        float xv[8][2], hv[8][2];
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            xv[r][0] = x_s[r * HID + 2 * lane]; xv[r][1] = x_s[r * HID + 2 * lane + 1];
            hv[r][0] = h_s[r * HID + 2 * lane]; hv[r][1] = h_s[r * HID + 2 * lane + 1];
        }
#pragma unroll 4
        for (int jj = warp; jj < 2 * G3; jj += AS_WARPS) {
            const bool hh = jj >= G3;
            const int j = hh ? jj - G3 : jj;
            const float2 wv = ldg_f2<POOL>(reinterpret_cast<const float2 *>(P + (hh ? L.w_hh : L.w_ih) + (int64_t)j * HID) + lane);
            float acc[8];
#pragma unroll
            for (int r = 0; r < 8; ++r)
                acc[r] = hh ? fmaf(wv.y, hv[r][1], wv.x * hv[r][0]) : fmaf(wv.y, xv[r][1], wv.x * xv[r][0]);
            float s = warp_fold8(acc, lane);
            if ((lane & 3) == 0) g_s[(lane >> 2) * 2 * G3 + jj] = s + __ldg(P + (hh ? L.b_hh : L.b_ih) + j);
        }
    }
    __syncthreads();

    // ---- gate math: r,z,n ; h' = n + z (h - n)        (DQN: q = fc2(relu(fc1(.))), dqn_agent.py:34-37)
    if (!rnn) {
        for (int idx = tid; idx < AS_ROWS * HID; idx += AS_THREADS) hn_s[idx] = x_s[idx];
    } else
    for (int idx = tid; idx < AS_ROWS * HID; idx += AS_THREADS) {
        int r = idx >> 6, i = idx & 63, row = cta_row<POOL>(r0, rl, r, a.rows);
        const float *g = g_s + r * 2 * G3;
        float rr = sigmoidf_acc(g[i] + g[G3 + i]);
        float zz = sigmoidf_acc(g[HID + i] + g[G3 + HID + i]);
        float nn = tanhf(g[2 * HID + i] + rr * g[G3 + 2 * HID + i]);
        float hp = h_s[idx];
        float hn = nn + zz * (hp - nn);
        hn_s[idx] = hn;
        if (row < a.rows) a.h_out[(int64_t)row * HID + i] = hn;
    }
    __syncthreads();

    // ---- fc2
    {
        float hv[8][2];
#pragma unroll
        for (int r = 0; r < 8; ++r) { hv[r][0] = hn_s[r * HID + 2 * lane]; hv[r][1] = hn_s[r * HID + 2 * lane + 1]; }
        for (int j = warp; j < a.A; j += AS_WARPS) {
            const float2 wv = ldg_f2<POOL>(reinterpret_cast<const float2 *>(P + L.fc2_w + (int64_t)j * HID) + lane);
            float acc[8];
#pragma unroll
            for (int r = 0; r < 8; ++r) acc[r] = fmaf(wv.y, hv[r][1], wv.x * hv[r][0]);
            float s = warp_fold8(acc, lane);
            if ((lane & 3) == 0) {
                int r = lane >> 2, row = cta_row<POOL>(r0, rl, r, a.rows);
                s += __ldg(P + L.fc2_b + j);
                q_s[r * 32 + j] = s;
                if (row < a.rows) a.q[(int64_t)row * a.A + j] = s;
            }
        }
    }
    if (!a.do_select) return;
    __syncthreads();
    // ---- epsilon-greedy selection: one warp per row
    {
        int row = cta_row<POOL>(r0, rl, warp, a.rows);
        if (row < a.rows) select_row(a.sel, row, a.A, lane, lane < a.A ? q_s[warp * 32 + lane] : 0.0f, a.io.enabled ? &a.io : nullptr);
    }
}
