// Weight-gradient reductions on the tensor cores:  dW[n, k] = sum_m dY[m, n] * A[m, k]   (split over row chunks of m)
// -- the `addmm` weight-gradient nodes of the reference's autograd graph (q_learner.py:103) as a split-M tcgen05 GEMM.
//
// The contraction runs over the ROW index m, so both MMA operands are the TRANSPOSES of what lies in memory.  Per
// 32-row block every warp loads four rows of the [32 x 128] dY and [32 x 64] A tiles (coalesced float4), parks them in
// its private shared-memory scratch, reads them back column-wise (lanes along n / k: conflict-free), splits each value into TF32 hi + lo
// (3xTF32, as in tc_gemm.cuh) and writes 16-byte pieces into the K-major SWIZZLE_128B operand tiles
// (row = n or k, the 128-byte row = the block's 32 m values).  Two operand stages: the 12 MMAs of block j
// (M = 128, N = 64, K = 8 x 4 k-steps x {hi*hi, lo*hi, hi*lo}) run while block j+1 is loaded, transposed and split.
// TMEM accumulators (hi*hi and the correction terms apart) are folded into fp32 REGISTER accumulators every RT_FLUSH
// blocks, so the tensor core's truncating accumulation never spans more than a few hundred rows.
// Output: per-chunk partials [chunk][Nout][K] (+ per-chunk column sums of dY for the bias gradient), gathered in a
// fixed order by k_grad_reduce exactly like the FFMA kernel's.
#pragma once
#include "tc_gemm.cuh"

#define RT_BM 32                          // rows (m) per block: one 128-byte swizzle row of the contraction dimension
#define RT_NT 128                         // n-tile (MMA M)
#define RT_KT 64                          // k-tile (MMA N)
#define RT_OP_A (RT_NT * 128)             // 16 KB: one of hi / lo of the dY^T operand
#define RT_OP_B (RT_KT * 128)             //  8 KB
#define RT_STAGE (2 * RT_OP_A + 2 * RT_OP_B)          // 48 KB
#define RT_RAW_Y (RT_BM * RT_NT * 4)      // 16 KB
#define RT_RAW_A (RT_BM * RT_KT * 4)      //  8 KB
#define RT_SMEM_BYTES (2 * RT_STAGE + RT_RAW_Y + RT_RAW_A)   // 120 KB
#define RT_FLUSH 8                        // blocks between TMEM -> register folds (256 rows)
#define RT_NS 4                           // MNM = 2: operand stages (blocks j+1, j+2 are in flight while block j is split and multiplied)
#define RT_AHEAD 2
#define RT_SMEM_BYTES_PIPE (RT_NS * RT_STAGE)                 // 192 KB

// SWAP = 1 computes the transposed tile dW^T[k, n] (MMA rows <- 128 columns of A, MMA columns <- 64 columns of dY): for
// narrow outputs with a wide inner dimension (fc1: Nout = 64, K = d_in up to 246) this fills the 128-row operand
// instead of padding half of it, and halves the number of tiles.
//
// MNM = 1 (default): the operands are handed to the tensor core in MN-MAJOR form, i.e. exactly as they lie in memory
// (the contraction index m is the slow one): a 32-row block is staged as [32-column slab][m row][128 bytes] straight
// from the registers the coalesced float4 loads landed in.  No scratch, no column-wise read-back, no __syncwarp; a
// k-step (8 rows of m) is 1 KB further into every slab.
// For MN-major TF32 operands the only layout the tensor core accepts is SWIZZLE_128B_BASE32B (descriptor layout type 1;
// with type 2 the MMA reads zeros -- decoded with tools/mn_probe.cu, which makes the tensor core report the shared-memory
// offset it fetches for every (mn, k)): atoms of 4 m rows x 128 bytes, the 32-byte granule index XOR-ed with (m & 3),
// SBO = 512 B between 4-row groups, LBO = the slab stride between 32-column groups.
// MNM = 0 keeps the round-1 in-shared-memory transposition into K-major tiles (mal_set_option "reduce_mn" = 0) for A/B checks.
__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;     // next 32-column slab of the MN dimension
    d |= (uint64_t)(512 >> 4) << 32;                      // next group of four m rows
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)1 << 61;                               // SWIZZLE_128B_BASE32B
    return d;
}
// byte offset of 16-byte piece c (0..7) of m row kr inside one [32 m rows x 32 columns] MN-major slab
__device__ __forceinline__ uint32_t mn_off(int kr, int c) { return (uint32_t)kr * 128u + (uint32_t)((c ^ ((kr & 3) << 1)) << 4); }
#define RT_SLAB (RT_BM * 128)             // 4 KB: [32 m rows x 32 columns] of one operand piece (MN-major staging)

template <int AK, int SWAP, int MNM>
__global__ void __launch_bounds__(256, 1) k_reduce_tc(const __grid_constant__ RedGroup g) {
    extern __shared__ __align__(1024) uint8_t rt_smem[];
    __shared__ __align__(8) uint64_t st_bar[RT_NS];
    __shared__ uint32_t tmem_base_s;
    __shared__ __align__(16) float bsum_s[8][RT_NT];
    int pi = 0;
    while (pi + 1 < g.n && (int)blockIdx.y >= g.p[pi + 1].tile0) ++pi;
    const RedProb p = g.p[pi];
    const BatchView &bv = g.bv;
    const int chunk = blockIdx.x;
    if (chunk >= p.n_chunks) return;
    const int tile = blockIdx.y - p.tile0;
    // wide operand (128 MMA rows) / narrow operand (64 MMA columns): dY / A, or A / dY when SWAP
    const int n_narrow = SWAP ? (p.Nout + RT_KT - 1) / RT_KT : p.n_ktiles;
    const int wt = tile / n_narrow, st_ = tile - wt * n_narrow;
    const int n0 = SWAP ? st_ * RT_KT : wt * RT_NT;      // first dY column of this tile
    const int k0 = SWAP ? wt * RT_NT : st_ * RT_KT;      // first A column of this tile
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t mb = p.M0 + (int64_t)chunk * p.rows_per_chunk;
    int64_t me = mb + p.rows_per_chunk;
    if (me > p.M) me = p.M;
    const int nblk = me > mb ? (int)((me - mb + RT_BM - 1) / RT_BM) : 0;
    const bool want_bias = p.partB && (SWAP ? wt == 0 : st_ == 0);

    float *rawY = reinterpret_cast<float *>(rt_smem + 2 * RT_STAGE);
    float *rawA = reinterpret_cast<float *>(rt_smem + 2 * RT_STAGE + RT_RAW_Y);
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(128u));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < RT_NS; ++i) mbar_init(&st_bar[i], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = tmem_base_s;
    pdl_wait();

    const bool y_vec = ((p.ldy & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.dY + n0) & 15) == 0);
    const bool a_vec = AK == A_DENSE && ((p.lda & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.A + k0) & 15) == 0);
    const bool fast_ok = p.M < (1 << 24);
    const float invR = 1.0f / (float)(bv.R > 0 ? bv.R : 1), invN = 1.0f / (float)(bv.N > 0 ? bv.N : 1);
    const float invT = 1.0f / (float)(bv.T > 0 ? bv.T : 1);
    const bool s_vec = AK == A_STATE && (bv.state.sb & 3) == 0 && (bv.state.st & 3) == 0 && (k0 & 3) == 0 &&
                       ((reinterpret_cast<uintptr_t>(bv.state.ptr) & 15) == 0);
    const bool o_vec = AK == A_AGENT_IN && (bv.OBS & 3) == 0 && (bv.obs.sb & 3) == 0 && (bv.obs.st & 3) == 0 &&
                       ((reinterpret_cast<uintptr_t>(bv.obs.ptr) & 15) == 0);
    auto load_dy4 = [&](int64_t m, int n) -> float4 {      // dY[m, n .. n+3]
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (m < me && n < p.Nout) {
            const float *src = p.dY + m * p.ldy + n;
            if (y_vec && n + 4 <= p.Nout) v = __ldg(reinterpret_cast<const float4 *>(src));
            else {
                v.x = __ldg(src);
                if (n + 1 < p.Nout) v.y = __ldg(src + 1);
                if (n + 2 < p.Nout) v.z = __ldg(src + 2);
                if (n + 3 < p.Nout) v.w = __ldg(src + 3);
            }
        }
        return v;
    };
    auto load_a4 = [&](int64_t m, int k) -> float4 {       // A[m, k .. k+3] through the fused loaders
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (m < me && k < p.K) {
            if (AK == A_DENSE) {
                if (m >= p.shift) {
                    const float *src = p.A + (m - p.shift) * p.lda + k;
                    if (a_vec && k + 4 <= p.K) v = __ldg(reinterpret_cast<const float4 *>(src));
                    else {
                        v.x = __ldg(src);
                        if (k + 1 < p.K) v.y = __ldg(src + 1);
                        if (k + 2 < p.K) v.z = __ldg(src + 2);
                        if (k + 3 < p.K) v.w = __ldg(src + 3);
                    }
                }
            } else if (AK == A_STATE) {
                int b, t;
                if (fast_ok) fast_divmod((int)m, bv.T, invT, b, t);
                else { b = (int)((unsigned)m / (unsigned)bv.T); t = (int)m - b * bv.T; }
                const float *src = field_ptr<float>(bv.state, b, t + p.shift) + k;
                if (s_vec && k + 4 <= p.K) v = __ldg(reinterpret_cast<const float4 *>(src));
                else {
                    v.x = __ldg(src);
                    if (k + 1 < p.K) v.y = __ldg(src + 1);
                    if (k + 2 < p.K) v.z = __ldg(src + 2);
                    if (k + 3 < p.K) v.w = __ldg(src + 3);
                }
            } else {   // [obs | last-action one-hot | agent-id one-hot]: float4 over the obs part
                int t, rr, b, n;
                if (fast_ok) { fast_divmod((int)m, bv.R, invR, t, rr); fast_divmod(rr, bv.N, invN, b, n); }
                else { t = (int)((unsigned)m / (unsigned)bv.R); rr = (int)m - t * bv.R; b = rr / bv.N; n = rr - b * bv.N; }
                if (o_vec && k + 4 <= bv.OBS) {
                    v = __ldg(reinterpret_cast<const float4 *>(field_ptr<float>(bv.obs, b, t) + (int64_t)n * bv.OBS + k));
                } else {
                    RowSrc rs;
                    rs.agent = n;
                    rs.p0 = field_ptr<float>(bv.obs, b, t) + (int64_t)n * bv.OBS;
                    rs.p1 = t > 0 ? field_ptr<float>(bv.onehot, b, t - 1) + (int64_t)n * bv.A : nullptr;
                    v.x = row_elem(A_AGENT_IN, bv, rs, k);
                    if (k + 1 < p.K) v.y = row_elem(A_AGENT_IN, bv, rs, k + 1);
                    if (k + 2 < p.K) v.z = row_elem(A_AGENT_IN, bv, rs, k + 2);
                    if (k + 3 < p.K) v.w = row_elem(A_AGENT_IN, bv, rs, k + 3);
                }
            }
        }
        return v;
    };
    float4 py[4], pa[2];                              // wide rows (32 float4 each) / narrow rows (16 float4 each)
    float4 qy[4], qa[2];                              // MNM: second register set (block j+1 is requested before block j is staged)
    auto load_block_into = [&](int j, float4 (&py)[4], float4 (&pa)[2]) {
        const int64_t mm = mb + (int64_t)j * RT_BM;
#pragma unroll
        for (int i = 0; i < 4; ++i) {                 // warp w owns rows 4w .. 4w+3 (one 16-byte piece of every operand row)
            const int64_t m = mm + 4 * warp + i;
            py[i] = SWAP ? load_a4(m, k0 + 4 * lane) : load_dy4(m, n0 + 4 * lane);
        }
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int64_t m = mm + 4 * warp + 2 * i + (lane >> 4);
            const int c = lane & 15;
            pa[i] = SWAP ? load_dy4(m, n0 + 4 * c) : load_a4(m, k0 + 4 * c);
        }
    };
    auto load_block = [&](int j) { load_block_into(j, py, pa); };

    const int q = warp & 3, half = warp >> 2;         // accumulator ownership: TMEM lane quarter q, columns half*32 .. +32
    float acc[32];
#pragma unroll
    for (int c = 0; c < 32; ++c) acc[c] = 0.0f;
    float bsum[4] = {0.0f, 0.0f, 0.0f, 0.0f};     // column sums of dY (bias gradient) over this warp's rows: columns lane + 32 i
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(RT_KT >> 3) << 17) | ((uint32_t)(RT_NT >> 4) << 24) |
                           (MNM ? ((1u << 15) | (1u << 16)) : 0u);       // bits 15 / 16: A / B operand MN-major
    bool fresh = true;                                // the next MMA overwrites the TMEM accumulators
    constexpr int NSTAGE = MNM == 2 ? RT_NS : 2;
    auto fold = [&](int j) {                          // all MMAs up to block j -> register accumulators
        mbar_wait(&st_bar[j % NSTAGE], (uint32_t)((j / NSTAGE) & 1));
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        uint32_t d1[32], d2[32];
        const uint32_t tl = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(half * 32);
        tmem_ld32_nowait(tl, d1);
        tmem_ld32_nowait(tl + RT_KT, d2);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int c = 0; c < 32; ++c) acc[c] += __uint_as_float(d1[c]) + __uint_as_float(d2[c]);
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    };

    if (MNM == 2) {
        // ---- asynchronous pipeline: the raw fp32 rows of block j + RT_AHEAD are requested with cp.async (16-byte pieces,
        //      zero fill past the edges) straight into the hi tiles of a free stage; when block j's own pieces have landed
        //      the thread that requested them rounds them to TF32 in place and writes the remainders into the lo tiles.
        float4 bs4 = make_float4(0.f, 0.f, 0.f, 0.f);
        auto add4 = [&](const float4 &v) { bs4.x += v.x; bs4.y += v.y; bs4.z += v.z; bs4.w += v.w; };
        auto issue_dy = [&](uint8_t *dst, int64_t m, int n) {              // dY[m, n .. n+3] -> dst
            if (m < me && n < p.Nout) {
                const float *src = p.dY + m * p.ldy + n;
                if (y_vec && n + 4 <= p.Nout) { cp_async16(dst, src); return; }
#pragma unroll
                for (int e = 0; e < 4; ++e) cp_async4(dst + 4 * e, n + e < p.Nout ? src + e : p.dY, n + e < p.Nout ? 4 : 0);
            } else cp_async16(dst, p.dY, 0);
        };
        auto issue_a = [&](uint8_t *dst, int64_t m, int k) {               // A[m, k .. k+3] through the fused loaders -> dst
            if (!(m < me && k < p.K)) { cp_async16(dst, p.dY, 0); return; }
            if (AK == A_DENSE) {
                if (m < p.shift) { cp_async16(dst, p.dY, 0); return; }
                const float *src = p.A + (m - p.shift) * p.lda + k;
                if (a_vec && k + 4 <= p.K) { cp_async16(dst, src); return; }
#pragma unroll
                for (int e = 0; e < 4; ++e) cp_async4(dst + 4 * e, k + e < p.K ? src + e : p.dY, k + e < p.K ? 4 : 0);
            } else if (AK == A_STATE) {
                int b, t;
                if (fast_ok) fast_divmod((int)m, bv.T, invT, b, t);
                else { b = (int)((unsigned)m / (unsigned)bv.T); t = (int)m - b * bv.T; }
                const float *src = field_ptr<float>(bv.state, b, t + p.shift) + k;
                if (s_vec && k + 4 <= p.K) { cp_async16(dst, src); return; }
#pragma unroll
                for (int e = 0; e < 4; ++e) cp_async4(dst + 4 * e, k + e < p.K ? src + e : p.dY, k + e < p.K ? 4 : 0);
            } else {   // [obs | last-action one-hot | agent-id one-hot]
                int t, rr, b, n;
                if (fast_ok) { fast_divmod((int)m, bv.R, invR, t, rr); fast_divmod(rr, bv.N, invN, b, n); }
                else { t = (int)((unsigned)m / (unsigned)bv.R); rr = (int)m - t * bv.R; b = rr / bv.N; n = rr - b * bv.N; }
                const float *ob = field_ptr<float>(bv.obs, b, t) + (int64_t)n * bv.OBS;
                if (o_vec && k + 4 <= bv.OBS) { cp_async16(dst, ob + k); return; }
                const float *oh = t > 0 ? field_ptr<float>(bv.onehot, b, t - 1) + (int64_t)n * bv.A : nullptr;
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int kk = k + e;
                    if (kk < bv.OBS) cp_async4(dst + 4 * e, ob + kk);
                    else if (kk < bv.OBS + bv.in.last) cp_async4(dst + 4 * e, oh ? oh + (kk - bv.OBS) : p.dY, oh ? 4 : 0);
                    else *reinterpret_cast<float *>(dst + 4 * e) = (kk < p.K && kk - bv.OBS - bv.in.last == n) ? 1.0f : 0.0f;   // computed, not loaded
                }
            }
        };
        auto stage_base = [&](int j) { return rt_smem + (size_t)(j % RT_NS) * RT_STAGE; };
        auto issue_block = [&](int j) {
            uint8_t *Ah = stage_base(j), *Bh = Ah + 2 * RT_OP_A;
            const int64_t mm = mb + (int64_t)j * RT_BM;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int kr = 4 * warp + i;
                uint8_t *dst = Ah + (uint32_t)(lane >> 3) * RT_SLAB + mn_off(kr, lane & 7);
                if (SWAP) issue_a(dst, mm + kr, k0 + 4 * lane); else issue_dy(dst, mm + kr, n0 + 4 * lane);
            }
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int kr = 4 * warp + 2 * i + (lane >> 4), c = lane & 15;
                uint8_t *dst = Bh + (uint32_t)(c >> 3) * RT_SLAB + mn_off(kr, c & 7);
                if (SWAP) issue_dy(dst, mm + kr, n0 + 4 * c); else issue_a(dst, mm + kr, k0 + 4 * c);
            }
        };
#pragma unroll
        for (int jj = 0; jj < RT_AHEAD; ++jj) {
            if (jj < nblk) issue_block(jj);
            cp_async_commit();
        }
        for (int j = 0; j < nblk; ++j) {
            const int s = j % RT_NS;
            uint8_t *Ah = stage_base(j), *Al = Ah + RT_OP_A, *Bh = Al + RT_OP_A, *Bl = Bh + RT_OP_B;
            const int ja = j + RT_AHEAD;
            if (ja < nblk) {
                if (ja >= RT_NS) mbar_wait(&st_bar[ja % RT_NS], (uint32_t)(((ja / RT_NS) - 1) & 1));   // the MMAs of block ja - RT_NS released that stage
                issue_block(ja);
            }
            cp_async_commit();
            cp_async_wait<RT_AHEAD>();                                       // this thread's pieces of block j have landed
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int kr = 4 * warp + i;
                const uint32_t off = (uint32_t)(lane >> 3) * RT_SLAB + mn_off(kr, lane & 7);
                const float4 v = *reinterpret_cast<const float4 *>(Ah + off);
                if (!SWAP) add4(v);
                split_store_fast(Ah, Al, off, v);
            }
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int kr = 4 * warp + 2 * i + (lane >> 4), c = lane & 15;
                const uint32_t off = (uint32_t)(c >> 3) * RT_SLAB + mn_off(kr, c & 7);
                const float4 v = *reinterpret_cast<const float4 *>(Bh + off);
                if (SWAP) add4(v);
                split_store_fast(Bh, Bl, off, v);
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncthreads();
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (tid == 0) {
                const uint64_t dAh = umma_desc_mn_sw128(smem_u32(Ah), RT_SLAB), dAl = umma_desc_mn_sw128(smem_u32(Al), RT_SLAB);
                const uint64_t dBh = umma_desc_mn_sw128(smem_u32(Bh), RT_SLAB), dBl = umma_desc_mn_sw128(smem_u32(Bl), RT_SLAB);
#pragma unroll
                for (int ks = 0; ks < RT_BM / 8; ++ks) {
                    const uint64_t o = (uint64_t)((ks * 1024) >> 4);
                    const uint32_t first = (fresh && ks == 0) ? 0u : 1u;
                    umma_tf32(tmem_base, dAh + o, dBh + o, idesc, first);
                    umma_tf32(tmem_base + RT_KT, dAl + o, dBh + o, idesc, first);
                    umma_tf32(tmem_base + RT_KT, dAh + o, dBl + o, idesc, 1u);
                }
                umma_commit(&st_bar[s]);
            }
            fresh = false;
            if ((j % RT_FLUSH) == RT_FLUSH - 1 || j == nblk - 1) {
                fold(j);
                fresh = true;
            }
        }
        if (SWAP) {
            bs4.x += __shfl_xor_sync(0xffffffffu, bs4.x, 16); bs4.y += __shfl_xor_sync(0xffffffffu, bs4.y, 16);
            bs4.z += __shfl_xor_sync(0xffffffffu, bs4.z, 16); bs4.w += __shfl_xor_sync(0xffffffffu, bs4.w, 16);
        }
        if (want_bias && (!SWAP || lane < 16)) *reinterpret_cast<float4 *>(&bsum_s[warp][4 * lane]) = bs4;
    } else if (MNM) {
        float4 bs4 = make_float4(0.f, 0.f, 0.f, 0.f);     // column sums of dY over this thread's rows: columns 4 lane .. +3 (wide) / 4 (lane & 15) .. +3 (narrow)
        auto add4 = [&](const float4 &v) { bs4.x += v.x; bs4.y += v.y; bs4.z += v.z; bs4.w += v.w; };
        auto body = [&](int j, float4 (&cy)[4], float4 (&ca)[2], float4 (&ny)[4], float4 (&na)[2]) {
            const int s = j & 1;
            uint8_t *Ah = rt_smem + (size_t)s * RT_STAGE, *Al = Ah + RT_OP_A, *Bh = Al + RT_OP_A, *Bl = Bh + RT_OP_B;
            if (j + 1 < nblk) load_block_into(j + 1, ny, na);                    // flies under the staging + MMAs of block j
            if (j >= 2) mbar_wait(&st_bar[s], (uint32_t)(((j - 2) >> 1) & 1));   // the MMAs of block j-2 released this stage
#pragma unroll
            for (int i = 0; i < 4; ++i) {                                        // wide operand: row m = 4 warp + i, columns 4 lane .. +3
                const int kr = 4 * warp + i;
                if (!SWAP) add4(cy[i]);
                split_store_fast(Ah, Al, (uint32_t)(lane >> 3) * RT_SLAB + mn_off(kr, lane & 7), cy[i]);
            }
#pragma unroll
            for (int i = 0; i < 2; ++i) {                                        // narrow operand: rows 4 warp + 2 i + (lane >> 4)
                const int kr = 4 * warp + 2 * i + (lane >> 4), c = lane & 15;
                if (SWAP) add4(ca[i]);
                split_store_fast(Bh, Bl, (uint32_t)(c >> 3) * RT_SLAB + mn_off(kr, c & 7), ca[i]);
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncthreads();
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (tid == 0) {
                const uint64_t dAh = umma_desc_mn_sw128(smem_u32(Ah), RT_SLAB), dAl = umma_desc_mn_sw128(smem_u32(Al), RT_SLAB);
                const uint64_t dBh = umma_desc_mn_sw128(smem_u32(Bh), RT_SLAB), dBl = umma_desc_mn_sw128(smem_u32(Bl), RT_SLAB);
#pragma unroll
                for (int ks = 0; ks < RT_BM / 8; ++ks) {
                    const uint64_t o = (uint64_t)((ks * 1024) >> 4);             // eight m rows = one atom further
                    const uint32_t first = (fresh && ks == 0) ? 0u : 1u;
                    umma_tf32(tmem_base, dAh + o, dBh + o, idesc, first);
                    umma_tf32(tmem_base + RT_KT, dAl + o, dBh + o, idesc, first);
                    umma_tf32(tmem_base + RT_KT, dAh + o, dBl + o, idesc, 1u);
                }
                umma_commit(&st_bar[s]);
            }
            fresh = false;
            if ((j % RT_FLUSH) == RT_FLUSH - 1 || j == nblk - 1) {
                fold(j);
                fresh = true;
            }
        };
        if (nblk > 0) load_block_into(0, py, pa);
        for (int j = 0; j < nblk; j += 2) {
            body(j, py, pa, qy, qa);
            if (j + 1 < nblk) body(j + 1, qy, qa, py, pa);
        }
        if (SWAP) {                                       // lanes c and c + 16 hold the same narrow columns
            bs4.x += __shfl_xor_sync(0xffffffffu, bs4.x, 16); bs4.y += __shfl_xor_sync(0xffffffffu, bs4.y, 16);
            bs4.z += __shfl_xor_sync(0xffffffffu, bs4.z, 16); bs4.w += __shfl_xor_sync(0xffffffffu, bs4.w, 16);
        }
        if (want_bias && (!SWAP || lane < 16)) *reinterpret_cast<float4 *>(&bsum_s[warp][4 * lane]) = bs4;
    } else {
        if (nblk > 0) load_block(0);
        for (int j = 0; j < nblk; ++j) {
            const int s = j & 1;
            uint8_t *Ah = rt_smem + (size_t)s * RT_STAGE, *Al = Ah + RT_OP_A, *Bh = Al + RT_OP_A, *Bl = Bh + RT_OP_B;
            // ---- raw rows (coalesced) -> the warp's private scratch; only this warp reads them back: __syncwarp suffices
            float *ry = rawY + warp * (4 * RT_NT), *ra = rawA + warp * (4 * RT_KT);
    #pragma unroll
            for (int i = 0; i < 4; ++i) reinterpret_cast<float4 *>(ry)[i * 32 + lane] = py[i];
    #pragma unroll
            for (int i = 0; i < 2; ++i) reinterpret_cast<float4 *>(ra)[(2 * i + (lane >> 4)) * 16 + (lane & 15)] = pa[i];
            __syncwarp();
            if (j + 1 < nblk) load_block(j + 1);                             // flies under the transposition + MMAs
            if (j >= 2) mbar_wait(&st_bar[s], (uint32_t)(((j - 2) >> 1) & 1));   // the MMAs of block j-2 released this stage
            // ---- transpose + split: the warp's four rows are 16-byte piece `warp` of every operand row
    #pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int n = lane + 32 * i;
                const float4 v = make_float4(ry[n], ry[RT_NT + n], ry[2 * RT_NT + n], ry[3 * RT_NT + n]);
                if (!SWAP) bsum[i] += (v.x + v.y) + (v.z + v.w);
                split_store_fast(Ah, Al, (uint32_t)n * 128u + (uint32_t)((warp ^ (n & 7)) << 4), v);
            }
    #pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int k = lane + 32 * i;
                const float4 v = make_float4(ra[k], ra[RT_KT + k], ra[2 * RT_KT + k], ra[3 * RT_KT + k]);
                if (SWAP) bsum[i] += (v.x + v.y) + (v.z + v.w);
                split_store_fast(Bh, Bl, (uint32_t)k * 128u + (uint32_t)((warp ^ (k & 7)) << 4), v);
            }
            __syncwarp();                                                    // scratch is rewritten by the next block
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncthreads();
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (tid == 0) {
                const uint64_t dAh = umma_desc_sw128(smem_u32(Ah)), dAl = umma_desc_sw128(smem_u32(Al));
                const uint64_t dBh = umma_desc_sw128(smem_u32(Bh)), dBl = umma_desc_sw128(smem_u32(Bl));
    #pragma unroll
                for (int ks = 0; ks < RT_BM / 8; ++ks) {
                    const uint64_t o = (uint64_t)((ks * 32) >> 4);
                    const uint32_t first = (fresh && ks == 0) ? 0u : 1u;
                    umma_tf32(tmem_base, dAh + o, dBh + o, idesc, first);
                    umma_tf32(tmem_base + RT_KT, dAl + o, dBh + o, idesc, first);
                    umma_tf32(tmem_base + RT_KT, dAh + o, dBl + o, idesc, 1u);
                }
                umma_commit(&st_bar[s]);
            }
            fresh = false;
            if ((j % RT_FLUSH) == RT_FLUSH - 1 || j == nblk - 1) {
                fold(j);
                fresh = true;
            }
        }
    }
    // ---- partials: partW[chunk][n][k]; TMEM lane = wide-operand row, columns = narrow-operand rows
    if (!SWAP) {
        const int n = n0 + q * 32 + lane;
        if (n < p.Nout) {
            float *pw = p.partW + ((int64_t)chunk * p.Nout + n) * p.K + k0 + half * 32;
#pragma unroll
            for (int c = 0; c < 32; ++c)
                if (k0 + half * 32 + c < p.K) pw[c] = acc[c];
        }
    } else {
        const int k = k0 + q * 32 + lane;
        if (k < p.K) {
#pragma unroll
            for (int c = 0; c < 32; ++c) {
                const int n = n0 + half * 32 + c;
                if (n < p.Nout) p.partW[((int64_t)chunk * p.Nout + n) * p.K + k] = acc[c];
            }
        }
    }
    if (want_bias) {
        if (!MNM) {
#pragma unroll
            for (int i = 0; i < 4; ++i) bsum_s[warp][lane + 32 * i] = bsum[i];
        }
        __syncthreads();
        if (tid < (SWAP ? RT_KT : RT_NT) && n0 + tid < p.Nout) {
            float sacc = 0.0f;
#pragma unroll
            for (int w = 0; w < 8; ++w) sacc += bsum_s[w][tid];
            p.partB[(int64_t)chunk * p.Nout + n0 + tid] = sacc;
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(128u));
}

// =====================================================================================================================
// k_reduce_tc3: the MN-major pipeline (MNM = 2 above) rebuilt around what its profile showed (profiles/
// r02_reduce_notes.txt): with 8 warps per SM the kernel was bound by INSTRUCTION ISSUE of two warps per sub-partition --
// ~380 instructions per warp and 32-row block (cvt.rna.tf32 expands to ~5 instructions, 64-bit address arithmetic and
// multi-way branches in the loaders), one instruction every ~4 cycles per warp, 2 470 cycles per block against 384 cycles of
// MMA and a shared-memory / DRAM time well below that.  Here:
//   * 512 threads (4 warps per sub-partition): a thread owns 2 + 1 sixteen-byte pieces per block instead of 4 + 2;
//   * everything that does not change from block to block is computed once: piece offsets, column validity, the vector /
//     scalar decision of a piece, and for plain row-major operands the global pointer, which then advances by a constant;
//   * the common pieces are ONE predicated cp.async (or a 16-byte zero store); the TF32 split is 2 integer + 1 FADD per value.
// Same stages, descriptors, MMA order, fold cadence and partial layout as k_reduce_tc<.., 2>.
// =====================================================================================================================
#define RT3_THREADS 512
#define RT3_WARPS 16

__device__ __forceinline__ void cp_async16_plain(void *smem_dst, const void *gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async4_plain(void *smem_dst, const void *gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}

template <int AK, int SWAP>
__global__ void __launch_bounds__(RT3_THREADS, 1) k_reduce_tc3(const __grid_constant__ RedGroup g) {
    extern __shared__ __align__(1024) uint8_t rt_smem[];
    __shared__ __align__(8) uint64_t st_bar[RT_NS];
    __shared__ uint32_t tmem_base_s;
    __shared__ __align__(16) float bsum_s[RT3_WARPS][RT_NT];
    int pi = 0;
    while (pi + 1 < g.n && (int)blockIdx.y >= g.p[pi + 1].tile0) ++pi;
    const RedProb &p = g.p[pi];
    const BatchView &bv = g.bv;
    const int chunk = blockIdx.x;
    if (chunk >= p.n_chunks) return;
    const int tile = blockIdx.y - p.tile0;
    const int n_narrow = SWAP ? (p.Nout + RT_KT - 1) / RT_KT : p.n_ktiles;
    const int wt = tile / n_narrow, st_ = tile - wt * n_narrow;
    const int n0 = SWAP ? st_ * RT_KT : wt * RT_NT;      // first dY column of this tile
    const int k0 = SWAP ? wt * RT_NT : st_ * RT_KT;      // first A column of this tile
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t mb = p.M0 + (int64_t)chunk * p.rows_per_chunk;
    int64_t me = mb + p.rows_per_chunk;
    if (me > p.M) me = p.M;
    const int nblk = me > mb ? (int)((me - mb + RT_BM - 1) / RT_BM) : 0;
    const bool want_bias = p.partB && (SWAP ? wt == 0 : st_ == 0);

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(128u));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < RT_NS; ++i) mbar_init(&st_bar[i], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = tmem_base_s;
    pdl_wait();

    // ---- this thread's three pieces: wide rows 2 warp, 2 warp + 1 (piece = lane), narrow row 2 warp + (lane >> 4) (piece = lane & 15)
    const int cw = (SWAP ? k0 : n0) + 4 * lane;          // first column of the wide pieces (A column if SWAP, else dY column)
    const int cn = (SWAP ? n0 : k0) + 4 * (lane & 15);   // first column of the narrow piece
    const int krn = 2 * warp + (lane >> 4);
    const uint32_t offw0 = (uint32_t)(lane >> 3) * RT_SLAB + mn_off(2 * warp, lane & 7);
    const uint32_t offw1 = (uint32_t)(lane >> 3) * RT_SLAB + mn_off(2 * warp + 1, lane & 7);
    const uint32_t offn = (uint32_t)((lane & 15) >> 3) * RT_SLAB + mn_off(krn, lane & 7);
    // per-piece class: 0 = always zero (column past the edge), 1 = one 16-byte copy, 2 = element-wise assembly
    const bool y_vec = ((p.ldy & 3) == 0) && ((p.Nout & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.dY) & 15) == 0);
    auto a_class = [&](int k) -> int {
        if (k >= p.K) return 0;
        if (AK == A_DENSE) return (((p.lda & 3) == 0) && ((p.K & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.A) & 15) == 0)) ? 1 : 2;
        if (AK == A_STATE) return ((bv.state.sb & 3) == 0 && (bv.state.st & 3) == 0 && (p.K & 3) == 0 &&
                                   ((reinterpret_cast<uintptr_t>(bv.state.ptr) & 15) == 0)) ? 1 : 2;
        return ((bv.OBS & 3) == 0 && (bv.obs.sb & 3) == 0 && (bv.obs.st & 3) == 0 && ((reinterpret_cast<uintptr_t>(bv.obs.ptr) & 15) == 0) &&
                k + 4 <= bv.OBS) ? 1 : 2;
    };
    auto y_class = [&](int nn) -> int { return nn >= p.Nout ? 0 : (y_vec ? 1 : 2); };
    const int cls_w = SWAP ? a_class(cw) : y_class(cw);
    const int cls_n = SWAP ? y_class(cn) : a_class(cn);
    const bool fast_ok = p.M < (1 << 24);
    const float invR = 1.0f / (float)(bv.R > 0 ? bv.R : 1), invN = 1.0f / (float)(bv.N > 0 ? bv.N : 1);
    const float invT = 1.0f / (float)(bv.T > 0 ? bv.T : 1);

    // source of dY[m, n ..] / A[m, k ..]; `ok` = the row exists (and, for shifted dense operands, has a predecessor)
    auto y_src = [&](int64_t m, int nn, bool &ok) -> const float * { ok = m < me; return p.dY + m * p.ldy + nn; };
    auto a_row = [&](int64_t m, bool &ok, int &agent, const float *&oh) -> const float * {   // row base (column 0)
        agent = 0; oh = nullptr;
        ok = m < me;
        const int64_t mc = ok ? m : mb;                                        // keep the address arithmetic in range
        if (AK == A_DENSE) { ok = ok && mc >= p.shift; return p.A + (mc >= p.shift ? mc - p.shift : 0) * p.lda; }
        if (AK == A_STATE) {
            int b, t;
            if (fast_ok) fast_divmod((int)mc, bv.T, invT, b, t);
            else { b = (int)((unsigned)mc / (unsigned)bv.T); t = (int)mc - b * bv.T; }
            return field_ptr<float>(bv.state, b, t + p.shift);
        }
        int t, rr, b, n;
        if (fast_ok) { fast_divmod((int)mc, bv.R, invR, t, rr); fast_divmod(rr, bv.N, invN, b, n); }
        else { t = (int)((unsigned)mc / (unsigned)bv.R); rr = (int)mc - t * bv.R; b = rr / bv.N; n = rr - b * bv.N; }
        agent = n;
        oh = t > 0 ? field_ptr<float>(bv.onehot, b, t - 1) + (int64_t)n * bv.A : nullptr;
        return field_ptr<float>(bv.obs, b, t) + (int64_t)n * bv.OBS;
    };
    auto zero16 = [&](uint8_t *dst) { *reinterpret_cast<float4 *>(dst) = make_float4(0.f, 0.f, 0.f, 0.f); };
    auto issue_y = [&](uint8_t *dst, int64_t m, int nn, int cls) {
        bool ok;
        const float *src = y_src(m, nn, ok);
        if (cls == 1 && ok) cp_async16_plain(dst, src);
        else if (cls == 2 && ok) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                if (nn + e < p.Nout) cp_async4_plain(dst + 4 * e, src + e); else *reinterpret_cast<float *>(dst + 4 * e) = 0.0f;
            }
        } else zero16(dst);
    };
    auto issue_a = [&](uint8_t *dst, int64_t m, int k, int cls) {
        bool ok; int agent; const float *oh;
        const float *src = a_row(m, ok, agent, oh);
        if (cls == 1 && ok) cp_async16_plain(dst, src + k);
        else if (cls == 2 && ok) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int kk = k + e;
                float *d = reinterpret_cast<float *>(dst + 4 * e);
                if (kk >= p.K) *d = 0.0f;
                else if (AK != A_AGENT_IN || kk < bv.OBS) cp_async4_plain(d, src + kk);
                else if (kk < bv.OBS + bv.in.last) { if (oh) cp_async4_plain(d, oh + (kk - bv.OBS)); else *d = 0.0f; }
                else *d = (kk - bv.OBS - bv.in.last == agent) ? 1.0f : 0.0f;         // agent-id one-hot: computed, not loaded
            }
        } else zero16(dst);
    };
    auto stage_base = [&](int j) { return rt_smem + (size_t)(j % RT_NS) * RT_STAGE; };
    auto issue_block = [&](int j) {
        uint8_t *Ah = stage_base(j), *Bh = Ah + 2 * RT_OP_A;
        const int64_t mm = mb + (int64_t)j * RT_BM;
        if (SWAP) {
            issue_a(Ah + offw0, mm + 2 * warp, cw, cls_w);
            issue_a(Ah + offw1, mm + 2 * warp + 1, cw, cls_w);
            issue_y(Bh + offn, mm + krn, cn, cls_n);
        } else {
            issue_y(Ah + offw0, mm + 2 * warp, cw, cls_w);
            issue_y(Ah + offw1, mm + 2 * warp + 1, cw, cls_w);
            issue_a(Bh + offn, mm + krn, cn, cls_n);
        }
    };

    const int q = warp & 3, cg = warp >> 2;             // accumulator ownership: TMEM lane quarter q, columns 16 cg .. +16
    float acc[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) acc[c] = 0.0f;
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(RT_KT >> 3) << 17) | ((uint32_t)(RT_NT >> 4) << 24);
    bool fresh = true;
    auto fold = [&](int j) {
        mbar_wait(&st_bar[j % RT_NS], (uint32_t)((j / RT_NS) & 1));
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        uint32_t d1[32], d2[32];
        const uint32_t tl = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(cg * 16);
        tmem_ld16_nowait(tl, d1);
        tmem_ld16_nowait(tl + RT_KT, d2);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int c = 0; c < 16; ++c) acc[c] += __uint_as_float(d1[c]) + __uint_as_float(d2[c]);
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    };
    float4 bs4 = make_float4(0.f, 0.f, 0.f, 0.f);       // column sums of dY over this thread's rows
    auto add4 = [&](const float4 &v) { bs4.x += v.x; bs4.y += v.y; bs4.z += v.z; bs4.w += v.w; };

#pragma unroll
    for (int jj = 0; jj < RT_AHEAD; ++jj) {
        if (jj < nblk) issue_block(jj);
        cp_async_commit();
    }
    for (int j = 0; j < nblk; ++j) {
        const int s = j % RT_NS;
        uint8_t *Ah = stage_base(j), *Al = Ah + RT_OP_A, *Bh = Al + RT_OP_A, *Bl = Bh + RT_OP_B;
        const int ja = j + RT_AHEAD;
        if (ja < nblk) {
            if (ja >= RT_NS) mbar_wait(&st_bar[ja % RT_NS], (uint32_t)(((ja / RT_NS) - 1) & 1));   // the MMAs of block ja - RT_NS released that stage
            issue_block(ja);
        }
        cp_async_commit();
        cp_async_wait<RT_AHEAD>();                       // this thread's pieces of block j have landed
        {
            const float4 v0 = *reinterpret_cast<const float4 *>(Ah + offw0);
            const float4 v1 = *reinterpret_cast<const float4 *>(Ah + offw1);
            const float4 v2 = *reinterpret_cast<const float4 *>(Bh + offn);
            if (!SWAP) { add4(v0); add4(v1); } else add4(v2);
            split_store_fast(Ah, Al, offw0, v0);
            split_store_fast(Ah, Al, offw1, v1);
            split_store_fast(Bh, Bl, offn, v2);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (tid == 0) {
            const uint64_t dAh = umma_desc_mn_sw128(smem_u32(Ah), RT_SLAB), dAl = umma_desc_mn_sw128(smem_u32(Al), RT_SLAB);
            const uint64_t dBh = umma_desc_mn_sw128(smem_u32(Bh), RT_SLAB), dBl = umma_desc_mn_sw128(smem_u32(Bl), RT_SLAB);
#pragma unroll
            for (int ks = 0; ks < RT_BM / 8; ++ks) {
                const uint64_t o = (uint64_t)((ks * 1024) >> 4);
                const uint32_t first = (fresh && ks == 0) ? 0u : 1u;
                umma_tf32(tmem_base, dAh + o, dBh + o, idesc, first);
                umma_tf32(tmem_base + RT_KT, dAl + o, dBh + o, idesc, first);
                umma_tf32(tmem_base + RT_KT, dAh + o, dBl + o, idesc, 1u);
            }
            umma_commit(&st_bar[s]);
        }
        fresh = false;
        if ((j % RT_FLUSH) == RT_FLUSH - 1 || j == nblk - 1) {
            fold(j);
            fresh = true;
        }
    }
    // ---- partials: partW[chunk][n][k]; TMEM lane = wide-operand row, columns = narrow-operand rows
    if (!SWAP) {
        const int n = n0 + q * 32 + lane;
        if (n < p.Nout) {
            float *pw = p.partW + ((int64_t)chunk * p.Nout + n) * p.K + k0 + cg * 16;
#pragma unroll
            for (int c = 0; c < 16; ++c)
                if (k0 + cg * 16 + c < p.K) pw[c] = acc[c];
        }
    } else {
        const int k = k0 + q * 32 + lane;
        if (k < p.K) {
#pragma unroll
            for (int c = 0; c < 16; ++c) {
                const int n = n0 + cg * 16 + c;
                if (n < p.Nout) p.partW[((int64_t)chunk * p.Nout + n) * p.K + k] = acc[c];
            }
        }
    }
    if (want_bias) {
        if (SWAP) {                                      // lanes c and c + 16 hold the same narrow columns
            bs4.x += __shfl_xor_sync(0xffffffffu, bs4.x, 16); bs4.y += __shfl_xor_sync(0xffffffffu, bs4.y, 16);
            bs4.z += __shfl_xor_sync(0xffffffffu, bs4.z, 16); bs4.w += __shfl_xor_sync(0xffffffffu, bs4.w, 16);
        }
        if (!SWAP || lane < 16) *reinterpret_cast<float4 *>(&bsum_s[warp][4 * lane]) = bs4;
        __syncthreads();
        if (tid < (SWAP ? RT_KT : RT_NT) && n0 + tid < p.Nout) {
            float sacc = 0.0f;
#pragma unroll
            for (int w = 0; w < RT3_WARPS; ++w) sacc += bsum_s[w][tid];
            p.partB[(int64_t)chunk * p.Nout + n0 + tid] = sacc;
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(128u));
}

// =====================================================================================================================
// k_reduce_gru: the W_ih / W_hh / b_ih / b_hh gradients of the GRU in ONE split-M GEMM per 32-row block,
//     D[128 x 256] += [x | h_{t-1}]^T [32 x 128]  .  d_g [32 x 256]          (d_g = d gi_r | d gi_z | d gi_n | d gh_n)
// instead of four 128 x 64 tiles on four CTAs.  The generic tiles above are bound by SHARED-MEMORY bandwidth, not by the
// tensor pipe or HBM (tools/mma_chain_probe.cu: an M128 x N64 x K8 TF32 MMA takes 53 cycles while reading 6 KB of operands,
// i.e. ~115 B/clk of the 128 B/clk an SM has, and every operand byte is also written and re-read once by the 3xTF32
// split); the fused shape reads 12 KB per 132-cycle MMA, stages d_g / x / h once instead of once per tile and touches every
// row from HBM exactly once.  Three quarters of D are used: x rows x (r, z, n) columns -> W_ih, h rows x (r, z) and
// x (gh_n) columns -> W_hh.
//   hi operands = the raw fp32 rows where cp.async lands them (the tensor core drops the 13 low mantissa bits itself),
//   lo operands = v - trunc(v), written by the thread that requested the piece; both biases this leaves (|lo| slightly
//   larger, lo.lo dropped) are proportional to every product with the same sign and factor (< 5e-7), i.e. a relative
//   error of the SUM of that size, immune to cancellation.
//   16-row blocks; smem: five hi stages (24 KB each: block j-1 still being read by the tensor core, block j, blocks j+1 .. j+3
//   landing) + two lo stages, so that block j is split while block j-1 is multiplied; TMEM: D1 | D2 = 256 + 256 columns.
// =====================================================================================================================
#define RG_BM 16                                         // rows (m) per block: two K = 8 MMA steps
#define RG_SLAB (RG_BM * 128)                            // 2 KB: [16 m rows x 32 columns]
#define RG_STAGE (12 * RG_SLAB)                          // 24 KB: xh (4 slabs) | d_g (8 slabs)
#define RG_NHI 5                                         // hi stages: block j (multiplied), j-1 (still being read), j+1 .. j+3 (landing)
#define RG_NLO 2
#define RG_AHEAD 3
#define RG_FLUSH 16                                      // blocks between TMEM -> register folds (256 rows)
#define RG_SMEM_BYTES ((RG_NHI + RG_NLO) * RG_STAGE)     // 168 KB
struct ReduceGruArgs {
    const float *x, *hout, *d_g;      // [M1, 64], [M1, 64] (h_t; h_{t-1} = row m - R, zero for m < R), [M1, 256]
    float *wih_w, *wih_b;             // [n_chunks][192][64], [n_chunks][192]
    float *whha_w, *whha_b;           // [n_chunks][128][64], [n_chunks][128]
    float *whhb_w, *whhb_b;           // [n_chunks][64][64],  [n_chunks][64]
    int64_t M1, rows_per_chunk;
    int n_chunks, R;
};

__global__ void __launch_bounds__(RT3_THREADS, 1) k_reduce_gru(const __grid_constant__ ReduceGruArgs a) {
    extern __shared__ __align__(1024) uint8_t rt_smem[];
    __shared__ __align__(8) uint64_t mma_bar[2];
    __shared__ uint32_t tmem_base_s;
    const int chunk = blockIdx.x;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t mb = (int64_t)chunk * a.rows_per_chunk;
    int64_t me = mb + a.rows_per_chunk;
    if (me > a.M1) me = a.M1;
    const int nblk = me > mb ? (int)((me - mb + RG_BM - 1) / RG_BM) : 0;
    uint8_t *lo_base = rt_smem + RG_NHI * RG_STAGE;

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(512u));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    if (tid == 0) {
        mbar_init(&mma_bar[0], 1);
        mbar_init(&mma_bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = tmem_base_s;
    pdl_wait();

    // ---- this thread's three pieces of a block: row `warp`; xh piece `lane` (x: lanes 0-15, h: 16-31), d_g pieces `lane`, `lane + 32`
    const uint32_t off_xh = (uint32_t)(lane >> 3) * RG_SLAB + mn_off(warp, lane & 7);
    const uint32_t off_g0 = (uint32_t)(4 + (lane >> 3)) * RG_SLAB + mn_off(warp, lane & 7);
    const uint32_t off_g1 = off_g0 + 4 * RG_SLAB;
    const bool is_h = lane >= 16;
    const float *src_xh = (is_h ? a.hout - (int64_t)a.R * HID : a.x) + (mb + warp) * HID + 4 * (lane & 15);
    const float *src_g = a.d_g + (mb + warp) * (4 * HID) + 4 * lane;
    int64_t m_next = mb + warp;                          // this thread's row of the next block to request
    auto zero16 = [&](uint8_t *dst) { *reinterpret_cast<float4 *>(dst) = make_float4(0.f, 0.f, 0.f, 0.f); };
    auto issue_block = [&](int j) {
        uint8_t *hi = rt_smem + (size_t)(j % RG_NHI) * RG_STAGE;
        const bool ok = m_next < me;
        if (ok && !(is_h && m_next < a.R)) cp_async16_plain(hi + off_xh, src_xh); else zero16(hi + off_xh);
        if (ok) {
            cp_async16_plain(hi + off_g0, src_g);
            cp_async16_plain(hi + off_g1, src_g + 2 * HID);
        } else { zero16(hi + off_g0); zero16(hi + off_g1); }
        m_next += RG_BM; src_xh += RG_BM * HID; src_g += RG_BM * 4 * HID;
    };

    const int q = warp & 3, cg = warp >> 2;              // TMEM lane quarter q (xh column 32 q + lane), d_g columns 64 cg .. +64
    float acc[64];
#pragma unroll
    for (int c = 0; c < 64; ++c) acc[c] = 0.0f;
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(256 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    bool fresh = true;
    auto wait_block = [&](int j) {                       // the MMAs of block j (and of every earlier block) are complete
        mbar_wait(&mma_bar[j & 1], (uint32_t)((j >> 1) & 1));
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    };
    auto fold = [&]() {                                  // TMEM -> register accumulators (16 columns at a time)
        const uint32_t tl = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(cg * 64);
#pragma unroll
        for (int h = 0; h < 4; ++h) {
            uint32_t d1[32], d2[32];
            tmem_ld16_nowait(tl + 16 * h, d1);
            tmem_ld16_nowait(tl + 256 + 16 * h, d2);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int c = 0; c < 16; ++c) acc[16 * h + c] += __uint_as_float(d1[c]) + __uint_as_float(d2[c]);
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    };
    float4 bs0 = make_float4(0.f, 0.f, 0.f, 0.f), bs1 = bs0;   // column sums of d_g: columns 4 lane .. +3 and 128 + 4 lane .. +3
    auto lo_of = [&](const float4 &v) {
        float4 l;
        l.x = v.x - __uint_as_float(__float_as_uint(v.x) & 0xFFFFE000u); l.y = v.y - __uint_as_float(__float_as_uint(v.y) & 0xFFFFE000u);
        l.z = v.z - __uint_as_float(__float_as_uint(v.z) & 0xFFFFE000u); l.w = v.w - __uint_as_float(__float_as_uint(v.w) & 0xFFFFE000u);
        return l;
    };

#pragma unroll
    for (int jj = 0; jj < RG_AHEAD; ++jj) {
        if (jj < nblk) issue_block(jj);
        cp_async_commit();
    }
    for (int j = 0; j < nblk; ++j) {
        uint8_t *hi = rt_smem + (size_t)(j % RG_NHI) * RG_STAGE;
        uint8_t *lo = lo_base + (size_t)(j & 1) * RG_STAGE;
        // block j-2 is done: its hi stage (the one block j+3 lands in) and this lo stage are free; the tensor pipe
        // still holds block j-1 while this block is split
        if (j >= 2) wait_block(j - 2);
        if (j + RG_AHEAD < nblk) issue_block(j + RG_AHEAD);
        cp_async_commit();
        cp_async_wait<RG_AHEAD>();                       // this thread's pieces of block j have landed
        {
            const float4 vx = *reinterpret_cast<const float4 *>(hi + off_xh);
            const float4 g0 = *reinterpret_cast<const float4 *>(hi + off_g0);
            const float4 g1 = *reinterpret_cast<const float4 *>(hi + off_g1);
            bs0.x += g0.x; bs0.y += g0.y; bs0.z += g0.z; bs0.w += g0.w;
            bs1.x += g1.x; bs1.y += g1.y; bs1.z += g1.z; bs1.w += g1.w;
            *reinterpret_cast<float4 *>(lo + off_xh) = lo_of(vx);
            *reinterpret_cast<float4 *>(lo + off_g0) = lo_of(g0);
            *reinterpret_cast<float4 *>(lo + off_g1) = lo_of(g1);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (tid == 0) {
            const uint64_t dAh = umma_desc_mn_sw128(smem_u32(hi), RG_SLAB), dAl = umma_desc_mn_sw128(smem_u32(lo), RG_SLAB);
            const uint64_t dBh = umma_desc_mn_sw128(smem_u32(hi + 4 * RG_SLAB), RG_SLAB), dBl = umma_desc_mn_sw128(smem_u32(lo + 4 * RG_SLAB), RG_SLAB);
#pragma unroll
            for (int ks = 0; ks < RG_BM / 8; ++ks) {
                const uint64_t o = (uint64_t)((ks * 1024) >> 4);
                const uint32_t first = (fresh && ks == 0) ? 0u : 1u;
                umma_tf32(tmem_base, dAh + o, dBh + o, idesc, first);
                umma_tf32(tmem_base + 256, dAl + o, dBh + o, idesc, first);
                umma_tf32(tmem_base + 256, dAh + o, dBl + o, idesc, 1u);
            }
            umma_commit(&mma_bar[j & 1]);
        }
        fresh = false;
        if ((j % RG_FLUSH) == RG_FLUSH - 1 && j + 1 < nblk) {   // the accumulation so far leaves the tensor core's truncating adder
            wait_block(j);
            fold();
            fresh = true;
        }
    }
    if (nblk > 0) { wait_block(nblk - 1); fold(); }
    // ---- partials.  TMEM lane = xh column: lanes 0-63 -> W_ih[n][k = lane], lanes 64-127 -> W_hh[n][k = lane - 64]
    {
        const int r = q * 32 + lane, k = r & 63;
        const bool hrow = r >= 64;
        float *dst = nullptr;                            // &part[chunk][n = first column of this warp's group][k]
        if (!hrow && cg < 3) dst = a.wih_w + ((int64_t)chunk * G3 + 64 * cg) * HID + k;
        else if (hrow && cg < 2) dst = a.whha_w + ((int64_t)chunk * 128 + 64 * cg) * HID + k;
        else if (hrow && cg == 3) dst = a.whhb_w + (int64_t)chunk * 64 * HID + k;
        if (dst) {
#pragma unroll
            for (int c = 0; c < 64; ++c) dst[(int64_t)c * HID] = acc[c];
        }
    }
    // ---- bias partials: column sums of d_g over the chunk (cross-warp sum through the free shared memory)
    __syncthreads();
    float *bsum = reinterpret_cast<float *>(rt_smem);    // [16 warps][256]
    *reinterpret_cast<float4 *>(bsum + warp * 256 + 4 * lane) = bs0;
    *reinterpret_cast<float4 *>(bsum + warp * 256 + 128 + 4 * lane) = bs1;
    __syncthreads();
    if (tid < 256) {
        float s = 0.0f;
#pragma unroll
        for (int w = 0; w < RT3_WARPS; ++w) s += bsum[w * 256 + tid];
        if (tid < G3) a.wih_b[(int64_t)chunk * G3 + tid] = s;
        if (tid < 128) a.whha_b[(int64_t)chunk * 128 + tid] = s;
        if (tid >= G3) a.whhb_b[(int64_t)chunk * 64 + tid - G3] = s;
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
}

// =====================================================================================================================
// k_reduce_fc1: the fc1 weight / bias gradient  dW1[n][k] = sum_m d_x[m][n] in[m][k]  (in = [obs | last-action one-hot |
// agent-id one-hot], never materialised) as ONE split-M GEMM per 16-row block and row chunk, built like k_reduce_gru:
//     D[256 x 64] += in^T [16 x 256]  .  d_x [16 x 64]            (two M = 128 halves when d_in > 128, N = 64)
// k_reduce_tc3 runs this problem as 128-column tiles on separate CTAs (d_x re-read per tile, 32-row blocks of 24 KB with
// three pieces per thread and two divisions per piece): 4.0 ms at 20v20 / B = 1024 = 16 % of the HBM peak.  Here one CTA
// owns a row chunk over the FULL input width: warp = row of the block, its (t, b, n) advance incrementally, a lane copies
// pieces `lane` and `lane + 32` of the input row (16-byte cp.async inside the obs part, 4-byte copies / computed values
// for the one-hot tail) and, lanes 0-15, one piece of the d_x row.  hi = the raw fp32 bits where they land, lo = v - trunc(v).
// TMEM: D1 halves at 0 | 64, D2 halves at 128 | 192.   smem: five hi + two lo stages of 20 KB.
// =====================================================================================================================
#define RF_STAGE (10 * RG_SLAB)                          // 20 KB: input (8 slabs of 32 columns) | d_x (2 slabs)
#define RF_SMEM_BYTES ((RG_NHI + RG_NLO) * RF_STAGE)     // 140 KB
struct ReduceFc1Args {
    const float *d_x;                 // [M, 64]
    float *partW, *partB;             // [n_chunks][64][d_in], [n_chunks][64]
    int64_t M, rows_per_chunk;
    int n_chunks, d_in;
    BatchView bv;
};

__global__ void __launch_bounds__(RT3_THREADS, 1) k_reduce_fc1(const __grid_constant__ ReduceFc1Args a) {
    extern __shared__ __align__(1024) uint8_t rt_smem[];
    __shared__ __align__(8) uint64_t mma_bar[2];
    __shared__ uint32_t tmem_base_s;
    const BatchView &bv = a.bv;
    const int chunk = blockIdx.x;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t mb = (int64_t)chunk * a.rows_per_chunk;
    int64_t me = mb + a.rows_per_chunk;
    if (me > a.M) me = a.M;
    const int nblk = me > mb ? (int)((me - mb + RG_BM - 1) / RG_BM) : 0;
    const int halves = a.d_in > 128 ? 2 : 1;
    uint8_t *lo_base = rt_smem + RG_NHI * RF_STAGE;

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(256u));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    if (tid == 0) {
        mbar_init(&mma_bar[0], 1);
        mbar_init(&mma_bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = tmem_base_s;

    // ---- this thread's pieces of a block: row `warp`; input pieces `lane` and `lane + 32`, d_x piece `lane` (lanes 0-15)
    const int KA = bv.OBS + bv.in.last;                  // first agent-id column (columns < d_in only)
    const bool obs_vec = (bv.OBS & 3) == 0 && (bv.obs.sb & 3) == 0 && (bv.obs.st & 3) == 0 && ((reinterpret_cast<uintptr_t>(bv.obs.ptr) & 15) == 0);
    uint32_t off_in[2];
    int col_in[2], cls_in[2];                            // class 0: zero, 1: one 16-byte copy from the obs row, 2: element-wise
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int pc = lane + 32 * h;
        off_in[h] = (uint32_t)(pc >> 3) * RG_SLAB + mn_off(warp, pc & 7);
        col_in[h] = 4 * pc;
        cls_in[h] = col_in[h] >= a.d_in ? 0 : ((obs_vec && col_in[h] + 4 <= bv.OBS) ? 1 : 2);
    }
    const uint32_t off_dx = (uint32_t)(8 + ((lane & 15) >> 3)) * RG_SLAB + mn_off(warp, lane & 7);
    const bool has_dx = lane < 16;
    // row bookkeeping: m = mb + warp + 16 j  ->  (t, b, n), advanced incrementally
    int64_t m_next = mb + warp;
    int t_, b_, n_, rr_;
    {
        const int64_t mc = m_next < a.M ? m_next : 0;
        t_ = (int)(mc / bv.R); rr_ = (int)(mc - (int64_t)t_ * bv.R); b_ = rr_ / bv.N; n_ = rr_ - b_ * bv.N;
    }
    const int q16 = RG_BM / bv.N, r16 = RG_BM - q16 * bv.N;
    const float *src_dx = a.d_x + (mb + warp) * HID + 4 * (lane & 15);
    auto zero16 = [&](uint8_t *dst) { *reinterpret_cast<float4 *>(dst) = make_float4(0.f, 0.f, 0.f, 0.f); };
    auto issue_block = [&](int j) {
        uint8_t *hi = rt_smem + (size_t)(j % RG_NHI) * RF_STAGE;
        const bool ok = m_next < me;
        const float *obs = field_ptr<float>(bv.obs, b_, t_) + (int64_t)n_ * bv.OBS;
        const float *oh = t_ > 0 ? field_ptr<float>(bv.onehot, b_, t_ - 1) + (int64_t)n_ * bv.A : nullptr;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            uint8_t *dst = hi + off_in[h];
            if (h >= halves) break;
            if (!ok || cls_in[h] == 0) zero16(dst);
            else if (cls_in[h] == 1) cp_async16_plain(dst, obs + col_in[h]);
            else {
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int kk = col_in[h] + e;
                    float *d = reinterpret_cast<float *>(dst + 4 * e);
                    if (kk < bv.OBS) cp_async4_plain(d, obs + kk);
                    else if (kk < KA) { if (oh) cp_async4_plain(d, oh + (kk - bv.OBS)); else *d = 0.0f; }
                    else *d = (kk < a.d_in && kk - KA == n_) ? 1.0f : 0.0f;      // agent-id one-hot: computed, not loaded
                }
            }
        }
        if (has_dx) { if (ok) cp_async16_plain(hi + off_dx, src_dx); else zero16(hi + off_dx); }
        // next block: row + 16
        m_next += RG_BM; src_dx += RG_BM * HID;
        rr_ += RG_BM; b_ += q16; n_ += r16;
        if (n_ >= bv.N) { n_ -= bv.N; ++b_; }
        if (rr_ >= bv.R) {
            do { rr_ -= bv.R; ++t_; } while (rr_ >= bv.R);
            b_ = rr_ / bv.N; n_ = rr_ - b_ * bv.N;
        }
    };

    const int q = warp & 3, cg = warp >> 2;              // TMEM lane quarter q (input column 32 q + lane of a half), d_x columns 16 cg .. +16
    float acc[2][16];
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int c = 0; c < 16; ++c) acc[h][c] = 0.0f;
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(64 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    bool fresh = true;
    auto wait_block = [&](int j) {
        mbar_wait(&mma_bar[j & 1], (uint32_t)((j >> 1) & 1));
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    };
    auto fold = [&]() {
        const uint32_t tl = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(cg * 16);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            if (h >= halves) break;
            uint32_t d1[32], d2[32];
            tmem_ld16_nowait(tl + 64 * h, d1);
            tmem_ld16_nowait(tl + 128 + 64 * h, d2);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int c = 0; c < 16; ++c) acc[h][c] += __uint_as_float(d1[c]) + __uint_as_float(d2[c]);
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    };
    float4 bs = make_float4(0.f, 0.f, 0.f, 0.f);         // column sums of d_x: columns 4 lane .. +3 (lanes 0-15)
    auto lo_of = [&](const float4 &v) {
        float4 l;
        l.x = v.x - __uint_as_float(__float_as_uint(v.x) & 0xFFFFE000u); l.y = v.y - __uint_as_float(__float_as_uint(v.y) & 0xFFFFE000u);
        l.z = v.z - __uint_as_float(__float_as_uint(v.z) & 0xFFFFE000u); l.w = v.w - __uint_as_float(__float_as_uint(v.w) & 0xFFFFE000u);
        return l;
    };

    pdl_wait();                                          // d_x comes from the stream predecessor (the dx GEMM)
#pragma unroll
    for (int jj = 0; jj < RG_AHEAD; ++jj) {
        if (jj < nblk) issue_block(jj);
        cp_async_commit();
    }
    for (int j = 0; j < nblk; ++j) {
        uint8_t *hi = rt_smem + (size_t)(j % RG_NHI) * RF_STAGE;
        uint8_t *lo = lo_base + (size_t)(j & 1) * RF_STAGE;
        if (j + 1 == nblk) pdl_trigger();                // the gradient gather may start its prologue
        if (j >= 2) wait_block(j - 2);                   // frees the hi stage block j+3 lands in and this lo stage
        if (j + RG_AHEAD < nblk) issue_block(j + RG_AHEAD);
        cp_async_commit();
        cp_async_wait<RG_AHEAD>();                       // this thread's pieces of block j have landed
        {
            const float4 v0 = *reinterpret_cast<const float4 *>(hi + off_in[0]);
            *reinterpret_cast<float4 *>(lo + off_in[0]) = lo_of(v0);
            if (halves > 1) {
                const float4 v1 = *reinterpret_cast<const float4 *>(hi + off_in[1]);
                *reinterpret_cast<float4 *>(lo + off_in[1]) = lo_of(v1);
            }
            if (has_dx) {
                const float4 g = *reinterpret_cast<const float4 *>(hi + off_dx);
                bs.x += g.x; bs.y += g.y; bs.z += g.z; bs.w += g.w;
                *reinterpret_cast<float4 *>(lo + off_dx) = lo_of(g);
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (tid == 0) {
            const uint64_t dBh = umma_desc_mn_sw128(smem_u32(hi + 8 * RG_SLAB), RG_SLAB), dBl = umma_desc_mn_sw128(smem_u32(lo + 8 * RG_SLAB), RG_SLAB);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                if (h >= halves) break;
                const uint64_t dAh = umma_desc_mn_sw128(smem_u32(hi + h * 4 * RG_SLAB), RG_SLAB), dAl = umma_desc_mn_sw128(smem_u32(lo + h * 4 * RG_SLAB), RG_SLAB);
#pragma unroll
                for (int ks = 0; ks < RG_BM / 8; ++ks) {
                    const uint64_t o = (uint64_t)((ks * 1024) >> 4);
                    const uint32_t first = (fresh && ks == 0) ? 0u : 1u;
                    umma_tf32(tmem_base + 64 * h, dAh + o, dBh + o, idesc, first);
                    umma_tf32(tmem_base + 128 + 64 * h, dAl + o, dBh + o, idesc, first);
                    umma_tf32(tmem_base + 128 + 64 * h, dAh + o, dBl + o, idesc, 1u);
                }
            }
            umma_commit(&mma_bar[j & 1]);
        }
        fresh = false;
        if ((j % RG_FLUSH) == RG_FLUSH - 1 && j + 1 < nblk) {   // the accumulation so far leaves the tensor core's truncating adder
            wait_block(j);
            fold();
            fresh = true;
        }
    }
    if (nblk > 0) { wait_block(nblk - 1); fold(); }
    // ---- partials: partW[chunk][n][k]; TMEM lane = input column k of a half, accumulator column = n
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int k = 128 * h + q * 32 + lane;
        if (h < halves && k < a.d_in) {
            float *dst = a.partW + ((int64_t)chunk * HID + cg * 16) * a.d_in + k;
#pragma unroll
            for (int c = 0; c < 16; ++c) dst[(int64_t)c * a.d_in] = acc[h][c];
        }
    }
    // ---- bias partials: column sums of d_x over the chunk
    __syncthreads();
    float *bsum = reinterpret_cast<float *>(rt_smem);    // [16 warps][64]
    if (has_dx) *reinterpret_cast<float4 *>(bsum + warp * HID + 4 * lane) = bs;
    __syncthreads();
    if (tid < HID) {
        float s = 0.0f;
#pragma unroll
        for (int w = 0; w < RT3_WARPS; ++w) s += bsum[w * HID + tid];
        a.partB[(int64_t)chunk * HID + tid] = s;
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(256u));
}
