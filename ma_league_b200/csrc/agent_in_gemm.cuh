// Fused agent-input projection:  gi = W_ih relu(fc1([obs | onehot(a_{t-1}) | agent id])) + b_ih  for all (t, b, n) rows of
// both nets, in ONE launch (basic_controller.py:80-92 + drqn_agent.py:30-31 + the W_ih half of GRUCell).
//
// Same 3xTF32 tcgen05 building blocks as tc_gemm.cuh; what the fusion buys on top of two k_linear_tc launches:
//   * x = relu(fc1(.)) goes from the first accumulator (TMEM) through registers straight into the A-operand staging of
//     the second MMA -- it is written to global once (the backward needs it) and never read back;
//   * one kernel skeleton (launch, TMEM allocation, weight staging, pipeline fill) instead of two, and one M-tile walk;
//   * W_ih (192 x 64, hi + lo = 96 KB) stays resident in shared memory, N = 192 is a single MMA.
// One persistent CTA per SM and net: 256 threads, M tiles of 128 rows.
//   TMEM (512 columns): fc1 D1 | D2 at 0 | 64, W_ih D1 | D2 at 128 | 320.
//   smem: A staging (input chunk, later x; hi + lo = 64 KB, reused as the epilogue's transposition scratch) |
//         W_fc1 chunk slot(s) (hi + lo = 32 KB each: one when the input fits a 64-wide chunk, else two) | W_ih (96 KB).
// Inputs wider than one chunk (10v10: 2, 20v20: 4 chunks) are software-pipelined: right after a chunk's MMAs are issued
// the next chunk's rows are requested into registers and its fc1 weight chunk is staged into the other slot, so both
// fly under the MMAs; with two chunks both stay resident for the whole kernel.
#pragma once
#include "tc_gemm.cuh"

#define AI_SLAB_A (TC_M * 128)            // 16 KB: [128 rows x 32 floats]
#define AI_SLAB_W1 (HID * 128)            //  8 KB: [64 rows x 32 floats]
#define AI_SLAB_W2 (G3 * 128)             // 24 KB: [192 rows x 32 floats]
#define AI_OFF_W1 (4 * AI_SLAB_A)
#define AI_W1_SLOT (4 * AI_SLAB_W1)                    // one fc1 weight chunk, hi + lo: 32 KB
// one fc1 chunk slot when the input fits one 64-wide chunk, two when it does not (the next chunk is staged under the MMA)
__host__ __device__ inline int ai_w1_slots(int K1) { return K1 > TC_KC ? 2 : 1; }
__host__ __device__ inline size_t ai_smem_bytes(int K1) { return AI_OFF_W1 + (size_t)ai_w1_slots(K1) * AI_W1_SLOT + 4 * AI_SLAB_W2; }   // 192 / 224 KB
#define AI_THREADS 512                    // 16 warps: four per sub-partition hide the load / TMEM / shared-memory latencies of the staging and epilogue phases (r2: 256 threads left ~20 K of a tile's 23 K cycles to those phases)
#define AI_RSTEP (AI_THREADS / 16)        // rows between two staging pieces of a thread (32)
#define AI_RPT (TC_M / AI_RSTEP)          // staging rows per thread (4)
#define AI_REM_MAX 4                      // widest K remainder handled in the epilogue instead of an extra k-chunk
#define AI_COL_X1 0
#define AI_COL_X2 64
#define AI_COL_G1 128
#define AI_COL_G2 320

struct AgentInArgs {
    const float *params[2];    // online, target flat agent buffers
    float *x[2];               // [M1, 64]
    float *gi[2];              // [M1, 192]
    int64_t M1;
    int64_t m_begin, m_end;    // row range of this launch (time-chunked forward: rows of t in [t0, t1))
    int d_in, n_actions;
    int gi_tiled;              // 1: gi leaves as gi_tiled[m / 32][chunk 0..47][m % 32][4] for k_gru_fwd_tc (R % 32 == 0)
    BatchView bv;
};

// DEFAULT_IN: the input layout is [obs | last action | agent id] (both switches on), compiled in; otherwise the column
// bounds come from a.bv.in at run time.  A template parameter rather than a branch: the kernel sits at its register cap
// (128 at 512 threads), and the default instance keeps the exact code of the fixed layout (DESIGN.md section 4).
template <bool DEFAULT_IN>
__global__ void __launch_bounds__(AI_THREADS, 1) k_agent_in_tc(const __grid_constant__ AgentInArgs a) {
    extern __shared__ __align__(1024) uint8_t tc_smem[];
    __shared__ __align__(8) uint64_t mma_bar;
    __shared__ uint32_t tmem_base_s;
    __shared__ __align__(16) float b1_s[HID], bih_s[G3];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, net = blockIdx.y;
    const AgentLayout L = agent_layout(a.d_in, a.n_actions);
    const float *P = a.params[net];
    const int64_t M = a.m_end;                          // rows >= m_end belong to another launch
    const int n_mtiles = (int)((a.m_end - a.m_begin + TC_M - 1) / TC_M);
    if ((int)blockIdx.x >= n_mtiles) return;
    const BatchView &bv = a.bv;
    const int K1f = bv.OBS + (DEFAULT_IN ? bv.A : bv.in.last);   // the agent-id columns are a bias gather in the epilogue
    const bool has_id = DEFAULT_IN || bv.in.id;
    // A short remainder past the last full 64-column chunk (20v20: 194 = 3 x 64 + 2) would cost a whole extra load / stage /
    // MMA / wait round for a handful of columns: those columns (of the one-hot part) join the agent-id term as rank-1
    // updates in epilogue 1 instead, and the MMA runs over K1 = the full chunks only.  Obs columns never do: without the
    // last-action block K1f = OBS, and the remainder rule requires K1 >= OBS.
    const int rem1 = (K1f > TC_KC && (K1f % TC_KC) != 0 && (K1f % TC_KC) <= AI_REM_MAX && K1f - (K1f % TC_KC) >= bv.OBS) ? K1f % TC_KC : 0;
    const int K1 = K1f - rem1;
    const int nkc1 = (K1 + TC_KC - 1) / TC_KC;
    const bool two_slots = ai_w1_slots(K1f) == 2;
    uint8_t *A_hi = tc_smem, *A_lo = tc_smem + 2 * AI_SLAB_A;
    uint8_t *W1_base = tc_smem + AI_OFF_W1;             // slot s: hi at + s * AI_W1_SLOT, lo 2 slabs further
    uint8_t *W2_hi = W1_base + (two_slots ? 2 : 1) * AI_W1_SLOT, *W2_lo = W2_hi + 2 * AI_SLAB_W2;

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(512u));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    if (tid == 0) {
        mbar_init(&mma_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (tid < HID) b1_s[tid] = __ldg(P + L.fc1_b + tid);
    // tiled mode (tensor-core recurrence): the r / z halves of b_hh ride along, only b_hh_n is applied inside the recurrence
    if (tid < G3) bih_s[tid] = __ldg(P + L.b_ih + tid) + ((a.gi_tiled && tid < 2 * HID) ? __ldg(P + L.b_hh + tid) : 0.0f);
    const int c4 = tid & 15, rbase = tid >> 4;          // staging map: float4 column c4 of a 64-wide chunk, rows rbase + AI_RSTEP i
    const uint32_t a_slab = (uint32_t)(c4 >> 3) * AI_SLAB_A;
    // W_ih [192 x 64], resident for the whole kernel (all twelve loads of a thread in flight before the first split)
    {
        float4 wv[G3 / AI_RSTEP];
#pragma unroll
        for (int i = 0; i < G3 / AI_RSTEP; ++i)
            wv[i] = __ldg(reinterpret_cast<const float4 *>(P + L.w_ih + (int64_t)(rbase + AI_RSTEP * i) * HID + 4 * c4));
#pragma unroll
        for (int i = 0; i < G3 / AI_RSTEP; ++i) {
            const int j = rbase + AI_RSTEP * i;
            split_store_fast(W2_hi, W2_lo, (uint32_t)(c4 >> 3) * AI_SLAB_W2 + (uint32_t)j * 128u + (uint32_t)(((c4 & 7) ^ (j & 7)) << 4), wv[i]);
        }
    }
    auto stage_w1 = [&](int kc, int slot) {             // fc1.weight[:, kc*64 .. +64) (columns >= K1 are zero)
        uint8_t *W1_hi = W1_base + slot * AI_W1_SLOT, *W1_lo = W1_hi + 2 * AI_SLAB_W1;
        const int kcol = kc * TC_KC + 4 * c4;
        float4 wv[HID / AI_RSTEP];
#pragma unroll
        for (int i = 0; i < HID / AI_RSTEP; ++i) {
            const float *wr = P + L.fc1_w + (int64_t)(rbase + AI_RSTEP * i) * a.d_in + kcol;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (kcol < K1) v.x = __ldg(wr);             // d_in is not a multiple of 4 in general: scalar loads
            if (kcol + 1 < K1) v.y = __ldg(wr + 1);
            if (kcol + 2 < K1) v.z = __ldg(wr + 2);
            if (kcol + 3 < K1) v.w = __ldg(wr + 3);
            wv[i] = v;
        }
#pragma unroll
        for (int i = 0; i < HID / AI_RSTEP; ++i) {
            const int j = rbase + AI_RSTEP * i;
            split_store_fast(W1_hi, W1_lo, (uint32_t)(c4 >> 3) * AI_SLAB_W1 + (uint32_t)j * 128u + (uint32_t)(((c4 & 7) ^ (j & 7)) << 4), wv[i]);
        }
    };
    int slot_chunk0 = -1, slot_chunk1 = -1;             // fc1 chunk held by each slot
    int step = 0;                                       // running (tile, chunk) counter: slot = step & 1 with two slots
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = tmem_base_s;
    uint32_t bar_phase = 0;
    const float invR = 1.0f / (float)bv.R, invN = 1.0f / (float)bv.N;

    const int q16 = AI_RSTEP / bv.N, r16 = AI_RSTEP - q16 * bv.N;   // a thread's rows are AI_RSTEP apart: (t, b, n) advance incrementally
    auto load_in = [&](int64_t m0, int kc, float4 (&v)[AI_RPT]) {   // [obs | last-action one-hot] rows, float4 over the obs part
        const int kcol = kc * TC_KC + 4 * c4;
        int t, rr, b, n;
        fast_divmod((int)m0 + rbase, bv.R, invR, t, rr);
        fast_divmod(rr, bv.N, invN, b, n);
#pragma unroll
        for (int i = 0; i < AI_RPT; ++i) {
            const int64_t m = m0 + rbase + AI_RSTEP * i;
            v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i > 0) {                                // row m = row (m - AI_RSTEP) + AI_RSTEP
                rr += AI_RSTEP; b += q16; n += r16;
                while (n >= bv.N) { n -= bv.N; ++b; }
                if (rr >= bv.R) {                       // next timestep(s): rare, recompute (b, n)
                    do { rr -= bv.R; ++t; } while (rr >= bv.R);
                    fast_divmod(rr, bv.N, invN, b, n);
                }
            }
            if (m < M && kcol < K1) {
                if (kcol < bv.OBS) {                    // OBS % 4 == 0 (host-checked)
                    v[i] = __ldg(reinterpret_cast<const float4 *>(field_ptr<float>(bv.obs, b, t) + (int64_t)n * bv.OBS + kcol));
                } else if (t > 0) {
                    const float *oh = field_ptr<float>(bv.onehot, b, t - 1) + (int64_t)n * bv.A;
                    const int a0 = kcol - bv.OBS;
                    if (a0 < bv.A) v[i].x = __ldg(oh + a0);
                    if (a0 + 1 < bv.A) v[i].y = __ldg(oh + a0 + 1);
                    if (a0 + 2 < bv.A) v[i].z = __ldg(oh + a0 + 2);
                    if (a0 + 3 < bv.A) v[i].w = __ldg(oh + a0 + 3);
                }
            }
        }
    };
    auto wait_mma = [&]() {
        mbar_wait(&mma_bar, bar_phase);
        bar_phase ^= 1u;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    };
    const uint32_t idesc1 = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(HID >> 3) << 17) | ((uint32_t)(TC_M >> 4) << 24);
    const uint32_t idesc2 = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(G3 >> 3) << 17) | ((uint32_t)(TC_M >> 4) << 24);

    float4 pre[AI_RPT];
    bool have_pre = false;
    for (int mt = blockIdx.x; mt < n_mtiles; mt += gridDim.x) {
        const int64_t m0 = a.m_begin + (int64_t)mt * TC_M;
        if (mt + (int)gridDim.x >= n_mtiles) pdl_trigger();   // last tile of this CTA: the recurrence may be scheduled and load W_hh
        // ---------------------------------------------------------------- x = fc1(input): nkc1 k-chunks into acc 1
        for (int kc = 0; kc < nkc1; ++kc) {
            float4 v[AI_RPT];
            if (have_pre) {
#pragma unroll
                for (int i = 0; i < AI_RPT; ++i) v[i] = pre[i];
            } else {
                load_in(m0, kc, v);
            }
#pragma unroll
            for (int i = 0; i < AI_RPT; ++i) {
                const int r = rbase + AI_RSTEP * i;
                split_store_fast(A_hi, A_lo, a_slab + (uint32_t)r * 128u + (uint32_t)(((c4 & 7) ^ (r & 7)) << 4), v[i]);
            }
            const int sl = two_slots ? (step & 1) : 0;
            if ((sl ? slot_chunk1 : slot_chunk0) != kc) {   // first chunks of the kernel, or the single-slot layout
                stage_w1(kc, sl);
                if (sl) slot_chunk1 = kc; else slot_chunk0 = kc;
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncthreads();
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (tid == 0) {
                const uint8_t *W1_hi = W1_base + sl * AI_W1_SLOT, *W1_lo = W1_hi + 2 * AI_SLAB_W1;
                const uint64_t dA_hi = umma_desc_sw128(smem_u32(A_hi)), dA_lo = umma_desc_sw128(smem_u32(A_lo));
                const uint64_t dW_hi = umma_desc_sw128(smem_u32(W1_hi)), dW_lo = umma_desc_sw128(smem_u32(W1_lo));
                const int k0 = kc * TC_KC;
                const int ksteps = ((K1 - k0 < TC_KC ? K1 - k0 : TC_KC) + 7) / 8;
#pragma unroll
                for (int ks = 0; ks < TC_KC / 8; ++ks) {
                    if (ks < ksteps) {
                        const uint64_t ao = (uint64_t)(((ks >> 2) * AI_SLAB_A + (ks & 3) * 32) >> 4);
                        const uint64_t wo = (uint64_t)(((ks >> 2) * AI_SLAB_W1 + (ks & 3) * 32) >> 4);
                        const uint32_t first = (kc == 0 && ks == 0) ? 0u : 1u;
                        umma_tf32(tmem_base + AI_COL_X1, dA_hi + ao, dW_hi + wo, idesc1, first);
                        umma_tf32(tmem_base + AI_COL_X2, dA_lo + ao, dW_hi + wo, idesc1, first);
                        umma_tf32(tmem_base + AI_COL_X2, dA_hi + ao, dW_lo + wo, idesc1, 1u);
                    }
                }
                umma_commit(&mma_bar);
            }
            // The next chunk in sequence (this tile's kc + 1, else the next tile's first) is requested now: its rows fly
            // under this chunk's MMAs (and, for a tile's last chunk, under the rest of the tile), and with two slots
            // its fc1 weight chunk is staged into the slot the previous chunk's MMAs have released.
            {
                const bool same_tile = kc + 1 < nkc1;
                const bool next_tile = mt + (int)gridDim.x < n_mtiles;
                have_pre = same_tile || next_tile;
                if (have_pre) {
                    const int kcn = same_tile ? kc + 1 : 0;
                    load_in(same_tile ? m0 : a.m_begin + (int64_t)(mt + (int)gridDim.x) * TC_M, kcn, pre);
                    if (two_slots) {
                        const int nsl = (step + 1) & 1;
                        if ((nsl ? slot_chunk1 : slot_chunk0) != kcn) {
                            stage_w1(kcn, nsl);
                            if (nsl) slot_chunk1 = kcn; else slot_chunk0 = kcn;
                        }
                    }
                }
            }
            ++step;
            wait_mma();
        }
        // ---------------------------------------------------------------- epilogue 1: x = relu(. + b1 + W1[:, K1 + agent])
        // lane = row (TMEM lane quarter warp & 3); warp group warp >> 2 takes columns 16 (warp >> 2) .. +16.  x goes to global
        // (backward) and, split hi/lo, into the A staging of the second MMA (the input chunk there is consumed).
        {
            const int q = warp & 3, cgp = warp >> 2;
            const int r = q * 32 + lane;
            const int64_t m = m0 + r;
            uint32_t d1[32], d2[32];
            const uint32_t tl = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(cgp * 16);
            tmem_ld16_nowait(tl + AI_COL_X1, d1);
            tmem_ld16_nowait(tl + AI_COL_X2, d2);
            int agent = 0, t_r = 0, b_r = 0;
            if (m < M) { int rr; fast_divmod((int)m, bv.R, invR, t_r, rr); fast_divmod(rr, bv.N, invN, b_r, agent); }
            const float *wid = P + L.fc1_w + K1f + agent;         // fc1.weight[n, K1f + agent] (when has_id)
            float wa[16];
#pragma unroll
            for (int e = 0; e < 16; ++e) wa[e] = has_id ? __ldg(wid + (int64_t)(cgp * 16 + e) * a.d_in) : 0.0f;   // in flight under the TMEM load
            if (rem1 > 0) {                                       // remainder columns K1 .. K1f-1 (one-hot part): x += in[k] W1[n, k]
                const float *oh = (m < M && t_r > 0) ? field_ptr<float>(bv.onehot, b_r, t_r - 1) + (int64_t)agent * bv.A + (K1 - bv.OBS) : nullptr;
#pragma unroll
                for (int j = 0; j < AI_REM_MAX; ++j) {
                    if (j < rem1) {
                        const float v = oh ? __ldg(oh + j) : 0.0f;
                        const float *wr = P + L.fc1_w + K1 + j;
#pragma unroll
                        for (int e = 0; e < 16; ++e) wa[e] = fmaf(v, __ldg(wr + (int64_t)(cgp * 16 + e) * a.d_in), wa[e]);
                    }
                }
            }
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            float *xrow = a.x[net] + m * HID + cgp * 16;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                float4 xv;
                float *xp = &xv.x;
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int n = cgp * 16 + 4 * c + e;
                    const float s = (__uint_as_float(d1[4 * c + e]) + __uint_as_float(d2[4 * c + e])) + b1_s[n] + wa[4 * c + e];
                    xp[e] = m < M ? fmaxf(s, 0.0f) : 0.0f;
                }
                if (m < M) *reinterpret_cast<float4 *>(xrow + 4 * c) = xv;
                const int cc = cgp * 4 + c;                       // 16-byte chunk of the 64-float row: slab cc >> 3
                split_store_fast(A_hi, A_lo, (uint32_t)(cc >> 3) * AI_SLAB_A + (uint32_t)r * 128u + (uint32_t)(((cc & 7) ^ (r & 7)) << 4), xv);
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        // ---------------------------------------------------------------- gi = W_ih x: one N = 192 MMA chain into acc 2
        if (tid == 0) {
            const uint64_t dA_hi = umma_desc_sw128(smem_u32(A_hi)), dA_lo = umma_desc_sw128(smem_u32(A_lo));
            const uint64_t dW_hi = umma_desc_sw128(smem_u32(W2_hi)), dW_lo = umma_desc_sw128(smem_u32(W2_lo));
#pragma unroll
            for (int ks = 0; ks < TC_KC / 8; ++ks) {
                const uint64_t ao = (uint64_t)(((ks >> 2) * AI_SLAB_A + (ks & 3) * 32) >> 4);
                const uint64_t wo = (uint64_t)(((ks >> 2) * AI_SLAB_W2 + (ks & 3) * 32) >> 4);
                const uint32_t first = ks == 0 ? 0u : 1u;
                umma_tf32(tmem_base + AI_COL_G1, dA_hi + ao, dW_hi + wo, idesc2, first);
                umma_tf32(tmem_base + AI_COL_G2, dA_lo + ao, dW_hi + wo, idesc2, first);
                umma_tf32(tmem_base + AI_COL_G2, dA_hi + ao, dW_lo + wo, idesc2, 1u);
            }
            umma_commit(&mma_bar);
        }
        wait_mma();
        // ---------------------------------------------------------------- epilogue 2: gi = . + b_ih
        if (a.gi_tiled) {
            // tiled layout for the tensor-core recurrence: TMEM lane = row = position inside the 32-row group, so every
            // float4 chunk of the warp is one contiguous 512-byte store -- no transposition
            const int q = warp & 3;
            const int64_t m = m0 + q * 32 + lane;
            const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16);
            float4 *gt = reinterpret_cast<float4 *>(a.gi[net]) + (m >> 5) * (int64_t)(G3 / 4) * 32 + (m & 31);
#pragma unroll 1
            for (int c0 = (warp >> 2) * 16; c0 < G3; c0 += 64) {
                uint32_t d1[32], d2[32];
                tmem_ld16_nowait(tlane + (uint32_t)(AI_COL_G1 + c0), d1);
                tmem_ld16_nowait(tlane + (uint32_t)(AI_COL_G2 + c0), d2);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (m < M) {
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const float4 b4 = *reinterpret_cast<const float4 *>(&bih_s[c0 + 4 * c]);
                        gt[((c0 >> 2) + c) * 32] =
                            make_float4((__uint_as_float(d1[4 * c]) + __uint_as_float(d2[4 * c])) + b4.x,
                                        (__uint_as_float(d1[4 * c + 1]) + __uint_as_float(d2[4 * c + 1])) + b4.y,
                                        (__uint_as_float(d1[4 * c + 2]) + __uint_as_float(d2[4 * c + 2])) + b4.z,
                                        (__uint_as_float(d1[4 * c + 3]) + __uint_as_float(d2[4 * c + 3])) + b4.w);
                    }
                }
            }
        } else {
            const int q = warp & 3;
            const int64_t mw = m0 + q * 32;
            const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16);
            float4 *stg = reinterpret_cast<float4 *>(A_hi) + warp * 256;      // the x operand is consumed: 4 KB per warp (16 warps = the 64 KB of A staging)
            TcEpi e;
            e.Y = a.gi[net]; e.aux = nullptr; e.W = nullptr; e.ldy = G3; e.ld_aux = 0; e.ldw = 0;
            e.M = (int)M; e.Nout = G3; e.K = 0; e.R = bv.R; e.N = bv.N; e.relu = false; e.vec_ok = true;
#pragma unroll 1
            for (int c0 = (warp >> 2) * 16; c0 < G3; c0 += 64) {
                uint32_t d1[32], d2[32];
                tmem_ld16_nowait(tlane + (uint32_t)(AI_COL_G1 + c0), d1);
                tmem_ld16_nowait(tlane + (uint32_t)(AI_COL_G2 + c0), d2);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                tc_epilogue_group<TCE_BIAS_ACT>(e, stg, d1, d2, 16, c0, mw, lane, bih_s, false);
            }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    }
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
}
