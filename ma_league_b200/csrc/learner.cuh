// K0-K8: the QLearner.train step (marl/learners/q_learner.py:34-131) as hand-written sm_100a kernels.
//
// Decomposition (cuDNN-RNN style, but fp32-exact and fused around the reference's glue ops):
//   * everything that does NOT depend on h_{t-1} is hoisted out of the time loop into grouped panel GEMMs over
//     all (t, b, n) rows at once:  x = relu(fc1 [obs | last action | agent id]),  gi = W_ih x + b_ih;
//   * the serial part (gh = W_hh h, gate math) runs in a lean recurrence kernel that keeps W_hh in REGISTERS
//     (one gate row per thread) and h in shared memory: 2 barriers per timestep, no weight traffic at all;
//   * q = fc2 h, the chosen-action gather and the avail-masked (double-Q) target max are one warp-per-row epilogue;
//   * the QMIX hypernetworks are two grouped panel GEMMs; abs/bmm/ELU/bmm + TD error + masked loss + the whole
//     element-wise part of the mixer backward are ONE warp-per-(b,t) kernel;
//   * BPTT mirrors the forward: a reverse recurrence with W_hh^T in registers emits d(gates); all weight
//     gradients are split-M reductions (deterministic two-pass: per-chunk partials, then a flat gather);
//   * clip_grad_norm_ + RMSprop are one pass over the flat parameter / gradient / square_avg buffers.
#pragma once
#include "mal_common.cuh"

// =============================================================================================
// Data-parallel exchange fused with the optimiser prologue (SURVEY.md 8e): every rank reads the un-normalised gradient
// of ALL ranks straight out of their symmetric (peer-mapped) buffers over NVLink, sums in rank order (so every rank gets
// bit-identical values), divides by the global mask sum -- itself the rank-order sum of one tail element -- writes the
// normalised gradient to its LOCAL buffer and leaves the per-block sums of squares for the clip.  One-shot all-reduce:
// 0.6 MB per rank at 20v20, latency-bound, so every rank pulling W x its share beats a ring; no NCCL call on the path.
// =============================================================================================
#define PEER_MAX 16
struct PeerBufs {
    const float *p[PEER_MAX];   // rank r's [n_total + tail] buffer (peer pointers from the symmetric-memory rendezvous)
    int world;
};

__global__ void __launch_bounds__(256) k_peer_allreduce_grad(const __grid_constant__ PeerBufs peers, int64_t n_total, int tail,
                                                             float *grad_out, float *tail_out, float *norm_part,
                                                             int64_t n_frozen) {
    __shared__ float s_sq[8];
    const int64_t p = (int64_t)blockIdx.x * 256 + threadIdx.x;
    float denom = 0.0f;
    for (int r = 0; r < peers.world; ++r) denom += __ldcg(peers.p[r] + n_total + 4);      // global mask.sum()
    float v = 0.0f;
    if (p < n_total) {
        if (p >= n_frozen) {                       // frozen prefix (freeze_agent_weights): no gradient, not in the norm
            for (int r = 0; r < peers.world; ++r) v += __ldcg(peers.p[r] + p);
            v = v / denom;
        }
        grad_out[p] = v;
    }
    if (blockIdx.x == 0 && threadIdx.x < tail) {
        float t = 0.0f;
        for (int r = 0; r < peers.world; ++r) t += __ldcg(peers.p[r] + n_total + threadIdx.x);
        tail_out[threadIdx.x] = t;
    }
    const float sq = warp_sum(v * v);
    if ((threadIdx.x & 31) == 0) s_sq[threadIdx.x >> 5] = sq;
    __syncthreads();
    if (threadIdx.x == 0) {
        float sacc = 0;
        for (int w = 0; w < 8; ++w) sacc += s_sq[w];
        norm_part[blockIdx.x] = sacc;
    }
}

// =============================================================================================
// row loaders shared by the panel GEMM and the split reduction
// =============================================================================================
struct BatchView {
    int B, TT, T, N, A, OBS, S, R;
    mal_field_t obs, onehot, state, actions;
    AgentInput in;        // column layout of the A_AGENT_IN rows
};

enum { A_DENSE = 0, A_AGENT_IN = 1, A_STATE = 2 };

struct RowSrc {           // resolved per row
    const float *p0;      // dense row / obs row / state row
    const float *p1;      // last-action one-hot row (may be null)
    int agent;
};

__device__ __forceinline__ RowSrc resolve_row(int kind, const BatchView &bv, const float *A, int64_t lda, int shift,
                                              int64_t m) {
    RowSrc r;
    r.p1 = nullptr;
    r.agent = 0;
    if (kind == A_DENSE) {
        r.p0 = A + (m - shift) * lda;   // shift = row shift (h_{t-1} pairing); callers guard m >= shift
    } else if (kind == A_AGENT_IN) {
        int t = (int)((unsigned)m / (unsigned)bv.R), rr = (int)m - t * bv.R;   // rows < 2^31
        int b = rr / bv.N, n = rr - b * bv.N;
        r.agent = n;
        r.p0 = field_ptr<float>(bv.obs, b, t) + (int64_t)n * bv.OBS;
        r.p1 = t > 0 ? field_ptr<float>(bv.onehot, b, t - 1) + (int64_t)n * bv.A : nullptr;
    } else {
        int b = (int)((unsigned)m / (unsigned)bv.T), t = (int)m - b * bv.T;
        r.p0 = field_ptr<float>(bv.state, b, t + shift);
    }
    return r;
}

// element k < d_in of the logical input row; for A_AGENT_IN: [obs | last-action one-hot | agent-id one-hot] (bv.in)
__device__ __forceinline__ float row_elem(int kind, const BatchView &bv, const RowSrc &r, int k) {
    if (kind != A_AGENT_IN) return r.p0[k];
    if (k < bv.OBS) return r.p0[k];
    k -= bv.OBS;
    if (k < bv.in.last) return r.p1 ? r.p1[k] : 0.0f;
    return (k - bv.in.last) == r.agent ? 1.0f : 0.0f;
}

// =============================================================================================
// grouped panel GEMM:  Y[m, n] = epi( sum_k A[m,k] * W[n,k] )      (tile 64x64, 256 threads, 4x4 micro-tile)
// =============================================================================================
enum { EPI_BIAS = 0, EPI_RELU = 1, EPI_MASKPOS = 2, EPI_FC1 = 3 };

struct LinProb {
    int M, K, Nout;
    int a_kind, shift;
    const float *A; int64_t lda;
    const float *W; int64_t ldw; int w_trans;     // w_trans: W(n,k) = W[k*ldw + n]
    const float *bias;
    int epi;
    const float *aux; int64_t ld_aux;             // EPI_MASKPOS: multiply by (aux[m,n] > 0)
    float *Y; int64_t ldy;
};
#define LIN_MAX_PROBS 20   // 20v20 hypernet layer 2: 2 nets x (8 + 1) column pieces of <= 80 (kernel parameter block: 20 x 112 B + view < 4 KB)
struct LinGroup {
    int n;
    int dbg;   // probe switches of k_linear_tc2 (0 in production): 1 no epilogue stores, 2 no A loads, 4 no A split/STS, 8 no MMAs
    LinProb p[LIN_MAX_PROBS];
    BatchView bv;
};

#define LIN_TM 64
#define LIN_TN 64
#define LIN_KC 64
#define LIN_LDW (LIN_KC + 4)

__global__ void __launch_bounds__(256) k_linear_group(const __grid_constant__ LinGroup g) {
    extern __shared__ __align__(16) float lin_smem[];
    const LinProb &p = g.p[blockIdx.y];
    const int64_t m0 = (int64_t)blockIdx.x * LIN_TM;
    if (m0 >= p.M) return;
    const int nkc = (p.K + LIN_KC - 1) / LIN_KC;
    const int KA = nkc * LIN_KC + 4;
    float *A_s = lin_smem;                 // [64][KA]
    float *W_s = lin_smem + LIN_TM * KA;   // [64][68]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int ty = tid >> 4, tx = tid & 15;

    // ---- stage the whole A row-panel once (zero padded)
    for (int r = warp; r < LIN_TM; r += 8) {
        const int64_t m = m0 + r;
        float *dst = A_s + r * KA;
        if (m < p.M) {
            RowSrc rs = resolve_row(p.a_kind, g.bv, p.A, p.lda, p.shift, m);
            for (int k = lane; k < nkc * LIN_KC; k += 32) dst[k] = k < p.K ? row_elem(p.a_kind, g.bv, rs, k) : 0.0f;
        } else {
            for (int k = lane; k < nkc * LIN_KC; k += 32) dst[k] = 0.0f;
        }
    }

    for (int n0 = 0; n0 < p.Nout; n0 += LIN_TN) {
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
        for (int kc = 0; kc < nkc; ++kc) {
            const int k0 = kc * LIN_KC;
            __syncthreads();   // previous W chunk fully consumed (and A panel staged on the first pass)
#pragma unroll 4
            for (int q = 0; q < (LIN_TN * LIN_KC) / 256; ++q) {
                int idx = tid + 256 * q;
                int j, kk;
                if (!p.w_trans) { j = idx >> 6; kk = idx & 63; } else { j = idx & 63; kk = idx >> 6; }
                int n = n0 + j, k = k0 + kk;
                float v = 0.0f;
                if (n < p.Nout && k < p.K) v = p.w_trans ? __ldg(p.W + (int64_t)k * p.ldw + n) : __ldg(p.W + (int64_t)n * p.ldw + k);
                W_s[j * LIN_LDW + kk] = v;
            }
            __syncthreads();
            const float *a_base = A_s + ty * KA + k0;
            const float *w_base = W_s + tx * LIN_LDW;
#pragma unroll 4
            for (int k4 = 0; k4 < LIN_KC / 4; ++k4) {
                float4 av[4], wv[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) av[i] = *reinterpret_cast<const float4 *>(a_base + i * 16 * KA + 4 * k4);
#pragma unroll
                for (int j = 0; j < 4; ++j) wv[j] = *reinterpret_cast<const float4 *>(w_base + j * 16 * LIN_LDW + 4 * k4);
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        acc[i][j] = fmaf(av[i].x, wv[j].x, acc[i][j]);
                        acc[i][j] = fmaf(av[i].y, wv[j].y, acc[i][j]);
                        acc[i][j] = fmaf(av[i].z, wv[j].z, acc[i][j]);
                        acc[i][j] = fmaf(av[i].w, wv[j].w, acc[i][j]);
                    }
            }
        }
        // ---- epilogue
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int64_t m = m0 + ty + 16 * i;
            if (m >= p.M) continue;
            int agent = 0;
            if (p.epi == EPI_FC1) agent = (int)((m % g.bv.R) % g.bv.N);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int n = n0 + tx + 16 * j;
                if (n >= p.Nout) continue;
                float v = acc[i][j];
                if (p.bias) v += __ldg(p.bias + n);
                if (p.epi == EPI_FC1) { v += __ldg(p.W + (int64_t)n * p.ldw + p.K + agent); v = fmaxf(v, 0.0f); }
                else if (p.epi == EPI_RELU) v = fmaxf(v, 0.0f);
                else if (p.epi == EPI_MASKPOS) v = (p.aux[m * p.ld_aux + n] > 0.0f) ? v : 0.0f;
                p.Y[m * p.ldy + n] = v;
            }
        }
    }
}

// =============================================================================================
// grouped split-M reduction:  part[c][n][k] = sum_{m in chunk c} dY[m,n] * A[m,k] ;  partB[c][n] = sum dY[m,n]
// =============================================================================================
struct RedProb {
    int64_t M0, M;            // rows [M0, M)
    int K, Nout;
    const float *dY; int64_t ldy;
    int dy_kind;              // 0: dense dY[m*ldy + n];  1: one-hot(action[m]) * d_chosen[m]  (fc2 / gather backward)
    int a_kind, shift;
    const float *A; int64_t lda;
    float *partW, *partB;     // [n_chunks][Nout][K], [n_chunks][Nout] (partB may be null)
    int n_chunks; int64_t rows_per_chunk;
    int tile0, n_ktiles;      // first tile id of this problem, number of k tiles
};
#define RED_MAX_PROBS 12
struct RedGroup {
    int n;
    RedProb p[RED_MAX_PROBS];
    BatchView bv;
};
#define RED_MR 64
#define RED_LD 68
#define RED_EPT (RED_MR * 64 / 256)   // elements of each operand a thread stages per block (16)

// AK: loader of the A operand (A_DENSE / A_STATE / A_AGENT_IN); DK: dY kind (0 dense, 1 one-hot(action) * d_chosen).
// Specialised so that each instance is straight-line code: all 32 staging loads of a thread issue back to back.
template <int AK, int DK>
__global__ void __launch_bounds__(256) k_reduce_group(const __grid_constant__ RedGroup g) {
    __shared__ __align__(16) float dY_s[RED_MR * RED_LD];
    __shared__ __align__(16) float A_s[RED_MR * RED_LD];
    int pi = 0;
    while (pi + 1 < g.n && (int)blockIdx.y >= g.p[pi + 1].tile0) ++pi;
    const RedProb p = g.p[pi];          // copy the descriptor to registers once
    const BatchView bv = g.bv;
    const int chunk = blockIdx.x;
    if (chunk >= p.n_chunks) return;
    const int tile = blockIdx.y - p.tile0;
    const int nt = tile / p.n_ktiles, kt = tile - nt * p.n_ktiles;
    const int n0 = nt * 64, k0 = kt * 64;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int ty = tid >> 4, tx = tid & 15;
    const int64_t mb = p.M0 + (int64_t)chunk * p.rows_per_chunk;
    int64_t me = mb + p.rows_per_chunk;
    if (me > p.M) me = p.M;
    const bool want_bias = p.partB && kt == 0;
    pdl_wait();

    float acc[4][4];
    float bsum[4] = {0, 0, 0, 0};
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;

    // staging map: warp w owns rows w, w+8, ... (8 rows per block), lane owns columns lane and lane+32
    const int c0 = lane, c1 = lane + 32;
    const bool n_ok0 = n0 + c0 < p.Nout, n_ok1 = n0 + c1 < p.Nout;
    const bool k_ok0 = k0 + c0 < p.K, k_ok1 = k0 + c1 < p.K;
    float rdy[RED_EPT], ra[RED_EPT];
    auto prefetch = [&](int64_t mm) {
#pragma unroll
        for (int u = 0; u < RED_MR / 8; ++u) {
            const int64_t m = mm + warp + 8 * u;
            const bool ok = m < me;
            // ---- dY
            if (DK == 0) {
                const float *dyp = p.dY + m * p.ldy + n0;
                rdy[2 * u] = (ok && n_ok0) ? __ldg(dyp + c0) : 0.0f;
                rdy[2 * u + 1] = (ok && n_ok1) ? __ldg(dyp + c1) : 0.0f;
            } else {   // row m = t*R + b*N + n of the [T*R] transition rows
                const int t = (int)((unsigned)m / (unsigned)bv.R), rr = (int)m - t * bv.R;   // rows < 2^31 (host-checked): 32-bit division
                const int b = rr / bv.N, n = rr - b * bv.N;
                float dsel = 0.0f;
                int asel = -1;
                if (ok) {
                    dsel = __ldg(p.dY + ((int64_t)b * bv.T + t) * bv.N + n);
                    asel = (int)(field_ptr<long long>(bv.actions, b, t)[n]);
                }
                rdy[2 * u] = (n0 + c0 == asel) ? dsel : 0.0f;
                rdy[2 * u + 1] = (n0 + c1 == asel) ? dsel : 0.0f;
            }
            // ---- A
            if (AK == A_DENSE) {
                const bool oka = ok && m >= p.shift;
                const float *ap = p.A + (m - p.shift) * p.lda + k0;
                ra[2 * u] = (oka && k_ok0) ? __ldg(ap + c0) : 0.0f;
                ra[2 * u + 1] = (oka && k_ok1) ? __ldg(ap + c1) : 0.0f;
            } else if (AK == A_STATE) {
                const int b = (int)((unsigned)m / (unsigned)bv.T), t = (int)m - b * bv.T;
                const float *ap = field_ptr<float>(bv.state, b, t + p.shift) + k0;
                ra[2 * u] = (ok && k_ok0) ? __ldg(ap + c0) : 0.0f;
                ra[2 * u + 1] = (ok && k_ok1) ? __ldg(ap + c1) : 0.0f;
            } else {   // [obs | last-action one-hot | agent-id one-hot], bounds from bv.in (K = d_in)
                const int t = (int)((unsigned)m / (unsigned)bv.R), rr = (int)m - t * bv.R;   // rows < 2^31 (host-checked): 32-bit division
                const int b = rr / bv.N, n = rr - b * bv.N;
                const float *po = field_ptr<float>(bv.obs, b, t) + (int64_t)n * bv.OBS;
                const float *ph = field_ptr<float>(bv.onehot, b, t > 0 ? t - 1 : 0) + (int64_t)n * bv.A;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int k = k0 + (h ? c1 : c0);
                    float v = 0.0f;
                    if (ok && k < p.K) {
                        if (k < bv.OBS) v = __ldg(po + k);
                        else if (k < bv.OBS + bv.in.last) v = t > 0 ? __ldg(ph + (k - bv.OBS)) : 0.0f;
                        else v = (k - bv.OBS - bv.in.last) == n ? 1.0f : 0.0f;
                    }
                    ra[2 * u + h] = v;
                }
            }
        }
    };
    if (mb < me) prefetch(mb);
    for (int64_t mm = mb; mm < me; mm += RED_MR) {
        __syncthreads();   // previous block fully consumed
#pragma unroll
        for (int u = 0; u < RED_MR / 8; ++u)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                dY_s[(warp + 8 * u) * RED_LD + lane + 32 * h] = rdy[2 * u + h];
                A_s[(warp + 8 * u) * RED_LD + lane + 32 * h] = ra[2 * u + h];
            }
        __syncthreads();
        if (mm + RED_MR < me) prefetch(mm + RED_MR);   // next block's global loads fly while this one is reduced
#pragma unroll 8
        for (int r = 0; r < RED_MR; ++r) {
            const float4 d = *reinterpret_cast<const float4 *>(dY_s + r * RED_LD + 4 * ty);
            const float4 av4 = *reinterpret_cast<const float4 *>(A_s + r * RED_LD + 4 * tx);
            const float dv[4] = {d.x, d.y, d.z, d.w}, avv[4] = {av4.x, av4.y, av4.z, av4.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(dv[i], avv[j], acc[i][j]);
            if (want_bias) {
#pragma unroll
                for (int i = 0; i < 4; ++i) bsum[i] += dv[i];
            }
        }
    }
    float *pw = p.partW + (int64_t)chunk * p.Nout * p.K;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int n = n0 + 4 * ty + i;
        if (n >= p.Nout) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int k = k0 + 4 * tx + j;
            if (k < p.K) pw[(int64_t)n * p.K + k] = acc[i][j];
        }
        if (want_bias && tx == 0) p.partB[(int64_t)chunk * p.Nout + n] = bsum[i];
    }
}

// =============================================================================================
// GRU recurrence: argument blocks
// =============================================================================================
struct GruFwdArgs {
    const float *params[2];    // online, target (flat agent buffers)
    const float *gi[2];        // [TT*R,192]
    float *hout[2];            // [TT*R,64]
    float *gates;              // [TT*R,64,4] online only: (r, z, n, gh_n) per unit
    int TT, R, d_in, n_actions;
    int t0, t1;                // timesteps of this launch: [t0, t1); h_{t0-1} comes from hout (zeros for t0 = 0)
    // balanced mode of k_gru_fwd9 (bal_D > 0; grid = workers x 1, t0 = 0, t1 = TT): the nets * R chains of TT steps each are
    // laid end to end and worker w runs steps [w bal_D, (w + 1) bal_D) of that sequence, LAST piece first, so the head of a
    // chain that is split between two workers is finished (chain_flags) before the neighbour reaches its tail
    int bal_D = 0, bal_chains = 0;
    int *chain_flags = nullptr;   // [bal_chains] zero between launches (the consumer resets what the producer sets)
};

__device__ __forceinline__ float sigmoid_fast(float x) { return __fdividef(1.0f, 1.0f + expf(-x)); }
// MUFU-only forms (ex2.approx + rcp.approx): ~2^-22 relative error on sigmoid, ~1.5e-7 absolute on tanh
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float sigmoid_mufu(float x) { return rcp_approx(1.0f + ex2_approx(-1.4426950408889634f * x)); }
__device__ __forceinline__ float tanh_mufu(float x) { return fmaf(2.0f, rcp_approx(1.0f + ex2_approx(-2.8853900817779268f * x)), -1.0f); }

#ifndef PDL_LEAD_STEPS
#define PDL_LEAD_STEPS 6   // timesteps before the end of a recurrence at which its dependent kernel may start its prologue
#endif
// (the recurrence kernels k_gru_fwd7 / k_gru_bwd7 live in gru_rec.cuh)

// out[c][r] = in[r][c] for up to three small weight matrices (grid: 32x32 tiles, problem); see mal_plan_t.w_t
struct TransArgs {
    const float *in[3];
    float *out[3];
    int rows[3], cols[3];
    int n;
};
__global__ void __launch_bounds__(256) k_transpose_w(TransArgs a) {
    __shared__ float tile[32][33];
    const int pi = blockIdx.y;
    const int rows = a.rows[pi], cols = a.cols[pi];
    const int tc = (cols + 31) / 32;
    if ((int)blockIdx.x >= ((rows + 31) / 32) * tc) return;
    const int r0 = ((int)blockIdx.x / tc) * 32, c0 = ((int)blockIdx.x % tc) * 32;
    for (int i = threadIdx.y; i < 32; i += 8) {
        const int r = r0 + i, c = c0 + threadIdx.x;
        tile[i][threadIdx.x] = (r < rows && c < cols) ? __ldg(a.in[pi] + (int64_t)r * cols + c) : 0.0f;
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += 8) {
        const int c = c0 + i, r = r0 + threadIdx.x;
        if (r < rows && c < cols) a.out[pi][(int64_t)c * rows + r] = tile[threadIdx.x][i];
    }
}

// =============================================================================================
// q = fc2 h for both nets, chosen-action gather, avail-masked (double-Q) target max.   q_learner.py:52-78
// =============================================================================================
struct HeadArgs {
    const float *params[2];
    const float *hout[2];
    int B, TT, N, A, R, d_in, double_q, kind;
    mal_field_t actions, avail;
    float *mac_out, *target_mac_out;   // [B,TT,N,A] or null
    float *chosen, *target_max;        // [B,T,N]
    int *argmax;                       // [B,T,N]
};

// A CTA stages both nets' fc2 once and then walks 64-row tiles.  Warps 0-1 serve the online net, warps 2-3 the target
// net, thread = row: the tile's h rows (both nets) arrive through a cp.async stage (coalesced 16-byte copies), each
// thread takes its row into registers, and the stage is refilled with the next tile right away, so that copy flies under
// the dot products.  The actions are walked four at a time with the fc2 rows broadcast from shared memory (the net is
// warp-uniform, so an LDS.128 is a single-address broadcast: one wavefront per 16 FMAs) -- four independent FMA chains,
// each in ascending k and seeded with the bias: the summation order of the fixtures.  Q goes through shared memory to
// the epilogue: thread r < 64 runs row r's avail-masked (double-Q) arg-max scan in index order (ties -> lowest index)
// on avail rows that were requested (4-byte cp.async) before the dot products; thread 64 + r picks row r's
// chosen-action Q.
#define QH_NET_F4 (64 * 17)         // float4 pitch between the two nets' h tiles (17-float4 rows: conflict-free per 8-lane phase)
#define QH_HS_F4 (2 * QH_NET_F4)
__host__ __device__ inline int qh_w2_pitch(int A) { return ((A + 3) & ~3) * HID; }       // floats between the nets' fc2 copies
__host__ __device__ inline int qh_q_pitch(int A) { return ((A + 3) & ~3) | 1; }          // odd: row-per-lane accesses are conflict-free
__host__ __device__ inline size_t qh_smem_bytes(int A) {
    return sizeof(float4) * QH_HS_F4 + sizeof(float) * (2 * (size_t)qh_w2_pitch(A) + 3 * 64 * (size_t)qh_q_pitch(A));
}

__global__ void __launch_bounds__(128, 3) k_q_head(HeadArgs a) {
    extern __shared__ __align__(16) float4 qh_smem[];        // hs_s [QH_HS_F4] | w2_s [2][w2_pitch] | q_s [2][64*qpitch] | av_s [64*qpitch]
    __shared__ float b2_s[2][MAL_MAX_ACTIONS];
    float4 *hs_s = qh_smem;
    const AgentLayout L = agent_layout(a.d_in, a.A, a.kind);
    const int tid = threadIdx.x;
    const int Apad = (a.A + 3) & ~3, w2_pitch = qh_w2_pitch(a.A), qpitch = qh_q_pitch(a.A);
    float *w2_all = reinterpret_cast<float *>(qh_smem + QH_HS_F4);
    float *q_s = w2_all + 2 * w2_pitch;
    const int q_net = 64 * qpitch;                           // floats between the nets' Q tiles
    int *av_s = reinterpret_cast<int *>(q_s + 2 * q_net);    // [64][qpitch] avail rows of the tile
    const int T = a.TT - 1;
    const int64_t total = (int64_t)a.TT * a.R;
    const int64_t n_tiles = (total + 63) >> 6;
    auto issue_h = [&](int64_t tile) {                       // 2 nets x 64 rows x 16 float4, rows past the end shadow the last row
        const int64_t m_base = tile * 64;
#pragma unroll
        for (int it = 0; it < 16; ++it) {
            const int idx = tid + 128 * it;
            const int nn = idx >> 10, r = (idx >> 4) & 63, c = idx & 15;
            const int64_t mm = m_base + r < total ? m_base + r : total - 1;
            cp_async16(hs_s + nn * QH_NET_F4 + r * 17 + c, (nn ? a.hout[1] : a.hout[0]) + mm * HID + 4 * c);
        }
        cp_async_commit();
    };
    int64_t tile = blockIdx.x;
    {   // fc2.weight of both nets (rows >= A zero), fc2.bias
        const bool vec = ((reinterpret_cast<uintptr_t>(a.params[0] + L.fc2_w) | reinterpret_cast<uintptr_t>(a.params[1] + L.fc2_w)) & 15) == 0;
        for (int idx = tid; idx < 2 * Apad * 16; idx += 128) {
            const int nn = idx >= Apad * 16, rem = idx - nn * Apad * 16;     // rem = action * 16 + float4 column
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if ((rem >> 4) < a.A) {
                const float *src = a.params[nn] + L.fc2_w + rem * 4;
                if (vec) v = __ldg(reinterpret_cast<const float4 *>(src));
                else { v.x = __ldg(src); v.y = __ldg(src + 1); v.z = __ldg(src + 2); v.w = __ldg(src + 3); }
            }
            *reinterpret_cast<float4 *>(w2_all + nn * w2_pitch + rem * 4) = v;
        }
        if (tid < 2 * MAL_MAX_ACTIONS) {
            const int nn = tid / MAL_MAX_ACTIONS, j = tid - nn * MAL_MAX_ACTIONS;
            b2_s[nn][j] = j < a.A ? __ldg(a.params[nn] + L.fc2_b + j) : 0.0f;
        }
    }
    pdl_wait();                                              // fc2 is a step constant; the h rows come from the recurrence
    if (tile < n_tiles) issue_h(tile);
    const int net = tid >> 6, r = tid & 63;                  // warp-uniform net
    const float4 *w2 = reinterpret_cast<const float4 *>(w2_all + net * w2_pitch);
    for (; tile < n_tiles; tile += gridDim.x) {
        // this thread's row: the same row for the dot products (net = tid >> 6) and for the epilogue
        const int64_t m = tile * 64 + r;
        int t = -1, b = 0, n = 0;
        if (m < total) {
            t = (int)((unsigned)m / (unsigned)a.R);
            const int row = (int)m - t * a.R;
            b = row / a.N; n = row - b * a.N;
        }
        cp_async_wait<0>();
        __syncthreads();                                     // the tile (and, first time round, fc2) is in shared memory
        float4 hv[HID / 4];
        {
            const float4 *hp = hs_s + net * QH_NET_F4 + r * 17;
#pragma unroll
            for (int k4 = 0; k4 < HID / 4; ++k4) hv[k4] = hp[k4];
        }
        __syncthreads();                                     // every thread holds its row: the stage is free
        // the epilogue's operands are requested now and fly under the dot products: the row's avail flags
        // (thread r < 64, 4-byte cp.async) and its action (thread 64 + r, a register), then the next tile's h rows
        long long act_ll = 0;
        if (tid < 64) {
            if (t >= 1) {
                const int *av = field_ptr<int>(a.avail, b, t) + (int64_t)n * a.A;
                for (int j = 0; j < a.A; ++j) cp_async4(av_s + r * qpitch + j, av + j);
            }
        } else if (t >= 0 && t < T) {
            act_ll = field_ptr<long long>(a.actions, b, t)[n];
        }
        cp_async_commit();
        const bool more = tile + gridDim.x < n_tiles;
        if (more) issue_h(tile + gridDim.x);
        else pdl_trigger();                                  // last tile of this CTA
        float *qp = q_s + net * q_net + r * qpitch;
#pragma unroll 1
        for (int a0 = 0; a0 < Apad; a0 += 4) {
            float q[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) q[j] = b2_s[net][a0 + j];
            const float4 *wj = w2 + a0 * (HID / 4);
#pragma unroll
            for (int k4 = 0; k4 < HID / 4; ++k4) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {                // one chain per action in ascending k
                    const float4 wa = wj[j * (HID / 4) + k4];
                    q[j] = fmaf(wa.x, hv[k4].x, q[j]);
                    q[j] = fmaf(wa.y, hv[k4].y, q[j]);
                    q[j] = fmaf(wa.z, hv[k4].z, q[j]);
                    q[j] = fmaf(wa.w, hv[k4].w, q[j]);
                }
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) qp[a0 + j] = q[j];
        }
        if (more) cp_async_wait<1>(); else cp_async_wait<0>();   // the avail rows (the next tile's h may still be in flight)
        __syncthreads();                                     // Q of the tile is complete
        if (t >= 0) {
            const float *qo_s = q_s + r * qpitch, *qt_s = q_s + q_net + r * qpitch;
            if (tid < 64) {
                if (t >= 1) {                                // targets use step t's Q for transition t-1
                    const int *av = av_s + r * qpitch;
                    float best_sel = 0.0f, best_mt = 0.0f;
                    int best_i = -1;
                    for (int j = 0; j < a.A; ++j) {
                        const int avv = av[j];
                        const float mt = avv == 0 ? -9999999.0f : qt_s[j];
                        const float sel = a.double_q ? (avv == 0 ? -9999999.0f : qo_s[j]) : mt;
                        if (best_i < 0 || arg_better(sel, j, best_sel, best_i)) { best_sel = sel; best_i = j; best_mt = mt; }
                    }
                    const int64_t o = ((int64_t)b * T + (t - 1)) * a.N + n;
                    a.target_max[o] = best_mt;
                    a.argmax[o] = best_i;
                }
            } else if (t < T) {                              // gather(mac_out[:, :-1], 3, actions)
                const int act = (int)act_ll;
                a.chosen[((int64_t)b * T + t) * a.N + n] = (act >= 0 && act < a.A) ? qo_s[act] : 0.0f;
            }
            if (a.mac_out) {                                 // save_q only (not on the training path)
                const int64_t qoff = (((int64_t)b * a.TT + t) * a.N + n) * a.A;
                float *dst = tid < 64 ? a.mac_out : a.target_mac_out;
                const float *src = tid < 64 ? qo_s : qt_s;
                if (dst) for (int j = 0; j < a.A; ++j) dst[qoff + j] = src[j];
            }
        }
    }
    cp_async_wait<0>();
}

// =============================================================================================
// mask + mixer (VDN / QMIX) + TD target + masked L2 loss + element-wise part of the mixer backward + the
// fc2/gather backward injection d h_t += d_chosen * W2[a_t].   One warp per (b,t); lane = embed index.
//                                            q_learner.py:40-42,81-98, qmix.py:41-59, vdn.py:9-10
// All seeds are UN-normalised (without the 1/mask.sum() factor); k_grad_reduce applies it once at the end.
// No mixer (IQL): lane n is agent n's own transition: its TD error against the shared reward, its q_tot / targets / td
// entry [m*N + n], its seed, and its share of the statistics, so that the block sums come out over the mask expanded to
// [B,T,N] (q_learner.py:92): sum m and the count are N times the per-transition values.
// =============================================================================================
#define MIX_NSTAT 6   // sum mtd^2, sum |mtd|, sum q_tot*m, sum targets*m, sum m, count(m != 0)
struct MixArgs {
    int mixer, B, T, N, E, HE, S, R, A, d_in, kind;
    const float *relu_src;             // feed-forward agent: x = relu(fc1) [TT*R,64]; the head seed is multiplied by (x > 0)
    const float *y1[2], *a2[2];        // online, target
    const float *mparams[2];
    const float *agent;                // online agent parameters (fc2.weight for the dh injection)
    const float *chosen, *target_max;  // [B*T,N]
    mal_field_t reward, terminated, filled, actions;
    float gamma;
    float *mask;                       // [B*T] out
    float *q_tot, *target_q_tot, *targets, *td;
    float *d_a2, *d_y1, *d_chosen;     // backward seeds (un-normalised)
    float *dh_head;                    // [TT*R,64]: rows of t < T: d_chosen * fc2.weight[a_t, :] (gather + fc2 backward)
    float *part_stats;                 // [gridDim.x][MIX_NSTAT]
    float *part_v2;                    // [gridDim.x][E+1] d V.2.weight | d V.2.bias
    mal_field_t weight;                // k_mix_td<true>: f32 [B] importance weights (batch stride sb)
};

// q(n): agent n's Q-value of row m (an array read, or a shuffle from the lane that holds it)
template <class QOf>
__device__ __forceinline__ float qmix_row(const MixArgs &a, int net, int64_t m, QOf q, int lane,
                                          float *pre_out, float *hidden_out, float *wf_out, float *v1_out) {
    const MixerLayout ML = mixer_layout(a.mixer, a.S, a.N, a.E, a.HE);
    const int two = (ML.layers == 2);
    const int ld1 = two ? 2 * a.HE + 2 * a.E : 2 * a.E;
    const int ld2 = a.E * a.N + a.E;
    const float *y1 = a.y1[net] + m * ld1 + (two ? 2 * a.HE : 0);   // -> [b1 | v1]
    const float *a2 = a.a2[net] + m * ld2;
    const bool act = lane < a.E;
    float pre = act ? y1[lane] : 0.0f;
    for (int n = 0; n < a.N; ++n) {
        float w1 = act ? fabsf(a2[n * a.E + lane]) : 0.0f;
        pre = fmaf(q(n), w1, pre);
    }
    float hidden = pre > 0.0f ? pre : expm1f(pre);
    float wf = act ? fabsf(a2[a.N * a.E + lane]) : 0.0f;
    float v1 = act ? y1[a.E + lane] : 0.0f;
    float v2w = act ? __ldg(a.mparams[net] + ML.v2_w + lane) : 0.0f;
    float y = warp_sum(act ? fmaf(hidden, wf, v1 * v2w) : 0.0f) + __ldg(a.mparams[net] + ML.v2_b);
    *pre_out = pre; *hidden_out = hidden; *wf_out = wf; *v1_out = v1;
    return y;
}

// WEIGHTED: prioritized replay's importance weights w_b scale episode b's loss term and seed (the <false> instance is the
// unweighted step, unchanged); multiplying by w_b = 1.0f is exact, so weights of one reproduce it bit for bit.
// GIVEN_TARGETS (TD(lambda), k_mix_td_lambda): the targets were formed by k_td_lambda and are read, not computed; the
// target mixer row is then not evaluated here (k_mix_tq wrote target_q_tot).
template <bool WEIGHTED, bool GIVEN_TARGETS>
__device__ __forceinline__ void mix_td_body(MixArgs a) {
    __shared__ float s_stats[8][MIX_NSTAT];
    __shared__ float s_v2[8][MAL_MAX_EMBED + 1];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t total = (int64_t)a.B * a.T;
    const MixerLayout ML = mixer_layout(a.mixer, a.S, a.N, a.E, a.HE);
    const int two = (ML.layers == 2);
    const int ld1 = two ? 2 * a.HE + 2 * a.E : 2 * a.E;
    const int ld2 = a.E * a.N + a.E;
    const int yo = two ? 2 * a.HE : 0;                    // column of [b1 | v1] inside a y1 row
    const float *w2p = a.agent + agent_layout(a.d_in, a.A, a.kind).fc2_w;
    const bool act = lane < a.E;
    float st[MIX_NSTAT] = {0, 0, 0, 0, 0, 0};
    float dv2w = 0, dv2b = 0;
    float v2w_o = 0.0f, v2w_t = 0.0f, v2b_o = 0.0f, v2b_t = 0.0f;
    if (mixer_has_hypernet(a.mixer)) {
        v2w_o = act ? __ldg(a.mparams[0] + ML.v2_w + lane) : 0.0f;
        v2w_t = act ? __ldg(a.mparams[1] + ML.v2_w + lane) : 0.0f;
        v2b_o = __ldg(a.mparams[0] + ML.v2_b);
        v2b_t = __ldg(a.mparams[1] + ML.v2_b);
    }
    pdl_wait();

    for (int64_t m = (int64_t)blockIdx.x * 8 + warp; m < total; m += (int64_t)gridDim.x * 8) {
        const int b = (int)((unsigned)m / (unsigned)a.T), t = (int)m - b * a.T;
        // lane n holds agent n's chosen / target Q (N <= 32): one coalesced load each, broadcast by shuffle
        const float qc = lane < a.N ? a.chosen[m * a.N + lane] : 0.0f;
        const float qt = !GIVEN_TARGETS && lane < a.N ? a.target_max[m * a.N + lane] : 0.0f;
        // per-transition scalars (issued early: independent of the mixing arithmetic)
        float mk = (float)(*field_ptr<long long>(a.filled, b, t));
        if (t > 0) mk = mk * (1.0f - (float)(*field_ptr<unsigned char>(a.terminated, b, t - 1)));   // mask[:, 1:] *= 1 - terminated[:, :-1]
        const float rew = *field_ptr<float>(a.reward, b, t);
        const float term = (float)(*field_ptr<unsigned char>(a.terminated, b, t));
        float y, ty = 0.0f, pre = 0, hidden = 0, wf = 0, v1 = 0;
        const float *a2o = a.a2[0] + m * ld2;
        const bool iql = a.mixer == MAL_MIXER_NONE;       // warp-uniform
        if (a.mixer == MAL_MIXER_VDN) {
            y = warp_sum(qc);
            if (!GIVEN_TARGETS) ty = warp_sum(qt);
        } else if (iql) {
            y = qc; ty = qt;                             // lane n: agent n's chosen / target Q (lanes >= N carry zeros)
        } else if (GIVEN_TARGETS) {
            y = qmix_row(a, 0, m, [&](int n) { return __shfl_sync(0xffffffffu, qc, n); }, lane, &pre, &hidden, &wf, &v1);
        } else {
            // online and target mixer rows side by side (lane = embed unit): hidden = elu(q . |w1| + b1), y = hidden . |w_f| + V(s)
            const float *a2t = a.a2[1] + m * ld2;
            const float *y1o = a.y1[0] + m * ld1 + yo, *y1t = a.y1[1] + m * ld1 + yo;
            float pre_t = act ? y1t[lane] : 0.0f;
            pre = act ? y1o[lane] : 0.0f;
            const float wf_t = act ? fabsf(a2t[a.N * a.E + lane]) : 0.0f;
            wf = act ? fabsf(a2o[a.N * a.E + lane]) : 0.0f;
            const float v1_t = act ? y1t[a.E + lane] : 0.0f;
            v1 = act ? y1o[a.E + lane] : 0.0f;
#pragma unroll 8
            for (int n = 0; n < a.N; ++n) {
                const float w1o = act ? fabsf(a2o[n * a.E + lane]) : 0.0f;
                const float w1t = act ? fabsf(a2t[n * a.E + lane]) : 0.0f;
                pre = fmaf(__shfl_sync(0xffffffffu, qc, n), w1o, pre);
                pre_t = fmaf(__shfl_sync(0xffffffffu, qt, n), w1t, pre_t);
            }
            hidden = pre > 0.0f ? pre : expm1f(pre);
            const float hidden_t = pre_t > 0.0f ? pre_t : expm1f(pre_t);
            y = warp_sum(act ? fmaf(hidden, wf, v1 * v2w_o) : 0.0f) + v2b_o;
            ty = warp_sum(act ? fmaf(hidden_t, wf_t, v1_t * v2w_t) : 0.0f) + v2b_t;
        }
        float target;
        if (GIVEN_TARGETS) target = iql ? (lane < a.N ? a.targets[m * a.N + lane] : 0.0f) : a.targets[m];
        else target = rew + a.gamma * (1.0f - term) * ty;
        const float tdv = y - target;
        const float mtd = tdv * mk;
        float gseed = 2.0f * mtd * mk;         // (d loss / d q_tot) * mask.sum()
        float lterm = mtd * mtd;
        if (WEIGHTED) {
            const float wb = *(reinterpret_cast<const float *>(a.weight.ptr) + (int64_t)b * a.weight.sb);
            gseed *= wb; lterm *= wb;
        }
        if (iql) {
            if (lane == 0) a.mask[m] = mk;
            if (lane < a.N) {
                const int64_t e = m * a.N + lane;
                a.q_tot[e] = y;
                if (!GIVEN_TARGETS) { a.target_q_tot[e] = ty; a.targets[e] = target; }
                a.td[e] = tdv;
                st[0] += lterm; st[1] += fabsf(mtd); st[2] += y * mk; st[3] += target * mk;
                st[4] += mk; st[5] += (mk != 0.0f) ? 1.0f : 0.0f;
            }
        } else if (lane == 0) {
            a.mask[m] = mk;
            a.q_tot[m] = y;
            if (!GIVEN_TARGETS) { a.target_q_tot[m] = ty; a.targets[m] = target; }
            a.td[m] = tdv;
            st[0] += lterm; st[1] += fabsf(mtd); st[2] += y * mk; st[3] += target * mk;
            st[4] += mk; st[5] += (mk != 0.0f) ? 1.0f : 0.0f;
        }
        int act_mine = lane < a.N ? (int)(field_ptr<long long>(a.actions, b, t)[lane]) : 0;
        act_mine = act_mine < 0 ? 0 : (act_mine >= a.A ? a.A - 1 : act_mine);            // never read outside fc2.weight
        // gather + fc2 backward: d h_t[row n] = d_chosen[n] * fc2.weight[a_t[n], :]   (consumed by the BPTT kernel)
        auto head_inject = [&](float dq_lane) {
            float *dh = a.dh_head + ((int64_t)t * a.R + (int64_t)b * a.N) * HID;
            const float *xr = a.relu_src ? a.relu_src + ((int64_t)t * a.R + (int64_t)b * a.N) * HID : nullptr;
#pragma unroll 8
            for (int n = 0; n < a.N; ++n) {
                const float dq = __shfl_sync(0xffffffffu, dq_lane, n);
                const float2 w2 = __ldg(reinterpret_cast<const float2 *>(w2p + (int64_t)__shfl_sync(0xffffffffu, act_mine, n) * HID) + lane);
                float2 v = make_float2(dq * w2.x, dq * w2.y);
                if (xr) {                                     // d relu(fc1): the seed becomes d(fc1 pre-activation)
                    const float2 xv = reinterpret_cast<const float2 *>(xr + (int64_t)n * HID)[lane];
                    v.x = xv.x > 0.0f ? v.x : 0.0f; v.y = xv.y > 0.0f ? v.y : 0.0f;
                }
                reinterpret_cast<float2 *>(dh + (int64_t)n * HID)[lane] = v;
            }
        };
        if (!mixer_has_hypernet(a.mixer)) {
            if (lane < a.N) a.d_chosen[m * a.N + lane] = gseed;   // VDN: d q_tot / d q_n = 1; IQL: lane n's own seed
            head_inject(gseed);
            continue;
        }
        // element-wise mixer backward
        float *da2 = a.d_a2 + m * ld2;
        float *dy1 = a.d_y1 + m * ld1 + yo;
        const float dhidden = gseed * wf;
        const float dwf = gseed * hidden;
        const float dpre = dhidden * (pre > 0.0f ? 1.0f : expf(pre));
        if (act) {
            const float af = a2o[a.N * a.E + lane];
            da2[a.N * a.E + lane] = dwf * (af > 0.0f ? 1.0f : (af < 0.0f ? -1.0f : 0.0f));
            dy1[lane] = dpre;                                                          // d hyper_b_1 out
            dy1[a.E + lane] = v1 > 0.0f ? gseed * v2w_o : 0.0f;                         // d V.0 pre-activation
            dv2w += gseed * v1;
        }
        if (lane == 0) dv2b += gseed;
        float dq_mine = 0.0f;                 // lane n ends up with d q_tot / d q_n * seed
#pragma unroll 8
        for (int n = 0; n < a.N; ++n) {
            const float a1 = act ? a2o[n * a.E + lane] : 0.0f;
            const float dq = warp_sum(act ? dpre * fabsf(a1) : 0.0f);
            const float qn = __shfl_sync(0xffffffffu, qc, n);
            if (act) da2[n * a.E + lane] = qn * dpre * (a1 > 0.0f ? 1.0f : (a1 < 0.0f ? -1.0f : 0.0f));
            if (lane == n) dq_mine = dq;
        }
        if (lane < a.N) a.d_chosen[m * a.N + lane] = dq_mine;
        head_inject(dq_mine);
    }
    // ---- deterministic block partials
    if (a.mixer == MAL_MIXER_NONE)                // IQL: every lane holds its agent's sums (fixed shuffle order)
        for (int k = 0; k < MIX_NSTAT; ++k) st[k] = warp_sum(st[k]);
    if (lane == 0)
        for (int k = 0; k < MIX_NSTAT; ++k) s_stats[warp][k] = st[k];
    if (mixer_has_hypernet(a.mixer)) {
        if (lane < a.E) s_v2[warp][lane] = dv2w;
        if (lane == 0) s_v2[warp][a.E] = dv2b;
    }
    pdl_trigger();                               // the BPTT recurrence may be scheduled and load W_hh under this tail
    __syncthreads();
    if (tid < MIX_NSTAT) {
        float s = 0;
        for (int w = 0; w < 8; ++w) s += s_stats[w][tid];
        a.part_stats[blockIdx.x * MIX_NSTAT + tid] = s;
    }
    if (mixer_has_hypernet(a.mixer) && tid <= a.E) {
        float s = 0;
        for (int w = 0; w < 8; ++w) s += s_v2[w][tid];
        a.part_v2[(int64_t)blockIdx.x * (a.E + 1) + tid] = s;
    }
}

template <bool WEIGHTED>
__global__ void __launch_bounds__(256, 4) k_mix_td(MixArgs a) { mix_td_body<WEIGHTED, false>(a); }

// TD(lambda): the mixing / TD / seed step over the targets k_td_lambda left in a.targets
template <bool WEIGHTED>
__global__ void __launch_bounds__(256, 4) k_mix_td_lambda(MixArgs a) { mix_td_body<WEIGHTED, true>(a); }

// stand-alone mixer forward (QMixer.forward / VDNMixer.forward called outside the learner)
__global__ void __launch_bounds__(256) k_mix_fwd(MixArgs a) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t total = (int64_t)a.B * a.T;
    float q[MAL_MAX_ACTIONS];
    for (int64_t m = (int64_t)blockIdx.x * 8 + warp; m < total; m += (int64_t)gridDim.x * 8) {
        float y;
        if (a.mixer == MAL_MIXER_VDN) {
            y = 0.0f;
            for (int n = 0; n < a.N; ++n) y += a.chosen[m * a.N + n];
        } else {
            float d0, d1, d2, d3;
            for (int n = 0; n < a.N; ++n) q[n] = a.chosen[m * a.N + n];
            y = qmix_row(a, 0, m, [&](int n) { return q[n]; }, lane, &d0, &d1, &d2, &d3);
        }
        if (lane == 0) a.q_tot[m] = y;
    }
}

// mask.sum(), loss and the logging scalars from the block partials (q_learner.py:98,112,117-124): block 0, one warp
// per statistic.  Blocks >= 1 fold the per-block d V.2 partials into one row (one warp per output, fixed order).
__global__ void __launch_bounds__(256) k_stats_finalize(const float *part_stats, int nblk, int n_agents, float *scalars,
                                                        const float *part_v2, int n_v2, float *v2_out) {
    __shared__ float s[MIX_NSTAT];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (blockIdx.x > 0) {
        const int o = (blockIdx.x - 1) * 8 + warp;
        if (o < n_v2) {
            float v = 0.0f;
            for (int i = lane; i < nblk; i += 32) v += part_v2[(int64_t)i * n_v2 + o];
            v = warp_sum(v);
            if (lane == 0) v2_out[o] = v;
        }
        return;
    }
    if (warp < MIX_NSTAT) {
        float v = 0.0f;
        for (int i = lane; i < nblk; i += 32) v += part_stats[i * MIX_NSTAT + warp];
        v = warp_sum(v);
        if (lane == 0) s[warp] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const float msum = s[4];
        scalars[MAL_SC_MASK_SUM] = msum;
        scalars[MAL_SC_LOSS] = s[0] / msum;
        scalars[MAL_SC_TD_ABS] = s[1] / msum;
        scalars[MAL_SC_Q_TAKEN] = s[2] / (msum * n_agents);
        scalars[MAL_SC_TARGET] = s[3] / (msum * n_agents);
        reinterpret_cast<int *>(scalars)[MAL_SC_MASK_COUNT] = (int)(s[5] + 0.5f);
        for (int k = 0; k < MIX_NSTAT; ++k) scalars[MAL_SC_RAW0 + k] = s[k];
    }
}

struct GruBwdArgs {
    const float *params;       // online agent
    const float *hout;         // [TT*R,64]
    const float *gates;        // [TT*R,64,4]
    const float *dh_head;      // [TT*R,64] (rows of t < TT-1 are valid)
    float *d_g;                // [TT*R,256]: d gi_r | d gi_z | d gi_n | d gh_n
    int TT, R, d_in, n_actions;
};

// =============================================================================================
// fc2 gradients:  dW2[a, :] = sum_m [a_m == a] d_chosen[m] h_m ,  db2[a] = sum_m [a_m == a] d_chosen[m]
// (the backward of `gather(mac_out, actions)` through fc2: only the chosen action's row receives a gradient).
// A segmented scatter-add, HBM-bound on the h rows: warp per row (lanes along the 64 hidden units, one coalesced
// 256-byte load), warp-private [A][64] accumulators in shared memory, a fixed row -> warp assignment and a fixed
// cross-warp summation order (bit-reproducible); per-CTA partials go through k_grad_reduce like every other gradient.
// =============================================================================================
struct Fc2GradArgs {
    const float *d_chosen;     // [B,T,N]
    mal_field_t actions;       // int64 [B,TT,N]
    const float *hout;         // [TT*R,64]
    float *partW, *partB;      // [gridDim.x][A*64], [gridDim.x][A]
    int T, N, A, R;
    int64_t rows;              // T*R
};

__global__ void __launch_bounds__(256) k_fc2_grad(Fc2GradArgs a) {
    extern __shared__ __align__(16) float f2_s[];            // [8 warps][A*64 + 32]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int ld = a.A * HID + 32;
    float *acc = f2_s + warp * ld;
    for (int e = lane; e < ld; e += 32) acc[e] = 0.0f;
    __syncwarp();
    const int64_t stride = (int64_t)gridDim.x * 8;
    constexpr int U = 8;                                      // rows in flight per warp
    for (int64_t m0 = (int64_t)blockIdx.x * 8 + warp; m0 < a.rows; m0 += U * stride) {
        float d[U];
        long long act64[U];
        int act[U];
        float2 h[U];
        // all 3 U loads are requested UNCONDITIONALLY (row clamped into range) and before any of them is used: with the loads
        // inside `if (m < rows)` blocks and the index clamp right behind them, every row cost its own DRAM latency (r2
        // profile: 46 % of all stall samples on the eight clamp compares)
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t m = m0 + u * stride;
            const int64_t mc = m < a.rows ? m : a.rows - 1;
            const int t = (int)((unsigned)mc / (unsigned)a.R), rr = (int)mc - t * a.R;   // rows < 2^31 (host-checked)
            const int b = rr / a.N, n = rr - b * a.N;
            d[u] = __ldg(a.d_chosen + ((int64_t)b * a.T + t) * a.N + n);
            act64[u] = __ldg(field_ptr<long long>(a.actions, b, t) + n);
            h[u] = __ldg(reinterpret_cast<const float2 *>(a.hout + mc * HID) + lane);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (m0 + u * stride >= a.rows) d[u] = 0.0f;           // rows past the end contribute nothing
            act[u] = (int)act64[u];
            act[u] = act[u] < 0 ? 0 : (act[u] >= a.A ? a.A - 1 : act[u]);   // never index outside the accumulators
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            float2 *p = reinterpret_cast<float2 *>(acc + act[u] * HID) + lane;
            float2 v = *p;
            v.x = fmaf(d[u], h[u].x, v.x);
            v.y = fmaf(d[u], h[u].y, v.y);
            *p = v;
            if (lane == 0) acc[a.A * HID + act[u]] += d[u];
            __syncwarp();
        }
    }
    __syncthreads();
    for (int e = tid; e < a.A * HID; e += 256) {
        float s = 0.0f;
#pragma unroll
        for (int w = 0; w < 8; ++w) s += f2_s[w * ld + e];
        a.partW[(int64_t)blockIdx.x * a.A * HID + e] = s;
    }
    if (tid < a.A) {
        float s = 0.0f;
#pragma unroll
        for (int w = 0; w < 8; ++w) s += f2_s[w * ld + a.A * HID + tid];
        a.partB[(int64_t)blockIdx.x * a.A + tid] = s;
    }
}

// =============================================================================================
// gather per-chunk partials into the flat gradient (fixed summation order), apply 1/mask.sum(),
// per-block sum of squares for the global norm
// =============================================================================================
struct GradSeg {
    int64_t grad_off;
    int count;
    const float *part;
    int n_chunks;
    int64_t chunk_stride;
};
#define GRAD_MAX_SEGS 32
struct GradReduceArgs {
    int n;
    GradSeg s[GRAD_MAX_SEGS];
    int64_t total;
    float *grad;
    float *norm_part;        // [gridDim.x]
    const float *scalars;    // mask sum
    int unnormalized;        // leave out the 1/mask.sum() factor (data-parallel mode)
    int64_t n_frozen;        // parameters [0, n_frozen) are frozen: gradient 0 (their partials are not even read)
};

#define GRED_EPB 64   // gradient elements per block: 256 threads = 64 elements x 4 chunk slices
__global__ void __launch_bounds__(256) k_grad_reduce(const __grid_constant__ GradReduceArgs a) {
    pdl_wait();
    pdl_trigger();
    __shared__ float part_s[4][GRED_EPB];
    __shared__ float s_sq[2];
    const int e = threadIdx.x & (GRED_EPB - 1), slice = threadIdx.x >> 6;   // slice is warp-uniform
    const int64_t p = (int64_t)blockIdx.x * GRED_EPB + e;
    float v = 0.0f;
    if (p < a.total && p >= a.n_frozen) {
        int si = 0;
        while (si + 1 < a.n && p >= a.s[si + 1].grad_off) ++si;
        const GradSeg &s = a.s[si];
        const int64_t off = p - s.grad_off;
        if (off < s.count) {
            // this thread's slice of the chunk partials: c = slice, slice + 4, ...; four loads in flight
            const float *src = s.part + off;
            float v0 = 0.0f, v1 = 0.0f, v2 = 0.0f, v3 = 0.0f;
            int c = slice;
            for (; c + 12 < s.n_chunks; c += 16) {
                v0 += src[(int64_t)c * s.chunk_stride];
                v1 += src[(int64_t)(c + 4) * s.chunk_stride];
                v2 += src[(int64_t)(c + 8) * s.chunk_stride];
                v3 += src[(int64_t)(c + 12) * s.chunk_stride];
            }
            for (; c < s.n_chunks; c += 4) v0 += src[(int64_t)c * s.chunk_stride];
            v = (v0 + v1) + (v2 + v3);
        }
    }
    part_s[slice][e] = v;
    __syncthreads();
    if (threadIdx.x < GRED_EPB) {
        const float inv = a.unnormalized ? 1.0f : 1.0f / a.scalars[MAL_SC_MASK_SUM];
        v = ((part_s[0][e] + part_s[1][e]) + (part_s[2][e] + part_s[3][e])) * inv;   // fixed order: bit-reproducible
        if (p < a.total) a.grad[p] = v; else v = 0.0f;
        const float sq = warp_sum(v * v);
        if ((threadIdx.x & 31) == 0) s_sq[threadIdx.x >> 5] = sq;
    }
    __syncthreads();
    if (threadIdx.x == 0) a.norm_part[blockIdx.x] = s_sq[0] + s_sq[1];
}

// sum of squares of an arbitrary flat gradient (used when mal_clip_rmsprop is called stand-alone)
__global__ void __launch_bounds__(256) k_sumsq(float *g, int64_t n, float *norm_part, const float *denominator, int64_t n_frozen) {
    __shared__ float s_sq[8];
    const int64_t p = (int64_t)blockIdx.x * 256 + threadIdx.x;
    const float inv = denominator ? 1.0f / denominator[0] : 1.0f;
    if (p < n_frozen && p < n) g[p] = 0.0f;       // frozen prefix: no gradient, not in the norm
    float v = (p < n && p >= n_frozen) ? g[p] * inv : 0.0f;
    float sq = warp_sum(v * v);
    if ((threadIdx.x & 31) == 0) s_sq[threadIdx.x >> 5] = sq;
    __syncthreads();
    if (threadIdx.x == 0) {
        float s = 0;
        for (int w = 0; w < 8; ++w) s += s_sq[w];
        norm_part[blockIdx.x] = s;
    }
}

// =============================================================================================
// clip_grad_norm_ (q_learner.py:104) + RMSprop.step (learner.py:25-31), one pass over the flat buffers
// =============================================================================================
// The clip prologue of k_clip_rmsprop and k_clip_adam: every block recomputes the global norm from the per-block
// partials in the same fixed order; thread 0 leaves min(clip / (norm + 1e-6), 1) in s_coef (read after a barrier).
__device__ __forceinline__ void clip_coef_prologue(const float *norm_part, int n_part, float clip, float *scalars,
                                                   float *s_red, float &s_coef) {
    float s = 0.0f;
    for (int i = threadIdx.x; i < n_part; i += 256) s += norm_part[i];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        float tot = 0;
        for (int w = 0; w < 8; ++w) tot += s_red[w];
        const float norm = sqrtf(tot);
        float coef = clip / (norm + 1e-6f);
        s_coef = coef < 1.0f ? coef : 1.0f;
        if (blockIdx.x == 0) scalars[MAL_SC_GRAD_NORM] = norm;
    }
}

// Soft target update of the SOFT optimiser instances: after the step, target = fp32(fp32(target * c1) + fp32(p_new * c2))
// with c1 = fp32(1 - tau) (subtraction in double), c2 = fp32(tau): `target.data.copy_(target.data * (1.0 - tau) +
// param.data * tau)` on fp32 tensors.  The target flats have the online flats' layout (agent | mixer).
struct SoftBlend {
    float *agent, *mixer;
    float c1, c2;
};

__device__ __forceinline__ void soft_blend(const SoftBlend &s, int64_t p, int64_t n_agent, float p_new) {
    float *t = p < n_agent ? s.agent + p : s.mixer + (p - n_agent);
    *t = __fadd_rn(__fmul_rn(*t, s.c1), __fmul_rn(p_new, s.c2));   // _rn intrinsics: never contracted into an FMA
}

// SOFT = false ignores `soft`; SOFT = true also blends every parameter's target, the frozen prefix included (its
// parameters do not move, so the blend reads them unchanged).
template <bool SOFT>
__global__ void __launch_bounds__(256) k_clip_rmsprop(float *agent, int64_t n_agent, float *mixer, int64_t n_mixer,
                                                      float *grad, float *sq, const float *norm_part, int n_part,
                                                      float lr, float alpha, float eps, float clip, float *scalars,
                                                      const float *denominator, int64_t n_frozen, SoftBlend soft) {
    __shared__ float s_red[8];
    __shared__ float s_coef;
    pdl_wait();
    clip_coef_prologue(norm_part, n_part, clip, scalars, s_red, s_coef);
    __syncthreads();
    const float coef = s_coef;
    const int64_t p = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (p >= n_agent + n_mixer) return;
    float *param = p < n_agent ? agent + p : mixer + (p - n_agent);
    if (p < n_frozen) {                                   // frozen parameters: RMSprop skips them (p.grad is None)
        if constexpr (SOFT) soft_blend(soft, p, n_agent, *param);
        return;
    }
    const float gv = grad[p] * (denominator ? 1.0f / denominator[0] : 1.0f) * coef;
    grad[p] = gv;   // clip_grad_norm_ scales .grad in place
    const float v = alpha * sq[p] + (1.0f - alpha) * gv * gv;
    sq[p] = v;
    const float pn = *param - lr * gv / (sqrtf(v) + eps);
    *param = pn;
    if constexpr (SOFT) soft_blend(soft, p, n_agent, pn);
}

// clip_grad_norm_ + torch.optim.Adam.step (amsgrad = False, maximize = False, L2 weight decay added to the gradient),
// one pass over the flat buffers.  state = exp_avg[P] | exp_avg_sq[P] | step (f32) | ticket (u32).  The step counter
// lives on the device so that a replayed CUDA graph advances it: every block reads the old step, then takes a ticket;
// the last block to arrive (all others have read by then) re-arms the ticket and writes step + 1.
template <bool SOFT>
__global__ void __launch_bounds__(256) k_clip_adam(float *agent, int64_t n_agent, float *mixer, int64_t n_mixer,
                                                   float *grad, float *state, const float *norm_part, int n_part,
                                                   mal_adam_t h, float *scalars, const float *denominator, int64_t n_frozen,
                                                   SoftBlend soft) {
    __shared__ float s_red[8];
    __shared__ float s_coef, s_step_size, s_bc2_sqrt;
    pdl_wait();
    const int64_t P = n_agent + n_mixer;
    clip_coef_prologue(norm_part, n_part, h.clip, scalars, s_red, s_coef);
    if (threadIdx.x == 0) {
        const float step = state[2 * P];
        const double t = (double)step + 1.0;
        // bias corrections in double, as torch's non-capturable Adam computes them on the host
        s_step_size = (float)(-h.lr / (1.0 - pow(h.beta1, t)));
        s_bc2_sqrt = (float)sqrt(1.0 - pow(h.beta2, t));
        unsigned *ticket = reinterpret_cast<unsigned *>(state + 2 * P + 1);
        __threadfence();                                          // this block's read of step precedes its ticket
        if (atomicAdd(ticket, 1u) == gridDim.x - 1) {
            __threadfence();
            *ticket = 0u;
            state[2 * P] = step + 1.0f;
        }
    }
    __syncthreads();
    const float coef = s_coef, step_size = s_step_size, bc2_sqrt = s_bc2_sqrt;
    const int64_t p = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (p >= P) return;
    float *param = p < n_agent ? agent + p : mixer + (p - n_agent);
    if (p < n_frozen) {                                           // frozen parameters: Adam skips them (p.grad is None)
        if constexpr (SOFT) soft_blend(soft, p, n_agent, *param);
        return;
    }
    float g = grad[p] * (denominator ? 1.0f / denominator[0] : 1.0f) * coef;
    grad[p] = g;                                                  // clip_grad_norm_ scales .grad in place
    const float pv = *param;
    if (h.weight_decay != 0.0) g += (float)h.weight_decay * pv;  // grad.add(param, alpha=weight_decay): not written back
    const float m = state[p], v = state[P + p];
    const float mn = m + (float)(1.0 - h.beta1) * (g - m);                 // exp_avg.lerp_(grad, 1 - beta1)
    const float vn = v * (float)h.beta2 + (float)(1.0 - h.beta2) * g * g;  // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
    state[p] = mn;
    state[P + p] = vn;
    const float pn = pv + step_size * (mn / (sqrtf(vn) / bc2_sqrt + (float)h.eps));   // addcdiv_(exp_avg, denom, -step_size)
    *param = pn;
    if constexpr (SOFT) soft_blend(soft, p, n_agent, pn);
}

__global__ void __launch_bounds__(256) k_copy_f32(float *dst, const float *src, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    const int64_t n4 = n / 4;
    if ((((uintptr_t)dst | (uintptr_t)src) & 15) == 0) {
        for (int64_t j = i; j < n4; j += (int64_t)gridDim.x * 256)
            reinterpret_cast<float4 *>(dst)[j] = reinterpret_cast<const float4 *>(src)[j];
        for (int64_t j = n4 * 4 + i; j < n; j += (int64_t)gridDim.x * 256) dst[j] = src[j];
    } else {
        for (int64_t j = i; j < n; j += (int64_t)gridDim.x * 256) dst[j] = src[j];
    }
}
