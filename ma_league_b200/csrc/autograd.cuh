// Backward of the stand-alone module calls (BasicMAC.forward / agent.forward one step, QMixer.forward) for torch autograd:
// element-wise / per-row kernels only.  The weight gradients are row reductions that go through the learner's own
// split reductions (k_reduce_group / k_reduce_tc) and its fixed-order gather k_grad_reduce, so every gradient is
// bit-reproducible (no float atomics).
#pragma once
#include "mal_common.cuh"

// =============================================================================================
// one agent step, backward: recompute fc1 -> ReLU -> GRUCell (or fc1 -> ReLU for the DQN agent) from the input and h_in,
// then push d q / d h_out back through fc2, the GRU gates and the ReLU.  ABR_ROWS rows per CTA, staged in shared memory;
// thread item = (output unit, group of 8 rows), weights read through the L1 (one pass per CTA and matrix).
// =============================================================================================
#define ABR_ROWS 16
#define ABR_THREADS 256
struct AgentBwdArgs {
    const float *params;
    int kind, rows, N, OBS, A, dense;
    AgentInput in;                 // fc1 input columns (dense: obs = d_in, last = id = 0)
    const float *obs; int64_t obs_sb;
    const float *onehot; int64_t onehot_sb;   // NULL: zeros (t == 0)
    const float *h_in;             // [rows,64] or NULL (zeros)
    const float *d_q;              // [rows,A] or NULL (zeros)
    const float *d_h_out;          // [rows,64] or NULL (zeros)
    float *xin; int ldi;           // assembled input [rows, ldi] (fused assembly only; NULL in dense mode)
    float *x1;                     // relu(fc1) [rows,64]
    float *hp;                     // h_in with zeros for NULL [rows,64] (written only when h_in == NULL)
    float *hn;                     // h_out [rows,64] (recurrent agent)
    float *dq;                     // d_q, zeros for NULL [rows,A]
    float *d_g;                    // [rows,256]: d gi_r | d gi_z | d gi_n | d gh_n (the learner's layout)
    float *d_x;                    // d fc1 pre-activation [rows,64]
    float *d_h_in;                 // [rows,64] or NULL
};

// out[r][n] (+)= sum_k in[r][k] * W(n,k) for the CTA's rows; W(n,k) = W[n*ldw + k] (TRANS: W[k*ldw + n]).
// Items (n, 8-row group) are spread over the threads; the k order is fixed, so results are reproducible.
template <bool TRANS>
__device__ __forceinline__ void abr_mv(const float *__restrict__ W, int64_t ldw, const float *__restrict__ bias,
                                       const float *in, int ld_in, int K, int Nout, float *out, int ld_out) {
    for (int it = threadIdx.x; it < Nout * (ABR_ROWS / 8); it += ABR_THREADS) {
        const int n = it % Nout, g = it / Nout;
        const float b = bias ? __ldg(bias + n) : 0.0f;
        float acc[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) acc[r] = b;
        const float *ip = in + (g * 8) * ld_in;
        for (int k = 0; k < K; ++k) {
            const float w = TRANS ? __ldg(W + (int64_t)k * ldw + n) : __ldg(W + (int64_t)n * ldw + k);
#pragma unroll
            for (int r = 0; r < 8; ++r) acc[r] = fmaf(ip[r * ld_in + k], w, acc[r]);
        }
#pragma unroll
        for (int r = 0; r < 8; ++r) out[(g * 8 + r) * ld_out + n] = acc[r];
    }
}

__global__ void __launch_bounds__(ABR_THREADS) k_agent_step_bwd(const __grid_constant__ AgentBwdArgs a) {
    extern __shared__ __align__(16) float abr_smem[];
    const bool rnn = a.kind == MAL_AGENT_RNN;
    const int d_in = a.in.d_in, A = a.A;
    const AgentLayout L = agent_layout(d_in, A, a.kind);
    const int ld_in = d_in + 1;                                    // odd stride: the row groups hit different banks
    float *s_in = abr_smem;                                        // [16][d_in+1], later [16][64] (d h_prev sums)
    float *s_x1 = s_in + ABR_ROWS * (ld_in > HID ? ld_in : HID);   // [16][64]
    float *s_h = s_x1 + ABR_ROWS * HID;                            // [16][64]   h_{t-1}
    float *s_g = s_h + ABR_ROWS * HID;                             // [16][384]  gi | gh, then d gi | d gh
    float *s_dh = s_g + ABR_ROWS * 2 * G3;                         // [16][64]   d h_out, then d h'
    float *s_dq = s_dh + ABR_ROWS * HID;                           // [16][32]
    float *s_t = s_dq + ABR_ROWS * MAL_MAX_ACTIONS;                // [16][64]   scratch (fc2^T . d q, dh_prev / d x sums)
    const int64_t r0 = (int64_t)blockIdx.x * ABR_ROWS;
    const int tid = threadIdx.x;

    // ---- stage the rows (rows past the end are zeros and never stored)
    for (int e = tid; e < ABR_ROWS * d_in; e += ABR_THREADS) {
        const int r = e / d_in, k = e - r * d_in;
        const int64_t row = r0 + r;
        float v = 0.0f;
        if (row < a.rows) {
            if (a.dense) v = a.obs[row * a.obs_sb + k];
            else {
                const int64_t b = row / a.N; const int n = (int)(row - b * a.N);
                if (k < a.in.obs) v = a.obs[b * a.obs_sb + (int64_t)n * a.OBS + k];
                else if (k < a.in.last_end()) v = a.onehot ? a.onehot[b * a.onehot_sb + (int64_t)n * A + (k - a.in.obs)] : 0.0f;
                else v = (k - a.in.last_end()) == n ? 1.0f : 0.0f;
                a.xin[row * a.ldi + k] = v;
            }
        }
        s_in[r * ld_in + k] = v;
    }
    for (int e = tid; e < ABR_ROWS * HID; e += ABR_THREADS) {
        const int r = e / HID;
        const int64_t row = r0 + r;
        const bool ok = row < a.rows;
        float h = 0.0f, dh = 0.0f;
        if (ok && rnn) {
            h = a.h_in ? a.h_in[r0 * HID + e] : 0.0f;
            if (!a.h_in) a.hp[r0 * HID + e] = 0.0f;
            dh = a.d_h_out ? a.d_h_out[r0 * HID + e] : 0.0f;
        }
        s_h[e] = h; s_dh[e] = dh;
    }
    for (int e = tid; e < ABR_ROWS * A; e += ABR_THREADS) {
        const int r = e / A, c = e - r * A;
        const int64_t row = r0 + r;
        float v = 0.0f;
        if (row < a.rows) { v = a.d_q ? a.d_q[row * A + c] : 0.0f; a.dq[row * A + c] = v; }
        s_dq[r * MAL_MAX_ACTIONS + c] = v;
    }
    __syncthreads();

    // ---- forward recompute: x1 = relu(fc1 in), gi = W_ih x1 + b_ih, gh = W_hh h + b_hh
    abr_mv<false>(a.params + L.fc1_w, d_in, a.params + L.fc1_b, s_in, ld_in, d_in, HID, s_x1, HID);
    // fc2^T . d q (independent of the recompute)
    abr_mv<true>(a.params + L.fc2_w, HID, nullptr, s_dq, MAL_MAX_ACTIONS, A, HID, s_t, HID);
    __syncthreads();
    for (int e = tid; e < ABR_ROWS * HID; e += ABR_THREADS) {
        const float x = fmaxf(s_x1[e], 0.0f);
        s_x1[e] = x;
        const int64_t row = r0 + e / HID;
        if (row < a.rows) a.x1[r0 * HID + e] = x;
    }
    __syncthreads();
    if (!rnn) {   // DQN: d x = (fc2^T . d q) * (x > 0)
        for (int e = tid; e < ABR_ROWS * HID; e += ABR_THREADS) {
            const int64_t row = r0 + e / HID;
            if (row < a.rows) a.d_x[r0 * HID + e] = s_x1[e] > 0.0f ? s_t[e] : 0.0f;
        }
        return;
    }
    abr_mv<false>(a.params + L.w_ih, HID, a.params + L.b_ih, s_x1, HID, HID, G3, s_g, 2 * G3);
    abr_mv<false>(a.params + L.w_hh, HID, a.params + L.b_hh, s_h, HID, HID, G3, s_g + G3, 2 * G3);
    __syncthreads();

    // ---- GRUCell gates (torch: r, z, n = tanh(gi_n + r * (W_hn h + b_hn)), h' = n + z (h - n)) and their gradients
    for (int e = tid; e < ABR_ROWS * HID; e += ABR_THREADS) {
        const int r = e / HID, j = e - r * HID;
        float *g = s_g + r * 2 * G3;
        const float rg = sigmoidf_acc(g[j] + g[G3 + j]);
        const float zg = sigmoidf_acc(g[HID + j] + g[G3 + HID + j]);
        const float ghn = g[G3 + 2 * HID + j];
        const float ng = tanhf(g[2 * HID + j] + rg * ghn);
        const float hprev = s_h[e];
        const float hnew = ng + zg * (hprev - ng);
        const float dh = s_dh[e] + s_t[e];                             // d h' = d h_out + fc2^T . d q
        const float dn_pre = dh * (1.0f - zg) * (1.0f - ng * ng);
        const float dz_pre = dh * (hprev - ng) * zg * (1.0f - zg);
        const float dr_pre = dn_pre * ghn * rg * (1.0f - rg);
        g[j] = dr_pre; g[HID + j] = dz_pre; g[2 * HID + j] = dn_pre;   // d gi
        g[G3 + j] = dr_pre; g[G3 + HID + j] = dz_pre; g[G3 + 2 * HID + j] = dn_pre * rg;   // d gh
        s_dh[e] = dh * zg;                                             // direct path of d h_prev
        const int64_t row = r0 + r;
        if (row < a.rows) {
            a.hn[row * HID + j] = hnew;
            float *dg = a.d_g + row * 4 * HID;
            dg[j] = dr_pre; dg[HID + j] = dz_pre; dg[2 * HID + j] = dn_pre; dg[3 * HID + j] = dn_pre * rg;
        }
    }
    __syncthreads();
    // ---- d x = (d gi . W_ih) * (x1 > 0);  d h_prev = d h' z + d gh . W_hh
    abr_mv<true>(a.params + L.w_ih, HID, nullptr, s_g, 2 * G3, G3, HID, s_t, HID);
    if (a.d_h_in) abr_mv<true>(a.params + L.w_hh, HID, nullptr, s_g + G3, 2 * G3, G3, HID, s_in, HID);   // s_in is free now
    __syncthreads();
    for (int e = tid; e < ABR_ROWS * HID; e += ABR_THREADS) {
        const int64_t row = r0 + e / HID;
        if (row >= a.rows) continue;
        a.d_x[r0 * HID + e] = s_x1[e] > 0.0f ? s_t[e] : 0.0f;
        if (a.d_h_in) a.d_h_in[r0 * HID + e] = s_dh[e] + s_in[e];
    }
}

static inline size_t agent_bwd_smem(int d_in) {
    return sizeof(float) * (size_t)ABR_ROWS * ((d_in + 1 > HID ? d_in + 1 : HID) + HID * 4 + 2 * G3 + MAL_MAX_ACTIONS);
}

// =============================================================================================
// QMixer.forward backward, element-wise part (one warp per (b,t) row, lane = embed unit, like qmix_row): from the forward
// call's scratch (y1: [h1 | hf | b1 | v1] after their activations, a2: [a1 | af] before abs) and the upstream d q_tot:
// d agent_qs, the seeds d a2 / d y1 of the hypernet GEMM backward (abs' = sign of the raw value, 0 at 0, as torch),
// and per-block d V.2 partials [gridDim.x][E+1].
// =============================================================================================
struct MixBwdArgs {
    int mixer, B, T, N, E, HE, S;
    const float *params, *agent_qs, *y1, *a2, *d_q_tot;
    float *d_agent_qs, *d_a2, *d_y1, *part_v2;
};

__global__ void __launch_bounds__(256) k_mix_bwd(MixBwdArgs a) {
    __shared__ float s_v2[8][MAL_MAX_EMBED + 1];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t total = (int64_t)a.B * a.T;
    const MixerLayout ML = mixer_layout(a.mixer, a.S, a.N, a.E, a.HE);
    const int two = (ML.layers == 2);
    const int ld1 = two ? 2 * a.HE + 2 * a.E : 2 * a.E;
    const int ld2 = a.E * a.N + a.E;
    const int yo = two ? 2 * a.HE : 0;
    const bool act = lane < a.E;
    const float v2w = act ? __ldg(a.params + ML.v2_w + lane) : 0.0f;
    float dv2w = 0.0f, dv2b = 0.0f;
    for (int64_t m = (int64_t)blockIdx.x * 8 + warp; m < total; m += (int64_t)gridDim.x * 8) {
        const float qc = lane < a.N ? a.agent_qs[m * a.N + lane] : 0.0f;
        const float gseed = a.d_q_tot[m];
        const float *a2 = a.a2 + m * ld2;
        const float *y1 = a.y1 + m * ld1 + yo;
        float pre = act ? y1[lane] : 0.0f;
        const float af = act ? a2[a.N * a.E + lane] : 0.0f;
        const float wf = fabsf(af);
        const float v1 = act ? y1[a.E + lane] : 0.0f;
        for (int n = 0; n < a.N; ++n) {
            const float w1 = act ? fabsf(a2[n * a.E + lane]) : 0.0f;
            pre = fmaf(__shfl_sync(0xffffffffu, qc, n), w1, pre);
        }
        const float hidden = pre > 0.0f ? pre : expm1f(pre);
        const float dpre = gseed * wf * (pre > 0.0f ? 1.0f : expf(pre));
        float *da2 = a.d_a2 + m * ld2;
        float *dy1 = a.d_y1 + m * ld1 + yo;
        if (act) {
            da2[a.N * a.E + lane] = gseed * hidden * (af > 0.0f ? 1.0f : (af < 0.0f ? -1.0f : 0.0f));
            dy1[lane] = dpre;                                       // d hyper_b_1 out
            dy1[a.E + lane] = v1 > 0.0f ? gseed * v2w : 0.0f;       // d V.0 pre-activation
            dv2w += gseed * v1;
        }
        if (lane == 0) dv2b += gseed;
        float dq_mine = 0.0f;
        for (int n = 0; n < a.N; ++n) {
            const float a1 = act ? a2[n * a.E + lane] : 0.0f;
            const float dq = warp_sum(act ? dpre * fabsf(a1) : 0.0f);
            const float qn = __shfl_sync(0xffffffffu, qc, n);
            if (act) da2[n * a.E + lane] = qn * dpre * (a1 > 0.0f ? 1.0f : (a1 < 0.0f ? -1.0f : 0.0f));
            if (lane == n) dq_mine = dq;
        }
        if (lane < a.N) a.d_agent_qs[m * a.N + lane] = dq_mine;
    }
    if (lane < a.E) s_v2[warp][lane] = dv2w;
    if (lane == 0) s_v2[warp][a.E] = dv2b;
    __syncthreads();
    if (tid <= a.E) {
        float s = 0.0f;
        for (int w = 0; w < 8; ++w) s += s_v2[w][tid];
        a.part_v2[(int64_t)blockIdx.x * (a.E + 1) + tid] = s;
    }
}
