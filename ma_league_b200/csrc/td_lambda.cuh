// TD(lambda) targets of the learner step (build_td_lambda_targets, coma_learner.py:10-21, over the [B,T] target array).
//
// The 1-step step forms each row's target inside k_mix_td.  A lambda-return depends on every later row of its episode,
// so the lambda step runs three kernels where the 1-step step runs one:
//   k_mix_tq          one warp per (b,t): the target mixer row only -> target_q_tot (the target half of k_mix_td, through
//                     the shared qmix_row); IQL copies target_max
//   k_td_lambda       one warp per episode (per (b, agent) for IQL): the reverse recursion in fp64 -> targets
//   k_mix_td_lambda   k_mix_td reading those targets (online mixer row, TD error, loss terms, seeds, statistics)
#pragma once
#include "mal_common.cuh"
#include "learner.cuh"

__global__ void __launch_bounds__(256) k_mix_tq(MixArgs a) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t total = (int64_t)a.B * a.T;
    pdl_wait();
    for (int64_t m = (int64_t)blockIdx.x * 8 + warp; m < total; m += (int64_t)gridDim.x * 8) {
        const float qt = lane < a.N ? a.target_max[m * a.N + lane] : 0.0f;
        if (a.mixer == MAL_MIXER_NONE) {                  // warp-uniform
            if (lane < a.N) a.target_q_tot[m * a.N + lane] = qt;
            continue;
        }
        float ty;
        if (a.mixer == MAL_MIXER_VDN) {
            ty = warp_sum(qt);
        } else {
            float d0, d1, d2, d3;
            ty = qmix_row(a, 1, m, [&](int n) { return __shfl_sync(0xffffffffu, qt, n); }, lane, &d0, &d1, &d2, &d3);
        }
        if (lane == 0) a.target_q_tot[m] = ty;
    }
    pdl_trigger();
}

struct TdLambdaArgs {
    const float *tq;               // target_q_tot [B,T,Q]
    float *targets;                // [B,T,Q] out
    mal_field_t reward, terminated, filled;
    int B, T, Q;                   // Q = N for IQL, else 1
    double lg, xg;                 // lambda * gamma, (1 - lambda) * gamma
};

#define TDL_WARPS 2                // warps (episodes) per CTA: B = 32 spreads over 16 SMs

// R[T] = tq[T-1] (1 - sum_t term[t]);  R[t] = lg R[t+1] + m[t] (r[t] + xg (1 - term[t]) tq[t]),  t = T-1 .. 0.
// Chunks of 32 steps from the end: lane i holds step t = 32k + i; a suffix scan over the chunk (Hillis-Steele, factor lg^d
// at distance d) gives S[t] = sum_{t <= s < end} lg^(s-t) x[s], and R[t] = S[t] + lg^(end-t) R[end] with the carry R[end]
// from the chunk after it.  fp64 throughout, fixed order, no atomics: deterministic.
__global__ void __launch_bounds__(32 * TDL_WARPS) k_td_lambda(TdLambdaArgs a) {
    const int lane = threadIdx.x & 31;
    const int64_t e = (int64_t)blockIdx.x * TDL_WARPS + (threadIdx.x >> 5);
    pdl_wait();
    if (e < (int64_t)a.B * a.Q) {                         // warp-uniform
        const int b = (int)(e / a.Q), n = (int)(e - (int64_t)b * a.Q);
        const float *tq = a.tq + (int64_t)b * a.T * a.Q + n;   // step t at tq[t * Q]
        int nterm = 0;
        for (int t = lane; t < a.T; t += 32) nterm += *field_ptr<unsigned char>(a.terminated, b, t);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) nterm += __shfl_xor_sync(0xffffffffu, nterm, o);
        double carry = (double)tq[(int64_t)(a.T - 1) * a.Q] * (1.0 - (double)nterm);
        auto x_of = [&](int k) -> double {                // this lane's x of chunk k (0 past the end)
            const int t = k * 32 + lane;
            if (t >= a.T) return 0.0;
            float mk = (float)(*field_ptr<long long>(a.filled, b, t));
            if (t > 0) mk = mk * (1.0f - (float)(*field_ptr<unsigned char>(a.terminated, b, t - 1)));   // make_mask
            const double r = *field_ptr<float>(a.reward, b, t);
            const double term = *field_ptr<unsigned char>(a.terminated, b, t);
            return (double)mk * (r + a.xg * (1.0 - term) * (double)tq[(int64_t)t * a.Q]);
        };
        const int nch = (a.T + 31) / 32;
        double x = x_of(nch - 1);
        for (int k = nch - 1; k >= 0; --k) {
            const double x_next = k > 0 ? x_of(k - 1) : 0.0;   // the next chunk's loads fly under this chunk's scan
            double s = x, cd = a.lg;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const double y = __shfl_down_sync(0xffffffffu, s, d);
                if (lane + d < 32) s = fma(cd, y, s);
                cd *= cd;
            }
            const int t = k * 32 + lane, end = min(k * 32 + 32, a.T);
            const double R = t < a.T ? fma(pow(a.lg, (double)(end - t)), carry, s) : 0.0;
            if (t < a.T) a.targets[((int64_t)b * a.T + t) * a.Q + n] = (float)R;
            carry = __shfl_sync(0xffffffffu, R, 0);
            x = x_next;
        }
    }
    pdl_trigger();
}
