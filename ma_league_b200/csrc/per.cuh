// Proportional prioritized episode replay (Schaul et al., 2016) over the slots of a device-resident replay buffer.
//
// k_per_sample: ONE CTA per sample.  Thread k owns the contiguous slice [k*per, (k+1)*per) of the n live priorities;
// the slice sums are accumulated sequentially in fp64 and scanned across the CTA in a fixed shuffle order, so two calls
// on the same priorities and uniforms give bit-identical ids.  Draw j lands at x_j = (j + u_j) * total / B (stratified,
// one uniform per draw); the CTA finds the first slice whose inclusive prefix exceeds x_j by binary search over the slice
// prefixes in shared memory, then the drawing thread rescans that slice.  A single CTA is enough up to 10^6 episodes
// (DESIGN.md section 4 has the measurement).
// k_per_update: one warp per sampled episode: (sum_t |td*m| / sum_t m + eps)^alpha written to its slot, and the running
// maximum raised with an integer atomicMax on the (non-negative) float bits, which is exact and order-independent.
#pragma once
#include "mal_common.cuh"

#define PER_THREADS 1024

struct PerSampleArgs {
    const float *p;            // [n] priorities of the live slots, 16-byte aligned
    int64_t n, per;            // live slots, slice length per thread (multiple of 4)
    int B;
    float beta;
    const float *u;            // [B] injected uniforms, or NULL: Philox (seed, offset) in th.rand(B)'s layout
    uint64_t seed, offset;
    uint32_t grid;             // grid of torch's uniform kernel for B elements
    int64_t *ids;              // [B] out
    float *w;                  // [B] out
};

__global__ void __launch_bounds__(PER_THREADS) k_per_sample(PerSampleArgs a) {
    __shared__ double s_pref[PER_THREADS];     // inclusive prefix of the slice sums
    __shared__ double s_wsum[32];
    __shared__ float s_wmin[32];
    __shared__ long long s_wlast[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t lo = min(a.n, (int64_t)tid * a.per), hi = min(a.n, lo + a.per);
    double s = 0.0;
    float mn = INFINITY;
    long long last = -1;                         // last slot of the slice with a positive priority
    int64_t i = lo;
    for (; i + 4 <= hi; i += 4) {
        const float4 v = *reinterpret_cast<const float4 *>(a.p + i);
        s += (double)v.x; s += (double)v.y; s += (double)v.z; s += (double)v.w;
        mn = fminf(fminf(mn, v.x), fminf(v.y, fminf(v.z, v.w)));
        if (v.w > 0.0f) last = i + 3; else if (v.z > 0.0f) last = i + 2; else if (v.y > 0.0f) last = i + 1;
        else if (v.x > 0.0f) last = i;
    }
    for (; i < hi; ++i) {
        const float v = a.p[i];
        s += (double)v; mn = fminf(mn, v);
        if (v > 0.0f) last = i;
    }
    double x = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
    }
    if (lane == 31) s_wsum[warp] = x;
    if (lane == 0) { s_wmin[warp] = mn; s_wlast[warp] = last; }
    __syncthreads();
    if (warp == 0) {
        double v = s_wsum[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double y = __shfl_up_sync(0xffffffffu, v, o);
            if (lane >= o) v += y;
        }
        s_wsum[lane] = v;
        float m = s_wmin[lane];
        long long l = s_wlast[lane];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            m = fminf(m, __shfl_xor_sync(0xffffffffu, m, o));
            l = max(l, __shfl_xor_sync(0xffffffffu, l, o));
        }
        if (lane == 0) { s_wmin[0] = m; s_wlast[0] = l; }
    }
    __syncthreads();
    s_pref[tid] = x + (warp > 0 ? s_wsum[warp - 1] : 0.0);
    __syncthreads();
    const double total = s_pref[PER_THREADS - 1];
    const float pmin = s_wmin[0];
    const long long any_last = s_wlast[0];
    for (int j = tid; j < a.B; j += PER_THREADS) {
        const float u = a.u ? a.u[j] : torch_uniform01(torch_philox_uniform(a.seed, a.offset, a.grid, (uint64_t)j));
        const double pt = ((double)j + (double)u) * total / (double)a.B;
        int k = 0, kh = PER_THREADS;             // first slice with s_pref[k] > pt (kh: none)
        while (k < kh) {
            const int mid = (k + kh) >> 1;
            if (s_pref[mid] > pt) kh = mid; else k = mid + 1;
        }
        long long id = -1;
        if (k < PER_THREADS) {
            double r = k > 0 ? s_pref[k - 1] : 0.0;
            const int64_t l0 = (int64_t)k * a.per, l1 = min(a.n, l0 + a.per);
            long long pos = -1;
            for (int64_t e = l0; e < l1; ++e) {
                const float v = a.p[e];
                r += (double)v;
                if (v > 0.0f) pos = e;
                if (r > pt) { id = e; break; }
            }
            if (id < 0) id = pos;                // rounding at the slice's end: its last positive slot
        }
        if (id < 0) id = any_last >= 0 ? any_last : a.n - 1;   // x at total by rounding, or no positive priority at all
        const float pid = a.p[id];
        a.ids[j] = id;
        a.w[j] = pid > 0.0f ? (float)pow((double)pmin / (double)pid, (double)a.beta) : 1.0f;
    }
}

struct PerUpdateArgs {
    const float *td;           // [B*T*nq], row m = b*T + t
    const float *mask;         // [B*T]
    int B, T, nq;
    const int64_t *ids;        // [B]
    int64_t capacity;          // slots of `priorities`; ids outside [0, capacity) are skipped
    float alpha, eps;
    float *priorities;
    float *max_priority;       // [1]
};

__global__ void __launch_bounds__(256) k_per_update(PerUpdateArgs a) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * 8 + warp;
    if (b >= a.B) return;
    const long long id = a.ids[b];
    bool later = false;                          // a later batch index samples the same slot: that occurrence wins
    for (int k = b + 1 + lane; k < a.B; k += 32) later |= (a.ids[k] == id);
    if (__any_sync(0xffffffffu, later) || id < 0 || id >= a.capacity) return;
    float s = 0.0f, ms = 0.0f;
    for (int t = lane; t < a.T; t += 32) {
        const int64_t m = (int64_t)b * a.T + t;
        const float mk = a.mask[m];
        ms += mk;
        for (int n = 0; n < a.nq; ++n) s += fabsf(a.td[m * a.nq + n] * mk);
    }
    s = warp_sum(s);
    ms = warp_sum(ms) * (float)a.nq;
    if (lane == 0) {
        const double mean = ms > 0.0f ? (double)s / (double)ms : 0.0;
        const float pr = (float)pow(mean + (double)a.eps, (double)a.alpha);
        a.priorities[id] = pr;
        atomicMax(reinterpret_cast<int *>(a.max_priority), __float_as_int(pr));
    }
}
