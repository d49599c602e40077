// Common device/host helpers for libmal_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <math.h>
#include "../../include/mal_b200.h"

#define HID MAL_HID          // rnn_hidden_dim
#define G3 (3 * MAL_HID)     // GRU gate rows (r|z|n)

// ---------------------------------------------------------------------------------------------
// error plumbing (host)
// ---------------------------------------------------------------------------------------------
void mal_set_error(const char *fmt, ...);

#define MAL_REQUIRE(cond, ...)                 \
    do {                                       \
        if (!(cond)) {                         \
            mal_set_error(__VA_ARGS__);        \
            return 1;                          \
        }                                      \
    } while (0)

#define MAL_CUDA(expr)                                                                     \
    do {                                                                                   \
        cudaError_t _e = (expr);                                                           \
        if (_e != cudaSuccess) {                                                           \
            mal_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return 2;                                                                      \
        }                                                                                  \
    } while (0)

#define MAL_LAUNCH_CHECK(name)                                                             \
    do {                                                                                   \
        cudaError_t _e = cudaGetLastError();                                               \
        if (_e != cudaSuccess) {                                                           \
            mal_set_error("launch of %s failed: %s", name, cudaGetErrorString(_e));        \
            return 3;                                                                      \
        }                                                                                  \
    } while (0)

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline int64_t align_up64(int64_t a, int64_t b) { return ceil_div64(a, b) * b; }

// ---------------------------------------------------------------------------------------------
// parameter layouts (offsets in floats inside the flat state_dict-ordered buffers)
// ---------------------------------------------------------------------------------------------
struct AgentLayout {   // drqn_agent.py:21-23
    int d_in, n_actions;
    int64_t fc1_w, fc1_b, w_ih, w_hh, b_ih, b_hh, fc2_w, fc2_b, total;
};
// kind MAL_AGENT_RNN: fc1 | gru | fc2 (drqn_agent.py:21-23); MAL_AGENT_DQN: fc1 | fc2 (dqn_agent.py:24-25)
__host__ __device__ inline AgentLayout agent_layout(int d_in, int n_actions, int kind = MAL_AGENT_RNN) {
    AgentLayout L;
    L.d_in = d_in; L.n_actions = n_actions;
    int64_t o = 0;
    L.fc1_w = o; o += (int64_t)HID * d_in;
    L.fc1_b = o; o += HID;
    L.w_ih = L.w_hh = L.b_ih = L.b_hh = -1;
    if (kind == MAL_AGENT_RNN) {
        L.w_ih = o;  o += (int64_t)G3 * HID;
        L.w_hh = o;  o += (int64_t)G3 * HID;
        L.b_ih = o;  o += G3;
        L.b_hh = o;  o += G3;
    }
    L.fc2_w = o; o += (int64_t)n_actions * HID;
    L.fc2_b = o; o += n_actions;
    L.total = o;
    return L;
}

// Column layout of fc1's input, basic_controller.py:80-101:  [obs | one-hot(a_{t-1}) | one-hot(agent id)], the last two
// blocks switched by obs_last_action / obs_agent_id.  Every loader and epilogue that touches fc1's input takes its
// column bounds from here: obs columns [0, obs), last-action columns [obs, obs + last), agent-id columns
// [obs + last, d_in).  The blocks are given as widths so that the kernels keep the arithmetic of the fixed layout, with
// `last` / `id` where they read n_actions / n_agents.
struct AgentInput {
    int obs;        // OBS
    int last;       // width of the last-action block: A * obs_last_action
    int id;         // width of the agent-id block: N * obs_agent_id
    int d_in;       // fc1 input width, obs + last + id
    __host__ __device__ int last_end() const { return obs + last; }
};
__host__ __device__ inline AgentInput agent_input(int OBS, int A, int N, int flags) {   // flags: MAL_IN_* bits
    AgentInput in;
    in.obs = OBS;
    in.last = (flags & MAL_IN_NO_LAST_ACTION) ? 0 : A;
    in.id = (flags & MAL_IN_NO_AGENT_ID) ? 0 : N;
    in.d_in = OBS + in.last + in.id;
    return in;
}

// QMIX (1- or 2-layer hypernetworks) is the only mixer with parameters, hypernet intermediates and a mixer backward;
// VDN and the absent mixer (IQL, MAL_MIXER_NONE) have none.  Every "is there a hypernetwork" branch tests this.
__host__ __device__ inline bool mixer_has_hypernet(int mixer) { return mixer == MAL_MIXER_QMIX2 || mixer == MAL_MIXER_QMIX1; }

struct MixerLayout {   // qmix.py:16-39 (layers == 2: Linear-ReLU-Linear hypernets; == 1: single Linear)
    int S, N, E, HE, layers;
    int64_t w1a_w, w1a_b, w1b_w, w1b_b;   // hyper_w_1.{0,2}  (layers==1: only w1b = hyper_w_1, K = S)
    int64_t wfa_w, wfa_b, wfb_w, wfb_b;   // hyper_w_final.{0,2}
    int64_t b1_w, b1_b, v0_w, v0_b, v2_w, v2_b, total;
};
__host__ __device__ inline MixerLayout mixer_layout(int mixer, int S, int N, int E, int HE) {
    MixerLayout L;
    L.S = S; L.N = N; L.E = E; L.HE = HE; L.layers = (mixer == MAL_MIXER_QMIX2) ? 2 : 1;
    int64_t o = 0;
    if (!mixer_has_hypernet(mixer)) { L.total = 0; L.layers = 0; return L; }
    if (L.layers == 2) {
        L.w1a_w = o; o += (int64_t)HE * S;  L.w1a_b = o; o += HE;
        L.w1b_w = o; o += (int64_t)E * N * HE; L.w1b_b = o; o += E * N;
        L.wfa_w = o; o += (int64_t)HE * S;  L.wfa_b = o; o += HE;
        L.wfb_w = o; o += (int64_t)E * HE;  L.wfb_b = o; o += E;
    } else {
        L.w1a_w = L.w1a_b = -1;
        L.w1b_w = o; o += (int64_t)E * N * S; L.w1b_b = o; o += E * N;
        L.wfa_w = L.wfa_b = -1;
        L.wfb_w = o; o += (int64_t)E * S;   L.wfb_b = o; o += E;
    }
    L.b1_w = o; o += (int64_t)E * S; L.b1_b = o; o += E;
    L.v0_w = o; o += (int64_t)E * S; L.v0_b = o; o += E;
    L.v2_w = o; o += E;              L.v2_b = o; o += 1;
    L.total = o;
    return L;
}

// ---------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ float sigmoidf_acc(float x) { return 1.0f / (1.0f + expf(-x)); }

// torch.max / argmax ordering: NaN beats everything, ties resolve to the lowest index.
__device__ __forceinline__ bool arg_better(float av, int ai, float bv, int bi) {
    bool an = (av != av), bn = (bv != bv);
    if (an || bn) {
        if (an && bn) return ai < bi;
        return an;
    }
    if (av > bv) return true;
    if (av < bv) return false;
    return ai < bi;
}

__device__ __forceinline__ void warp_argmax(float &v, int &i) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        float ov = __shfl_xor_sync(0xffffffffu, v, o);
        int oi = __shfl_xor_sync(0xffffffffu, i, o);
        if (arg_better(ov, oi, v, i)) { v = ov; i = oi; }
    }
}

template <typename T>
__device__ __forceinline__ const T *field_ptr(const mal_field_t &f, int64_t b, int64_t t) {
    return reinterpret_cast<const T *>(f.ptr) + b * f.sb + t * f.st;
}

// ---------------------------------------------------------------------------------------------
// mbarrier + bulk-copy engine (TMA, non-tensor form) helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE;\n"
        "bra WAIT_LOOP;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gsrc, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void bulk_s2g(void *gdst, const void *smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(smem_src)),
                 "r"(bytes)
                 : "memory");
}
// packed fp32x2 FMA (sm_100 FFMA2): two independent IEEE fp32 fused multiply-adds per instruction
__device__ __forceinline__ unsigned long long pack2(float lo, float hi) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(unsigned long long v, float &lo, float &hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long fma2(unsigned long long a, unsigned long long b, unsigned long long c) {
    unsigned long long d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}

// per-thread asynchronous copies (LDGSTS): src_bytes < size zero-fills the rest (src_bytes = 0: pure zero fill)
__device__ __forceinline__ void cp_async4(void *smem_dst, const void *gsrc, int src_bytes = 4) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gsrc, int src_bytes = 16) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
// programmatic dependent launch: a kernel launched with the programmatic-serialization attribute may start while its
// stream predecessor is still running; it may only touch what the predecessor produces after pdl_wait() (a no-op when
// the kernel was launched without the attribute).  pdl_trigger() in the predecessor lets the dependent grid be scheduled
// as soon as every CTA of the predecessor has issued it (or exited).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
// read-only loads that keep their program position relative to pdl_wait() (the compiler is free to sink a plain __ldg
// below the wait, which would serialise the weight loads behind the predecessor kernel again)
__device__ __forceinline__ float ldg_ordered(const float *p) {
    float v;
    asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ float4 ldg_ordered(const float4 *p) {
    float4 v;
    asm volatile("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

