// Shared device helpers for the relation-autoencoder kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace rae {

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;

// ---- programmatic dependent launch (the step is a chain of ~20 dependent kernels, most of them 5-60 us) ----
// Every kernel of the step starts with pdl_enter(): it lets the NEXT kernel of the stream be scheduled already (its CTAs
// become resident as SM resources free up and park in griddepcontrol.wait) and then waits until the PREVIOUS kernel of the
// stream has completed and flushed its memory - before this kernel's first global access, so the data dependencies are
// exactly those of plain stream order.  What overlaps is launch latency, CTA placement and the tail of the previous
// kernel's last wave.  A kernel launched without the attribute executes both instructions as no-ops.
__device__ __forceinline__ void pdl_enter() {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
}

#ifdef __CUDACC__
extern bool g_pdl_enabled;      // rae_engine.cu; cleared by RAE_FLAG_NO_PDL (A/B measurements)
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = g_pdl_enabled ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, KArgs(static_cast<Args&&>(args))...);
}
#endif

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(kFull, v, o));
    return v;
}

// log(sigmoid(x)) = -softplus(-x), stable for both signs (Bilinear.py:38,47 after Theano's own rewrite)
__device__ __forceinline__ float log_sigmoid(float x) {
    return fminf(x, 0.f) - log1pf(expf(-fabsf(x)));
}
__device__ __forceinline__ float sigmoidf(float x) {
    // 1/(1+exp(-x)) without overflow for large |x|
    float e = expf(-fabsf(x));
    float s = 1.f / (1.f + e);
    return x >= 0.f ? s : e * s;
}

__device__ __forceinline__ float ld_nc(const float* p) { return __ldg(p); }
// 16-byte read-only load that stays where it is written (volatile asm keeps program order): a run of these is issued back
// to back, so the loads of a thread cost one memory latency instead of one each
__device__ __forceinline__ float4 ldg_stream4(const float* p) {
    float4 v;
    asm volatile("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}

// AdaGrad row rule, Optimizers.py:29-32: acc' = acc + g^2 ; p' = p - lr*g/(sqrt(acc') + 1e-6)
// sqrt.approx / rcp.approx (1 ulp each, MUFU) instead of the IEEE sequences: the update kernels are instruction-bound and
// the rule is checked against its float64 evaluation at 2e-6 relative (tests/test_gpu_parity.py), 3 ulp is 4e-7.
__device__ __forceinline__ void adagrad_apply(float& p, float& acc, float g, float lr) {
    acc = fmaf(g, g, acc);
    float r, inv;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(acc));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(r + 1e-6f));
    p = fmaf(-lr * g, inv, p);
}

// the handle's optimiser rule on one element: AdaGrad (above) or SGD, Optimizers.py:51 (p' = p - lr*g; acc untouched)
__device__ __forceinline__ void opt_step(float& w, float& a, float g, float lr, int adagrad) {
    if (adagrad) adagrad_apply(w, a, g, lr);
    else w -= lr * g;
}
__device__ __forceinline__ void opt_step(float4& w, float4& a, const float4& g, float lr, int adagrad) {
    opt_step(w.x, a.x, g.x, lr, adagrad); opt_step(w.y, a.y, g.y, lr, adagrad);
    opt_step(w.z, a.z, g.z, lr, adagrad); opt_step(w.w, a.w, g.w, lr, adagrad);
}

// v[b,j], w[b,j] of the tensor-core contraction from its partial buffers (rae_decoder_tc.cu):
//   vg [2][B][dp]          DP=128: both epilogue groups hold a half-row partial; DP=64: group j%2; DP=32: group (j/2)%2
//   wp [slot][2][B][dp]    sum over the NS = tcs_nslots(schedule, b / 128) slots of the example's tile of the group
//                          partials (DP=128: only group j/64 holds column j)
// The consumers (scoring, backward finish) read them directly: no separate combine pass.
__device__ __forceinline__ void tc_combined_vw(const float* __restrict__ vg, const float* __restrict__ wp, int B, int dp, int DP,
                                               int NS, int b, int j, float& v, float& w) {
    const size_t total = (size_t)B * dp, idx = (size_t)b * dp + j;
    if (DP == 128) v = vg[idx] + vg[total + idx];
    else if (DP == 64) v = vg[(size_t)(j & 1) * total + idx];
    else v = vg[(size_t)((j >> 1) & 1) * total + idx];
    w = 0.f;
    if (DP == 128) {
        const int g = j >> 6;
        for (int s = 0; s < NS; ++s) w += wp[(size_t)(2 * s + g) * total + idx];
    } else {
        for (int s = 0; s < 2 * NS; ++s) w += wp[(size_t)s * total + idx];
    }
}

}  // namespace rae
