// Small device helpers shared by the SIMT kernels (reductions, activations, bf16 packing).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cstdint>

namespace b200 {

__device__ __forceinline__ float gelu_exact(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }
__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

// GELU of every stored inference activation: 0.5 x (1 + tanh(x (c0 + c1 x^2))) with the hardware tanh (MUFU.TANH),
// two elements per instruction on the packed fp32x2 pipe: 5 packed instructions + 2 MUFU per pair.  The 8-term
// polynomial erf it replaced (exact to 9e-5) cost 13 packed + 4 FMNMX per pair, and the GEMM epilogues of the 1x1
// layers are instruction-issue bound: block tail 0.709 -> 0.634 ms, C3 step -5 %, C4 -3 % on the same box.
// Deviation from nn.GELU() (erf): <= 4.7e-4 from the tanh form plus the 2^-11
// relative error of MUFU.TANH on (1 + tanh), together <= 1.2e-3 ABSOLUTE (largest around x = -3 .. -2, where
// gelu ~ -0.01 .. -0.05) - below the bf16 rounding step of every output with |y| >= 0.3, and 2e-4 of a typical map's
// range.  Measured effect on parity with the trained weights: fusion logits 5.6e-3 (was 5.7e-3), argmax agreement
// unchanged (tests/test_trained_gpu.py).  The training path keeps the exact erf GELU and its derivative.
__device__ __forceinline__ float2 gelu_fast2(float2 x) {
    const float2 t = __fmul2_rn(x, x);
    const float2 p = __ffma2_rn(t, make_float2(0.0356774081f, 0.0356774081f), make_float2(0.7978845608f, 0.7978845608f));
    const float2 u = __fmul2_rn(x, p);
    float2 th;
    asm("tanh.approx.f32 %0, %1;" : "=f"(th.x) : "f"(u.x));
    asm("tanh.approx.f32 %0, %1;" : "=f"(th.y) : "f"(u.y));
    const float2 h = __fmul2_rn(x, make_float2(0.5f, 0.5f));
    return __ffma2_rn(h, th, h);
}

template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Block-wide sum of per-thread fp32 partials: fp32 shuffles inside a warp, fp64 across warps.
__device__ __forceinline__ double block_sum_f(float v, double* scratch) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
    v = warp_sum(v);
    __syncthreads();  // protect scratch from a previous use
    if (lane == 0) scratch[warp] = static_cast<double>(v);
    __syncthreads();
    double t = 0.0;
    for (int w = 0; w < nwarps; ++w) t += scratch[w];  // broadcast reads, identical order in every thread
    return t;
}

// Sum over the whole block; every thread gets the result.  `scratch` needs 33 elements.
template <typename T>
__device__ __forceinline__ T block_sum(T v, T* scratch) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
    v = warp_sum(v);
    __syncthreads();  // protect scratch from a previous use
    if (lane == 0) scratch[warp] = v;
    __syncthreads();
    if (warp == 0) {
        T t = lane < nwarps ? scratch[lane] : T(0);
        t = warp_sum(t);
        if (lane == 0) scratch[32] = t;
    }
    __syncthreads();
    return scratch[32];
}

__device__ __forceinline__ void unpack_bf16x8(const uint4& u, float (&f)[8]) {
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(&w[i]);
        f[2 * i] = __low2float(h);
        f[2 * i + 1] = __high2float(h);
    }
}
__device__ __forceinline__ uint4 pack_bf16x8(const float (&f)[8]) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const __nv_bfloat162 h = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
        w[i] = *reinterpret_cast<const uint32_t*>(&h);
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

inline int launch_status() { return static_cast<int>(cudaGetLastError()); }

// Philox4x32 with 7 rounds (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3"; 7 rounds pass BigCrush):
// counter-based, so a dropout decision is a pure function of (seed, element index) - no state, any launch shape.
__device__ __forceinline__ uint4 philox4x32_7(unsigned long long ctr, uint32_t key0, uint32_t key1) {
    uint32_t c0 = static_cast<uint32_t>(ctr), c1 = static_cast<uint32_t>(ctr >> 32), c2 = 0x2545f491u, c3 = 0x9e3779b9u;
#pragma unroll
    for (int r = 0; r < 7; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ key0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ key1;
        c3 = lo0;
        key0 += 0x9E3779B9u;
        key1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}

// MC-dropout request of one launch (b200_conv_gemm_mc / b200_stem_mc): probability, Philox seed, and which output
// segments it applies to (0 = none).  Passed by value in the argument list; there is no ambient state.
struct DropoutArgs {
    float p = 0.f;
    unsigned long long seed = 0;
    int seg = 0;
};
inline bool dropout_args_valid(float p, int segments) { return p >= 0.f && p < 1.f && segments >= 0 && segments <= 3; }
inline unsigned int dropout_threshold(float p) {
    const double t = static_cast<double>(p) * 4294967296.0;
    return t >= 4294967295.0 ? 4294967295u : static_cast<unsigned int>(t);
}

}  // namespace b200
