// Training-mode element-wise / reduction kernels of the encoders and the fusion head (sm_100a, HBM-bound SIMT):
// batch-statistic BatchNorm forward / backward fused with the activation, the residual add and dropout; the
// squeeze-excite, mask-attention, 1-channel convolution, stem and pooling backward passes; and the loss terms of the
// reference's training steps with their gradients.  Maps are NHWC bf16 [rows = B*H*W][ld] (C % 8 == 0 channels used),
// per-channel / per-case vectors fp32, reductions over the batch accumulate in fp64.
//
// Reference: torch autograd over code/model_module.py:25-43 (SEBlock), :49-97 (MaskGuidedSpatialAttention),
// :100-125 (ReconHead), :220-316 (ResNetLiteBlock_withRecon), :323-369 (Projector, ClassificationHead),
// nn.BatchNorm2d in training mode; losses code/train.py:991-1048, code/loss.py:45-62, :133-213.
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cfloat>
#include <cstdint>

#include <type_traits>

#include "b200_fusion.h"
#include "common.cuh"

namespace b200 {

constexpr int kTeThreads = 256;

__device__ __forceinline__ float gelu_grad(float y) {
    // d/dy [0.5 y (1 + erf(y / sqrt 2))] = 0.5 (1 + erf(y / sqrt 2)) + y exp(-y^2 / 2) / sqrt(2 pi)
    return 0.5f * (1.0f + erff(y * 0.70710678118654752f)) + y * 0.3989422804014327f * __expf(-0.5f * y * y);
}
__device__ __forceinline__ float act_fwd(float y, int act) {
    return act == 1 ? gelu_exact(y) : (act == 2 ? fmaxf(y, 0.f) : y);
}
__device__ __forceinline__ float act_bwd(float y, int act) {
    return act == 1 ? gelu_grad(y) : (act == 2 ? (y > 0.f ? 1.f : 0.f) : 1.f);
}
static inline int blocks_for(long long items, int threads = kTeThreads, int cap = 148 * 8) {
    long long b = (items + threads - 1) / threads;
    if (b < 1) b = 1;
    return static_cast<int>(b < cap ? b : cap);
}

// ------------------------------------------------------------------------------------------------ BN statistics --
// sum / sum of squares per channel of a bf16 map, accumulated into fp64 [C] buffers (caller zeroes them).
// Thread = one 8-channel group x a strided set of rows; partials are combined across the row-threads of the CTA in
// shared memory and leave with one fp64 atomic per channel and CTA.
__global__ void __launch_bounds__(kTeThreads, 4)
bn_stats_kernel(const __nv_bfloat16* __restrict__ z, long long R, int C, int ld, double* __restrict__ sum,
                double* __restrict__ sumsq) {
    extern __shared__ float s_part[];  // [rows_par][C][2]
    const int CG = C / 8;
    const int rows_par = kTeThreads / CG;
    const int tid = threadIdx.x;
    const int cg = tid % CG, rp = tid / CG;
    float s[8], q[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) s[i] = q[i] = 0.f;
    if (rp < rows_par) {
        // four rows per trip with all loads issued first (same pattern and reason as map_dot_kernel below)
        constexpr int NR = 4;
        const long long step = static_cast<long long>(gridDim.x) * rows_par;
        for (long long r = static_cast<long long>(blockIdx.x) * rows_par + rp; r < R; r += NR * step) {
            uint4 zq[NR];
#pragma unroll
            for (int h = 0; h < NR; ++h)
                if (r + h * step < R) zq[h] = __ldg(reinterpret_cast<const uint4*>(z + (r + h * step) * ld + cg * 8));
#pragma unroll
            for (int h = 0; h < NR; ++h) {
                if (r + h * step >= R) break;
                float f[8];
                unpack_bf16x8(zq[h], f);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    s[i] += f[i];
                    q[i] = fmaf(f[i], f[i], q[i]);
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            s_part[(rp * C + cg * 8 + i) * 2 + 0] = s[i];
            s_part[(rp * C + cg * 8 + i) * 2 + 1] = q[i];
        }
    }
    __syncthreads();
    for (int c = tid; c < C; c += kTeThreads) {
        double a = 0.0, b = 0.0;
        for (int k = 0; k < rows_par; ++k) {
            a += static_cast<double>(s_part[(k * C + c) * 2 + 0]);
            b += static_cast<double>(s_part[(k * C + c) * 2 + 1]);
        }
        atomicAdd(sum + c, a);
        atomicAdd(sumsq + c, b);
    }
}

// mean / 1/sqrt(var + eps) (biased variance, what normalises the batch) and the running-statistics update of
// nn.BatchNorm2d in training mode: running = (1 - momentum) * running + momentum * (mean | unbiased variance).
__global__ void bn_finalize_kernel(const double* __restrict__ sum, const double* __restrict__ sumsq, int C, double count,
                                   float eps, float momentum, float* __restrict__ running_mean,
                                   float* __restrict__ running_var, float* __restrict__ mean_out,
                                   float* __restrict__ invstd_out) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const double m = sum[c] / count;
    double v = sumsq[c] / count - m * m;
    if (v < 0.0) v = 0.0;
    mean_out[c] = static_cast<float>(m);
    invstd_out[c] = static_cast<float>(1.0 / sqrt(v + static_cast<double>(eps)));
    if (running_mean != nullptr) {
        const double unbiased = count > 1.0 ? v * count / (count - 1.0) : v;
        running_mean[c] = static_cast<float>((1.0 - momentum) * running_mean[c] + momentum * m);
        running_var[c] = static_cast<float>((1.0 - momentum) * running_var[c] + momentum * unbiased);
    }
}

struct BnAct {
    const __nv_bfloat16* z;   // conv output [R, ldz]
    int ldz;
    const __nv_bfloat16* res; // residual added before the activation, or nullptr
    int ldres;
    const float *mean, *invstd, *gamma, *beta;  // any may be nullptr (0, 1, 1, 0)
    int act;
    unsigned int drop_thresh;  // 0 = no dropout
    float drop_scale;
    unsigned int seed_lo, seed_hi;
    long long R;
    int C;
};

// erf(z) ~= z * P(z^2) on |z| <= 3 (the 8-term odd minimax polynomial of the GEMM epilogue's GELU, |err| < 9e-5)
__device__ __forceinline__ float erf_poly(float zc) {
    const float t = zc * zc;
    float q = -3.901667185e-07f;
    q = fmaf(q, t, 1.668003461e-05f);
    q = fmaf(q, t, -3.086500801e-04f);
    q = fmaf(q, t, 3.281538375e-03f);
    q = fmaf(q, t, -2.256273106e-02f);
    q = fmaf(q, t, 1.075116023e-01f);
    q = fmaf(q, t, -3.730817735e-01f);
    q = fmaf(q, t, 1.127865076e+00f);
    return zc * q;
}
__device__ __forceinline__ float act_fwd_fast(float y, int act) {
    if (act == 1) {
        const float zc = fminf(fmaxf(y * 0.70710678118654752f, -3.0f), 3.0f);
        const float h = 0.5f * y;
        return fmaf(h, erf_poly(zc), h);
    }
    return act == 2 ? fmaxf(y, 0.f) : y;
}
__device__ __forceinline__ float act_bwd_fast(float y, int act) {
    if (act == 1) {
        const float zc = fminf(fmaxf(y * 0.70710678118654752f, -3.0f), 3.0f);
        // 0.5 (1 + erf) + y phi(y);  phi = exp(-y^2 / 2) / sqrt(2 pi) = 2^(-y^2 * log2(e) / 2) / sqrt(2 pi)
        float e;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-0.72134752044448170f * y * y));
        return fmaf(0.5f, erf_poly(zc), 0.5f) + y * 0.3989422804014327f * e;
    }
    return act == 2 ? (y > 0.f ? 1.f : 0.f) : 1.f;
}

// Thread layout shared by the BN kernels: a thread owns ONE 4-channel group (its BatchNorm constants stay in a handful
// of registers: the kernels run at 5-6 CTAs per SM - at 8 channels per thread and 80-130 registers ncu showed 24 % of
// the warp slots active and the kernels latency bound) and walks rows r = first, first + stride, ...; a warp's 32
// lanes cover 32 consecutive 8-byte groups.  One Philox call yields the 4 dropout decisions of the group.
#define BN_ROW_WALK(CG_)                                                                             \
    const int CG = (CG_);                                                                              \
    const int rows_par = kTeThreads / CG;                                                              \
    const int cg = threadIdx.x % CG, rp = threadIdx.x / CG;                                            \
    const int c0 = cg * 4;                                                                             \
    const long long row_first = static_cast<long long>(blockIdx.x) * rows_par + rp;                    \
    const long long row_step = static_cast<long long>(gridDim.x) * rows_par;

__device__ __forceinline__ void unpack_bf16x4(const uint2& u, float (&f)[4]) {
    f[0] = __uint_as_float(u.x << 16);
    f[1] = __uint_as_float(u.x & 0xffff0000u);
    f[2] = __uint_as_float(u.y << 16);
    f[3] = __uint_as_float(u.y & 0xffff0000u);
}
__device__ __forceinline__ uint2 pack_bf16x4(const float (&f)[4]) {
    const __nv_bfloat162 h0 = __floats2bfloat162_rn(f[0], f[1]), h1 = __floats2bfloat162_rn(f[2], f[3]);
    return make_uint2(*reinterpret_cast<const uint32_t*>(&h0), *reinterpret_cast<const uint32_t*>(&h1));
}
// y = z * a + b per channel (BatchNorm folded with its batch statistics)
__device__ __forceinline__ void bnact_ab(const BnAct& p, int c0, float (&a)[4], float (&b)[4]) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float is = p.invstd != nullptr ? p.invstd[c0 + i] : 1.f;
        const float g = p.gamma != nullptr ? p.gamma[c0 + i] : 1.f;
        const float m = p.mean != nullptr ? p.mean[c0 + i] : 0.f;
        const float be = p.beta != nullptr ? p.beta[c0 + i] : 0.f;
        a[i] = is * g;
        b[i] = be - m * is * g;
    }
}
__device__ __forceinline__ uint4 drop_bits4(const BnAct& p, long long r, int c0) {
    return philox4x32_7((static_cast<unsigned long long>(r) * p.C + c0) / 4, p.seed_lo, p.seed_hi);
}

// out = dropout(act(bn(z) + res)).  The activation / residual / dropout options are template parameters: as run-time
// fields they sat in the per-element loop as uniform branches (cf. the first-layer kernel, DESIGN 4.3).
template <int ACT, bool RES, bool DROP>
__global__ void __launch_bounds__(kTeThreads, 4)
bn_act_fwd_kernel(const BnAct p, __nv_bfloat16* __restrict__ out, int ldo) {
    BN_ROW_WALK(p.C / 4)
    if (rp >= rows_par) return;
    float ka[4], kb[4];
    bnact_ab(p, c0, ka, kb);
    constexpr int NR = 4;  // rows per trip: all loads of a trip are issued before its arithmetic
    for (long long r = row_first; r < p.R; r += NR * row_step) {
        uint2 zq[NR], rq[NR];
#pragma unroll
        for (int h = 0; h < NR; ++h) {
            const long long rh = r + h * row_step;
            if (rh < p.R) {
                zq[h] = __ldg(reinterpret_cast<const uint2*>(p.z + rh * p.ldz + c0));
                if (RES) rq[h] = __ldg(reinterpret_cast<const uint2*>(p.res + rh * p.ldres + c0));
            }
        }
#pragma unroll
        for (int h = 0; h < NR; ++h) {
            const long long rh = r + h * row_step;
            if (rh >= p.R) break;
            float f[4], rr[4];
            unpack_bf16x4(zq[h], f);
            if (RES) unpack_bf16x4(rq[h], rr);
            uint4 rn = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
            if (DROP) rn = drop_bits4(p, rh, c0);
            const unsigned int rnv[4] = {rn.x, rn.y, rn.z, rn.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float y = fmaf(f[j], ka[j], kb[j]);
                if (RES) y += rr[j];
                y = act_fwd_fast(y, ACT);
                if (DROP) y = rnv[j] < p.drop_thresh ? 0.f : y * p.drop_scale;
                f[j] = y;
            }
            *reinterpret_cast<uint2*>(out + rh * ldo + c0) = pack_bf16x4(f);
        }
    }
}

// Backward, pass 1: dY = dA * dropout_mask * act'(y), y = bn(z) + res, WRITTEN to dy_out (and dy_out2: the residual
// branch's gradient); with batch statistics s1[c] += sum dY, s2[c] += sum dY * xhat; without them dy_out receives
// dz = a * dY directly and only s1 / s2 (when requested) feed dbeta / dgamma.
template <int ACT, bool RES, bool DROP>
__global__ void __launch_bounds__(kTeThreads, 4)
bn_act_bwd_pass1_kernel(const BnAct p, const __nv_bfloat16* __restrict__ dA, int ldd, int batch_stats,
                        __nv_bfloat16* __restrict__ dy_out, int ldo, __nv_bfloat16* __restrict__ dy_out2, int ldo2,
                        double* __restrict__ s1, double* __restrict__ s2) {
    extern __shared__ float s_part[];
    BN_ROW_WALK(p.C / 4)
    float u[4], v[4];  // sum dY, sum dY * z (xhat = (z - mu) * invstd is applied once, after the reduction)
#pragma unroll
    for (int i = 0; i < 4; ++i) u[i] = v[i] = 0.f;
    if (rp < rows_par) {
        float ka[4], kb[4];
        bnact_ab(p, c0, ka, kb);
        constexpr int NR = 2;
        for (long long r = row_first; r < p.R; r += NR * row_step) {
            uint2 zq[NR], dq[NR], rq[NR];
#pragma unroll
            for (int h = 0; h < NR; ++h) {
                const long long rh = r + h * row_step;
                if (rh < p.R) {
                    zq[h] = __ldg(reinterpret_cast<const uint2*>(p.z + rh * p.ldz + c0));
                    dq[h] = __ldg(reinterpret_cast<const uint2*>(dA + rh * ldd + c0));
                    if (RES) rq[h] = __ldg(reinterpret_cast<const uint2*>(p.res + rh * p.ldres + c0));
                }
            }
#pragma unroll
            for (int h = 0; h < NR; ++h) {
                const long long rh = r + h * row_step;
                if (rh >= p.R) break;
                float f[4], d[4], rr[4];
                unpack_bf16x4(zq[h], f);
                unpack_bf16x4(dq[h], d);
                if (RES) unpack_bf16x4(rq[h], rr);
                uint4 rn = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
                if (DROP) rn = drop_bits4(p, rh, c0);
                const unsigned int rnv[4] = {rn.x, rn.y, rn.z, rn.w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float g = d[j];
                    if (DROP) g = rnv[j] < p.drop_thresh ? 0.f : g * p.drop_scale;
                    if (ACT != 0) {
                        float y = fmaf(f[j], ka[j], kb[j]);
                        if (RES) y += rr[j];
                        g *= act_bwd_fast(y, ACT);
                    }
                    u[j] += g;
                    v[j] = fmaf(g, f[j], v[j]);
                    d[j] = g;
                }
                if (dy_out2 != nullptr) *reinterpret_cast<uint2*>(dy_out2 + rh * ldo2 + c0) = pack_bf16x4(d);
                if (dy_out != nullptr) {
                    if (!batch_stats) {
#pragma unroll
                        for (int j = 0; j < 4; ++j) d[j] *= ka[j];
                    }
                    *reinterpret_cast<uint2*>(dy_out + rh * ldo + c0) = pack_bf16x4(d);
                }
            }
        }
        if (s1 != nullptr) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                s_part[(rp * p.C + c0 + i) * 2 + 0] = u[i];
                s_part[(rp * p.C + c0 + i) * 2 + 1] = v[i];
            }
        }
    }
    if (s1 == nullptr) return;
    __syncthreads();
    for (int c = threadIdx.x; c < p.C; c += kTeThreads) {
        double a = 0.0, b = 0.0;
        for (int kk = 0; kk < rows_par; ++kk) {
            a += static_cast<double>(s_part[(kk * p.C + c) * 2 + 0]);
            b += static_cast<double>(s_part[(kk * p.C + c) * 2 + 1]);
        }
        const double mu = p.mean != nullptr ? static_cast<double>(p.mean[c]) : 0.0;
        const double is = p.invstd != nullptr ? static_cast<double>(p.invstd[c]) : 1.0;
        atomicAdd(s1 + c, a);
        atomicAdd(s2 + c, (b - mu * a) * is);  // sum dY * xhat
    }
}

// Backward, pass 2 (batch statistics only), in place on the dY map pass 1 wrote:
// dz = gamma * invstd * (dY - s1/N - xhat * s2/N).  Block 0 also accumulates dgamma += s2, dbeta += s1.
__global__ void __launch_bounds__(kTeThreads, 4)
bn_act_bwd_pass2_kernel(const BnAct p, const double* __restrict__ s1, const double* __restrict__ s2, double count,
                        __nv_bfloat16* __restrict__ dz, int lddz, float* __restrict__ dgamma, float* __restrict__ dbeta,
                        int map_pass) {
    if (blockIdx.x == 0) {
        for (int c = threadIdx.x; c < p.C; c += kTeThreads) {
            if (dgamma != nullptr) dgamma[c] += static_cast<float>(s2[c]);
            if (dbeta != nullptr) dbeta[c] += static_cast<float>(s1[c]);
        }
    }
    if (!map_pass) return;
    BN_ROW_WALK(p.C / 4)
    if (rp >= rows_par) return;
    // dz = a (dY - k1 - (z - mu) is k2) = A dY + Bz z + Cc with A = a, Bz = -a is k2, Cc = a (is k2 mu - k1)
    float kA[4], kB[4], kC[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float is = p.invstd != nullptr ? p.invstd[c0 + i] : 1.f;
        const float g = p.gamma != nullptr ? p.gamma[c0 + i] : 1.f;
        const float mu = p.mean != nullptr ? p.mean[c0 + i] : 0.f;
        const float k1 = static_cast<float>(s1[c0 + i] / count), k2 = static_cast<float>(s2[c0 + i] / count);
        kA[i] = is * g;
        kB[i] = -kA[i] * is * k2;
        kC[i] = kA[i] * (is * k2 * mu - k1);
    }
    constexpr int NR = 4;
    for (long long r = row_first; r < p.R; r += NR * row_step) {
        uint2 zq[NR], gq[NR];
#pragma unroll
        for (int h = 0; h < NR; ++h) {
            const long long rh = r + h * row_step;
            if (rh < p.R) {
                zq[h] = __ldg(reinterpret_cast<const uint2*>(p.z + rh * p.ldz + c0));
                gq[h] = *reinterpret_cast<const uint2*>(dz + rh * lddz + c0);
            }
        }
#pragma unroll
        for (int h = 0; h < NR; ++h) {
            const long long rh = r + h * row_step;
            if (rh >= p.R) break;
            float f[4], g[4];
            unpack_bf16x4(zq[h], f);
            unpack_bf16x4(gq[h], g);
#pragma unroll
            for (int j = 0; j < 4; ++j) g[j] = fmaf(kA[j], g[j], fmaf(kB[j], f[j], kC[j]));
            *reinterpret_cast<uint2*>(dz + rh * lddz + c0) = pack_bf16x4(g);
        }
    }
}

// ------------------------------------------------------------------------------------- generic map helpers -------
// out[b, c] = sum_p a[b, p, c] * b[b, p, c]   (b == nullptr: plain channel sums)       [fp32, overwritten]
__global__ void __launch_bounds__(kTeThreads, 4)
map_dot_kernel(const __nv_bfloat16* __restrict__ a, int lda, const __nv_bfloat16* __restrict__ bmap, int ldb, int npix,
               int C, float* __restrict__ out) {
    extern __shared__ float s_part[];  // [rows_par][C]
    const int CG = C / 8;
    const int rows_par = kTeThreads / CG;
    const int tid = threadIdx.x, cg = tid % CG, rp = tid / CG;
    const int bcase = blockIdx.x;
    float s[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) s[i] = 0.f;
    if (rp < rows_par) {
        // four rows per trip, every load issued before the first use (one 16-byte load in flight per thread left the
        // kernel latency bound at 40-57 % of the HBM peak); the accumulation order over the rows is unchanged
        constexpr int NR = 4;
        const long long row0 = static_cast<long long>(bcase) * npix;
        for (int pp = rp; pp < npix; pp += NR * rows_par) {
            uint4 aq[NR], bq[NR];
#pragma unroll
            for (int h = 0; h < NR; ++h) {
                const int ph = pp + h * rows_par;
                if (ph < npix) {
                    aq[h] = __ldg(reinterpret_cast<const uint4*>(a + (row0 + ph) * lda + cg * 8));
                    if (bmap != nullptr) bq[h] = __ldg(reinterpret_cast<const uint4*>(bmap + (row0 + ph) * ldb + cg * 8));
                }
            }
#pragma unroll
            for (int h = 0; h < NR; ++h) {
                if (pp + h * rows_par >= npix) break;
                float f[8], g[8];
                unpack_bf16x8(aq[h], f);
                if (bmap != nullptr) {
                    unpack_bf16x8(bq[h], g);
#pragma unroll
                    for (int i = 0; i < 8; ++i) s[i] = fmaf(f[i], g[i], s[i]);
                } else {
#pragma unroll
                    for (int i = 0; i < 8; ++i) s[i] += f[i];
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) s_part[rp * C + cg * 8 + i] = s[i];
    }
    __syncthreads();
    for (int c = tid; c < C; c += kTeThreads) {
        float t = 0.f;
        for (int k = 0; k < rows_par; ++k) t += s_part[k * C + c];
        out[static_cast<long long>(bcase) * C + c] = t;
    }
}

// out[b,p,c] = x[b,p,c] * gate[b,c] + add[b,c]  (x NULL: the gate alone, or 0 without a gate -> a pure broadcast of add)
// Per-case grid (chunks, B), 32-bit indices, the options as template parameters: the generic kernel below spends three
// 64-bit divisions (~150 instructions each) per 16 bytes and ran at 48-52 % of the HBM peak.  A thread's vectors all
// carry the same 8 channels when the CTA's stride is a multiple of C / 8 (every power-of-two width), so its gate / add
// values are loaded once.
template <bool HAS_X, bool HAS_GATE, bool HAS_ADD, bool ACC>
__global__ void __launch_bounds__(kTeThreads, 4)
map_scale_add_case_kernel(const __nv_bfloat16* __restrict__ x, int ldx, const float* __restrict__ gate,
                          const float* __restrict__ add, int npix, int C, __nv_bfloat16* __restrict__ out, int ldo) {
    const int CG = C >> 3, nvc = npix * CG, b = blockIdx.y;
    const int sh = (CG & (CG - 1)) == 0 ? 31 - __clz(CG) : -1;
    const int step = gridDim.x * kTeThreads;
    const bool fixed_c = (step % CG) == 0;  // the thread keeps one channel group for its whole walk
    const float* gr = HAS_GATE ? gate + static_cast<size_t>(b) * C : nullptr;
    const float* ar = HAS_ADD ? add + static_cast<size_t>(b) * C : nullptr;
    const size_t row0 = static_cast<size_t>(b) * npix;
    const int i_first = blockIdx.x * kTeThreads + threadIdx.x;
    float gk[8], ak[8];
    auto load_ga = [&](int c0) {
        if (HAS_GATE) {
            const float4 g0 = __ldg(reinterpret_cast<const float4*>(gr + c0)), g1 = __ldg(reinterpret_cast<const float4*>(gr + c0 + 4));
            gk[0] = g0.x; gk[1] = g0.y; gk[2] = g0.z; gk[3] = g0.w; gk[4] = g1.x; gk[5] = g1.y; gk[6] = g1.z; gk[7] = g1.w;
        }
        if (HAS_ADD) {
            const float4 a0 = __ldg(reinterpret_cast<const float4*>(ar + c0)), a1 = __ldg(reinterpret_cast<const float4*>(ar + c0 + 4));
            ak[0] = a0.x; ak[1] = a0.y; ak[2] = a0.z; ak[3] = a0.w; ak[4] = a1.x; ak[5] = a1.y; ak[6] = a1.z; ak[7] = a1.w;
        }
    };
    if (fixed_c && i_first < nvc) load_ga((sh >= 0 ? (i_first & (CG - 1)) : (i_first % CG)) << 3);
    constexpr int NI = 2;  // independent 16-byte loads in flight per thread
    for (int i0 = i_first; i0 < nvc; i0 += NI * step) {
        uint4 xq[NI], oq[NI];
        int pl[NI], c0[NI];
#pragma unroll
        for (int h = 0; h < NI; ++h) {
            const int i = i0 + h * step;
            pl[h] = sh >= 0 ? i >> sh : i / CG;
            c0[h] = (i - pl[h] * CG) << 3;
            if (i < nvc) {
                if (HAS_X) xq[h] = __ldg(reinterpret_cast<const uint4*>(x + (row0 + pl[h]) * ldx + c0[h]));
                if (ACC) oq[h] = *reinterpret_cast<const uint4*>(out + (row0 + pl[h]) * ldo + c0[h]);
            }
        }
#pragma unroll
        for (int h = 0; h < NI; ++h) {
            if (i0 + h * step >= nvc) break;
            if (!fixed_c) load_ga(c0[h]);
            float f[8], o[8];
            if (HAS_X) unpack_bf16x8(xq[h], f);
            if (ACC) unpack_bf16x8(oq[h], o);
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                float v = HAS_X ? f[k] : (HAS_GATE ? 1.f : 0.f);
                if (HAS_GATE) v *= gk[k];
                if (HAS_ADD) v += ak[k];
                o[k] = ACC ? o[k] + v : v;
            }
            *reinterpret_cast<uint4*>(out + (row0 + pl[h]) * ldo + c0[h]) = pack_bf16x8(o);
        }
    }
}

// generic form (any row count; kept for shapes whose per-case vector count does not fit 32 bits)
__global__ void __launch_bounds__(kTeThreads, 4)
map_scale_add_kernel(const __nv_bfloat16* __restrict__ x, int ldx, const float* __restrict__ gate,
                     const float* __restrict__ add, long long R, int npix, int C, __nv_bfloat16* __restrict__ out,
                     int ldo, int accumulate) {
    const int CG = C / 8;
    const long long total = R * CG;
    constexpr int NI = 1;
    const long long step = static_cast<long long>(gridDim.x) * kTeThreads;
    for (long long i0 = blockIdx.x * static_cast<long long>(kTeThreads) + threadIdx.x; i0 < total; i0 += NI * step) {
        uint4 xq[NI], oq[NI];
#pragma unroll
        for (int h = 0; h < NI; ++h) {
            const long long i = i0 + h * step;
            if (i < total) {
                const long long r = i / CG;
                const int c0 = static_cast<int>(i - r * CG) * 8;
                if (x != nullptr) xq[h] = __ldg(reinterpret_cast<const uint4*>(x + r * ldx + c0));
                if (accumulate) oq[h] = *reinterpret_cast<const uint4*>(out + r * ldo + c0);
            }
        }
#pragma unroll
        for (int h = 0; h < NI; ++h) {
            const long long i = i0 + h * step;
            if (i >= total) break;
            const long long r = i / CG;
            const int c0 = static_cast<int>(i - r * CG) * 8;
            const long long bc = (r / npix) * C + c0;
            float f[8], o[8];
            if (x != nullptr) unpack_bf16x8(xq[h], f);
            if (accumulate) unpack_bf16x8(oq[h], o);
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                float v = x != nullptr ? f[k] : (gate != nullptr ? 1.f : 0.f);
                if (gate != nullptr) v *= gate[bc + k];
                if (add != nullptr) v += add[bc + k];
                o[k] = accumulate ? o[k] + v : v;
            }
            *reinterpret_cast<uint4*>(out + r * ldo + c0) = pack_bf16x8(o);
        }
    }
}

// y = alpha * a + beta * b (bf16 maps with row strides; b may be nullptr)
template <typename I>  // I = int when R * C / 8 fits 31 bits: 32-bit index arithmetic, a shift for power-of-two widths
__global__ void __launch_bounds__(kTeThreads)
map_axpby_kernel(const __nv_bfloat16* __restrict__ a, int lda, float alpha, const __nv_bfloat16* __restrict__ b, int ldb,
                 float beta, long long R, int C, __nv_bfloat16* __restrict__ y, int ldy) {
    const int CG = C / 8;
    const I total = static_cast<I>(R * CG);
    const int sh = (CG & (CG - 1)) == 0 ? 31 - __clz(CG) : -1;
    for (I i = static_cast<I>(blockIdx.x) * kTeThreads + threadIdx.x; i < total; i += static_cast<I>(gridDim.x) * kTeThreads) {
        const long long r = sh >= 0 ? static_cast<long long>(i >> sh) : static_cast<long long>(i / CG);
        const int c0 = static_cast<int>(i - static_cast<I>(r) * CG) * 8;
        float f[8], g[8];
        unpack_bf16x8(__ldg(reinterpret_cast<const uint4*>(a + r * lda + c0)), f);
        if (b != nullptr) unpack_bf16x8(__ldg(reinterpret_cast<const uint4*>(b + r * ldb + c0)), g);
#pragma unroll
        for (int k = 0; k < 8; ++k) f[k] = alpha * f[k] + (b != nullptr ? beta * g[k] : 0.f);
        *reinterpret_cast<uint4*>(y + r * ldy + c0) = pack_bf16x8(f);
    }
}

// sum of squares of a bf16 map -> fp64 scalar (accumulated): the feature-norm regulariser, code/train.py:1021-1030
__global__ void __launch_bounds__(kTeThreads)
map_sumsq_kernel(const __nv_bfloat16* __restrict__ a, int lda, long long R, int C, double* __restrict__ out) {
    __shared__ double scratch[33];
    const int CG = C / 8;
    const long long total = R * CG;
    float s = 0.f;
    for (long long i = blockIdx.x * static_cast<long long>(kTeThreads) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * kTeThreads) {
        const long long r = i / CG;
        const int c0 = static_cast<int>(i - r * CG) * 8;
        float f[8];
        unpack_bf16x8(__ldg(reinterpret_cast<const uint4*>(a + r * lda + c0)), f);
#pragma unroll
        for (int k = 0; k < 8; ++k) s = fmaf(f[k], f[k], s);
    }
    const double t = block_sum<double>(static_cast<double>(s), scratch);
    if (threadIdx.x == 0) atomicAdd(out, t);
}

// ------------------------------------------------------------------------------------------- squeeze-excite ------
// y[i] = bias[i] + sum_j W[i * n_in + j] * v[j] for i < n_out, one warp per output row (coalesced weight reads)
template <typename F>
__device__ __forceinline__ void rows_dot(const float* __restrict__ Wm, const float* __restrict__ bias, const float* v,
                                         int n_out, int n_in, F store) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int i = warp; i < n_out; i += nw) {
        float a = 0.f;
        for (int j = lane; j < n_in; j += 32) a = fmaf(__ldg(Wm + static_cast<long long>(i) * n_in + j), v[j], a);
        a = warp_sum(a);
        if (lane == 0) store(i, a + (bias != nullptr ? bias[i] : 0.f));
    }
}

// Forward with the weights in their nn.Conv2d layouts (the training step re-reads the fp32 master weights every step,
// so nothing is pre-transposed): pooled = sums / npix (also written out), gate = sigmoid(W2 gelu(W1 pooled + b1) + b2).
__global__ void __launch_bounds__(kTeThreads)
se_fwd_kernel(const float* __restrict__ sums, float inv_npix, const float* __restrict__ w1, const float* __restrict__ b1,
              const float* __restrict__ w2, const float* __restrict__ b2, int C, int M, float* __restrict__ pooled,
              float* __restrict__ gate) {
    extern __shared__ float s_se[];  // pooled[C] | h[M]
    float* s_p = s_se;
    float* s_h = s_p + C;
    const int b = blockIdx.x, tid = threadIdx.x;
    for (int c = tid; c < C; c += kTeThreads) {
        s_p[c] = sums[static_cast<long long>(b) * C + c] * inv_npix;
        if (pooled != nullptr) pooled[static_cast<long long>(b) * C + c] = s_p[c];
    }
    __syncthreads();
    rows_dot(w1, b1, s_p, M, C, [&](int m, float a) { s_h[m] = gelu_exact(a); });
    __syncthreads();
    rows_dot(w2, b2, s_h, C, M, [&](int c, float a) { gate[static_cast<long long>(b) * C + c] = sigmoidf_(a); });
}

// One CTA per case: recomputes the SE MLP from the pooled vector and back-propagates dgate through it.
//   a1 = W1 pooled + b1, h = gelu(a1), a2 = W2 h + b2, gate = sigmoid(a2)
// Outputs (all fp32): dpooled [B,C] (gradient of the MEAN-pooled vector), da2 [B,C], da1 [B,M], h [B,M].
__global__ void __launch_bounds__(kTeThreads)
se_bwd_kernel(const float* __restrict__ pooled, const float* __restrict__ w1, const float* __restrict__ b1,
              const float* __restrict__ w2, const float* __restrict__ b2, const float* __restrict__ dgate, int C, int M,
              float* __restrict__ dpooled, float* __restrict__ da2, float* __restrict__ da1, float* __restrict__ h_out) {
    extern __shared__ float s_se[];  // pooled[C] | a1[M] | h[M] | da2[C] | da1[M]
    float* s_p = s_se;
    float* s_a1 = s_p + C;
    float* s_h = s_a1 + M;
    float* s_da2 = s_h + M;
    float* s_da1 = s_da2 + C;
    const int b = blockIdx.x, tid = threadIdx.x;
    for (int c = tid; c < C; c += kTeThreads) s_p[c] = pooled[static_cast<long long>(b) * C + c];
    __syncthreads();
    rows_dot(w1, b1, s_p, M, C, [&](int m, float a) {
        s_a1[m] = a;
        s_h[m] = gelu_exact(a);
        h_out[static_cast<long long>(b) * M + m] = s_h[m];
    });
    __syncthreads();
    rows_dot(w2, b2, s_h, C, M, [&](int c, float a) {
        const float g = sigmoidf_(a);
        const float d = dgate[static_cast<long long>(b) * C + c] * g * (1.f - g);
        s_da2[c] = d;
        da2[static_cast<long long>(b) * C + c] = d;
    });
    __syncthreads();
    for (int m = tid; m < M; m += kTeThreads) {
        float a = 0.f;
        for (int c = 0; c < C; ++c) a = fmaf(w2[c * M + m], s_da2[c], a);
        const float d = a * gelu_grad(s_a1[m]);
        s_da1[m] = d;
        da1[static_cast<long long>(b) * M + m] = d;
    }
    __syncthreads();
    for (int c = tid; c < C; c += kTeThreads) {
        float a = 0.f;
        for (int m = 0; m < M; ++m) a = fmaf(w1[m * C + c], s_da1[m], a);
        dpooled[static_cast<long long>(b) * C + c] = a;
    }
}

// --------------------------------------------------------------------------- C -> 1 convolutions (1x1 / 3x3) -----
// out[b,h,w] = bias + sum_{tap,c} x[b, h+dy, w+dx, c] * w[c * taps + tap]   (weights in the nn.Conv2d layout [1,C,kh,kw])
//
// One CTA per case.  A group of C/8 lanes owns a pixel: every lane loads 8 channels (one 16-byte load) and keeps its
// 8 x TAPS weights in registers.  Forward: the TAPS per-pixel dot products d[p][tap] go to shared memory, then
// out[q] = bias + sum_tap d[q + off(tap)][tap] - the map is read from HBM exactly once.  Backward: dout of the case sits
// in shared memory; dx[p][c] = sum_tap dout[p - off(tap)] w[c][tap] is written once, dw[c][tap] += sum_p dout[p - off] x[p][c]
// accumulates in registers over the CTA's pixels and leaves through shared memory with one atomic per (c, tap) and CTA.
template <int TAPS>
__global__ void __launch_bounds__(kTeThreads)
convc1_fwd_kernel(const __nv_bfloat16* __restrict__ x, int ldx, int H, int W, int C, const float* __restrict__ w,
                  const float* __restrict__ bias, float* __restrict__ out) {
    extern __shared__ float s_d[];  // [H*W][TAPS]
    const int b = blockIdx.x, npix = H * W;
    const int lpp = C / 8;                      // lanes per pixel (power of two, <= 32: C <= 256) or 32 (C > 256: loop)
    const int gl = lpp < 32 ? lpp : 32;
    const int lane = threadIdx.x & 31;
    const int sub = lane % gl, grp = lane / gl;  // lane's channel slice / pixel slot inside the warp
    const int ppw = 32 / gl;                     // pixels per warp and trip
    const int slot = (threadIdx.x >> 5) * ppw + grp, nslots = (kTeThreads >> 5) * ppw;
    for (int c0 = sub * 8; c0 < C; c0 += 256) {
        float wr[8][TAPS];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
#pragma unroll
            for (int t = 0; t < TAPS; ++t) wr[k][t] = __ldg(w + (c0 + k) * TAPS + t);
        }
        constexpr int NP = 4;  // pixels per trip: their loads are issued together (the loop is latency bound otherwise)
        // The trip / break conditions use the warp's first pixel slot so that every lane reaches the full-warp shuffles
        // below; a lane past the last pixel reduces zeros and stores nothing.
        const int wslot = slot - grp;
        for (int w0 = wslot; w0 < npix; w0 += NP * nslots) {
            uint4 q[NP];
#pragma unroll
            for (int h = 0; h < NP; ++h) {
                const int pix = w0 + grp + h * nslots;
                q[h] = pix < npix ? __ldg(reinterpret_cast<const uint4*>(x + (static_cast<long long>(b) * npix + pix) * ldx + c0))
                                  : make_uint4(0u, 0u, 0u, 0u);
            }
#pragma unroll
            for (int h = 0; h < NP; ++h) {
                if (w0 + h * nslots >= npix) break;
                const int pix = w0 + grp + h * nslots;
                float acc[TAPS];
#pragma unroll
                for (int t = 0; t < TAPS; ++t) acc[t] = 0.f;
                float f[8];
                unpack_bf16x8(q[h], f);
#pragma unroll
                for (int k = 0; k < 8; ++k) {
#pragma unroll
                    for (int t = 0; t < TAPS; ++t) acc[t] = fmaf(f[k], wr[k][t], acc[t]);
                }
#pragma unroll
                for (int t = 0; t < TAPS; ++t) {
                    float v = acc[t];
                    for (int o = gl >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                    acc[t] = v;
                }
                if (sub == 0 && pix < npix) {  // (C > 256: the same lane revisits the pixel with the next 256 channels)
#pragma unroll
                    for (int t = 0; t < TAPS; ++t) s_d[pix * TAPS + t] = (c0 < 256 ? 0.f : s_d[pix * TAPS + t]) + acc[t];
                }
            }
        }
    }
    __syncthreads();
    const float bv = bias != nullptr ? bias[0] : 0.f;
    for (int q = threadIdx.x; q < npix; q += kTeThreads) {
        float v = bv;
        if (TAPS == 1) {
            v += s_d[q];
        } else {
            const int hq = q / W, wq = q - hq * W;
#pragma unroll
            for (int t = 0; t < TAPS; ++t) {
                const int hh = hq + t / 3 - 1, ww = wq + t % 3 - 1;
                if (hh >= 0 && hh < H && ww >= 0 && ww < W) v += s_d[(hh * W + ww) * TAPS + t];
            }
        }
        out[static_cast<long long>(b) * npix + q] = v;
    }
}

template <int TAPS>
__global__ void __launch_bounds__(kTeThreads)
convc1_bwd_kernel(const float* __restrict__ dout, const __nv_bfloat16* __restrict__ x, int ldx, int H, int W, int C,
                  const float* __restrict__ w, __nv_bfloat16* __restrict__ dx, int lddx, int accumulate,
                  float* __restrict__ dw, float* __restrict__ dbias) {
    extern __shared__ float s_g[];  // [H*W] dout of this case | [C*TAPS] dw partials
    __shared__ double scratch[33];
    const int b = blockIdx.x, npix = H * W;
    float* s_dw = s_g + npix;
    float bsum = 0.f;
    for (int i = threadIdx.x; i < npix; i += kTeThreads) {
        const float g = dout[static_cast<long long>(b) * npix + i];
        s_g[i] = g;
        bsum += g;
    }
    for (int i = threadIdx.x; i < C * TAPS; i += kTeThreads) s_dw[i] = 0.f;
    __syncthreads();
    const int lpp = C / 8;
    const int gl = lpp < 32 ? lpp : 32;
    const int lane = threadIdx.x & 31;
    const int sub = lane % gl, grp = lane / gl;
    const int ppw = 32 / gl;
    const int slot = (threadIdx.x >> 5) * ppw + grp, nslots = (kTeThreads >> 5) * ppw;
    for (int c0 = sub * 8; c0 < C; c0 += 256) {
        float wr[8][TAPS], acc[8][TAPS];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
#pragma unroll
            for (int t = 0; t < TAPS; ++t) {
                wr[k][t] = __ldg(w + (c0 + k) * TAPS + t);
                acc[k][t] = 0.f;
            }
        }
        constexpr int NP = 4;
        for (int pix0 = slot; pix0 < npix; pix0 += NP * nslots) {
            uint4 q[NP], oq[NP];
#pragma unroll
            for (int h = 0; h < NP; ++h) {
                const int pix = pix0 + h * nslots;
                if (pix < npix) {
                    const long long row = static_cast<long long>(b) * npix + pix;
                    if (dw != nullptr) q[h] = __ldg(reinterpret_cast<const uint4*>(x + row * ldx + c0));
                    if (dx != nullptr && accumulate) oq[h] = *reinterpret_cast<const uint4*>(dx + row * lddx + c0);
                }
            }
#pragma unroll
            for (int h = 0; h < NP; ++h) {
                const int pix = pix0 + h * nslots;
                if (pix >= npix) break;
                const int hq = pix / W, wq = pix - hq * W;
                float g[TAPS];
#pragma unroll
                for (int t = 0; t < TAPS; ++t) {
                    const int hh = TAPS == 9 ? hq - (t / 3 - 1) : hq, ww = TAPS == 9 ? wq - (t % 3 - 1) : wq;
                    g[t] = (hh >= 0 && hh < H && ww >= 0 && ww < W) ? s_g[hh * W + ww] : 0.f;
                }
                const long long row = static_cast<long long>(b) * npix + pix;
                if (dw != nullptr) {
                    float f[8];
                    unpack_bf16x8(q[h], f);
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
#pragma unroll
                        for (int t = 0; t < TAPS; ++t) acc[k][t] = fmaf(g[t], f[k], acc[k][t]);
                    }
                }
                if (dx != nullptr) {
                    float o[8];
                    if (accumulate) unpack_bf16x8(oq[h], o);
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        float v = accumulate ? o[k] : 0.f;
#pragma unroll
                        for (int t = 0; t < TAPS; ++t) v = fmaf(g[t], wr[k][t], v);
                        o[k] = v;
                    }
                    *reinterpret_cast<uint4*>(dx + row * lddx + c0) = pack_bf16x8(o);
                }
            }
        }
        if (dw != nullptr) {
#pragma unroll
            for (int k = 0; k < 8; ++k) {
#pragma unroll
                for (int t = 0; t < TAPS; ++t) atomicAdd(&s_dw[(c0 + k) * TAPS + t], acc[k][t]);
            }
        }
    }
    if (dw != nullptr) {
        __syncthreads();
        for (int i = threadIdx.x; i < C * TAPS; i += kTeThreads) atomicAdd(dw + i, s_dw[i]);
    }
    if (dbias != nullptr) {
        const double t = block_sum<double>(static_cast<double>(bsum), scratch);
        if (threadIdx.x == 0) atomicAdd(dbias, static_cast<float>(t));
    }
}

// ------------------------------------------------------------------ 1 -> N "lift" convolution (Projector on r) ----
// z[p, n] = r[p] * w[n] (bf16 out);  backward: dw[n] += sum_p dz[p,n] r[p];  dr[p] = sum_n dz[p,n] w[n]
__global__ void __launch_bounds__(kTeThreads)
lift_fwd_kernel(const float* __restrict__ r, long long P, int N, const float* __restrict__ w, __nv_bfloat16* __restrict__ z) {
    const int NG = N / 8;
    const long long total = P * NG;
    for (long long i = blockIdx.x * static_cast<long long>(kTeThreads) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * kTeThreads) {
        const long long pix = i / NG;
        const int n0 = static_cast<int>(i - pix * NG) * 8;
        const float rv = r[pix];
        float f[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) f[k] = rv * w[n0 + k];
        *reinterpret_cast<uint4*>(z + pix * N + n0) = pack_bf16x8(f);
    }
}
__global__ void __launch_bounds__(kTeThreads)
lift_bwd_kernel(const __nv_bfloat16* __restrict__ dz, const float* __restrict__ r, long long P, int N,
                const float* __restrict__ w, float* __restrict__ dw, float* __restrict__ dr) {
    // one warp per pixel for dr; dw through shared-memory partials
    extern __shared__ float s_dw[];  // [N]
    for (int n = threadIdx.x; n < N; n += kTeThreads) s_dw[n] = 0.f;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long long warp = (blockIdx.x * static_cast<long long>(kTeThreads) + threadIdx.x) >> 5;
    const long long nwarps = (static_cast<long long>(gridDim.x) * kTeThreads) >> 5;
    float acc_w[4] = {0.f, 0.f, 0.f, 0.f};  // channels lane*2, lane*2+1 (+64)
    for (long long pix = warp; pix < P; pix += nwarps) {
        const float rv = r[pix];
        float d = 0.f;
        int k = 0;
        for (int n = lane * 2; n < N; n += 64, ++k) {
            const __nv_bfloat162 v = *reinterpret_cast<const __nv_bfloat162*>(dz + pix * N + n);
            const float v0 = __low2float(v), v1 = __high2float(v);
            d = fmaf(v0, w[n], d);
            d = fmaf(v1, w[n + 1], d);
            if (k < 2) {
                acc_w[2 * k] = fmaf(v0, rv, acc_w[2 * k]);
                acc_w[2 * k + 1] = fmaf(v1, rv, acc_w[2 * k + 1]);
            }
        }
        d = warp_sum(d);
        if (lane == 0 && dr != nullptr) dr[pix] = d;
    }
    int k = 0;
    for (int n = lane * 2; n < N && k < 2; n += 64, ++k) {
        atomicAdd(&s_dw[n], acc_w[2 * k]);
        atomicAdd(&s_dw[n + 1], acc_w[2 * k + 1]);
    }
    __syncthreads();
    for (int n = threadIdx.x; n < N; n += kTeThreads) atomicAdd(dw + n, s_dw[n]);
}

// --------------------------------------------------------------------------- mask-guided modulation backward -----
// forward: y = f * (1 + gamma * A[b,p]).   backward (one warp per pixel):
//   df[b,p,c] = dy * (1 + gamma A);  dA[b,p] = gamma * sum_c dy * f;  dgamma += sum dy * f * A
__global__ void __launch_bounds__(kTeThreads)
modulate_bwd_kernel(const __nv_bfloat16* __restrict__ dy, int lddy, const __nv_bfloat16* __restrict__ f, int ldf,
                    const float* __restrict__ A, const float* __restrict__ gamma, long long P, int C,
                    __nv_bfloat16* __restrict__ df, int lddf, float* __restrict__ dA, float* __restrict__ dgamma) {
    __shared__ double scratch[33];
    const int lane = threadIdx.x & 31;
    const long long warp = (blockIdx.x * static_cast<long long>(kTeThreads) + threadIdx.x) >> 5;
    const long long nwarps = (static_cast<long long>(gridDim.x) * kTeThreads) >> 5;
    const float gm = gamma[0];
    float dg = 0.f;
    for (long long pix = warp; pix < P; pix += nwarps) {
        const float a = A[pix];
        const float m = 1.f + gm * a;
        float dot = 0.f;
        for (int c = lane * 8; c < C; c += 256) {
            float u[8], v[8], o[8];
            unpack_bf16x8(__ldg(reinterpret_cast<const uint4*>(dy + pix * lddy + c)), u);
            unpack_bf16x8(__ldg(reinterpret_cast<const uint4*>(f + pix * ldf + c)), v);
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                dot = fmaf(u[k], v[k], dot);
                o[k] = u[k] * m;
            }
            *reinterpret_cast<uint4*>(df + pix * lddf + c) = pack_bf16x8(o);
        }
        dot = warp_sum(dot);
        if (lane == 0) {
            dA[pix] = gm * dot;
            dg = fmaf(dot, a, dg);
        }
    }
    const double t = block_sum<double>(static_cast<double>(dg), scratch);
    if (threadIdx.x == 0 && dgamma != nullptr) atomicAdd(dgamma, static_cast<float>(t));
}

// ------------------------------------------------------------------- mask attention (1 -> 16 -> 1) backward ------
// forward per case: u[p,k] = wa[k] m[p];  GroupNorm(1, K) over all (p, k);  g = gelu(gn);  s[p] = sum_k wb[k] g[p,k] + bb;
// A = clamp(sigmoid(s), 1e-4, 1 - 1e-4).  One CTA per case; K <= 32; the map is recomputed, nothing was saved.
// Outputs: dm[b,p] overwritten; dwa[K], dgnw[K], dgnb[K], dwb[K], dbb accumulated atomically.
__global__ void __launch_bounds__(kTeThreads)
mask_attn_bwd_kernel(const float* __restrict__ mask, const float* __restrict__ dA, int npix, int K,
                     const float* __restrict__ wa, const float* __restrict__ gnw, const float* __restrict__ gnb,
                     const float* __restrict__ wb, const float* __restrict__ bb, float eps, float* __restrict__ dm,
                     float* __restrict__ dwa, float* __restrict__ dgnw, float* __restrict__ dgnb,
                     float* __restrict__ dwb, float* __restrict__ dbb) {
    __shared__ double scratch[33];
    __shared__ float s_wa[32], s_gw[32], s_gb[32], s_wb[32];
    __shared__ float s_acc[5][32];
    const int b = blockIdx.x, tid = threadIdx.x;
    const float* m = mask + static_cast<long long>(b) * npix;
    const float* dAp = dA + static_cast<long long>(b) * npix;
    if (tid < 32) {
        s_wa[tid] = tid < K ? wa[tid] : 0.f;
        s_gw[tid] = tid < K ? gnw[tid] : 0.f;
        s_gb[tid] = tid < K ? gnb[tid] : 0.f;
        s_wb[tid] = tid < K ? wb[tid] : 0.f;
        for (int j = 0; j < 5; ++j) s_acc[j][tid] = 0.f;
    }
    __syncthreads();
    // group statistics: mean / var of u = wa[k] m[p] over (p, k)
    double sm = 0.0, sq = 0.0;
    for (int p = tid; p < npix; p += kTeThreads) {
        sm += m[p];
        sq += static_cast<double>(m[p]) * m[p];
    }
    const double Sm = block_sum<double>(sm, scratch);
    const double Sq = block_sum<double>(sq, scratch);
    double swa = 0.0, swa2 = 0.0;
    for (int k = 0; k < K; ++k) {
        swa += s_wa[k];
        swa2 += static_cast<double>(s_wa[k]) * s_wa[k];
    }
    const double n = static_cast<double>(npix) * K;
    const double mu = swa * Sm / n;
    double var = swa2 * Sq / n - mu * mu;
    if (var < 0.0) var = 0.0;
    const float mean = static_cast<float>(mu), rstd = static_cast<float>(1.0 / sqrt(var + eps));
    // pass 1: dxhat statistics for the GroupNorm backward (sum dxhat, sum dxhat * xhat) and the affine / wb / bb grads
    float t1 = 0.f, t2 = 0.f, tbb = 0.f;
    float agw[32], agb[32], awb[32];
    for (int k = 0; k < 32; ++k) agw[k] = agb[k] = awb[k] = 0.f;
    for (int p = tid; p < npix; p += kTeThreads) {
        float s = bb[0];
        for (int k = 0; k < K; ++k) s = fmaf(s_wb[k], gelu_exact(fmaf((s_wa[k] * m[p] - mean) * rstd, s_gw[k], s_gb[k])), s);
        const float a = sigmoidf_(s);
        const float ds = (a > 1e-4f && a < 1.f - 1e-4f) ? dAp[p] * a * (1.f - a) : 0.f;
        tbb += ds;
#pragma unroll
        for (int k = 0; k < 32; ++k) {
            if (k < K) {
                const float xh = (s_wa[k] * m[p] - mean) * rstd;
                const float y = fmaf(xh, s_gw[k], s_gb[k]);
                awb[k] = fmaf(ds, gelu_exact(y), awb[k]);
                const float dy = ds * s_wb[k] * gelu_grad(y);
                agw[k] = fmaf(dy, xh, agw[k]);
                agb[k] += dy;
                const float dxh = dy * s_gw[k];
                t1 += dxh;
                t2 = fmaf(dxh, xh, t2);
            }
        }
    }
    const float T1 = static_cast<float>(block_sum<double>(static_cast<double>(t1), scratch) / n);
    const float T2 = static_cast<float>(block_sum<double>(static_cast<double>(t2), scratch) / n);
    // pass 2: du = rstd * (dxhat - T1 - xhat T2);  dm[p] = sum_k du wa[k];  dwa[k] = sum_p du m[p]
    float awa[32];
    for (int k = 0; k < 32; ++k) awa[k] = 0.f;
    for (int p = tid; p < npix; p += kTeThreads) {
        float s = bb[0];
        for (int k = 0; k < K; ++k) s = fmaf(s_wb[k], gelu_exact(fmaf((s_wa[k] * m[p] - mean) * rstd, s_gw[k], s_gb[k])), s);
        const float a = sigmoidf_(s);
        const float ds = (a > 1e-4f && a < 1.f - 1e-4f) ? dAp[p] * a * (1.f - a) : 0.f;
        float dmp = 0.f;
#pragma unroll
        for (int k = 0; k < 32; ++k) {
            if (k < K) {
                const float xh = (s_wa[k] * m[p] - mean) * rstd;
                const float y = fmaf(xh, s_gw[k], s_gb[k]);
                const float dxh = ds * s_wb[k] * gelu_grad(y) * s_gw[k];
                const float du = rstd * (dxh - T1 - xh * T2);
                dmp = fmaf(du, s_wa[k], dmp);
                awa[k] = fmaf(du, m[p], awa[k]);
            }
        }
        dm[static_cast<long long>(b) * npix + p] = dmp;
    }
    for (int k = 0; k < K; ++k) {
        atomicAdd(&s_acc[0][k], awa[k]);
        atomicAdd(&s_acc[1][k], agw[k]);
        atomicAdd(&s_acc[2][k], agb[k]);
        atomicAdd(&s_acc[3][k], awb[k]);
    }
    const double Tbb = block_sum<double>(static_cast<double>(tbb), scratch);
    __syncthreads();
    if (tid < K) {
        atomicAdd(dwa + tid, s_acc[0][tid]);
        atomicAdd(dgnw + tid, s_acc[1][tid]);
        atomicAdd(dgnb + tid, s_acc[2][tid]);
        atomicAdd(dwb + tid, s_acc[3][tid]);
    }
    if (tid == 0) atomicAdd(dbb, static_cast<float>(Tbb));
}

// ---------------------------------------------------------------------------------------------- stem backward ----
// Forward (b200_stem_ex with every output channel in the un-activated segment): z[b,p,n] = sum_c wcat[n,c] x[b,c,s*p] gate[b,c].
// Backward from dz [B, npix, N] bf16:  dwcat[n,c] += gate[b,c] * sum_p dz[b,p,n] x[b,c,sp];
//   dgate[b,c] = sum_p x[b,c,sp] * sum_n dz[b,p,n] wcat[n,c].
// One CTA per case, 256-pixel tiles of x staged in shared memory (channels padded to CP).  Phase A: thread = pixel,
// t[c] = sum_n dz[p,n] w[n,c] with the weights broadcast from shared memory.  Phase B: thread = output channel n,
// acc[c] += dz[p,n] x[p,c] with dz read coalesced across n and x broadcast from shared memory.
template <int CP>
__global__ void __launch_bounds__(kTeThreads)
stem_bwd_kernel(const float* __restrict__ x, int C, int H, int W, int stride, const float* __restrict__ gate,
                const __nv_bfloat16* __restrict__ dz, int N, const float* __restrict__ wcat, float* __restrict__ dwcat,
                float* __restrict__ dgate) {
    extern __shared__ float s_st[];  // w[N][CP] | x[256][CP] | dg[CP]
    float* s_w = s_st;
    float* s_x = s_w + N * CP;
    float* s_dg = s_x + kTeThreads * CP;
    const int b = blockIdx.x, tid = threadIdx.x;
    const int Ho = H / stride, Wo = W / stride, npix = Ho * Wo;
    for (int i = tid; i < N * CP; i += kTeThreads) {
        const int n = i / CP, c = i - n * CP;
        s_w[i] = c < C ? wcat[n * C + c] : 0.f;
    }
    if (tid < CP) s_dg[tid] = 0.f;
    float dg[CP], acc[CP];
#pragma unroll
    for (int c = 0; c < CP; ++c) dg[c] = acc[c] = 0.f;
    const __nv_bfloat16* dzb = dz + static_cast<long long>(b) * npix * N;
    for (int pix0 = 0; pix0 < npix; pix0 += kTeThreads) {
        const int np = min(kTeThreads, npix - pix0);
        __syncthreads();  // previous tile's readers are done with s_x
        for (int i = tid; i < kTeThreads * CP; i += kTeThreads) {
            const int c = i / kTeThreads, pp = i - c * kTeThreads;
            float v = 0.f;
            if (c < C && pp < np) {
                const int pix = pix0 + pp;
                const int ho = pix / Wo, wo = pix - ho * Wo;
                v = __ldg(x + ((static_cast<long long>(b) * C + c) * H + ho * stride) * W + wo * stride);
            }
            s_x[pp * CP + c] = v;
        }
        __syncthreads();
        if (tid < np) {  // phase A
            float t[CP];
#pragma unroll
            for (int c = 0; c < CP; ++c) t[c] = 0.f;
            const __nv_bfloat16* row = dzb + static_cast<long long>(pix0 + tid) * N;
            for (int n0 = 0; n0 < N; n0 += 8) {
                float f[8];
                unpack_bf16x8(__ldg(reinterpret_cast<const uint4*>(row + n0)), f);
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const float4* w4 = reinterpret_cast<const float4*>(s_w + (n0 + k) * CP);
#pragma unroll
                    for (int c4 = 0; c4 < CP / 4; ++c4) {
                        const float4 wv = w4[c4];
                        t[4 * c4 + 0] = fmaf(f[k], wv.x, t[4 * c4 + 0]);
                        t[4 * c4 + 1] = fmaf(f[k], wv.y, t[4 * c4 + 1]);
                        t[4 * c4 + 2] = fmaf(f[k], wv.z, t[4 * c4 + 2]);
                        t[4 * c4 + 3] = fmaf(f[k], wv.w, t[4 * c4 + 3]);
                    }
                }
            }
#pragma unroll
            for (int c = 0; c < CP; ++c) dg[c] = fmaf(t[c], s_x[tid * CP + c], dg[c]);
        }
        if (tid < N) {  // phase B
            for (int pp = 0; pp < np; ++pp) {
                const float v = __bfloat162float(dzb[static_cast<long long>(pix0 + pp) * N + tid]);
                const float4* x4 = reinterpret_cast<const float4*>(s_x + pp * CP);
#pragma unroll
                for (int c4 = 0; c4 < CP / 4; ++c4) {
                    const float4 xv = x4[c4];
                    acc[4 * c4 + 0] = fmaf(v, xv.x, acc[4 * c4 + 0]);
                    acc[4 * c4 + 1] = fmaf(v, xv.y, acc[4 * c4 + 1]);
                    acc[4 * c4 + 2] = fmaf(v, xv.z, acc[4 * c4 + 2]);
                    acc[4 * c4 + 3] = fmaf(v, xv.w, acc[4 * c4 + 3]);
                }
            }
        }
    }
#pragma unroll
    for (int c = 0; c < CP; ++c) {
        const float v = warp_sum(dg[c]);
        if ((tid & 31) == 0 && c < C) atomicAdd(&s_dg[c], v);
    }
    if (tid < N) {
#pragma unroll
        for (int c = 0; c < CP; ++c)
            if (c < C) atomicAdd(dwcat + tid * C + c, acc[c] * (gate != nullptr ? gate[static_cast<long long>(b) * C + c] : 1.f));
    }
    __syncthreads();
    if (dgate != nullptr && tid < C) atomicAdd(dgate + static_cast<long long>(b) * C + tid, s_dg[tid]);
}

// --------------------------------------------------------------------------------------------- classifier head ---
// ClassificationHead (code/model_module.py:355-369): v = pooled (mean), u = v / max(||v||, 1e-12), logits = W u + b.
// Backward from dlogits: dW += dlogits^T u, db += dlogits, dpooled = (I - u u^T) W^T dlogits / ||v||.  One CTA per case.
__global__ void __launch_bounds__(kTeThreads)
cls_head_bwd_kernel(const float* __restrict__ pooled, const float* __restrict__ dlogits, const float* __restrict__ fcw,
                    int C, int K, int normalize, float* __restrict__ dfcw, float* __restrict__ dfcb,
                    float* __restrict__ dpooled) {
    extern __shared__ float s_cl[];  // u[C] | g[C]
    __shared__ double scratch[33];
    float* s_u = s_cl;
    float* s_g = s_u + C;
    const int b = blockIdx.x, tid = threadIdx.x;
    const float* v = pooled + static_cast<long long>(b) * C;
    const float* dl = dlogits + static_cast<long long>(b) * K;
    float ss = 0.f;
    for (int c = tid; c < C; c += kTeThreads) ss = fmaf(v[c], v[c], ss);
    const float nrm = normalize ? fmaxf(sqrtf(static_cast<float>(block_sum<double>(static_cast<double>(ss), scratch))), 1e-12f) : 1.f;
    float dot = 0.f;
    for (int c = tid; c < C; c += kTeThreads) {
        const float u = v[c] / nrm;
        float g = 0.f;
        for (int k = 0; k < K; ++k) {
            g = fmaf(fcw[k * C + c], dl[k], g);
            atomicAdd(dfcw + k * C + c, dl[k] * u);
        }
        s_u[c] = u;
        s_g[c] = g;
        dot = fmaf(g, u, dot);
    }
    const float D = normalize ? static_cast<float>(block_sum<double>(static_cast<double>(dot), scratch)) : 0.f;
    for (int c = tid; c < C; c += kTeThreads) dpooled[static_cast<long long>(b) * C + c] = (s_g[c] - s_u[c] * D) / nrm;
    if (tid < K) atomicAdd(dfcb + tid, dl[tid]);
}

// ----------------------------------------------------------------------------------------------------- losses ----
// LabelSmoothing + Soft(Weighted)FocalLoss, reduction "mean" (code/loss.py:133-213): loss += scale * sum_b l_b;
// dlogits[b,:] = scale * dl_b/dlogits.  One thread per case (K <= 16).
__global__ void focal_loss_kernel(const float* __restrict__ logits, const long long* __restrict__ labels, int B, int K,
                                  float smoothing, float gamma, const float* __restrict__ cw, float scale,
                                  float* __restrict__ loss, float* __restrict__ dlogits) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    float l = 0.f;
    if (b < B) {
        const float* z = logits + static_cast<long long>(b) * K;
        float mx = -FLT_MAX;
        for (int k = 0; k < K; ++k) mx = fmaxf(mx, z[k]);
        float se = 0.f;
        for (int k = 0; k < K; ++k) se += expf(z[k] - mx);
        const float lse = mx + logf(se);
        // l = -sum_k t_k w_k (1 - p_k)^gamma log p_k ;  dl/dlogp_k = -t_k w_k [ (1-p)^g - g p (1-p)^(g-1) log p ] =: a_k
        // dl/dz_j = a_j - p_j sum_k a_k
        float a[16], pr[16], sa = 0.f;
        for (int k = 0; k < K; ++k) {
            const float lp = z[k] - lse, p = expf(lp);
            const float t = (k == static_cast<int>(labels[b])) ? 1.f - smoothing : smoothing / (K - 1);
            const float w = cw != nullptr ? cw[k] : 1.f;
            const float om = fmaxf(1.f - p, 0.f);
            const float fw = powf(om, gamma);
            l -= t * w * fw * lp;
            const float dfw = om > 0.f ? gamma * powf(om, gamma - 1.f) : 0.f;
            a[k] = -t * w * (fw - dfw * p * lp);
            pr[k] = p;
            sa += a[k];
        }
        for (int k = 0; k < K; ++k) dlogits[static_cast<long long>(b) * K + k] = scale * (a[k] - pr[k] * sa);
    }
    l = warp_sum(l);
    if ((threadIdx.x & 31) == 0 && l != 0.f) atomicAdd(loss, scale * l);
}

// SoftDiceLoss (code/loss.py:45-62) on logits [B, n] vs targets [B, n]: loss += scale * sum_b (1 - dice_b);
// dlogits = scale * d(1 - dice_b)/dlogit.  One CTA per case.
__global__ void __launch_bounds__(kTeThreads)
dice_loss_kernel(const float* __restrict__ logits, const float* __restrict__ target, int n, float eps, float scale,
                 float* __restrict__ loss, float* __restrict__ dlogits) {
    __shared__ double scratch[33];
    const int b = blockIdx.x;
    const float* z = logits + static_cast<long long>(b) * n;
    const float* t = target + static_cast<long long>(b) * n;
    float si = 0.f, sp = 0.f, st = 0.f;
    for (int i = threadIdx.x; i < n; i += kTeThreads) {
        const float p = sigmoidf_(z[i]);
        si = fmaf(p, t[i], si);
        sp += p;
        st += t[i];
    }
    const float I = static_cast<float>(block_sum<double>(static_cast<double>(si), scratch));
    const float U = static_cast<float>(block_sum<double>(static_cast<double>(sp), scratch)) +
                    static_cast<float>(block_sum<double>(static_cast<double>(st), scratch));
    const float num = 2.f * I + eps, den = U + eps;
    if (threadIdx.x == 0) atomicAdd(loss, scale * (1.f - num / den));
    if (dlogits != nullptr) {
        for (int i = threadIdx.x; i < n; i += kTeThreads) {
            const float p = sigmoidf_(z[i]);
            // d(1 - num/den)/dp_i = -(2 t_i den - num) / den^2
            dlogits[static_cast<long long>(b) * n + i] = scale * (-(2.f * t[i] * den - num) / (den * den)) * p * (1.f - p);
        }
    }
}

// Reconstruction term (code/train.py:1041-1048, :446-454; code/train_fusion.py:709-745): r [B,h,w] fp32 (1 channel) is
// bilinearly up-sampled to the input size (align_corners = False), sigmoid, clamp(0,1), Charbonnier against the
// clamp(0,1) channel-MEAN of the fp32 input x [B,C,H,W]:  loss += scale * sum sqrt((s - t)^2 + eps^2)
// (scale = weight / (B H W)).  dr[b,i,j] = scale * sum over the output pixels it feeds.  One CTA per case; h*w <= 4096.
__global__ void __launch_bounds__(kTeThreads)
recon_loss_kernel(const float* __restrict__ r, int h, int w, const float* __restrict__ x, int C, const float* __restrict__ x2,
                  int C2, int H, int W, float eps, float scale, float* __restrict__ loss, float* __restrict__ dr) {
    extern __shared__ float s_dr[];  // [h*w]
    __shared__ double scratch[33];
    const int b = blockIdx.x;
    for (int i = threadIdx.x; i < h * w; i += kTeThreads) s_dr[i] = 0.f;
    __syncthreads();
    const float* rb = r + static_cast<long long>(b) * h * w;
    const float sy = static_cast<float>(h) / H, sx = static_cast<float>(w) / W;
    float acc = 0.f;
    for (int i = threadIdx.x; i < H * W; i += kTeThreads) {
        const int oy = i / W, ox = i - oy * W;
        const float fy = fmaxf((oy + 0.5f) * sy - 0.5f, 0.f), fx = fmaxf((ox + 0.5f) * sx - 0.5f, 0.f);
        const int y0 = min(static_cast<int>(fy), h - 1), x0 = min(static_cast<int>(fx), w - 1);
        const int y1 = min(y0 + 1, h - 1), x1 = min(x0 + 1, w - 1);
        const float ly = fy - y0, lx = fx - x0;
        const float w00 = (1.f - ly) * (1.f - lx), w01 = (1.f - ly) * lx, w10 = ly * (1.f - lx), w11 = ly * lx;
        const float v = w00 * rb[y0 * w + x0] + w01 * rb[y0 * w + x1] + w10 * rb[y1 * w + x0] + w11 * rb[y1 * w + x1];
        float t = 0.f;
        for (int c = 0; c < C; ++c) t += x[((static_cast<long long>(b) * C + c) * H + oy) * W + ox];
        for (int c = 0; c < C2; ++c) t += x2[((static_cast<long long>(b) * C2 + c) * H + oy) * W + ox];
        t = fminf(fmaxf(t / (C + C2), 0.f), 1.f);
        const float s = sigmoidf_(v);
        const float d = s - t;
        const float e = sqrtf(d * d + eps * eps);
        acc += e;
        const float g = scale * (d / e) * s * (1.f - s);
        atomicAdd(&s_dr[y0 * w + x0], g * w00);
        atomicAdd(&s_dr[y0 * w + x1], g * w01);
        atomicAdd(&s_dr[y1 * w + x0], g * w10);
        atomicAdd(&s_dr[y1 * w + x1], g * w11);
    }
    const double T = block_sum<double>(static_cast<double>(acc), scratch);
    if (threadIdx.x == 0) atomicAdd(loss, scale * static_cast<float>(T));
    __syncthreads();
    if (dr != nullptr)
        for (int i = threadIdx.x; i < h * w; i += kTeThreads) dr[static_cast<long long>(b) * h * w + i] = s_dr[i];
}

// Mimic term (code/train.py:1033-1038): per case cos = <s, t> / (|s| |t|) over the flattened maps (F.normalize eps
// 1e-12 on each norm), loss += scale * sum_b (1 - clamp(cos, -1 + 1e-6, 1 - 1e-6)); the teacher t is detached:
// ds = -scale * (t / (|s||t|) - cos * s / |s|^2) inside the clamp, 0 outside.  One CTA per case.
__global__ void __launch_bounds__(kTeThreads)
mimic_loss_kernel(const __nv_bfloat16* __restrict__ s, const __nv_bfloat16* __restrict__ t, long long n, float scale,
                  float* __restrict__ loss, __nv_bfloat16* __restrict__ ds) {
    __shared__ double scratch[33];
    const int b = blockIdx.x;
    const __nv_bfloat16* sb = s + b * n;
    const __nv_bfloat16* tb = t + b * n;
    float st = 0.f, ss = 0.f, tt = 0.f;
    for (long long i = threadIdx.x * 8LL; i < n; i += kTeThreads * 8LL) {
        float u[8], v[8];
        unpack_bf16x8(__ldg(reinterpret_cast<const uint4*>(sb + i)), u);
        unpack_bf16x8(__ldg(reinterpret_cast<const uint4*>(tb + i)), v);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            st = fmaf(u[k], v[k], st);
            ss = fmaf(u[k], u[k], ss);
            tt = fmaf(v[k], v[k], tt);
        }
    }
    const double ST = block_sum<double>(static_cast<double>(st), scratch);
    const double SS = block_sum<double>(static_cast<double>(ss), scratch);
    const double TT = block_sum<double>(static_cast<double>(tt), scratch);
    const double ns = fmax(sqrt(SS), 1e-12), nt = fmax(sqrt(TT), 1e-12);
    const double cosv = ST / (ns * nt);
    const bool inside = cosv > -1.0 + 1e-6 && cosv < 1.0 - 1e-6;
    const double cl = cosv < -1.0 + 1e-6 ? -1.0 + 1e-6 : (cosv > 1.0 - 1e-6 ? 1.0 - 1e-6 : cosv);
    if (threadIdx.x == 0) atomicAdd(loss, scale * static_cast<float>(1.0 - cl));
    if (ds != nullptr) {
        const float k1 = inside ? static_cast<float>(-scale / (ns * nt)) : 0.f;
        const float k2 = inside ? static_cast<float>(scale * cosv / (ns * ns)) : 0.f;
        for (long long i = threadIdx.x * 8LL; i < n; i += kTeThreads * 8LL) {
            float u[8], v[8], o[8];
            unpack_bf16x8(__ldg(reinterpret_cast<const uint4*>(sb + i)), u);
            unpack_bf16x8(__ldg(reinterpret_cast<const uint4*>(tb + i)), v);
#pragma unroll
            for (int k = 0; k < 8; ++k) o[k] = k1 * v[k] + k2 * u[k];
            *reinterpret_cast<uint4*>(ds + b * n + i) = pack_bf16x8(o);
        }
    }
}


// ------------------------------------------------------------------------------------------- fusion head ---------
// GatingAttention (code/model_module.py:745-780): gx = [pvec_dwi, pvec_dce, mean(mask_dwi), mean(mask_dce)],
// alpha = softmax(W gx + b) over the two modalities.  One CTA per case.  pvec_* are per-case channel SUMS (x inv_npix).
__global__ void __launch_bounds__(kTeThreads)
gating_fwd_kernel(const float* __restrict__ sum_d, const float* __restrict__ sum_c, float inv_npix,
                  const float* __restrict__ mask_d, const float* __restrict__ mask_c, int npix_mask, int C,
                  const float* __restrict__ w, const float* __restrict__ bias, float* __restrict__ gx,
                  float* __restrict__ alpha) {
    __shared__ double scratch[33];
    const int b = blockIdx.x, tid = threadIdx.x;
    const int D = 2 * C + (mask_d != nullptr ? 2 : 0);
    float* g = gx + static_cast<long long>(b) * D;
    float md = 0.f, mc = 0.f;
    if (mask_d != nullptr) {
        for (int i = tid; i < npix_mask; i += kTeThreads) {
            md += mask_d[static_cast<long long>(b) * npix_mask + i];
            mc += mask_c[static_cast<long long>(b) * npix_mask + i];
        }
        md = static_cast<float>(block_sum<double>(static_cast<double>(md), scratch) / npix_mask);
        mc = static_cast<float>(block_sum<double>(static_cast<double>(mc), scratch) / npix_mask);
    }
    float a0 = 0.f, a1 = 0.f;
    for (int i = tid; i < D; i += kTeThreads) {
        float v;
        if (i < C) v = sum_d[static_cast<long long>(b) * C + i] * inv_npix;
        else if (i < 2 * C) v = sum_c[static_cast<long long>(b) * C + i - C] * inv_npix;
        else v = i == 2 * C ? md : mc;
        g[i] = v;
        a0 = fmaf(w[i], v, a0);
        a1 = fmaf(w[D + i], v, a1);
    }
    const float l0 = static_cast<float>(block_sum<double>(static_cast<double>(a0), scratch)) + bias[0];
    const float l1 = static_cast<float>(block_sum<double>(static_cast<double>(a1), scratch)) + bias[1];
    if (tid == 0) {
        const float m = fmaxf(l0, l1);
        const float e0 = expf(l0 - m), e1 = expf(l1 - m);
        alpha[b * 2 + 0] = e0 / (e0 + e1);
        alpha[b * 2 + 1] = e1 / (e0 + e1);
    }
}
// softmax backward + input gradient: dgl = alpha * (dalpha - <alpha, dalpha>), dgx = dgl W.  (dW = dgl^T gx and db =
// column sums of dgl are taken by b200_sgemm / b200_colsum.)
__global__ void gating_bwd_kernel(const float* __restrict__ alpha, const float* __restrict__ dalpha,
                                  const float* __restrict__ w, int C, int D, float inv_npix, float* __restrict__ dgl,
                                  float* __restrict__ dgx, float* __restrict__ dpv_d, float* __restrict__ dpv_c) {
    const int b = blockIdx.x;
    const float a0 = alpha[b * 2], a1 = alpha[b * 2 + 1];
    const float d0 = dalpha[b * 2], d1 = dalpha[b * 2 + 1];
    const float dot = a0 * d0 + a1 * d1;
    const float g0 = a0 * (d0 - dot), g1 = a1 * (d1 - dot);
    if (threadIdx.x == 0) {
        dgl[b * 2] = g0;
        dgl[b * 2 + 1] = g1;
    }
    for (int i = threadIdx.x; i < D; i += blockDim.x) {
        const float v = g0 * w[i] + g1 * w[D + i];
        dgx[static_cast<long long>(b) * D + i] = v;
        // gradient w.r.t. the per-case channel SUMS' pixels: the pooled vectors are means over npix pixels
        if (i < C) dpv_d[static_cast<long long>(b) * C + i] = v * inv_npix;
        else if (i < 2 * C) dpv_c[static_cast<long long>(b) * C + i - C] = v * inv_npix;
    }
}

// pooled fused vector (GAP of alpha0 p_dwi + alpha1 p_dce + bilinear_up(lowres)), as channel "sums" with npix = 1:
// out[b,c] = alpha0 pvec_d + alpha1 pvec_c + sum_t up[t] lowres[b,t,c]
__global__ void fused_pool_kernel(const float* __restrict__ sum_d, const float* __restrict__ sum_c, float inv_npix,
                                  const float* __restrict__ alpha, const float* __restrict__ lowres,
                                  const float* __restrict__ up, int T, int C, float* __restrict__ out) {
    const int b = blockIdx.x;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float v = (alpha[b * 2] * sum_d[static_cast<long long>(b) * C + c] + alpha[b * 2 + 1] * sum_c[static_cast<long long>(b) * C + c]) * inv_npix;
        if (lowres != nullptr)
            for (int t = 0; t < T; ++t) v = fmaf(up[t], lowres[(static_cast<long long>(b) * T + t) * C + c], v);
        out[static_cast<long long>(b) * C + c] = v;
    }
}

// Backward of fused = alpha0 p_dwi + alpha1 p_dce + bilinear_up(lowres) from dfused [B,H,W,C] bf16.
// reduce pass: dalpha[b,m] += sum dfused * p_m;  dlowres[b,t,c] += sum_p U[p,t] dfused[b,p,c]   (grid: (slabs, B))
__global__ void __launch_bounds__(kTeThreads)
fusion_mix_bwd_reduce_kernel(const __nv_bfloat16* __restrict__ df, const __nv_bfloat16* __restrict__ pd,
                             const __nv_bfloat16* __restrict__ pc, int H, int W, int C, int Hp, int Wp,
                             float* __restrict__ dalpha, float* __restrict__ dlowres) {
    extern __shared__ float s_low[];  // [Hp*Wp][C]
    __shared__ double scratch[33];
    const int b = blockIdx.y, tid = threadIdx.x;
    const int T = Hp * Wp, CG = C / 8, npix = H * W;
    for (int i = tid; i < T * C; i += kTeThreads) s_low[i] = 0.f;
    __syncthreads();
    float ad = 0.f, ac = 0.f;
    const int per = (npix + gridDim.x - 1) / gridDim.x;
    const int p0 = blockIdx.x * per, p1 = min(p0 + per, npix);
    const float sy = static_cast<float>(Hp) / H, sx = static_cast<float>(Wp) / W;
    for (int i = p0 * CG + tid; i < p1 * CG; i += kTeThreads) {
        const int pix = i / CG, c0 = (i - pix * CG) * 8;
        const long long off = (static_cast<long long>(b) * npix + pix) * C + c0;
        float g[8], u[8], v[8];
        unpack_bf16x8(__ldg(reinterpret_cast<const uint4*>(df + off)), g);
        unpack_bf16x8(__ldg(reinterpret_cast<const uint4*>(pd + off)), u);
        unpack_bf16x8(__ldg(reinterpret_cast<const uint4*>(pc + off)), v);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            ad = fmaf(g[k], u[k], ad);
            ac = fmaf(g[k], v[k], ac);
        }
        if (dlowres != nullptr) {
            const int oy = pix / W, ox = pix - oy * W;
            const float fy = fmaxf((oy + 0.5f) * sy - 0.5f, 0.f), fx = fmaxf((ox + 0.5f) * sx - 0.5f, 0.f);
            const int y0 = min(static_cast<int>(fy), Hp - 1), x0 = min(static_cast<int>(fx), Wp - 1);
            const int y1 = min(y0 + 1, Hp - 1), x1 = min(x0 + 1, Wp - 1);
            const float ly = fy - y0, lx = fx - x0;
            const float wt[4] = {(1.f - ly) * (1.f - lx), (1.f - ly) * lx, ly * (1.f - lx), ly * lx};
            const int tk[4] = {y0 * Wp + x0, y0 * Wp + x1, y1 * Wp + x0, y1 * Wp + x1};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (wt[q] != 0.f) {
#pragma unroll
                    for (int k = 0; k < 8; ++k) atomicAdd(&s_low[tk[q] * C + c0 + k], wt[q] * g[k]);
                }
            }
        }
    }
    const double AD = block_sum<double>(static_cast<double>(ad), scratch);
    const double AC = block_sum<double>(static_cast<double>(ac), scratch);
    if (tid == 0) {
        atomicAdd(dalpha + b * 2, static_cast<float>(AD));
        atomicAdd(dalpha + b * 2 + 1, static_cast<float>(AC));
    }
    __syncthreads();
    if (dlowres != nullptr)
        for (int i = tid; i < T * C; i += kTeThreads) atomicAdd(dlowres + static_cast<long long>(b) * T * C + i, s_low[i]);
}
// apply pass: dp_m[b,p,c] = alpha_m dfused + dtok_m[b, bin(p), c] + dpvec_m[b,c]   (dtok already / bin size, dpvec / npix)
__global__ void __launch_bounds__(kTeThreads)
fusion_mix_bwd_apply_kernel(const __nv_bfloat16* __restrict__ df, const float* __restrict__ alpha,
                            const float* __restrict__ dtok_d, const float* __restrict__ dtok_c,
                            const float* __restrict__ dpv_d, const float* __restrict__ dpv_c, int B, int H, int W, int C,
                            int Hp, int Wp, __nv_bfloat16* __restrict__ dpd, __nv_bfloat16* __restrict__ dpc) {
    const int CG = C / 8, npix = H * W, T = Hp * Wp;
    const long long total = static_cast<long long>(B) * npix * CG;
    for (long long i = blockIdx.x * static_cast<long long>(kTeThreads) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * kTeThreads) {
        const int c0 = static_cast<int>(i % CG) * 8;
        const long long r = i / CG;
        const int pix = static_cast<int>(r % npix);
        const long long b = r / npix;
        const int oy = pix / W, ox = pix - oy * W;
        const int t = (oy * Hp / H) * Wp + (ox * Wp / W);
        float g[8], o0[8], o1[8];
        unpack_bf16x8(__ldg(reinterpret_cast<const uint4*>(df + r * C + c0)), g);
        const float a0 = alpha[b * 2], a1 = alpha[b * 2 + 1];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            float e0 = a0 * g[k], e1 = a1 * g[k];
            if (dtok_d != nullptr) {
                e0 += dtok_d[(b * T + t) * C + c0 + k];
                e1 += dtok_c[(b * T + t) * C + c0 + k];
            }
            if (dpv_d != nullptr) {
                e0 += dpv_d[b * C + c0 + k];
                e1 += dpv_c[b * C + c0 + k];
            }
            o0[k] = e0;
            o1[k] = e1;
        }
        *reinterpret_cast<uint4*>(dpd + r * C + c0) = pack_bf16x8(o0);
        *reinterpret_cast<uint4*>(dpc + r * C + c0) = pack_bf16x8(o1);
    }
}

// The fusion step's mimic term as the reference writes it (code/train_fusion.py:287-296): `proj_fused[:4]` unpacks the
// first four CASES of the fused projection as (p1, p1_r, p2, p2_r); mimic_feat_loss flattens a [C,H,W] tensor from dim
// 1, so the cosine is taken per CHANNEL over the pixels and averaged over channels.  map [B, npix, C] bf16 (B >= 4).
// loss += scale * (mean_c(1 - cos_c(case0, case1)) + mean_c(1 - cos_c(case2, case3))) / 2; dmap is zero except for
// the student cases 0 and 2.  grid = 2 (one CTA per pair), thread = channel.
__global__ void mimic_pairs_kernel(const __nv_bfloat16* __restrict__ map, int npix, int C, float scale,
                                   float* __restrict__ loss, __nv_bfloat16* __restrict__ dmap) {
    __shared__ double scratch[33];
    const int pair = blockIdx.x;
    const __nv_bfloat16* s = map + static_cast<long long>(2 * pair) * npix * C;
    const __nv_bfloat16* t = map + static_cast<long long>(2 * pair + 1) * npix * C;
    float acc = 0.f;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float st = 0.f, ss = 0.f, tt = 0.f;
        for (int p = 0; p < npix; ++p) {
            const float u = __bfloat162float(s[static_cast<long long>(p) * C + c]);
            const float v = __bfloat162float(t[static_cast<long long>(p) * C + c]);
            st = fmaf(u, v, st);
            ss = fmaf(u, u, ss);
            tt = fmaf(v, v, tt);
        }
        const float ns = fmaxf(sqrtf(ss), 1e-12f), nt = fmaxf(sqrtf(tt), 1e-12f);
        const float cosv = st / (ns * nt);
        const bool inside = cosv > -1.f + 1e-6f && cosv < 1.f - 1e-6f;
        acc += 1.f - fminf(fmaxf(cosv, -1.f + 1e-6f), 1.f - 1e-6f);
        if (dmap != nullptr) {
            const float w = scale * 0.5f / C;
            const float k1 = inside ? -w / (ns * nt) : 0.f, k2 = inside ? w * cosv / (ns * ns) : 0.f;
            __nv_bfloat16* d = dmap + static_cast<long long>(2 * pair) * npix * C;
            for (int p = 0; p < npix; ++p) {
                const float u = __bfloat162float(s[static_cast<long long>(p) * C + c]);
                const float v = __bfloat162float(t[static_cast<long long>(p) * C + c]);
                d[static_cast<long long>(p) * C + c] = __float2bfloat16_rn(k1 * v + k2 * u);
            }
        }
    }
    const double A = block_sum<double>(static_cast<double>(acc), scratch);
    if (threadIdx.x == 0) atomicAdd(loss, scale * 0.5f * static_cast<float>(A) / C);
}

// 2x2 replication (AdaptiveAvgPool2d to twice the size) backward: din[b,h,w,c] = sum of the four replicas of dout
__global__ void __launch_bounds__(kTeThreads)
up2_bwd_kernel(const __nv_bfloat16* __restrict__ dout, int B, int H, int W, int C, __nv_bfloat16* __restrict__ din) {
    const int CG = C / 8;
    const long long total = static_cast<long long>(B) * H * W * CG;
    for (long long i = blockIdx.x * static_cast<long long>(kTeThreads) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * kTeThreads) {
        const int cg = static_cast<int>(i % CG);
        const long long pix = i / CG;
        const int wq = static_cast<int>(pix % W), hq = static_cast<int>((pix / W) % H);
        const long long b = pix / (static_cast<long long>(W) * H);
        float o[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) o[k] = 0.f;
#pragma unroll
        for (int rep = 0; rep < 4; ++rep) {
            const long long op = (b * (2 * H) + 2 * hq + (rep >> 1)) * (2 * W) + 2 * wq + (rep & 1);
            float f[8];
            unpack_bf16x8(__ldg(reinterpret_cast<const uint4*>(dout + op * C + cg * 8)), f);
#pragma unroll
            for (int k = 0; k < 8; ++k) o[k] += f[k];
        }
        *reinterpret_cast<uint4*>(din + pix * C + cg * 8) = pack_bf16x8(o);
    }
}

// out[b, i] = v[b * v_stride] * scale for i < n (gradient of a per-case mean of an fp32 map)
__global__ void row_bcast_kernel(const float* __restrict__ v, int v_stride, float scale, int n, float* __restrict__ out) {
    const int b = blockIdx.x;
    const float s = v[static_cast<long long>(b) * v_stride] * scale;
    for (int i = threadIdx.x; i < n; i += blockDim.x) out[static_cast<long long>(b) * n + i] = s;
}

// fp32 vector helpers for the tiny per-case tensors: y = alpha * a + beta * y
__global__ void vec_axpby_kernel(const float* __restrict__ a, float alpha, float beta, long long n, float* __restrict__ y) {
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<long long>(gridDim.x) * blockDim.x)
        y[i] = alpha * a[i] + (beta != 0.f ? beta * y[i] : 0.f);
}

}  // namespace b200

// ================================================================================================== C ABI =======
using namespace b200;

#define TE_STREAM static_cast<cudaStream_t>(stream)

extern "C" int b200_bn_stats(const void* z, long long R, int C, int ld, double* sum, double* sumsq, void* stream) {
    if (z == nullptr || sum == nullptr || sumsq == nullptr || R <= 0 || C <= 0 || C % 8 != 0 || C > 2048 || ld % 8 != 0) return -1;
    const int CG = C / 8, rows_par = kTeThreads / CG;
    if (rows_par < 1) return -2;
    const size_t smem = static_cast<size_t>(rows_par) * C * 2 * sizeof(float);
    long long want = (R + rows_par * 16 - 1) / (rows_par * 16);
    const int grid = static_cast<int>(want < 1 ? 1 : (want > 148 * 4 ? 148 * 4 : want));
    bn_stats_kernel<<<grid, kTeThreads, smem, TE_STREAM>>>(static_cast<const __nv_bfloat16*>(z), R, C, ld, sum, sumsq);
    return launch_status();
}

extern "C" int b200_bn_finalize(const double* sum, const double* sumsq, int C, double count, float eps, float momentum,
                                float* running_mean, float* running_var, float* mean_out, float* invstd_out,
                                void* stream) {
    if (sum == nullptr || sumsq == nullptr || mean_out == nullptr || invstd_out == nullptr || C <= 0 || count <= 0) return -1;
    bn_finalize_kernel<<<(C + 127) / 128, 128, 0, TE_STREAM>>>(sum, sumsq, C, count, eps, momentum, running_mean,
                                                              running_var, mean_out, invstd_out);
    return launch_status();
}

static int fill_bnact(BnAct& p, const void* z, int ldz, const void* res, int ldres, const float* mean,
                      const float* invstd, const float* gamma, const float* beta, int act, float drop_p,
                      unsigned long long seed, long long R, int C) {
    if (z == nullptr || R <= 0 || C <= 0 || C % 8 != 0 || ldz % 8 != 0 || (res != nullptr && ldres % 8 != 0)) return -1;
    if (act < 0 || act > 2 || !(drop_p >= 0.f && drop_p < 1.f)) return -2;
    p.z = static_cast<const __nv_bfloat16*>(z);
    p.ldz = ldz;
    p.res = static_cast<const __nv_bfloat16*>(res);
    p.ldres = ldres;
    p.mean = mean;
    p.invstd = invstd;
    p.gamma = gamma;
    p.beta = beta;
    p.act = act;
    p.drop_thresh = drop_p > 0.f ? dropout_threshold(drop_p) : 0u;
    p.drop_scale = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
    p.seed_lo = static_cast<unsigned int>(seed);
    p.seed_hi = static_cast<unsigned int>(seed >> 32);
    p.R = R;
    p.C = C;
    return 0;
}

// (act, residual?, dropout?) -> compile-time kernel options
template <typename F>
static void bn_dispatch(const BnAct& p, F&& f) {
    auto with_act = [&](auto act) {
        const bool res = p.res != nullptr, drop = p.drop_thresh != 0u;
        if (res && drop) f(act, std::true_type{}, std::true_type{});
        else if (res) f(act, std::true_type{}, std::false_type{});
        else if (drop) f(act, std::false_type{}, std::true_type{});
        else f(act, std::false_type{}, std::false_type{});
    };
    if (p.act == 1) with_act(std::integral_constant<int, 1>{});
    else if (p.act == 2) with_act(std::integral_constant<int, 2>{});
    else with_act(std::integral_constant<int, 0>{});
}

static int bn_grid(long long R, int C, int& rows_par) {
    rows_par = kTeThreads / (C / 4);
    long long want = (R + rows_par * 4 - 1) / (rows_par * 4);
    return static_cast<int>(want < 1 ? 1 : (want > 148 * 8 ? 148 * 8 : want));
}

extern "C" int b200_bn_act_fwd(const void* z, int ldz, const void* res, int ldres, const float* mean, const float* invstd,
                               const float* gamma, const float* beta, int act, float drop_p, unsigned long long seed,
                               long long R, int C, void* out, int ldo, void* stream) {
    BnAct p;
    int rc = fill_bnact(p, z, ldz, res, ldres, mean, invstd, gamma, beta, act, drop_p, seed, R, C);
    if (rc != 0 || out == nullptr || ldo % 8 != 0 || C > 1024) return rc != 0 ? rc : -3;
    int rows_par;
    const int grid = bn_grid(R, C, rows_par);
    bn_dispatch(p, [&](auto act, auto res, auto drop) {
        bn_act_fwd_kernel<decltype(act)::value, decltype(res)::value, decltype(drop)::value>
            <<<grid, kTeThreads, 0, TE_STREAM>>>(p, static_cast<__nv_bfloat16*>(out), ldo);
    });
    return launch_status();
}

extern "C" int b200_bn_act_bwd(const void* z, int ldz, const void* res, int ldres, const float* mean, const float* invstd,
                               const float* gamma, const float* beta, int act, float drop_p, unsigned long long seed,
                               long long R, int C, const void* dA, int ldd, int batch_stats, double* scratch2C,
                               void* dz, int lddz, void* dres, int lddres, float* dgamma, float* dbeta, void* stream) {
    BnAct p;
    int rc = fill_bnact(p, z, ldz, res, ldres, mean, invstd, gamma, beta, act, drop_p, seed, R, C);
    if (rc != 0 || dA == nullptr || ldd % 8 != 0 || C > 1024) return rc != 0 ? rc : -3;
    if (batch_stats && dz == nullptr) return -5;  // pass 2 works in place on dz
    const bool need_sums = batch_stats || dgamma != nullptr || dbeta != nullptr;
    double *s1 = nullptr, *s2 = nullptr;
    int rows_par;
    const int grid = bn_grid(R, C, rows_par);
    size_t smem = 0;
    if (need_sums) {
        if (scratch2C == nullptr) return -4;
        s1 = scratch2C;
        s2 = scratch2C + C;
        cudaMemsetAsync(scratch2C, 0, 2 * C * sizeof(double), TE_STREAM);
        smem = static_cast<size_t>(rows_par) * C * 2 * sizeof(float);
    }
    bn_dispatch(p, [&](auto act, auto res, auto drop) {
        bn_act_bwd_pass1_kernel<decltype(act)::value, decltype(res)::value, decltype(drop)::value>
            <<<grid, kTeThreads, smem, TE_STREAM>>>(p, static_cast<const __nv_bfloat16*>(dA), ldd, batch_stats ? 1 : 0,
                                                    static_cast<__nv_bfloat16*>(dz), lddz,
                                                    static_cast<__nv_bfloat16*>(dres), lddres, s1, s2);
    });
    if (need_sums) {
        bn_act_bwd_pass2_kernel<<<batch_stats ? grid : 1, kTeThreads, 0, TE_STREAM>>>(
            p, s1, s2, static_cast<double>(R), static_cast<__nv_bfloat16*>(dz), lddz, dgamma, dbeta, batch_stats ? 1 : 0);
    }
    return launch_status();
}

extern "C" int b200_map_dot(const void* a, int lda, const void* b, int ldb, int B, int npix, int C, float* out,
                            void* stream) {
    if (a == nullptr || out == nullptr || B <= 0 || npix <= 0 || C <= 0 || C % 8 != 0 || C > 2048) return -1;
    const int rows_par = kTeThreads / (C / 8);
    if (rows_par < 1) return -2;
    map_dot_kernel<<<B, kTeThreads, static_cast<size_t>(rows_par) * C * sizeof(float), TE_STREAM>>>(
        static_cast<const __nv_bfloat16*>(a), lda, static_cast<const __nv_bfloat16*>(b), ldb, npix, C, out);
    return launch_status();
}

extern "C" int b200_map_scale_add(const void* x, int ldx, const float* gate, const float* add, int B, int npix, int C,
                                  void* out, int ldo, int accumulate, void* stream) {
    if (out == nullptr || B <= 0 || npix <= 0 || C <= 0 || C % 8 != 0) return -1;
    const long long R = static_cast<long long>(B) * npix;
    const long long nvc = static_cast<long long>(npix) * (C / 8);
    const bool aligned = (gate == nullptr || (reinterpret_cast<uintptr_t>(gate) & 15) == 0) &&
                         (add == nullptr || (reinterpret_cast<uintptr_t>(add) & 15) == 0);
    if (B <= 65535 && nvc < (1LL << 30) && aligned) {
        // chunks per case: enough CTAs to fill the machine, each walking >= 2 vectors per thread
        long long chunks = (nvc + 2 * kTeThreads - 1) / (2 * kTeThreads);
        const long long cap = (148LL * 8 + B - 1) / B;
        if (chunks > cap) chunks = cap;
        if (chunks < 1) chunks = 1;
        const dim3 grid(static_cast<unsigned>(chunks), static_cast<unsigned>(B));
        auto go = [&](auto hx, auto hg, auto ha, auto ac) {
            map_scale_add_case_kernel<decltype(hx)::value, decltype(hg)::value, decltype(ha)::value, decltype(ac)::value>
                <<<grid, kTeThreads, 0, TE_STREAM>>>(static_cast<const __nv_bfloat16*>(x), ldx, gate, add, npix, C,
                                                     static_cast<__nv_bfloat16*>(out), ldo);
        };
        auto d3 = [&](auto hx, auto hg, auto ha) {
            if (accumulate) go(hx, hg, ha, std::true_type{}); else go(hx, hg, ha, std::false_type{});
        };
        auto d2 = [&](auto hx, auto hg) {
            if (add != nullptr) d3(hx, hg, std::true_type{}); else d3(hx, hg, std::false_type{});
        };
        auto d1 = [&](auto hx) {
            if (gate != nullptr) d2(hx, std::true_type{}); else d2(hx, std::false_type{});
        };
        if (x != nullptr) d1(std::true_type{}); else d1(std::false_type{});
        return launch_status();
    }
    map_scale_add_kernel<<<blocks_for(R * (C / 8)), kTeThreads, 0, TE_STREAM>>>(
        static_cast<const __nv_bfloat16*>(x), ldx, gate, add, R, npix, C, static_cast<__nv_bfloat16*>(out), ldo, accumulate);
    return launch_status();
}

extern "C" int b200_map_axpby(const void* a, int lda, float alpha, const void* b, int ldb, float beta, long long R, int C,
                              void* y, int ldy, void* stream) {
    if (a == nullptr || y == nullptr || R <= 0 || C <= 0 || C % 8 != 0) return -1;
    if (R * (C / 8) < (1LL << 30))
        map_axpby_kernel<int><<<blocks_for(R * (C / 8)), kTeThreads, 0, TE_STREAM>>>(
            static_cast<const __nv_bfloat16*>(a), lda, alpha, static_cast<const __nv_bfloat16*>(b), ldb, beta, R, C,
            static_cast<__nv_bfloat16*>(y), ldy);
    else
        map_axpby_kernel<long long><<<blocks_for(R * (C / 8)), kTeThreads, 0, TE_STREAM>>>(
            static_cast<const __nv_bfloat16*>(a), lda, alpha, static_cast<const __nv_bfloat16*>(b), ldb, beta, R, C,
            static_cast<__nv_bfloat16*>(y), ldy);
    return launch_status();
}

extern "C" int b200_map_sumsq(const void* a, int lda, long long R, int C, double* out, void* stream) {
    if (a == nullptr || out == nullptr || R <= 0 || C <= 0 || C % 8 != 0) return -1;
    map_sumsq_kernel<<<blocks_for(R * (C / 8), kTeThreads, 148 * 4), kTeThreads, 0, TE_STREAM>>>(
        static_cast<const __nv_bfloat16*>(a), lda, R, C, out);
    return launch_status();
}

extern "C" int b200_se_fwd(const float* sums, int B, int C, int M, int npix, const float* w1, const float* b1,
                           const float* w2, const float* b2, float* pooled, float* gate, void* stream) {
    if (sums == nullptr || gate == nullptr || B <= 0 || C <= 0 || M <= 0 || npix <= 0) return -1;
    se_fwd_kernel<<<B, kTeThreads, static_cast<size_t>(C + M) * sizeof(float), TE_STREAM>>>(sums, 1.0f / npix, w1, b1, w2, b2,
                                                                                           C, M, pooled, gate);
    return launch_status();
}

extern "C" int b200_se_bwd(const float* pooled, const float* w1, const float* b1, const float* w2, const float* b2,
                           const float* dgate, int B, int C, int M, float* dpooled, float* da2, float* da1, float* h,
                           void* stream) {
    if (pooled == nullptr || dgate == nullptr || B <= 0 || C <= 0 || M <= 0) return -1;
    const size_t smem = static_cast<size_t>(2 * C + 3 * M) * sizeof(float);
    if (smem > 48 * 1024) return -2;
    se_bwd_kernel<<<B, kTeThreads, smem, TE_STREAM>>>(pooled, w1, b1, w2, b2, dgate, C, M, dpooled, da2, da1, h);
    return launch_status();
}

static bool convc1_shape_ok(int H, int W, int C, int taps) {
    const int lpp = C / 8;
    return C % 8 == 0 && (lpp >= 32 ? C % 256 == 0 : (lpp & (lpp - 1)) == 0) && (taps == 1 || taps == 9) &&
           static_cast<size_t>(H) * W * taps * sizeof(float) <= 200 * 1024;
}

extern "C" int b200_convc1_fwd(const void* x, int ldx, int B, int H, int W, int C, int taps, const float* w,
                               const float* bias, float* out, void* stream) {
    if (x == nullptr || w == nullptr || out == nullptr || B <= 0 || !convc1_shape_ok(H, W, C, taps) || ldx % 8 != 0) return -1;
    const size_t smem = static_cast<size_t>(H) * W * taps * sizeof(float);
    auto go = [&](auto kern) -> int {
        if (smem > 48 * 1024) {
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
            if (e != cudaSuccess) return static_cast<int>(e);
        }
        kern<<<B, kTeThreads, smem, TE_STREAM>>>(static_cast<const __nv_bfloat16*>(x), ldx, H, W, C, w, bias, out);
        return launch_status();
    };
    return taps == 9 ? go(convc1_fwd_kernel<9>) : go(convc1_fwd_kernel<1>);
}

extern "C" int b200_convc1_bwd(const void* x, int ldx, const float* dout, int B, int H, int W, int C, int taps,
                               const float* w, void* dx, int lddx, int accumulate_dx, float* dw, float* dbias,
                               void* stream) {
    if (x == nullptr || w == nullptr || dout == nullptr || B <= 0 || !convc1_shape_ok(H, W, C, taps) || ldx % 8 != 0) return -1;
    const size_t smem = (static_cast<size_t>(H) * W + static_cast<size_t>(C) * taps) * sizeof(float);
    if (smem > 200 * 1024) return -2;
    auto go = [&](auto kern) -> int {
        if (smem > 48 * 1024) {
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
            if (e != cudaSuccess) return static_cast<int>(e);
        }
        kern<<<B, kTeThreads, smem, TE_STREAM>>>(dout, static_cast<const __nv_bfloat16*>(x), ldx, H, W, C, w,
                                                static_cast<__nv_bfloat16*>(dx), lddx, accumulate_dx, dw, dbias);
        return launch_status();
    };
    return taps == 9 ? go(convc1_bwd_kernel<9>) : go(convc1_bwd_kernel<1>);
}

extern "C" int b200_lift_fwd(const float* r, long long P, int N, const float* w, void* z, void* stream) {
    if (r == nullptr || w == nullptr || z == nullptr || P <= 0 || N % 8 != 0) return -1;
    lift_fwd_kernel<<<blocks_for(P * (N / 8)), kTeThreads, 0, TE_STREAM>>>(r, P, N, w, static_cast<__nv_bfloat16*>(z));
    return launch_status();
}

extern "C" int b200_lift_bwd(const void* dz, const float* r, long long P, int N, const float* w, float* dw, float* dr,
                             void* stream) {
    if (dz == nullptr || r == nullptr || w == nullptr || dw == nullptr || N % 2 != 0 || N > 128) return -1;
    lift_bwd_kernel<<<blocks_for(P * 32, kTeThreads, 148 * 4), kTeThreads, N * sizeof(float), TE_STREAM>>>(
        static_cast<const __nv_bfloat16*>(dz), r, P, N, w, dw, dr);
    return launch_status();
}

extern "C" int b200_modulate_bwd(const void* dy, int lddy, const void* f, int ldf, const float* A, const float* gamma,
                                 long long P, int C, void* df, int lddf, float* dA, float* dgamma, void* stream) {
    if (dy == nullptr || f == nullptr || A == nullptr || gamma == nullptr || df == nullptr || dA == nullptr || C % 8 != 0) return -1;
    modulate_bwd_kernel<<<blocks_for(P * 32, kTeThreads, 148 * 8), kTeThreads, 0, TE_STREAM>>>(
        static_cast<const __nv_bfloat16*>(dy), lddy, static_cast<const __nv_bfloat16*>(f), ldf, A, gamma, P, C,
        static_cast<__nv_bfloat16*>(df), lddf, dA, dgamma);
    return launch_status();
}

extern "C" int b200_mask_attn_bwd(const float* mask, const float* dA, int B, int npix, int K, const float* wa,
                                  const float* gnw, const float* gnb, const float* wb, const float* bb, float eps,
                                  float* dm, float* dwa, float* dgnw, float* dgnb, float* dwb, float* dbb, void* stream) {
    if (mask == nullptr || dA == nullptr || dm == nullptr || K <= 0 || K > 32 || B <= 0) return -1;
    mask_attn_bwd_kernel<<<B, kTeThreads, 0, TE_STREAM>>>(mask, dA, npix, K, wa, gnw, gnb, wb, bb, eps, dm, dwa, dgnw, dgnb,
                                                         dwb, dbb);
    return launch_status();
}

extern "C" int b200_stem_bwd(const float* x, int B, int C, int H, int W, int stride, const float* gate, const void* dz,
                             int N, const float* wcat, float* dwcat, float* dgate, void* stream) {
    if (x == nullptr || dz == nullptr || wcat == nullptr || dwcat == nullptr || C <= 0 || C > 32 || N > kTeThreads || N % 8 != 0 ||
        B <= 0)
        return -1;
    // the forward (b200_stem_ex) takes every stride-th pixel of an H x W plane that the stride divides
    if (stride < 1 || H % stride != 0 || W % stride != 0) return -1;
    const int CP = C <= 8 ? 8 : (C <= 16 ? 16 : 32);
    const size_t smem = (static_cast<size_t>(N) * CP + static_cast<size_t>(kTeThreads) * CP + CP) * sizeof(float);
    auto go = [&](auto kern) -> int {
        if (smem > 48 * 1024) {
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
            if (e != cudaSuccess) return static_cast<int>(e);
        }
        kern<<<B, kTeThreads, smem, TE_STREAM>>>(x, C, H, W, stride, gate, static_cast<const __nv_bfloat16*>(dz), N, wcat, dwcat,
                                                dgate);
        return launch_status();
    };
    if (CP == 8) return go(stem_bwd_kernel<8>);
    if (CP == 16) return go(stem_bwd_kernel<16>);
    return go(stem_bwd_kernel<32>);
}

extern "C" int b200_cls_head_bwd(const float* pooled, const float* dlogits, const float* fcw, int B, int C, int K,
                                 int normalize, float* dfcw, float* dfcb, float* dpooled, void* stream) {
    if (pooled == nullptr || dlogits == nullptr || fcw == nullptr || B <= 0 || K > 16) return -1;
    cls_head_bwd_kernel<<<B, kTeThreads, 2 * C * sizeof(float), TE_STREAM>>>(pooled, dlogits, fcw, C, K, normalize, dfcw,
                                                                            dfcb, dpooled);
    return launch_status();
}

extern "C" int b200_focal_loss(const float* logits, const long long* labels, int B, int K, float smoothing, float gamma,
                               const float* class_weights, float scale, float* loss, float* dlogits, void* stream) {
    if (logits == nullptr || labels == nullptr || loss == nullptr || dlogits == nullptr || K > 16 || B <= 0) return -1;
    focal_loss_kernel<<<(B + 127) / 128, 128, 0, TE_STREAM>>>(logits, labels, B, K, smoothing, gamma, class_weights, scale,
                                                             loss, dlogits);
    return launch_status();
}

extern "C" int b200_dice_loss(const float* logits, const float* target, int B, int n, float eps, float scale, float* loss,
                              float* dlogits, void* stream) {
    if (logits == nullptr || target == nullptr || loss == nullptr || B <= 0 || n <= 0) return -1;
    dice_loss_kernel<<<B, kTeThreads, 0, TE_STREAM>>>(logits, target, n, eps, scale, loss, dlogits);
    return launch_status();
}

extern "C" int b200_recon_loss(const float* r, int B, int h, int w, const float* x, int C, const float* x2, int C2, int H,
                               int W, float eps, float scale, float* loss, float* dr, void* stream) {
    if (r == nullptr || x == nullptr || loss == nullptr || B <= 0 || h * w > 8192 || (x2 == nullptr && C2 != 0)) return -1;
    recon_loss_kernel<<<B, kTeThreads, static_cast<size_t>(h) * w * sizeof(float), TE_STREAM>>>(r, h, w, x, C, x2, C2, H, W,
                                                                                               eps, scale, loss, dr);
    return launch_status();
}

extern "C" int b200_mimic_loss(const void* s, const void* t, int B, long long n, float scale, float* loss, void* ds,
                               void* stream) {
    if (s == nullptr || t == nullptr || loss == nullptr || B <= 0 || n % 8 != 0) return -1;
    mimic_loss_kernel<<<B, kTeThreads, 0, TE_STREAM>>>(static_cast<const __nv_bfloat16*>(s),
                                                      static_cast<const __nv_bfloat16*>(t), n, scale, loss,
                                                      static_cast<__nv_bfloat16*>(ds));
    return launch_status();
}


extern "C" int b200_gating_fwd(const float* sum_d, const float* sum_c, int B, int C, int npix, const float* mask_d,
                               const float* mask_c, int npix_mask, const float* w, const float* bias, float* gx,
                               float* alpha, void* stream) {
    if (sum_d == nullptr || sum_c == nullptr || w == nullptr || bias == nullptr || gx == nullptr || alpha == nullptr || B <= 0) return -1;
    gating_fwd_kernel<<<B, kTeThreads, 0, TE_STREAM>>>(sum_d, sum_c, 1.0f / npix, mask_d, mask_c, npix_mask, C, w, bias, gx, alpha);
    return launch_status();
}
extern "C" int b200_gating_bwd(const float* alpha, const float* dalpha, const float* w, int B, int C, int D, int npix,
                               float* dgl, float* dgx, float* dpv_d, float* dpv_c, void* stream) {
    if (alpha == nullptr || dalpha == nullptr || w == nullptr || dgl == nullptr || dgx == nullptr || dpv_d == nullptr ||
        dpv_c == nullptr || B <= 0 || npix <= 0)
        return -1;
    gating_bwd_kernel<<<B, 128, 0, TE_STREAM>>>(alpha, dalpha, w, C, D, 1.0f / npix, dgl, dgx, dpv_d, dpv_c);
    return launch_status();
}
extern "C" int b200_fused_pool(const float* sum_d, const float* sum_c, int B, int C, int npix, const float* alpha,
                               const float* lowres, const float* up, int T, float* out, void* stream) {
    if (sum_d == nullptr || sum_c == nullptr || alpha == nullptr || out == nullptr || B <= 0) return -1;
    fused_pool_kernel<<<B, 128, 0, TE_STREAM>>>(sum_d, sum_c, 1.0f / npix, alpha, lowres, up, T, C, out);
    return launch_status();
}
extern "C" int b200_fusion_mix_bwd(const void* dfused, const void* p_dwi, const void* p_dce, const float* alpha, int B, int H,
                                   int W, int C, int Hp, int Wp, float* dalpha, float* dlowres, const float* dtok_d,
                                   const float* dtok_c, const float* dpv_d, const float* dpv_c, void* dp_dwi, void* dp_dce,
                                   int phase, void* stream) {
    if (dfused == nullptr || B <= 0 || C % 8 != 0) return -1;
    if (phase == 0) {  // reductions: dalpha, dlowres (caller zeroes both)
        if (p_dwi == nullptr || p_dce == nullptr || dalpha == nullptr) return -2;
        const size_t smem = static_cast<size_t>(Hp) * Wp * C * sizeof(float);
        if (smem > 48 * 1024) return -3;
        int slabs = (148 * 2 + B - 1) / B;
        if (slabs < 1) slabs = 1;
        if (slabs > 16) slabs = 16;
        fusion_mix_bwd_reduce_kernel<<<dim3(slabs, B), kTeThreads, smem, TE_STREAM>>>(
            static_cast<const __nv_bfloat16*>(dfused), static_cast<const __nv_bfloat16*>(p_dwi),
            static_cast<const __nv_bfloat16*>(p_dce), H, W, C, Hp, Wp, dalpha, dlowres);
    } else {
        if (alpha == nullptr || dp_dwi == nullptr || dp_dce == nullptr) return -2;
        if (dtok_d != nullptr && (H % Hp != 0 || W % Wp != 0)) return -4;
        fusion_mix_bwd_apply_kernel<<<blocks_for(static_cast<long long>(B) * H * W * (C / 8)), kTeThreads, 0, TE_STREAM>>>(
            static_cast<const __nv_bfloat16*>(dfused), alpha, dtok_d, dtok_c, dpv_d, dpv_c, B, H, W, C, Hp, Wp,
            static_cast<__nv_bfloat16*>(dp_dwi), static_cast<__nv_bfloat16*>(dp_dce));
    }
    return launch_status();
}
extern "C" int b200_mimic_pairs(const void* map, int B, int npix, int C, float scale, float* loss, void* dmap, void* stream) {
    if (map == nullptr || loss == nullptr || B < 4 || C <= 0) return -1;
    if (dmap != nullptr) cudaMemsetAsync(dmap, 0, static_cast<size_t>(B) * npix * C * 2, TE_STREAM);
    mimic_pairs_kernel<<<2, 128, 0, TE_STREAM>>>(static_cast<const __nv_bfloat16*>(map), npix, C, scale, loss,
                                                static_cast<__nv_bfloat16*>(dmap));
    return launch_status();
}

extern "C" int b200_up2_bwd(const void* dout, int B, int H, int W, int C, void* din, void* stream) {
    if (dout == nullptr || din == nullptr || C % 8 != 0) return -1;
    up2_bwd_kernel<<<blocks_for(static_cast<long long>(B) * H * W * (C / 8)), kTeThreads, 0, TE_STREAM>>>(
        static_cast<const __nv_bfloat16*>(dout), B, H, W, C, static_cast<__nv_bfloat16*>(din));
    return launch_status();
}

extern "C" int b200_row_bcast(const float* v, int v_stride, float scale, int B, int n, float* out, void* stream) {
    if (v == nullptr || out == nullptr || B <= 0 || n <= 0) return -1;
    row_bcast_kernel<<<B, 256, 0, TE_STREAM>>>(v, v_stride, scale, n, out);
    return launch_status();
}

extern "C" int b200_vec_axpby(const float* a, float alpha, float beta, long long n, float* y, void* stream) {
    if (a == nullptr || y == nullptr || n <= 0) return -1;
    vec_axpby_kernel<<<blocks_for(n), 256, 0, TE_STREAM>>>(a, alpha, beta, n, y);
    return launch_status();
}
