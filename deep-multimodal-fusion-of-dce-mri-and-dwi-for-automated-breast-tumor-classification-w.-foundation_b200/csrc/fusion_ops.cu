// Late-fusion head (code/model_module.py:919-1000, FusionModel.forward) - the per-case
// vector/token part and the elementwise mix.  The GEMM-shaped pieces (proj_in_*, mask
// head `pre`, recon head, projector) run through b200_conv_gemm_ex.
//
//   fusion_tokens : adaptive 4x4 average pooling of a projected map into tokens (:903-917)
//   fusion_core   : one CTA per case - gating softmax (:745-780, :952-956), multi-head
//                   cross-attention q=DWI, kv=DCE with head-averaged weights (:806, :816),
//                   residual FFN (:807-817), squeeze-excite gate (:977-978, SEBlock :25-43)
//                   and classifier (:895-899, :986) evaluated on the analytically pooled
//                   fused map: GAP(a0*p_dwi + a1*p_dce + up(lowres)) is linear in its parts
//   fusion_mix    : fused_refined = (a0*p_dwi + a1*p_dce + bilinear_up(lowres)) * gate (:958-978)
#include "b200_fusion.h"
#include "common.cuh"

namespace b200 {

// One CTA per (token, case): 16-byte loads (8 channels per thread), the bin's pixels split over the thread groups that
// do not fit the channel vectors, 4 loads in flight per thread, partial sums combined through shared memory.
constexpr int kTokThreads = 128;
__global__ void __launch_bounds__(kTokThreads)
fusion_tokens_kernel(const __nv_bfloat16* __restrict__ p, int H, int W, int C, int Hp, int Wp,
                     float* __restrict__ tokens) {
    __shared__ float part[kTokThreads][9];
    const int b = blockIdx.y;
    const int t = blockIdx.x;
    const int ti = t / Wp, tj = t % Wp;
    const int h0 = (ti * H) / Hp, h1 = ((ti + 1) * H + Hp - 1) / Hp;
    const int w0 = (tj * W) / Wp, w1 = ((tj + 1) * W + Wp - 1) / Wp;
    const int bw = w1 - w0, npx = (h1 - h0) * bw;
    const float inv = 1.0f / static_cast<float>(npx);
    const int nvec = C >> 3;
    float* dst = tokens + (static_cast<size_t>(b) * Hp * Wp + t) * C;
    for (int v0 = 0; v0 < nvec; v0 += kTokThreads) {  // one trip unless C > 1024
        const int nv = min(nvec - v0, kTokThreads);
        const int groups = kTokThreads / nv;           // pixel slices working on the same channel vectors
        const int vi = threadIdx.x % nv, grp = threadIdx.x / nv;
        float acc[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[k] = 0.f;
        if (grp < groups) {
#pragma unroll 4
            for (int q = grp; q < npx; q += groups) {
                const int h = h0 + q / bw, w = w0 + q % bw;
                float f[8];
                unpack_bf16x8(__ldg(reinterpret_cast<const uint4*>(p + ((static_cast<size_t>(b) * H + h) * W + w) * C) +
                                    v0 + vi), f);
#pragma unroll
                for (int k = 0; k < 8; ++k) acc[k] += f[k];
            }
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) part[threadIdx.x][k] = acc[k];
        __syncthreads();
        if (grp == 0) {
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                float s = 0.f;
                for (int g = 0; g < groups; ++g) s += part[g * nv + vi][k];
                dst[(v0 + vi) * 8 + k] = s * inv;
            }
        }
        __syncthreads();
    }
}

// Equal, non-overlapping bins (H % Hp == 0, W % Wp == 0): one CTA per (token row, case) streams the bin rows' contiguous
// H/Hp * W * C region; a thread owns (token column, 8 channels), so no cross-thread reduction is needed.
__global__ void __launch_bounds__(256)
fusion_tokens_rows_kernel(const __nv_bfloat16* __restrict__ p, int H, int W, int C, int Hp, int Wp,
                          float* __restrict__ tokens) {
    const int b = blockIdx.y, ti = blockIdx.x;
    const int nvec = C >> 3, bh = H / Hp, bw = W / Wp;
    const int vi = threadIdx.x % nvec, tj = threadIdx.x / nvec;
    const uint4* base = reinterpret_cast<const uint4*>(p + ((static_cast<size_t>(b) * H + ti * bh) * W + tj * bw) * C) + vi;
    float acc[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k] = 0.f;
    for (int h = 0; h < bh; ++h) {
        const uint4* row = base + static_cast<size_t>(h) * W * nvec;
        for (int w0 = 0; w0 < bw; w0 += 8) {  // 8 independent 16-byte loads issued before the first use
            uint4 r[8];
#pragma unroll
            for (int u = 0; u < 8; ++u)
                if (w0 + u < bw) r[u] = __ldg(row + static_cast<size_t>(w0 + u) * nvec);
#pragma unroll
            for (int u = 0; u < 8; ++u)
                if (w0 + u < bw) {
                    float f[8];
                    unpack_bf16x8(r[u], f);
#pragma unroll
                    for (int k = 0; k < 8; ++k) acc[k] += f[k];
                }
        }
    }
    const float inv = 1.0f / static_cast<float>(bh * bw);
    float4* dst = reinterpret_cast<float4*>(tokens + (static_cast<size_t>(b) * Hp * Wp + ti * Wp + tj) * C + vi * 8);
    dst[0] = make_float4(acc[0] * inv, acc[1] * inv, acc[2] * inv, acc[3] * inv);
    dst[1] = make_float4(acc[4] * inv, acc[5] * inv, acc[6] * inv, acc[7] * inv);
}

// Y[t][o] = act(sum_i X[t][i] * Wt[i][o] + bias[o]) for T <= 16 tokens held in shared memory.
__device__ __forceinline__ void linear_tokens(const float* X, int ldx, const float* __restrict__ Wt, int ldw,
                                              const float* __restrict__ bias, float* Y, int ldy, int T, int Cin,
                                              int Cout, int act) {
    const int TG = (T + 1) >> 1;  // tokens per thread group (<= 8)
    for (int idx = threadIdx.x; idx < Cout * 2; idx += blockDim.x) {
        const int o = idx % Cout, t0 = (idx / Cout) * TG;
        float acc[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[k] = 0.f;
        if (((Cin | ldx) & 3) == 0 && (reinterpret_cast<uintptr_t>(X) & 15) == 0) {
            // four input channels per trip: the token rows are read as one broadcast LDS.128 instead of four LDS.32
            // (the loop was shared-memory-issue bound: one LDS per FMA), four weight loads in flight; the
            // accumulation order over i is unchanged
#pragma unroll 2
            for (int i = 0; i < Cin; i += 4) {
                const float* wp = Wt + static_cast<size_t>(i) * ldw + o;
                const float w0 = __ldg(wp), w1 = __ldg(wp + ldw), w2 = __ldg(wp + 2 * ldw), w3 = __ldg(wp + 3 * ldw);
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    if (k < TG && t0 + k < T) {
                        const float4 xv = *reinterpret_cast<const float4*>(X + (t0 + k) * ldx + i);
                        acc[k] = fmaf(w0, xv.x, acc[k]);
                        acc[k] = fmaf(w1, xv.y, acc[k]);
                        acc[k] = fmaf(w2, xv.z, acc[k]);
                        acc[k] = fmaf(w3, xv.w, acc[k]);
                    }
            }
        } else {
#pragma unroll 8
            for (int i = 0; i < Cin; ++i) {
                const float w = __ldg(Wt + static_cast<size_t>(i) * ldw + o);
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    if (k < TG && t0 + k < T) acc[k] += w * X[(t0 + k) * ldx + i];
            }
        }
        const float bv = bias != nullptr ? bias[o] : 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k)
            if (k < TG && t0 + k < T) {
                float v = acc[k] + bv;
                if (act) v = gelu_exact(v);
                Y[(t0 + k) * ldy + o] = v;
            }
    }
}

__global__ void __launch_bounds__(256)
fusion_core_kernel(const b200_fusion_weights wts, const float* __restrict__ pvec_dwi_sum,
                   const float* __restrict__ pvec_dce_sum, float inv_npix, const float* __restrict__ mask_dwi,
                   const float* __restrict__ mask_dce, int npix_mask, const float* __restrict__ tok_dwi,
                   const float* __restrict__ tok_dce, float* __restrict__ gating_out, float* __restrict__ attn_out,
                   float* __restrict__ lowres_out, float* __restrict__ gate_out, float* __restrict__ logits_out) {
    extern __shared__ float sm[];
    const int C = wts.C, T = wts.T, NH = wts.heads, DH = C / NH, Cm = wts.se_mid, K = wts.num_classes;
    float* bufA = sm;
    float* bufB = bufA + T * C;
    float* bufC = bufB + T * C;
    float* bufD = bufC + T * C;
    float* bufE = bufD + T * C;
    float* S = bufE + T * C;           // [NH][T][T]
    float* s_pd = S + NH * T * T;      // [C] pooled p_dwi
    float* s_pc = s_pd + C;            // [C] pooled p_dce
    float* s_gf = s_pc + C;            // [C] pooled fused
    float* s_h = s_gf + C;             // [Cm]
    float* s_misc = s_h + Cm;          // [8]
    __shared__ double scratch[33];
    const int b = blockIdx.x;
    const int tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;

    for (int c = tid; c < C; c += blockDim.x) {
        s_pd[c] = pvec_dwi_sum[static_cast<size_t>(b) * C + c] * inv_npix;
        s_pc[c] = pvec_dce_sum[static_cast<size_t>(b) * C + c] * inv_npix;
    }
    // ---- gating ----
    const bool use_mask = wts.use_mask_attention && mask_dwi != nullptr && mask_dce != nullptr;
    double cd = 0.0, cc = 0.0;
    if (use_mask) {
        for (int p = tid; p < npix_mask; p += blockDim.x) {
            cd += mask_dwi[static_cast<size_t>(b) * npix_mask + p];
            cc += mask_dce[static_cast<size_t>(b) * npix_mask + p];
        }
        cd = block_sum<double>(cd, scratch) / npix_mask;
        cc = block_sum<double>(cc, scratch) / npix_mask;
    }
    __syncthreads();
    {
        const int in_dim = 2 * C + (wts.use_mask_attention ? 2 : 0);
        // The reference builds fc for 2C+2 inputs when use_mask_attention but feeds only 2C
        // values when a mask is missing (model_module.py:763-777) - that raises in torch, so
        // both masks are required by the host wrapper whenever use_mask_attention is set.
        float part[2] = {0.f, 0.f};
        for (int i = tid; i < 2 * C; i += blockDim.x) {
            const float xv = i < C ? s_pd[i] : s_pc[i - C];
            part[0] += wts.gate_w[i] * xv;
            part[1] += wts.gate_w[in_dim + i] * xv;
        }
        const double g0 = block_sum<double>(part[0], scratch);
        const double g1 = block_sum<double>(part[1], scratch);
        if (tid == 0) {
            float l0 = static_cast<float>(g0) + wts.gate_b[0], l1 = static_cast<float>(g1) + wts.gate_b[1];
            if (use_mask) {
                l0 += wts.gate_w[2 * C] * static_cast<float>(cd) + wts.gate_w[2 * C + 1] * static_cast<float>(cc);
                l1 += wts.gate_w[in_dim + 2 * C] * static_cast<float>(cd) +
                      wts.gate_w[in_dim + 2 * C + 1] * static_cast<float>(cc);
            }
            const float mx = fmaxf(l0, l1);
            const float e0 = expf(l0 - mx), e1 = expf(l1 - mx);
            s_misc[0] = e0 / (e0 + e1);
            s_misc[1] = e1 / (e0 + e1);
            gating_out[b * 2 + 0] = s_misc[0];
            gating_out[b * 2 + 1] = s_misc[1];
        }
    }
    __syncthreads();
    const float a0 = s_misc[0], a1 = s_misc[1];

    // ---- cross attention + FFN ----
    if (wts.use_cross_attention) {
        for (int i = tid; i < T * C; i += blockDim.x) {
            bufA[i] = tok_dwi[static_cast<size_t>(b) * T * C + i];
            bufB[i] = tok_dce[static_cast<size_t>(b) * T * C + i];
        }
        __syncthreads();
        linear_tokens(bufA, C, wts.in_proj_wt, 3 * C, wts.in_proj_b, bufC, C, T, C, C, 0);                  // Q
        linear_tokens(bufB, C, wts.in_proj_wt + C, 3 * C, wts.in_proj_b + C, bufD, C, T, C, C, 0);          // K
        linear_tokens(bufB, C, wts.in_proj_wt + 2 * C, 3 * C, wts.in_proj_b + 2 * C, bufE, C, T, C, C, 0);  // V
        __syncthreads();
        const float qscale = rsqrtf(static_cast<float>(DH));
        for (int idx = tid; idx < NH * T * T; idx += blockDim.x) {
            const int h = idx / (T * T), tq = (idx / T) % T, tk = idx % T;
            float acc = 0.f;
            for (int d = 0; d < DH; ++d) acc += bufC[tq * C + h * DH + d] * bufD[tk * C + h * DH + d];
            S[idx] = acc * qscale;
        }
        __syncthreads();
        for (int r = tid; r < NH * T; r += blockDim.x) {
            float* row = S + r * T;
            float mx = row[0];
            for (int k = 1; k < T; ++k) mx = fmaxf(mx, row[k]);
            float sum = 0.f;
            for (int k = 0; k < T; ++k) {
                row[k] = expf(row[k] - mx);
                sum += row[k];
            }
            const float inv = 1.0f / sum;
            for (int k = 0; k < T; ++k) row[k] *= inv;
        }
        __syncthreads();
        for (int idx = tid; idx < T * T; idx += blockDim.x) {
            float acc = 0.f;
            for (int h = 0; h < NH; ++h) acc += S[h * T * T + idx];
            attn_out[static_cast<size_t>(b) * T * T + idx] = acc / NH;
        }
        for (int idx = tid; idx < T * C; idx += blockDim.x) {  // ctx -> bufA
            const int tq = idx / C, col = idx % C, h = col / DH;
            float acc = 0.f;
            for (int tk = 0; tk < T; ++tk) acc += S[(h * T + tq) * T + tk] * bufE[tk * C + col];
            bufA[idx] = acc;
        }
        __syncthreads();
        linear_tokens(bufA, C, wts.out_proj_wt, C, wts.out_proj_b, bufB, C, T, C, C, 0);  // attn_out -> bufB
        __syncthreads();
        for (int t = warp; t < T; t += nwarps) {  // LayerNorm -> bufC
            float s1 = 0.f;
            for (int c = lane; c < C; c += 32) s1 += bufB[t * C + c];
            const float mean = warp_sum(s1) / C;
            float s2 = 0.f;
            for (int c = lane; c < C; c += 32) {
                const float d = bufB[t * C + c] - mean;
                s2 += d * d;
            }
            const float rstd = rsqrtf(warp_sum(s2) / C + wts.ln_eps);
            for (int c = lane; c < C; c += 32)
                bufC[t * C + c] = (bufB[t * C + c] - mean) * rstd * wts.ln_w[c] + wts.ln_b[c];
        }
        __syncthreads();
        linear_tokens(bufC, C, wts.ffn1_wt, C, wts.ffn1_b, bufD, C, T, C, C, 1);
        __syncthreads();
        linear_tokens(bufD, C, wts.ffn2_wt, C, wts.ffn2_b, bufE, C, T, C, C, 0);
        __syncthreads();
        for (int i = tid; i < T * C; i += blockDim.x) {
            const float v = bufB[i] + bufE[i];
            bufE[i] = v;
            lowres_out[static_cast<size_t>(b) * T * C + i] = v;
        }
        __syncthreads();
    }
    // ---- pooled fused map, SE gate, classifier ----
    for (int c = tid; c < C; c += blockDim.x) {
        float g = a0 * s_pd[c] + a1 * s_pc[c];
        if (wts.use_cross_attention)
            for (int t = 0; t < T; ++t) g += wts.up_coef[t] * bufE[t * C + c];
        s_gf[c] = g;
    }
    __syncthreads();
    if (wts.use_se) {
        for (int m = tid; m < Cm; m += blockDim.x) {
            float a = wts.se_b1[m];
            for (int c = 0; c < C; ++c) a += wts.se_w1t[c * Cm + m] * s_gf[c];
            s_h[m] = gelu_exact(a);
        }
        __syncthreads();
        for (int c = tid; c < C; c += blockDim.x) {
            float a = wts.se_b2[c];
            for (int m = 0; m < Cm; ++m) a += wts.se_w2t[m * C + c] * s_h[m];
            const float g = sigmoidf_(a);
            gate_out[static_cast<size_t>(b) * C + c] = g;
            s_gf[c] *= g;
        }
    } else {
        for (int c = tid; c < C; c += blockDim.x) gate_out[static_cast<size_t>(b) * C + c] = 1.f;
    }
    __syncthreads();
    for (int k = warp; k < K; k += nwarps) {
        float a = 0.f;
        for (int c = lane; c < C; c += 32) a += wts.cls_w[k * C + c] * s_gf[c];
        a = warp_sum(a);
        if (lane == 0) logits_out[static_cast<size_t>(b) * K + k] = a + wts.cls_b[k];
    }
}

// grid (chunks, B), 32-bit index arithmetic; a thread handles kMixUnroll vectors (8 channels of one pixel each) and
// issues all its map loads before the first use.
constexpr int kMixUnroll = 2;
__global__ void __launch_bounds__(256)
fusion_mix_kernel(const __nv_bfloat16* __restrict__ p_dwi, const __nv_bfloat16* __restrict__ p_dce,
                  const float* __restrict__ gating, const float* __restrict__ lowres, const float* __restrict__ gate,
                  int H, int W, int C, int Hp, int Wp, __nv_bfloat16* __restrict__ out) {
    const int cv = C >> 3, nvc = H * W * cv, b = blockIdx.y;
    const float sh = static_cast<float>(Hp) / H, sw = static_cast<float>(Wp) / W;
    const size_t case_off = static_cast<size_t>(b) * nvc;
    const uint4* xd = reinterpret_cast<const uint4*>(p_dwi) + case_off;
    const uint4* xc = reinterpret_cast<const uint4*>(p_dce) + case_off;
    uint4* ys = reinterpret_cast<uint4*>(out) + case_off;
    const float a0 = gating[b * 2], a1 = gating[b * 2 + 1];
    const float* low = lowres != nullptr ? lowres + static_cast<size_t>(b) * Hp * Wp * C : nullptr;
    const int i0 = blockIdx.x * (kMixUnroll * blockDim.x) + threadIdx.x;
    uint4 rd[kMixUnroll], rc[kMixUnroll];
#pragma unroll
    for (int u = 0; u < kMixUnroll; ++u) {
        const int i = i0 + u * blockDim.x;
        if (i < nvc) {
            rd[u] = __ldcs(xd + i);
            rc[u] = __ldcs(xc + i);
        }
    }
#pragma unroll
    for (int u = 0; u < kMixUnroll; ++u) {
        const int i = i0 + u * blockDim.x;
        if (i >= nvc) continue;
        const int c0 = (i % cv) << 3, px = i / cv, w = px % W, h = px / W;
        float fd[8], fc[8], r[8];
        unpack_bf16x8(rd[u], fd);
        unpack_bf16x8(rc[u], fc);
#pragma unroll
        for (int k = 0; k < 8; ++k) r[k] = a0 * fd[k] + a1 * fc[k];
        if (low != nullptr) {
            // F.interpolate(mode='bilinear', align_corners=False) source coordinates
            const float sy = fmaxf((h + 0.5f) * sh - 0.5f, 0.f), sx = fmaxf((w + 0.5f) * sw - 0.5f, 0.f);
            const int y0 = static_cast<int>(sy), x0 = static_cast<int>(sx);
            const int y1 = min(y0 + 1, Hp - 1), x1 = min(x0 + 1, Wp - 1);
            const float ly = sy - y0, lx = sx - x0;
            const float* base = low + c0;
            const float w00 = (1.f - ly) * (1.f - lx), w01 = (1.f - ly) * lx, w10 = ly * (1.f - lx), w11 = ly * lx;
            const float* q00 = base + (y0 * Wp + x0) * C;
            const float* q01 = base + (y0 * Wp + x1) * C;
            const float* q10 = base + (y1 * Wp + x0) * C;
            const float* q11 = base + (y1 * Wp + x1) * C;
            // 16-byte loads of the four taps (c0 is a multiple of 8 floats); same arithmetic order as before
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const float4 t00 = __ldg(reinterpret_cast<const float4*>(q00) + half);
                const float4 t01 = __ldg(reinterpret_cast<const float4*>(q01) + half);
                const float4 t10 = __ldg(reinterpret_cast<const float4*>(q10) + half);
                const float4 t11 = __ldg(reinterpret_cast<const float4*>(q11) + half);
                r[4 * half + 0] += w00 * t00.x + w01 * t01.x + w10 * t10.x + w11 * t11.x;
                r[4 * half + 1] += w00 * t00.y + w01 * t01.y + w10 * t10.y + w11 * t11.y;
                r[4 * half + 2] += w00 * t00.z + w01 * t01.z + w10 * t10.z + w11 * t11.z;
                r[4 * half + 3] += w00 * t00.w + w01 * t01.w + w10 * t10.w + w11 * t11.w;
            }
        }
        if (gate != nullptr) {
            const float4 g0 = __ldg(reinterpret_cast<const float4*>(gate + static_cast<size_t>(b) * C + c0));
            const float4 g1 = __ldg(reinterpret_cast<const float4*>(gate + static_cast<size_t>(b) * C + c0) + 1);
            r[0] *= g0.x; r[1] *= g0.y; r[2] *= g0.z; r[3] *= g0.w;
            r[4] *= g1.x; r[5] *= g1.y; r[6] *= g1.z; r[7] *= g1.w;
        }
        ys[i] = pack_bf16x8(r);
    }
}

}  // namespace b200

using namespace b200;

extern "C" int b200_fusion_tokens(const void* p, int B, int H, int W, int C, int Hp, int Wp, float* tokens,
                                  void* stream) {
    if (B < 0 || C <= 0 || C % 8 != 0 || Hp <= 0 || Wp <= 0 || H < Hp || W < Wp) return -1;
    if (B == 0) return 0;
    if (p == nullptr || tokens == nullptr) return -2;
    const int row_threads = (C / 8) * Wp;
    if (H % Hp == 0 && W % Wp == 0 && row_threads >= 32 && row_threads <= 256) {
        fusion_tokens_rows_kernel<<<dim3(Hp, B), row_threads, 0, static_cast<cudaStream_t>(stream)>>>(
            static_cast<const __nv_bfloat16*>(p), H, W, C, Hp, Wp, tokens);
        return launch_status();
    }
    dim3 grid(Hp * Wp, B);
    fusion_tokens_kernel<<<grid, kTokThreads, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __nv_bfloat16*>(p), H, W, C, Hp, Wp, tokens);
    return launch_status();
}

extern "C" int b200_fusion_core(const b200_fusion_weights* wts, int B, const float* pvec_dwi_sum,
                                const float* pvec_dce_sum, int npix, const float* mask_dwi, const float* mask_dce,
                                int npix_mask, const float* tok_dwi, const float* tok_dce, float* gating_out,
                                float* attn_out, float* lowres_out, float* gate_out, float* logits_out, void* stream) {
    if (wts == nullptr || B < 0) return -1;
    if (B == 0) return 0;
    const int C = wts->C, T = wts->T;
    if (C <= 0 || T <= 0 || T > 16 || wts->heads <= 0 || C % wts->heads != 0) return -2;
    if (pvec_dwi_sum == nullptr || pvec_dce_sum == nullptr || gating_out == nullptr || gate_out == nullptr ||
        logits_out == nullptr)
        return -3;
    if (wts->use_cross_attention && (tok_dwi == nullptr || tok_dce == nullptr || attn_out == nullptr ||
                                     lowres_out == nullptr))
        return -4;
    if (wts->use_mask_attention && (mask_dwi == nullptr || mask_dce == nullptr)) return -5;
    const size_t smem =
        (static_cast<size_t>(5) * T * C + static_cast<size_t>(wts->heads) * T * T + 3 * C + wts->se_mid + 8) *
        sizeof(float);
    if (smem > 200 * 1024) return -6;
    static size_t configured = 0;
    if (smem > 48 * 1024 && smem > configured) {
        cudaError_t e = cudaFuncSetAttribute(fusion_core_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             static_cast<int>(smem));
        if (e != cudaSuccess) return static_cast<int>(e);
        configured = smem;
    }
    fusion_core_kernel<<<B, 256, smem, static_cast<cudaStream_t>(stream)>>>(
        *wts, pvec_dwi_sum, pvec_dce_sum, 1.0f / npix, mask_dwi, mask_dce, npix_mask, tok_dwi, tok_dce, gating_out,
        attn_out, lowres_out, gate_out, logits_out);
    return launch_status();
}

extern "C" int b200_fusion_mix(const void* p_dwi, const void* p_dce, const float* gating, const float* lowres,
                               const float* gate, int B, int H, int W, int C, int Hp, int Wp, void* out, void* stream) {
    if (B < 0 || C % 8 != 0 || H <= 0 || W <= 0) return -1;
    if (B == 0) return 0;
    if (p_dwi == nullptr || p_dce == nullptr || gating == nullptr || out == nullptr) return -2;
    const long long nvc = static_cast<long long>(H) * W * (C / 8);
    if (nvc > 0x7fffffff / 2 || B > 65535) return -3;
    const unsigned chunks = static_cast<unsigned>((nvc + kMixUnroll * 256 - 1) / (kMixUnroll * 256));
    fusion_mix_kernel<<<dim3(chunks, B), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __nv_bfloat16*>(p_dwi), static_cast<const __nv_bfloat16*>(p_dce), gating, lowres, gate, H, W,
        C, Hp, Wp, static_cast<__nv_bfloat16*>(out));
    return launch_status();
}
