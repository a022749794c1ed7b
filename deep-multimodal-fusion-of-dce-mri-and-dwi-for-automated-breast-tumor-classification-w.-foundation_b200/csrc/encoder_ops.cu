// SIMT kernels of the DWI / DCE encoder that are not GEMM-shaped (K < 64, N == 1, or
// per-case vectors): modality-attention + first strided 1x1 convolutions ("stem"),
// squeeze-excite gates, channel rescaling, N=1 convolutions, the mask head tail with the
// mask-guided spatial attention, the 1->C projector lift and the classification head.
// Reference: code/model_module.py (line ranges cited per kernel).
#include "b200_fusion.h"
#include "common.cuh"

namespace b200 {

// ---------------------------------------------------------------- stem -----
// model_module.py:649-650 (modality SE, SEBlock :25-43) followed by the two stride-s 1x1
// convolutions of block1 that read the raw input: skip (:276-280) and the first
// bottleneck conv + BN + GELU (:260-262).  Input is fp32 NCHW (what the normalisers
// emit), outputs are NHWC bf16.  K = C <= 32 is far too thin for the tensor cores and the
// layer is write-bound, so this is fp32 SIMT: one CTA = one case x 64 consecutive output
// pixels; every thread owns one pixel and a quarter of the output channels, weights are
// broadcast from shared memory, and the [64 px][n_out] bf16 tile is staged in shared memory
// so that both maps leave the SM as fully coalesced 16-byte stores.
constexpr int kStemPix = 64;
constexpr int kStemMaxC = 32;
constexpr int kStemThreads = 256;
constexpr int kStemCB = 16;  // output channels per register block

template <int CMAX, bool FULL>  // FULL: C == CMAX, the input-channel loops carry no `c < C` tests
__global__ void __launch_bounds__(kStemThreads, CMAX <= 16 ? 4 : 2)  // 4 CTAs / SM (<= 64 registers) for C <= 16
stem_kernel(const float* __restrict__ x, int C, int H, int W, int stride,
            const float* __restrict__ plane_mean,  // [B, C]
            const float* __restrict__ se_w1, const float* __restrict__ se_b1,  // [Cm, C], [Cm]
            const float* __restrict__ se_w2, const float* __restrict__ se_b2,  // [C, Cm], [C]
            int Cm,
            const float* __restrict__ wcat,   // [n_out, C], n_out = n_skip + n_mid
            const float* __restrict__ scale,  // [n_out]
            const float* __restrict__ bias, int n_skip, int n_mid, __nv_bfloat16* __restrict__ skip_out,
            __nv_bfloat16* __restrict__ mid_out, float* __restrict__ mod_attn, unsigned int drop_thresh,
            float drop_scale, unsigned int seed_lo, unsigned int seed_hi,
            // normalisation fused into the operand load (x is then the RAW input):
            const float* __restrict__ in_affine,  // [B*C][4] {mean, 1/std, scale, offset} from b200_dwi_normalize_ex
            float z_lo, float z_hi,
            const double* __restrict__ in_table,  // [B*C][56] composed Nyul table from b200_nyul_transform_ex2
            int L) {
    extern __shared__ float s_dyn[];
    __shared__ float s_gate[kStemMaxC];
    __shared__ float s_hidden[kStemMaxC];
    const int n_out = n_skip + n_mid;       // multiple of 4 * kStemCB (host-checked)
    const int row_words = n_out / 2 + 1;    // staged row: n_out bf16 + one pad word -> odd stride, no bank conflicts
    // weights as one [w_rows][16] slab per 16-channel register block: inside a block every (input channel, vector)
    // offset is a compile-time constant, so the main loop's LDS.128 carry immediates instead of per-channel address
    // arithmetic (which, with the `c < C` tests and their uniform branches, was ~15 % of the kernel's instructions;
    // DWI, C = 16 = CMAX, runs the FULL instantiation without the tests: 0.404 -> 0.338 ms per 1 024 cases).
    const int w_rows = C;
    float* s_w = s_dyn;                     // [n_out / 16][w_rows][16]
    float* s_sc = s_w + w_rows * n_out;     // [n_out]
    float* s_bi = s_sc + n_out;             // [n_out]
    uint32_t* s_out = reinterpret_cast<uint32_t*>(s_bi + n_out);  // [kStemPix][row_words]
    // per-plane normaliser parameters of this case (8-byte aligned: after an even number of words)
    constexpr int kTabD = 3 * 16 + 8;  // doubles per plane: orig[16] | slope[16] | value[16] | up[16] as floats
    double* s_tab = reinterpret_cast<double*>(s_out + ((kStemPix * row_words + 1) & ~1));
    __shared__ float4 s_aff[kStemMaxC];
    __shared__ float s_in[kStemMaxC * kStemPix];
    const int b = blockIdx.y;
    const int Ho = H / stride, Wo = W / stride;
    const int npix = Ho * Wo;
    const int tid = threadIdx.x;

    if (se_w1 != nullptr) {
        if (tid < Cm) {
            float a = se_b1[tid];
            for (int c = 0; c < C; ++c) a += se_w1[tid * C + c] * plane_mean[b * C + c];
            s_hidden[tid] = gelu_exact(a);
        }
        __syncthreads();
        if (tid < C) {
            float a = se_b2[tid];
            for (int m = 0; m < Cm; ++m) a += se_w2[tid * Cm + m] * s_hidden[m];
            const float g = sigmoidf_(a);
            s_gate[tid] = g;
            if (blockIdx.x == 0 && mod_attn != nullptr) mod_attn[b * C + tid] = g;
        }
    } else if (tid < C) {
        s_gate[tid] = 1.f;
    }
    for (int i = tid; i < w_rows * n_out; i += kStemThreads) {
        const int c = i / n_out, n = i - c * n_out;
        s_w[(n / kStemCB) * (w_rows * kStemCB) + c * kStemCB + (n % kStemCB)] = c < C ? wcat[n * C + c] : 0.f;
    }
    for (int i = tid; i < n_out; i += kStemThreads) {
        s_sc[i] = scale[i];
        s_bi[i] = bias[i];
    }
    if (in_affine != nullptr && tid < C) s_aff[tid] = reinterpret_cast<const float4*>(in_affine)[b * C + tid];
    if (in_table != nullptr)
        for (int i = tid; i < C * kTabD; i += kStemThreads) s_tab[i] = in_table[static_cast<size_t>(b) * C * kTabD + i];
    __syncthreads();

    const int pp = tid % kStemPix;
    const int quarter = tid / kStemPix;  // 0..3
    // power-of-two map widths / vector counts (every shipped configuration): shifts instead of integer divisions
    const int wo_shift = (Wo & (Wo - 1)) == 0 ? 31 - __clz(Wo) : -1;
    // A CTA walks several 64-pixel tiles of its case: the weight staging / transposition and the SE gate above are
    // paid once per CTA, not once per tile (they cost about as much as one tile's arithmetic).
    const int n_tiles = (npix + kStemPix - 1) / kStemPix;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int pix0 = tile * kStemPix;
    const int pix = pix0 + pp;
    // the tile's inputs - normalised (when fused) and gated - are staged in shared memory ONCE per (pixel, channel);
    // the four threads that share a pixel then read them from there (they used to load and transform 4 x each)
    __syncthreads();  // the previous tile's readers are done with s_in
    for (int i = tid; i < C * kStemPix; i += kStemThreads) {
        const int c = i / kStemPix, q = i - c * kStemPix;
        const int px = pix0 + q;
        float v = 0.f;
        if (px < npix) {
            const int ho = wo_shift >= 0 ? px >> wo_shift : px / Wo, wo = px - ho * Wo;
            v = __ldg(x + ((static_cast<size_t>(b) * C + c) * H + static_cast<size_t>(ho) * stride) * W + wo * stride);
            if (in_affine != nullptr) {  // DWINormalize, the instructions of dwi_normalize_reg_kernel's apply step
                const float4 st = s_aff[c];
                v = fmaf(fminf(fmaxf((v - st.x) * st.y, z_lo), z_hi), st.z, st.w);
            } else if (in_table != nullptr) {  // Nyul: the composed piece-wise linear table (nyul_apply, fast path)
                const double* tb = s_tab + c * kTabD;
                const float* up = reinterpret_cast<const float*>(tb + 48);
                int j = 0;
                for (int t = 1; t < L; ++t) j += (v >= up[t]) ? 1 : 0;
                const double d = static_cast<double>(v) - tb[j];
                const float o = static_cast<float>(fma(tb[16 + j], d > 0.0 ? d : 0.0, tb[32 + j]));
                v = v != v ? v : o;
            }
            v *= s_gate[c];
        }
        s_in[c * kStemPix + q] = v;
    }
    __syncthreads();
    float2 xv[CMAX];  // the pixel's gated input, duplicated into both halves of a packed operand
#pragma unroll
    for (int c = 0; c < CMAX; ++c) {
        const float v = (FULL || c < C) ? s_in[c * kStemPix + pp] : 0.f;
        xv[c] = make_float2(v, v);
    }
    const int per_quarter = n_out / 4;
    for (int n0 = quarter * per_quarter; n0 < (quarter + 1) * per_quarter; n0 += kStemCB) {
        float2 acc[kStemCB / 2];
#pragma unroll
        for (int j = 0; j < kStemCB / 2; ++j) acc[j] = make_float2(0.f, 0.f);
#pragma unroll
        const float4* wb = reinterpret_cast<const float4*>(s_w + (n0 / kStemCB) * (w_rows * kStemCB));
#pragma unroll
        for (int c = 0; c < CMAX; ++c) {
            if (FULL || c < C) {
#pragma unroll
                for (int j = 0; j < kStemCB / 4; ++j) {
                    const float4 wv = wb[c * (kStemCB / 4) + j];
                    acc[2 * j + 0] = __ffma2_rn(xv[c], make_float2(wv.x, wv.y), acc[2 * j + 0]);
                    acc[2 * j + 1] = __ffma2_rn(xv[c], make_float2(wv.z, wv.w), acc[2 * j + 1]);
                }
            }
        }
        const bool is_mid = n0 >= n_skip;  // a 16-channel block never straddles the two maps (host-checked)
        // MC-dropout on the bottleneck's first activation (model_module.py:260): element index in the mid map
        const unsigned long long e0 = (static_cast<unsigned long long>(b) * npix + pix) * n_mid + (n0 - n_skip);
#pragma unroll
        for (int j = 0; j < kStemCB / 2; ++j) {
            const float2 sc = *reinterpret_cast<const float2*>(s_sc + n0 + 2 * j);
            const float2 bi = *reinterpret_cast<const float2*>(s_bi + n0 + 2 * j);
            float2 y = __ffma2_rn(acc[j], sc, bi);
            if (is_mid) y = gelu_fast2(y);
            if (is_mid && drop_thresh != 0u) {
                const uint4 rnd = philox4x32_7(e0 / 4 + (j >> 1), seed_lo, seed_hi);  // 4 channels per call
                const unsigned int r0 = (j & 1) ? rnd.z : rnd.x, r1 = (j & 1) ? rnd.w : rnd.y;
                y.x = r0 < drop_thresh ? 0.f : y.x * drop_scale;
                y.y = r1 < drop_thresh ? 0.f : y.y * drop_scale;
            }
            const __nv_bfloat162 h2 = __floats2bfloat162_rn(y.x, y.y);
            s_out[pp * row_words + n0 / 2 + j] = *reinterpret_cast<const uint32_t*>(&h2);
        }
    }
    __syncthreads();
    // copy out: the CTA's pixels are consecutive, so each map's slice is one contiguous block in HBM
    const int valid_pix = min(kStemPix, npix - pix0);
    {
        const int vec_per_pix = n_skip / 8;
        const int vsh = (vec_per_pix & (vec_per_pix - 1)) == 0 ? 31 - __clz(vec_per_pix) : -1;
        uint4* dst = reinterpret_cast<uint4*>(skip_out + (static_cast<size_t>(b) * npix + pix0) * n_skip);
        for (int i = tid; i < valid_pix * vec_per_pix; i += kStemThreads) {
            const int pq = vsh >= 0 ? i >> vsh : i / vec_per_pix, v = i - pq * vec_per_pix;
            const uint32_t* src = s_out + pq * row_words + v * 4;
            dst[i] = make_uint4(src[0], src[1], src[2], src[3]);
        }
    }
    {
        const int vec_per_pix = n_mid / 8;
        const int vsh = (vec_per_pix & (vec_per_pix - 1)) == 0 ? 31 - __clz(vec_per_pix) : -1;
        uint4* dst = reinterpret_cast<uint4*>(mid_out + (static_cast<size_t>(b) * npix + pix0) * n_mid);
        for (int i = tid; i < valid_pix * vec_per_pix; i += kStemThreads) {
            const int pq = vsh >= 0 ? i >> vsh : i / vec_per_pix, v = i - pq * vec_per_pix;
            const uint32_t* src = s_out + pq * row_words + n_skip / 2 + v * 4;
            dst[i] = make_uint4(src[0], src[1], src[2], src[3]);
        }
    }
    __syncthreads();  // s_out is rewritten by the next tile
    }  // tile loop
}

// ------------------------------------------------------------- SE gate -----
// SEBlock.fc on the pooled vector (model_module.py:34-40): gate = sigmoid(W2 gelu(W1 m + b1) + b2) with
// m = gap_sum / npix, as two small fp32 dense layers.  One CTA = 8 cases x 64 outputs; its 256 threads are
// 64 output columns x 4 quarters of every 128-long K slice, so a thread issues 32 independent weight loads
// per slice (the layer is L2-latency bound, not bandwidth bound) and reuses each for 8 cases; the four
// partial sums meet in shared memory.  Weights are passed transposed ([in, out]): consecutive threads read
// consecutive addresses.  ACT: 0 = GELU (hidden layer), 1 = sigmoid (gate).
constexpr int kSeCases = 8;

template <int ACT>
__global__ void __launch_bounds__(256)
se_dense_kernel(const float* __restrict__ in, float in_scale, int B, int K, int N, const float* __restrict__ wt,
                const float* __restrict__ bias, float* __restrict__ out) {
    __shared__ float s_in[kSeCases][128];
    __shared__ float s_part[4][kSeCases][64];
    const int tx = threadIdx.x & 63, kq = (threadIdx.x >> 6) * 32;
    const int n = blockIdx.x * 64 + tx;
    const int b0 = blockIdx.y * kSeCases;
    float acc[kSeCases];
#pragma unroll
    for (int c = 0; c < kSeCases; ++c) acc[c] = 0.f;
    for (int k0 = 0; k0 < K; k0 += 128) {
        __syncthreads();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int idx = threadIdx.x + i * 256;  // 8 cases x 128 k
            const int r = idx >> 7, kk = idx & 127;
            s_in[r][kk] = (b0 + r < B && k0 + kk < K) ? in[static_cast<size_t>(b0 + r) * K + k0 + kk] * in_scale : 0.f;
        }
        __syncthreads();
        if (n < N && k0 + kq < K) {
            float w[32];
#pragma unroll
            for (int kk = 0; kk < 32; ++kk)
                w[kk] = k0 + kq + kk < K ? __ldg(wt + static_cast<size_t>(k0 + kq + kk) * N + n) : 0.f;
#pragma unroll
            for (int kk = 0; kk < 32; ++kk) {
#pragma unroll
                for (int c = 0; c < kSeCases; ++c) acc[c] = fmaf(w[kk], s_in[c][kq + kk], acc[c]);
            }
        }
    }
#pragma unroll
    for (int c = 0; c < kSeCases; ++c) s_part[kq >> 5][c][tx] = acc[c];
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const int idx = threadIdx.x + i * 256;  // 8 cases x 64 columns
        const int c = idx >> 6, col = idx & 63;
        const int nn = blockIdx.x * 64 + col, bb = b0 + c;
        if (nn < N && bb < B) {
            const float v = s_part[0][c][col] + s_part[1][c][col] + s_part[2][c][col] + s_part[3][c][col] + bias[nn];
            out[static_cast<size_t>(bb) * N + nn] = ACT == 0 ? gelu_exact(v) : sigmoidf_(v);
        }
    }
}

// ------------------------------------------------- channel / pixel scale ---
// y[b,p,c] = x[b,p,c] * gate[b,c] * (1 + gamma * attn[b,p]); either factor optional.
// SE rescale (model_module.py:43) and mask-guided modulation (:96).
// grid (chunks, B): a CTA owns 4 * blockDim consecutive 8-channel vectors of one case; every thread issues its four
// 16-byte loads before the first use, and all index arithmetic is 32-bit.
constexpr int kScaleUnroll = 4;
__global__ void __launch_bounds__(256)
scale_map_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y, int C, int npix,
                 const float* __restrict__ gate, const float* __restrict__ attn, const float* __restrict__ gamma_ptr) {
    const int cv = C >> 3, nvc = npix * cv, b = blockIdx.y;
    const float gamma = gamma_ptr != nullptr ? *gamma_ptr : 0.f;
    const size_t case_off = static_cast<size_t>(b) * nvc;
    const uint4* xs = reinterpret_cast<const uint4*>(x) + case_off;
    uint4* ys = reinterpret_cast<uint4*>(y) + case_off;
    const float* gr = gate != nullptr ? gate + static_cast<size_t>(b) * C : nullptr;
    const float* ar = attn != nullptr ? attn + static_cast<size_t>(b) * npix : nullptr;
    const int i0 = blockIdx.x * (kScaleUnroll * blockDim.x) + threadIdx.x;
    uint4 r[kScaleUnroll];
#pragma unroll
    for (int u = 0; u < kScaleUnroll; ++u) {
        const int i = i0 + u * blockDim.x;
        if (i < nvc) r[u] = __ldcs(xs + i);
    }
    // C / 8 a power of two that divides the block size (every CNN width: 128 / 256 / 512 channels): the thread's four
    // vectors share one channel offset - one pair of gate loads instead of four, shifts instead of divisions
    const bool pow2 = (cv & (cv - 1)) == 0 && (blockDim.x % cv) == 0;
    const int sh = 31 - __clz(cv);
    float4 gs0 = make_float4(1.f, 1.f, 1.f, 1.f), gs1 = gs0;
    if (pow2 && gr != nullptr) {
        const int c0 = (i0 & (cv - 1)) << 3;
        gs0 = __ldg(reinterpret_cast<const float4*>(gr + c0));
        gs1 = __ldg(reinterpret_cast<const float4*>(gr + c0 + 4));
    }
#pragma unroll
    for (int u = 0; u < kScaleUnroll; ++u) {
        const int i = i0 + u * blockDim.x;
        if (i >= nvc) continue;
        const int c0 = (pow2 ? (i & (cv - 1)) : (i % cv)) << 3, px = pow2 ? (i >> sh) : (i / cv);
        float f[8];
        unpack_bf16x8(r[u], f);
        const float m = ar != nullptr ? 1.f + gamma * __ldg(ar + px) : 1.f;
        if (gr != nullptr) {
            const float4 g0 = pow2 ? gs0 : __ldg(reinterpret_cast<const float4*>(gr + c0));
            const float4 g1 = pow2 ? gs1 : __ldg(reinterpret_cast<const float4*>(gr + c0 + 4));
            f[0] *= g0.x * m; f[1] *= g0.y * m; f[2] *= g0.z * m; f[3] *= g0.w * m;
            f[4] *= g1.x * m; f[5] *= g1.y * m; f[6] *= g1.z * m; f[7] *= g1.w * m;
        } else {
#pragma unroll
            for (int k = 0; k < 8; ++k) f[k] *= m;
        }
        ys[i] = pack_bf16x8(f);
    }
}

// ------------------------------------------------------- conv 3x3, N=1 -----
// ReconHead's last conv (model_module.py:117): C -> 1, 3x3, pad 1, with bias, fp32 output
// [B,H,W].  One warp per output pixel; lanes split the channels, taps are L1/L2 re-reads.
__global__ void conv3x3_c1_kernel(const __nv_bfloat16* __restrict__ x, int H, int W, int C,
                                  const float* __restrict__ w,  // [9, C]
                                  const float* __restrict__ bias, float* __restrict__ out, size_t total_pix) {
    const int lane = threadIdx.x & 31;
    const size_t warp_global = (blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x) >> 5;
    if (warp_global >= total_pix) return;
    const int wq = static_cast<int>(warp_global % W);
    const int hq = static_cast<int>((warp_global / W) % H);
    const size_t b = warp_global / (static_cast<size_t>(W) * H);
    float acc = 0.f;
    for (int tap = 0; tap < 9; ++tap) {
        const int hh = hq + tap / 3 - 1, ww = wq + tap % 3 - 1;
        if (hh < 0 || hh >= H || ww < 0 || ww >= W) continue;
        const __nv_bfloat16* px = x + ((b * H + hh) * W + ww) * C;
        for (int c0 = lane * 8; c0 < C; c0 += 256) {
            float f[8];
            unpack_bf16x8(__ldg(reinterpret_cast<const uint4*>(px + c0)), f);
            const float4 w0 = *reinterpret_cast<const float4*>(w + tap * C + c0);
            const float4 w1 = *reinterpret_cast<const float4*>(w + tap * C + c0 + 4);
            acc += f[0] * w0.x + f[1] * w0.y + f[2] * w0.z + f[3] * w0.w + f[4] * w1.x + f[5] * w1.y + f[6] * w1.z +
                   f[7] * w1.w;
        }
    }
    acc = warp_sum(acc);
    if (lane == 0) out[warp_global] = acc + bias[0];
}

// ------------------------------------------------------ tap shift-sum ------
// Second half of a 3x3, C -> 1 convolution whose per-tap dot products d[p][k] = sum_c x[p,c] w[k,c]
// were produced by the preceding GEMM's epilogue (b200_conv_gemm_ex, dot_w):
// out[b,h,w] = bias + sum_k d[(b, h+ky-1, w+kx-1)][k] with zero padding.
__global__ void tapsum_kernel(const float* __restrict__ d, int H, int W, const float* __restrict__ bias,
                              float* __restrict__ out, size_t total_pix) {
    const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
    if (i >= total_pix) return;
    const int w = static_cast<int>(i % W);
    const int h = static_cast<int>((i / W) % H);
    float acc = bias[0];
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        const int hh = h + k / 3 - 1, ww = w + k % 3 - 1;
        if (hh >= 0 && hh < H && ww >= 0 && ww < W)
            acc += d[(i + static_cast<long long>(k / 3 - 1) * W + (k % 3 - 1)) * 9 + k];
    }
    out[i] = acc;
}

// ------------------------------------------------ 1-channel bilinear resize -
// F.interpolate(mode='bilinear', align_corners=False) of an fp32 1-channel map (MaskHeadResize's fallback
// path, model_module.py:205-211; it commutes with the 1x1 `out` convolution that follows it there, so it is
// applied to the 1-channel logits instead of the 64-channel map).
// block (64, 4): thread (tx, ty) produces outputs x = 4 tx .. 4 tx + 3 of row blockIdx.y * 4 + ty of plane blockIdx.z
// (grid.x strides over rows wider than 256); one 16-byte store per thread when the row allows it.
__global__ void __launch_bounds__(256)
resize_bilinear_c1_kernel(const float* __restrict__ in, int h, int w, float* __restrict__ out, int H, int W) {
    const int oy = blockIdx.y * 4 + threadIdx.y;
    const int ox0 = (blockIdx.x * 64 + threadIdx.x) * 4;
    if (oy >= H || ox0 >= W) return;
    const size_t plane = blockIdx.z;
    const float sy = fmaxf((oy + 0.5f) * (static_cast<float>(h) / H) - 0.5f, 0.f);
    const int y0 = min(static_cast<int>(sy), h - 1);
    const int y1 = min(y0 + 1, h - 1);
    const float ly = sy - y0;
    const float* r0 = in + (plane * h + y0) * w;
    const float* r1 = in + (plane * h + y1) * w;
    const float sxs = static_cast<float>(w) / W;
    float o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int ox = min(ox0 + k, W - 1);
        const float sx = fmaxf((ox + 0.5f) * sxs - 0.5f, 0.f);
        const int x0 = min(static_cast<int>(sx), w - 1);
        const int x1 = min(x0 + 1, w - 1);
        const float lx = sx - x0;
        o[k] = (1.f - ly) * ((1.f - lx) * __ldg(r0 + x0) + lx * __ldg(r0 + x1)) +
               ly * ((1.f - lx) * __ldg(r1 + x0) + lx * __ldg(r1 + x1));
    }
    float* dst = out + (plane * H + oy) * W + ox0;
    if ((W & 3) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0) {
        __stcs(reinterpret_cast<float4*>(dst), make_float4(o[0], o[1], o[2], o[3]));
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (ox0 + k < W) dst[k] = o[k];
    }
}

// --------------------------------- 1-channel antialiased bilinear resize ----
// torchvision `transforms.Resize(input_size)` / F.interpolate(mode='bilinear', align_corners=False, antialias=True)
// where a side SHRINKS (code/prepare_single_model.py:112-120 with ROIs larger than `input_size`): ATen's separable
// triangle filter (UpSampleKernel.cpp, `_compute_indices_min_size_weights_aa`) - per output index i:
//   scale = in / out,  support = max(scale, 1),  centre = scale (i + 0.5),
//   first = max(int(centre - support + 0.5), 0),  count = min(int(centre + support + 0.5), in) - first,
//   w_j = max(0, 1 - |(j + first - centre + 0.5) / max(scale, 1)|) / sum_j(...)
// horizontal pass first, then vertical, both accumulated in fp32 in tap order as ATen does.  A side that grows gets
// support 1, i.e. the plain bilinear taps, so mixed shrink / grow shapes go through the same code.
// block (64, 4): thread (tx, ty) produces output x = blockIdx.x * 64 + tx of row blockIdx.y * 4 + ty of plane
// blockIdx.z; the <= 2 support + 1 source rows / columns of neighbouring outputs overlap and are served by L1.
struct AaTaps {
    int first, count;
    float centre, inv, norm;
    __device__ __forceinline__ float weight(int j) const {
        return fmaxf(0.f, 1.f - fabsf((static_cast<float>(j + first) - centre + 0.5f) * inv)) * norm;
    }
};

__device__ __forceinline__ AaTaps aa_taps(int i, int in_size, int out_size) {
    const float scale = static_cast<float>(in_size) / static_cast<float>(out_size);
    const float support = scale >= 1.f ? scale : 1.f;
    AaTaps t;
    t.centre = scale * (static_cast<float>(i) + 0.5f);
    t.inv = scale >= 1.f ? 1.f / scale : 1.f;
    t.first = max(static_cast<int>(t.centre - support + 0.5f), 0);
    t.count = min(static_cast<int>(t.centre + support + 0.5f), in_size) - t.first;
    t.norm = 1.f;
    float total = 0.f;
    for (int j = 0; j < t.count; ++j) total += t.weight(j);
    t.norm = total != 0.f ? 1.f / total : 1.f;
    return t;
}

__global__ void __launch_bounds__(256)
resize_aa_c1_kernel(const float* __restrict__ in, int h, int w, float* __restrict__ out, int H, int W) {
    const int oy = blockIdx.y * 4 + threadIdx.y;
    const int ox = blockIdx.x * 64 + threadIdx.x;
    if (oy >= H || ox >= W) return;
    const size_t plane = blockIdx.z;
    const AaTaps ty = aa_taps(oy, h, H), tx = aa_taps(ox, w, W);
    const float* src = in + (plane * h + ty.first) * w + tx.first;
    float acc = 0.f;
    for (int r = 0; r < ty.count; ++r, src += w) {
        float row = __ldg(src) * tx.weight(0);
        for (int c = 1; c < tx.count; ++c) row = fmaf(__ldg(src + c), tx.weight(c), row);
        acc = r == 0 ? row * ty.weight(0) : fmaf(row, ty.weight(r), acc);
    }
    __stcs(out + (plane * H + oy) * W + ox, acc);
}

// ------------------------------------------- mask head tail + attention ----
// MaskHeadResize.out (model_module.py:187, 1x1 Cm->1 + bias) on the `pre` activations, then
// MaskGuidedSpatialAttention.mask_processor (:67-73, :92-93): 1x1 1->Hc (no bias),
// GroupNorm(1,Hc), GELU, 1x1 Hc->1 (+bias), sigmoid, clamp to [1e-4, 1-1e-4].
// GroupNorm(1,Hc) of u[c,p] = wa[c]*m[p] has mean = mean(wa)*mean(m) and
// E[u^2] = mean(wa^2)*mean(m^2), so two plane statistics of m suffice.  One CTA per case.
constexpr int kMaskHidden = 32;

__global__ void mask_tail_kernel(const __nv_bfloat16* __restrict__ pre, int Cm, int npix,
                                 const float* __restrict__ w_out, const float* __restrict__ b_out,
                                 float* __restrict__ mask_pred,  // [B, npix]
                                 int Hc, const float* __restrict__ wa, const float* __restrict__ gn_w,
                                 const float* __restrict__ gn_b, const float* __restrict__ wb,
                                 const float* __restrict__ bb, float gn_eps,
                                 float* __restrict__ attn) {  // [B, npix] or nullptr
    extern __shared__ float s_m[];  // npix floats
    __shared__ double scratch[33];
    const int b = blockIdx.x;
    // one thread per pixel: its Cm bf16 activations are one contiguous 2*Cm-byte row (16-byte loads);
    // with pre == nullptr the mask is already there (emitted by the producing GEMM's fused dot product)
    for (int p = threadIdx.x; p < npix; p += blockDim.x) {
        if (pre == nullptr) {
            s_m[p] = mask_pred[static_cast<size_t>(b) * npix + p];
            continue;
        }
        const uint4* px = reinterpret_cast<const uint4*>(pre + (static_cast<size_t>(b) * npix + p) * Cm);
        float acc = b_out[0];
        for (int v = 0; v < Cm / 8; ++v) {
            float f[8];
            unpack_bf16x8(__ldg(px + v), f);
#pragma unroll
            for (int k = 0; k < 8; ++k) acc = fmaf(f[k], __ldg(w_out + v * 8 + k), acc);
        }
        s_m[p] = acc;
        mask_pred[static_cast<size_t>(b) * npix + p] = acc;
    }
    __syncthreads();
    if (attn == nullptr) return;
    double s1 = 0.0, s2 = 0.0;
    for (int p = threadIdx.x; p < npix; p += blockDim.x) {
        const double m = s_m[p];
        s1 += m;
        s2 += m * m;
    }
    const double mean_m = block_sum<double>(s1, scratch) / npix;
    const double mean_m2 = block_sum<double>(s2, scratch) / npix;
    double wa1 = 0.0, wa2 = 0.0;
    for (int c = 0; c < Hc; ++c) {
        wa1 += wa[c];
        wa2 += static_cast<double>(wa[c]) * wa[c];
    }
    wa1 /= Hc;
    wa2 /= Hc;
    const double mu = wa1 * mean_m;
    const double var = fmax(wa2 * mean_m2 - mu * mu, 0.0);
    const float rstd = static_cast<float>(1.0 / sqrt(var + static_cast<double>(gn_eps)));
    const float muf = static_cast<float>(mu);
    for (int p = threadIdx.x; p < npix; p += blockDim.x) {
        const float m = s_m[p];
        float a = bb[0];
        for (int c = 0; c + 1 < Hc; c += 2) {
            const float2 g = gelu_fast2(make_float2((wa[c] * m - muf) * rstd * gn_w[c] + gn_b[c],
                                                    (wa[c + 1] * m - muf) * rstd * gn_w[c + 1] + gn_b[c + 1]));
            a += wb[c] * g.x + wb[c + 1] * g.y;
        }
        if (Hc & 1) a += wb[Hc - 1] * gelu_exact((wa[Hc - 1] * m - muf) * rstd * gn_w[Hc - 1] + gn_b[Hc - 1]);
        const float A = fminf(fmaxf(sigmoidf_(a), 1e-4f), 1.0f - 1e-4f);
        attn[static_cast<size_t>(b) * npix + p] = A;
    }
}

// ----------------------------------------------- 1 -> C pointwise lift -----
// First layer of Projector(1, proj_dim) (model_module.py:338-340) on a 1-channel fp32
// map: y[p, n] = gelu(r[p] * w[n] * scale[n] + bias[n]) as NHWC bf16.
// A thread keeps its 8 output channels' folded weights in registers and walks pixels (blockDim / nv pixels per CTA
// trip), 32-bit indices; requires blockDim % nv == 0.
__global__ void __launch_bounds__(256)
lift_c1_kernel(const float* __restrict__ r, int total_pix, int N, const float* __restrict__ w,
               const float* __restrict__ scale, const float* __restrict__ bias, __nv_bfloat16* __restrict__ y) {
    const int nv = N >> 3;
    const int vi = threadIdx.x % nv, pl = threadIdx.x / nv, ppb = blockDim.x / nv;
    const int n0 = vi << 3;
    float wr[8], sr[8], bs[8];  // ((r * w) * scale) + bias keeps the rounding order of the unfolded form
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        wr[k] = w[n0 + k];
        sr[k] = scale[n0 + k];
        bs[k] = bias[n0 + k];
    }
    uint4* out = reinterpret_cast<uint4*>(y);
    for (int p = blockIdx.x * ppb + pl; p < total_pix; p += gridDim.x * ppb) {
        const float rv = __ldg(r + p);
        float f[8];
#pragma unroll
        for (int k = 0; k < 8; k += 2) {
            const float2 g = gelu_fast2(make_float2(rv * wr[k] * sr[k] + bs[k], rv * wr[k + 1] * sr[k + 1] + bs[k + 1]));
            f[k] = g.x;
            f[k + 1] = g.y;
        }
        out[static_cast<size_t>(p) * nv + vi] = pack_bf16x8(f);
    }
}

// ------------------------------------------------- classification head -----
// ClassificationHead.forward (model_module.py:364-369): GAP -> L2 normalise -> Linear.
// The pooled vector comes from the fp32 channel sums of the producing GEMM epilogue,
// rescaled by the SE gate (GAP(x*g) = g*GAP(x)).  One warp per case.
__global__ void cls_head_kernel(const float* __restrict__ gap_sum, const float* __restrict__ gate, float inv_npix,
                                int C, int K, const float* __restrict__ fc_w, const float* __restrict__ fc_b,
                                int normalize, int B, float* __restrict__ logits, float* __restrict__ pooled_out) {
    const int lane = threadIdx.x & 31;
    const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (b >= B) return;
    float ss = 0.f;
    for (int c = lane; c < C; c += 32) {
        float v = gap_sum[static_cast<size_t>(b) * C + c] * inv_npix;
        if (gate != nullptr) v *= gate[static_cast<size_t>(b) * C + c];
        ss += v * v;
    }
    ss = warp_sum(ss);
    const float inv = normalize ? 1.0f / fmaxf(sqrtf(ss), 1e-12f) : 1.0f;
    for (int k = 0; k < K; ++k) {
        float a = 0.f;
        for (int c = lane; c < C; c += 32) {
            float v = gap_sum[static_cast<size_t>(b) * C + c] * inv_npix;
            if (gate != nullptr) v *= gate[static_cast<size_t>(b) * C + c];
            a += v * inv * fc_w[k * C + c];
        }
        a = warp_sum(a);
        if (lane == 0) logits[static_cast<size_t>(b) * K + k] = a + fc_b[k];
    }
    if (pooled_out != nullptr) {
        for (int c = lane; c < C; c += 32) {
            float v = gap_sum[static_cast<size_t>(b) * C + c] * inv_npix;
            if (gate != nullptr) v *= gate[static_cast<size_t>(b) * C + c];
            pooled_out[static_cast<size_t>(b) * C + c] = v * inv;
        }
    }
}

static inline int grid_for(size_t work_items, int threads, int max_blocks = 148 * 16) {
    size_t g = (work_items + threads - 1) / threads;
    if (g > static_cast<size_t>(max_blocks)) g = max_blocks;
    if (g == 0) g = 1;
    return static_cast<int>(g);
}

}  // namespace b200

using namespace b200;

static int stem_launch(const float* x, int B, int C, int H, int W, int stride, const float* plane_mean,
                       const float* se_w1, const float* se_b1, const float* se_w2, const float* se_b2, int Cm,
                       const float* wcat, const float* scale, const float* bias, int n_skip, int n_mid, void* skip_out,
                       void* mid_out, float* mod_attn, const float* in_affine, float z_lo, float z_hi,
                       const double* in_table, int L, b200::DropoutArgs drop, void* stream) {
    if (B < 0 || C <= 0 || C > kStemMaxC || Cm > kStemMaxC || H % stride != 0 || W % stride != 0) return -1;
    if (B == 0) return 0;
    if (x == nullptr || wcat == nullptr || scale == nullptr || bias == nullptr) return -2;
    if (se_w1 != nullptr && plane_mean == nullptr) return -3;
    const int n_out = n_skip + n_mid;
    // register blocks of 16 channels per quarter of the outputs, none straddling the skip / mid boundary
    if (n_out <= 0 || n_out % (4 * kStemCB) != 0 || n_skip % kStemCB != 0 || n_skip % 8 != 0 || n_mid % 8 != 0)
        return -4;
    if (skip_out == nullptr || mid_out == nullptr) return -5;
    const int npix = (H / stride) * (W / stride);
    if (in_affine != nullptr && in_table != nullptr) return -7;
    if (in_table != nullptr && (L < 2 || L > 16)) return -7;
    const size_t out_words = (static_cast<size_t>(kStemPix) * (n_out / 2 + 1) + 1) & ~static_cast<size_t>(1);
    const int w_rows = C;
    const size_t smem = (static_cast<size_t>(w_rows) * n_out + 2 * n_out) * sizeof(float) + out_words * sizeof(uint32_t) +
                        (in_table != nullptr ? static_cast<size_t>(C) * 56 * sizeof(double) : 0);
    if (((static_cast<size_t>(w_rows) * n_out + 2 * n_out) & 1) != 0) return -6;  // keeps the table 8-byte aligned
    if (smem > 48 * 1024) return -6;  // all supported shapes stay inside the default dynamic limit
    const int n_tiles = (npix + kStemPix - 1) / kStemPix;
    // tiles per CTA: as many as keeps >= ~8 CTAs per SM in the grid
    int gx = n_tiles;
    while (gx > 1 && static_cast<long long>(gx / 2) * B >= 148LL * 8) gx = (gx + 1) / 2;
    dim3 grid(gx, B);
    const unsigned int thresh = drop.seg != 0 ? b200::dropout_threshold(drop.p) : 0u;
    const float dscale = drop.seg != 0 ? 1.0f / (1.0f - drop.p) : 1.0f;
    auto go = [&](auto kern) {
        kern<<<grid, kStemThreads, smem, static_cast<cudaStream_t>(stream)>>>(
            x, C, H, W, stride, plane_mean, se_w1, se_b1, se_w2, se_b2, Cm, wcat, scale, bias, n_skip, n_mid,
            static_cast<__nv_bfloat16*>(skip_out), static_cast<__nv_bfloat16*>(mid_out), mod_attn, thresh, dscale,
            static_cast<unsigned int>(drop.seed), static_cast<unsigned int>(drop.seed >> 32), in_affine, z_lo, z_hi,
            in_table, L);
    };
    if (C == 8) go(stem_kernel<8, true>);
    else if (C < 8) go(stem_kernel<8, false>);
    else if (C == 16) go(stem_kernel<16, true>);
    else if (C < 16) go(stem_kernel<16, false>);
    else if (C == 32) go(stem_kernel<32, true>);
    else go(stem_kernel<32, false>);
    return launch_status();
}

extern "C" int b200_stem_ex(const float* x, int B, int C, int H, int W, int stride, const float* plane_mean,
                            const float* se_w1, const float* se_b1, const float* se_w2, const float* se_b2, int Cm,
                            const float* wcat, const float* scale, const float* bias, int n_skip, int n_mid,
                            void* skip_out, void* mid_out, float* mod_attn, const float* in_affine, float z_lo, float z_hi,
                            const double* in_table, int L, void* stream) {
    return stem_launch(x, B, C, H, W, stride, plane_mean, se_w1, se_b1, se_w2, se_b2, Cm, wcat, scale, bias, n_skip,
                       n_mid, skip_out, mid_out, mod_attn, in_affine, z_lo, z_hi, in_table, L, b200::DropoutArgs{}, stream);
}

// b200_stem_ex with MC dropout (probability drop_p, Philox seed drop_seed) on the bottleneck (mid) output, where the
// reference's first nn.Dropout sits (model_module.py:262).
extern "C" int b200_stem_mc(const float* x, int B, int C, int H, int W, int stride, const float* plane_mean,
                            const float* se_w1, const float* se_b1, const float* se_w2, const float* se_b2, int Cm,
                            const float* wcat, const float* scale, const float* bias, int n_skip, int n_mid,
                            void* skip_out, void* mid_out, float* mod_attn, const float* in_affine, float z_lo, float z_hi,
                            const double* in_table, int L, float drop_p, unsigned long long drop_seed, void* stream) {
    if (!b200::dropout_args_valid(drop_p, 1)) return -19;
    b200::DropoutArgs d;
    d.p = drop_p;
    d.seed = drop_seed;
    d.seg = drop_p > 0.f ? 1 : 0;
    return stem_launch(x, B, C, H, W, stride, plane_mean, se_w1, se_b1, se_w2, se_b2, Cm, wcat, scale, bias, n_skip,
                       n_mid, skip_out, mid_out, mod_attn, in_affine, z_lo, z_hi, in_table, L, d, stream);
}

extern "C" int b200_se_gate(const float* gap_sum, int B, int C, int Cm, int npix, const float* w1t, const float* b1,
                            const float* w2t, const float* b2, float* gate, float* hidden, void* stream) {
    if (B < 0 || C <= 0 || Cm <= 0 || npix <= 0) return -1;
    if (B == 0) return 0;
    if (gap_sum == nullptr || gate == nullptr || hidden == nullptr) return -2;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const unsigned rows = (B + kSeCases - 1) / kSeCases;
    se_dense_kernel<0><<<dim3((Cm + 63) / 64, rows), 256, 0, s>>>(gap_sum, 1.0f / npix, B, C, Cm, w1t, b1, hidden);
    se_dense_kernel<1><<<dim3((C + 63) / 64, rows), 256, 0, s>>>(hidden, 1.0f, B, Cm, C, w2t, b2, gate);
    return launch_status();
}

extern "C" int b200_scale_map(const void* x, void* y, int B, int npix, int C, const float* gate, const float* attn,
                              const float* gamma, void* stream) {
    if (B < 0 || C % 8 != 0 || npix <= 0) return -1;
    if (B == 0) return 0;
    if (x == nullptr || y == nullptr) return -2;
    const long long nvc = static_cast<long long>(npix) * (C / 8);
    if (nvc > 0x7fffffff / 2 || B > 65535) return -3;
    const unsigned chunks = static_cast<unsigned>((nvc + kScaleUnroll * 256 - 1) / (kScaleUnroll * 256));
    scale_map_kernel<<<dim3(chunks, B), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __nv_bfloat16*>(x), static_cast<__nv_bfloat16*>(y), C, npix, gate, attn, gamma);
    return launch_status();
}

extern "C" int b200_conv3x3_c1(const void* x, int B, int H, int W, int C, const float* w, const float* bias,
                               float* out, void* stream) {
    if (B < 0 || C % 8 != 0 || H <= 0 || W <= 0) return -1;
    if (B == 0) return 0;
    if (x == nullptr || w == nullptr || bias == nullptr || out == nullptr) return -2;
    const size_t total_pix = static_cast<size_t>(B) * H * W;
    const size_t blocks = (total_pix * 32 + 255) / 256;
    conv3x3_c1_kernel<<<static_cast<unsigned>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __nv_bfloat16*>(x), H, W, C, w, bias, out, total_pix);
    return launch_status();
}

extern "C" int b200_tapsum(const float* d, int B, int H, int W, const float* bias, float* out, void* stream) {
    if (B < 0 || H <= 0 || W <= 0) return -1;
    if (B == 0) return 0;
    if (d == nullptr || bias == nullptr || out == nullptr) return -2;
    const size_t total_pix = static_cast<size_t>(B) * H * W;
    tapsum_kernel<<<static_cast<unsigned>((total_pix + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        d, H, W, bias, out, total_pix);
    return launch_status();
}

extern "C" int b200_mask_tail(const void* pre, int B, int npix, int Cm, const float* w_out, const float* b_out,
                              float* mask_pred, int Hc, const float* wa, const float* gn_w, const float* gn_b,
                              const float* wb, const float* bb, float gn_eps, float* attn, void* stream) {
    if (B < 0 || npix <= 0 || Cm % 8 != 0 || npix > 12 * 1024) return -1;
    if (B == 0) return 0;
    if (pre == nullptr || w_out == nullptr || b_out == nullptr || mask_pred == nullptr) return -2;
    if (attn != nullptr && (wa == nullptr || gn_w == nullptr || gn_b == nullptr || wb == nullptr || bb == nullptr))
        return -3;
    mask_tail_kernel<<<B, 256, npix * sizeof(float), static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __nv_bfloat16*>(pre), Cm, npix, w_out, b_out, mask_pred, Hc, wa, gn_w, gn_b, wb, bb, gn_eps,
        attn);
    return launch_status();
}

extern "C" int b200_mask_attention(const float* mask, int B, int npix, int Hc, const float* wa, const float* gn_w,
                                   const float* gn_b, const float* wb, const float* bb, float gn_eps, float* attn,
                                   void* stream) {
    if (B < 0 || npix <= 0 || npix > 12 * 1024 || Hc <= 0) return -1;
    if (B == 0) return 0;
    if (mask == nullptr || attn == nullptr || wa == nullptr || gn_w == nullptr || gn_b == nullptr || wb == nullptr ||
        bb == nullptr)
        return -2;
    mask_tail_kernel<<<B, 256, npix * sizeof(float), static_cast<cudaStream_t>(stream)>>>(
        nullptr, 0, npix, nullptr, nullptr, const_cast<float*>(mask), Hc, wa, gn_w, gn_b, wb, bb, gn_eps, attn);
    return launch_status();
}

extern "C" int b200_resize_bilinear_c1(const float* in, int B, int h, int w, float* out, int H, int W, void* stream) {
    if (B < 0 || h <= 0 || w <= 0 || H <= 0 || W <= 0) return -1;
    if (B == 0) return 0;
    if (in == nullptr || out == nullptr) return -2;
    if (B > 65535 * 64 || (H + 3) / 4 > 65535) return -3;
    for (int b0 = 0; b0 < B; b0 += 65535) {  // gridDim.z limit
        const int nb = B - b0 < 65535 ? B - b0 : 65535;
        const dim3 grid((W + 255) / 256, (H + 3) / 4, nb);
        resize_bilinear_c1_kernel<<<grid, dim3(64, 4), 0, static_cast<cudaStream_t>(stream)>>>(
            in + static_cast<size_t>(b0) * h * w, h, w, out + static_cast<size_t>(b0) * H * W, H, W);
    }
    return launch_status();
}

extern "C" int b200_resize_aa_c1(const float* in, int B, int h, int w, float* out, int H, int W, void* stream) {
    if (B < 0 || h <= 0 || w <= 0 || H <= 0 || W <= 0) return -1;
    if (B == 0) return 0;
    if (in == nullptr || out == nullptr) return -2;
    if (B > 65535 * 64 || (H + 3) / 4 > 65535) return -3;
    for (int b0 = 0; b0 < B; b0 += 65535) {  // gridDim.z limit
        const int nb = B - b0 < 65535 ? B - b0 : 65535;
        const dim3 grid((W + 63) / 64, (H + 3) / 4, nb);
        resize_aa_c1_kernel<<<grid, dim3(64, 4), 0, static_cast<cudaStream_t>(stream)>>>(
            in + static_cast<size_t>(b0) * h * w, h, w, out + static_cast<size_t>(b0) * H * W, H, W);
    }
    return launch_status();
}

extern "C" int b200_lift_c1(const float* r, long long total_pix, int N, const float* w, const float* scale,
                            const float* bias, void* y, void* stream) {
    if (total_pix < 0 || N <= 0 || N % 8 != 0 || N > 2048 || total_pix > 0x7fffffffLL) return -1;
    if (total_pix == 0) return 0;
    if (r == nullptr || w == nullptr || scale == nullptr || bias == nullptr || y == nullptr) return -2;
    const int nv = N / 8, threads = nv * (256 / nv), ppb = threads / nv;
    long long blocks = (total_pix + ppb - 1) / ppb;
    if (blocks > 148 * 16) blocks = 148 * 16;
    lift_c1_kernel<<<static_cast<unsigned>(blocks), threads, 0, static_cast<cudaStream_t>(stream)>>>(
        r, static_cast<int>(total_pix), N, w, scale, bias, static_cast<__nv_bfloat16*>(y));
    return launch_status();
}

extern "C" int b200_cls_head(const float* gap_sum, const float* gate, int B, int C, int npix, int K, const float* fc_w,
                             const float* fc_b, int normalize, float* logits, float* pooled_out, void* stream) {
    if (B < 0 || C <= 0 || K <= 0 || npix <= 0) return -1;
    if (B == 0) return 0;
    if (gap_sum == nullptr || fc_w == nullptr || fc_b == nullptr || logits == nullptr) return -2;
    const int blocks = (B * 32 + 127) / 128;
    cls_head_kernel<<<blocks, 128, 0, static_cast<cudaStream_t>(stream)>>>(gap_sum, gate, 1.0f / npix, C, K, fc_w,
                                                                           fc_b, normalize, B, logits, pooled_out);
    return launch_status();
}
