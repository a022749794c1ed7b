// ResNet-50 backbone glue that is not GEMM shaped (timm / torchvision `resnet50`, reference
// code/foundation_model.py:15-68, :220-312): the 7x7 / stride-2 stem convolution on the few-channel fp32 input and
// the 3x3 / stride-2 max pool.  Everything after them (bottleneck 1x1 / 3x3 / dilated 3x3 convolutions with folded
// BatchNorm, ReLU and the residual) runs on the tcgen05 implicit-GEMM kernel.
#include "b200_fusion.h"
#include "common.cuh"

namespace b200 {

constexpr int kStemTile = 8;                        // 8 x 8 output pixels per CTA
constexpr int kStemPatch = kStemTile * 2 + 5;       // 21 x 21 input pixels feed them (7x7, stride 2)

// im2col of the 7x7 / stride-2 / padding-3 stem for the tensor-core route: row (b, oy, ox) of the bf16 patch matrix
// holds gate[b, c] * x[b, c, 2 oy + ky - 3, 2 ox + kx - 3] at column c * 49 + ky * 7 + kx (Conv2d weight order),
// zero-padded to Kp columns (a multiple of 64), so that conv1 + bn1 + ReLU is one GEMM with K = Kp.  One CTA
// produces the 64 rows of an 8 x 8 output tile: the [C][21][21] input patch is staged in shared memory with
// coalesced reads, a per-column offset table removes the divisions, and the rows go out as 16-byte stores that are
// contiguous across the CTA.
__global__ void __launch_bounds__(256)
im2col7x7_s2_kernel(const float* __restrict__ x, const float* __restrict__ gate, int C, int H, int W, int Kp,
                    __nv_bfloat16* __restrict__ out) {
    extern __shared__ float s_dyn[];
    float* s_patch = s_dyn;                                            // [C][21*21]
    short* s_off = reinterpret_cast<short*>(s_patch + C * kStemPatch * kStemPatch);  // [Kp] patch offset or -1
    const int Ho = H / 2, Wo = W / 2;
    const int b = blockIdx.z;
    const int oy0 = blockIdx.y * kStemTile, ox0 = blockIdx.x * kStemTile;
    const int tid = threadIdx.x;
    constexpr int kPP = kStemPatch * kStemPatch;
    for (int i = tid; i < C * kPP; i += 256) {
        const int c = i / kPP, q = i - c * kPP;
        const int iy = oy0 * 2 - 3 + q / kStemPatch, ix = ox0 * 2 - 3 + q % kStemPatch;
        float v = 0.f;
        if (iy >= 0 && iy < H && ix >= 0 && ix < W) {
            v = __ldg(x + ((static_cast<size_t>(b) * C + c) * H + iy) * W + ix);
            if (gate != nullptr) v *= __ldg(gate + b * C + c);
        }
        s_patch[i] = v;
    }
    for (int k = tid; k < Kp; k += 256) {
        short off = -1;
        if (k < C * 49) {
            const int c = k / 49, t = k - c * 49;
            off = static_cast<short>(c * kPP + (t / 7) * kStemPatch + t % 7);
        }
        s_off[k] = off;
    }
    __syncthreads();
    const int kv = Kp >> 3;
    for (int idx = tid; idx < kStemTile * kStemTile * kv; idx += 256) {
        const int rr = idx / kv, jc = idx - rr * kv;
        const int py = rr >> 3, px = rr & 7;
        const int oy = oy0 + py, ox = ox0 + px;
        if (oy >= Ho || ox >= Wo) continue;
        const int base = (py * 2) * kStemPatch + px * 2;
        float f[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int off = s_off[jc * 8 + e];
            f[e] = off >= 0 ? s_patch[off + base] : 0.f;
        }
        uint4* dst = reinterpret_cast<uint4*>(out + ((static_cast<size_t>(b) * Ho + oy) * Wo + ox) * Kp) + jc;
        *dst = pack_bf16x8(f);
    }
}

// nn.MaxPool2d(3, stride 2, padding 1) on an NHWC bf16 map (padding never wins: taps outside the map are skipped).
__global__ void maxpool3x3_s2_kernel(const __nv_bfloat16* __restrict__ x, int H, int W, int C,
                                     __nv_bfloat16* __restrict__ y, size_t total_vec) {
    const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
    if (i >= total_vec) return;
    const int Ho = H / 2, Wo = W / 2, cv = C >> 3;
    const int c0 = static_cast<int>(i % cv) << 3;
    size_t r = i / cv;
    const int ox = static_cast<int>(r % Wo); r /= Wo;
    const int oy = static_cast<int>(r % Ho);
    const size_t b = r / Ho;
    float m[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) m[k] = -INFINITY;
    for (int dy = -1; dy <= 1; ++dy) {
        const int iy = oy * 2 + dy;
        if (iy < 0 || iy >= H) continue;
        for (int dx = -1; dx <= 1; ++dx) {
            const int ix = ox * 2 + dx;
            if (ix < 0 || ix >= W) continue;
            float f[8];
            unpack_bf16x8(__ldg(reinterpret_cast<const uint4*>(x + ((b * H + iy) * W + ix) * C + c0)), f);
#pragma unroll
            for (int k = 0; k < 8; ++k) m[k] = fmaxf(m[k], f[k]);
        }
    }
    reinterpret_cast<uint4*>(y)[i] = pack_bf16x8(m);
}

}  // namespace b200

using namespace b200;

extern "C" int b200_maxpool3x3_s2(const void* x, int B, int H, int W, int C, void* y, void* stream) {
    if (B < 0 || H <= 0 || W <= 0 || H % 2 != 0 || W % 2 != 0 || C <= 0 || C % 8 != 0) return -1;
    if (B == 0) return 0;
    if (x == nullptr || y == nullptr) return -2;
    const size_t total_vec = static_cast<size_t>(B) * (H / 2) * (W / 2) * (C / 8);
    maxpool3x3_s2_kernel<<<static_cast<unsigned>((total_vec + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __nv_bfloat16*>(x), H, W, C, static_cast<__nv_bfloat16*>(y), total_vec);
    return launch_status();
}

extern "C" int b200_im2col7x7_s2(const float* x, const float* gate, int B, int C, int H, int W, int Kp, void* out,
                                 void* stream) {
    if (B < 0 || C <= 0 || C > 64 || H <= 0 || W <= 0 || H % 2 != 0 || W % 2 != 0 || Kp % 64 != 0 || Kp < C * 49 || B > 65535)
        return -1;
    if (B == 0) return 0;
    if (x == nullptr || out == nullptr) return -2;
    const size_t smem = static_cast<size_t>(C) * kStemPatch * kStemPatch * sizeof(float) + static_cast<size_t>(Kp) * sizeof(short);
    static size_t configured = 0;
    if (smem > 48 * 1024 && smem > configured) {
        cudaError_t e = cudaFuncSetAttribute(im2col7x7_s2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             static_cast<int>(smem));
        if (e != cudaSuccess) return static_cast<int>(e);
        configured = smem;
    }
    const dim3 grid((W / 2 + kStemTile - 1) / kStemTile, (H / 2 + kStemTile - 1) / kStemTile, B);
    im2col7x7_s2_kernel<<<grid, 256, smem, static_cast<cudaStream_t>(stream)>>>(x, gate, C, H, W, Kp,
                                                                                static_cast<__nv_bfloat16*>(out));
    return launch_status();
}
