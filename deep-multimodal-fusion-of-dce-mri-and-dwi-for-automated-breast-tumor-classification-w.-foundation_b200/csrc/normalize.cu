// Per-(case, channel) input normalisation: HBM-bound, one CTA per image plane.
//
//  * DWI: z-score with unbiased std (clamped at 1e-6), clip to [z_lo, z_hi], affine to
//    [0,1]; the last channel is written as zeros when `skip_last` (the reference's
//    adc=True default).  Follows code/dataset.py:14-41 (DWINormalize.__call__).
//  * DCE: Nyul histogram standardisation: 11 order-statistic landmarks of the plane
//    (numpy "linear" percentile rule) -> piece-wise linear map onto the fitted average
//    landmarks -> piece-wise linear map onto the standard scale, all in float64 with
//    numpy.interp's exact branch structure.  Follows code/preprocess_helpers.py:85-120
//    (NyulStandardizer.transform).
//
// Both kernels read every input element from HBM once and write every output once.
#include <cfloat>

#include "b200_fusion.h"
#include "common.cuh"

#include <cstdlib>

namespace b200 {

constexpr int kNormThreads = 256;

// ------------------------------------------------------------------ DWI ----
template <int VEC>
__global__ void __launch_bounds__(kNormThreads)
dwi_normalize_reg_kernel(const float* __restrict__ x, float* __restrict__ out, int planes, int C, int n,
                         int skip_last, float z_lo, float z_hi, float* __restrict__ plane_mean,
                         float* __restrict__ stats_out) {
    // out == nullptr: statistics only (the consumer applies the map while loading the raw plane: stats_out[plane] =
    // {mean, 1/std, scale, offset} with y = fma(clamp((x - mean) * (1/std), z_lo, z_hi), scale, offset); a skipped
    // plane carries {0, 0, 0, 0}, i.e. y = 0).  The arithmetic below and the consumer's are the same instructions.
    // One block-wide barrier per plane.  Each thread accumulates sum(d) and sum(d^2) of d = x - pivot in fp64
    // (pivot = the plane's first sample: shifting makes the one-pass variance as safe as the reference's two
    // passes; fp64 removes what cancellation is left), the block reduces both together with the OUTPUT sum of
    // the previous plane (the plane_mean by-product), and the scratch area is double buffered so that no
    // second barrier is needed before it is rewritten.
    constexpr int kWarps = kNormThreads / 32;
    __shared__ double red[2][kWarps][3];
    const int n4 = n >> 2;
    const float range = z_hi - z_lo;
    const float inv_range = 1.0f / range, off = -z_lo * inv_range;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    auto skipped = [&](int pl) { return skip_last && (pl % C) == C - 1; };
    auto load = [&](int pl, float4 (&v)[VEC], float& pivot) {
        const float4* src = reinterpret_cast<const float4*>(x + static_cast<size_t>(pl) * n);
        pivot = __ldg(reinterpret_cast<const float*>(src));
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
            const int i = threadIdx.x + j * kNormThreads;
            v[j] = (i < n4) ? __ldcs(src + i) : make_float4(pivot, pivot, pivot, pivot);  // d = 0 for padding lanes
        }
    };
    int plane = blockIdx.x;
    float4 v[VEC], vn[VEC];
    float pivot = 0.f, pivot_n = 0.f;
    if (plane < planes && !skipped(plane)) load(plane, v, pivot);
    double osum_prev = 0.0;  // this thread's share of the previous plane's output sum
    int prev_plane = -1;     // plane whose output mean is still to be written (-1: none)
    int buf = 0;
    for (; plane < planes; plane += gridDim.x) {
        // the next plane's loads are issued before this plane's barrier, so HBM reads stay in flight across it
        const int next = plane + gridDim.x;
        if (next < planes && !skipped(next)) load(next, vn, pivot_n);
        float4* dst = out != nullptr ? reinterpret_cast<float4*>(out + static_cast<size_t>(plane) * n) : nullptr;
        const bool skip = skipped(plane);
        double sd = 0.0, sq = 0.0;
        if (!skip) {
            // per-thread partial sums of d = x - pivot in fp32 (<= 32 samples per thread: ~1e-7 relative error, the
            // shift keeps the variance well conditioned); fp64 only across threads.  The fp64 per-element form made
            // the kernel issue bound (ncu: 67 % issue-active, 4 200 warp instructions per plane).
            float fs = 0.f, fq = 0.f;
#pragma unroll
            for (int j = 0; j < VEC; ++j) {
                const float a = v[j].x - pivot, b = v[j].y - pivot, c = v[j].z - pivot, d = v[j].w - pivot;
                fs += (a + b) + (c + d);
                fq = fmaf(a, a, fq);
                fq = fmaf(b, b, fq);
                fq = fmaf(c, c, fq);
                fq = fmaf(d, d, fq);
            }
            sd = static_cast<double>(fs);
            sq = static_cast<double>(fq);
        }
        // fp32 shuffles inside the warp (32 partials of <= 32 samples each), fp64 across the warps
        double r0 = static_cast<double>(warp_sum(static_cast<float>(sd))), r1 = static_cast<double>(warp_sum(static_cast<float>(sq)));
        double r2 = static_cast<double>(warp_sum(static_cast<float>(osum_prev)));
        if (lane == 0) {
            red[buf][warp][0] = r0;
            red[buf][warp][1] = r1;
            red[buf][warp][2] = r2;
        }
        __syncthreads();
        r0 = r1 = r2 = 0.0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) {  // broadcast reads, identical order in every thread
            r0 += red[buf][w][0];
            r1 += red[buf][w][1];
            r2 += red[buf][w][2];
        }
        buf ^= 1;
        if (plane_mean != nullptr && threadIdx.x == 0 && prev_plane >= 0) plane_mean[prev_plane] = static_cast<float>(r2 / n);
        float osum = 0.f;
        if (skip) {
            if (dst != nullptr)
                for (int i = threadIdx.x; i < n4; i += kNormThreads) __stcs(dst + i, make_float4(0.f, 0.f, 0.f, 0.f));
            if (stats_out != nullptr && threadIdx.x == 0)
                *reinterpret_cast<float4*>(stats_out + 4 * static_cast<size_t>(plane)) = make_float4(0.f, 0.f, 0.f, 0.f);
        } else {
            const double md = r0 / n;
            const float mean = static_cast<float>(static_cast<double>(pivot) + md);
            // torch.std(): unbiased (n-1); n == 1 gives NaN there as well.
            const double var = (r1 - r0 * md) / static_cast<double>(n - 1);
            const float sdev = fmaxf(static_cast<float>(sqrt(fmax(var, 0.0))), 1e-6f);
            // The two divisions of the reference become multiplications by correctly rounded reciprocals
            // (<= 2 ulp from the divided form, far inside the 1e-5 tolerance): IEEE fp32 division costs ~10
            // issue slots and would make this HBM-bound kernel ALU-bound.
            const float inv_sd = 1.0f / sdev;
            if (stats_out != nullptr && threadIdx.x == 0)
                *reinterpret_cast<float4*>(stats_out + 4 * static_cast<size_t>(plane)) = make_float4(mean, inv_sd, inv_range, off);
#pragma unroll
            for (int j = 0; j < VEC; ++j) {
                const int i = threadIdx.x + j * kNormThreads;
                if (i < n4) {
                    float4 o;
                    // (x - mean) * inv_sd as packed fp32x2 (FADD2 / FMUL2 / FFMA2 round exactly like the scalar forms)
                    const float2 nm = make_float2(-mean, -mean), is2 = make_float2(inv_sd, inv_sd);
                    const float2 ir2 = make_float2(inv_range, inv_range), of2 = make_float2(off, off);
                    float2 a = __fmul2_rn(__fadd2_rn(make_float2(v[j].x, v[j].y), nm), is2);
                    float2 b = __fmul2_rn(__fadd2_rn(make_float2(v[j].z, v[j].w), nm), is2);
                    a.x = fminf(fmaxf(a.x, z_lo), z_hi);
                    a.y = fminf(fmaxf(a.y, z_lo), z_hi);
                    b.x = fminf(fmaxf(b.x, z_lo), z_hi);
                    b.y = fminf(fmaxf(b.y, z_lo), z_hi);
                    a = __ffma2_rn(a, ir2, of2);
                    b = __ffma2_rn(b, ir2, of2);
                    o = make_float4(a.x, a.y, b.x, b.y);
                    const float2 s2 = __fadd2_rn(a, b);
                    osum += s2.x + s2.y;
                    if (dst != nullptr) __stcs(dst + i, o);
                }
            }
        }
        osum_prev = static_cast<double>(osum);
        prev_plane = plane;
        pivot = pivot_n;
#pragma unroll
        for (int j = 0; j < VEC; ++j) v[j] = vn[j];
    }
    if (plane_mean != nullptr && prev_plane >= 0) {  // the last plane's output mean
        const double r2 = warp_sum(osum_prev);
        if (lane == 0) red[buf][warp][2] = r2;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
            for (int w = 0; w < kWarps; ++w) t += red[buf][w][2];
            plane_mean[prev_plane] = static_cast<float>(t / n);
        }
    }
}

// Any plane size / alignment: three sweeps, the 2nd and 3rd hit L2 (a plane is <= 200 KB).
__global__ void __launch_bounds__(kNormThreads)
dwi_normalize_stream_kernel(const float* __restrict__ x, float* __restrict__ out, int C, int n, int skip_last,
                            float z_lo, float z_hi, float* __restrict__ plane_mean) {
    // Planes too large for registers (224 x 224 after the C4 resize): one statistics pass (pivot-shifted fp64
    // sum / sum of squares, see the register kernel) and one apply pass that re-reads the plane from L2;
    // 16-byte accesses when the plane allows it.
    __shared__ double scratch[33];
    const int plane = blockIdx.x;
    const int c = plane % C;
    const float* src = x + static_cast<size_t>(plane) * n;
    float* dst = out + static_cast<size_t>(plane) * n;
    const bool vec = (n & 3) == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0;
    const int n4 = vec ? n >> 2 : 0;
    if (skip_last && c == C - 1) {
        for (int i = threadIdx.x; i < n4; i += kNormThreads)
            __stcs(reinterpret_cast<float4*>(dst) + i, make_float4(0.f, 0.f, 0.f, 0.f));
        for (int i = n4 * 4 + threadIdx.x; i < n; i += kNormThreads) dst[i] = 0.f;
        if (plane_mean != nullptr && threadIdx.x == 0) plane_mean[plane] = 0.f;
        return;
    }
    const double pv = static_cast<double>(__ldg(src));
    double sd = 0.0, sq = 0.0;
    for (int i = threadIdx.x; i < n4; i += kNormThreads) {
        const float4 f = __ldg(reinterpret_cast<const float4*>(src) + i);
        const double a = f.x - pv, b = f.y - pv, cc = f.z - pv, d = f.w - pv;
        sd += (a + b) + (cc + d);
        sq = fma(a, a, fma(b, b, fma(cc, cc, fma(d, d, sq))));
    }
    for (int i = n4 * 4 + threadIdx.x; i < n; i += kNormThreads) {
        const double a = src[i] - pv;
        sd += a;
        sq = fma(a, a, sq);
    }
    const double r0 = block_sum<double>(sd, scratch);
    const double r1 = block_sum<double>(sq, scratch);
    const double md = r0 / n;
    const float mean = static_cast<float>(pv + md);
    const float sdev = fmaxf(static_cast<float>(sqrt(fmax((r1 - r0 * md) / static_cast<double>(n - 1), 0.0))), 1e-6f);
    const float inv_sd = 1.0f / sdev, inv_range = 1.0f / (z_hi - z_lo), off = -z_lo * inv_range;
    auto map = [&](float v) { return fmaf(fminf(fmaxf((v - mean) * inv_sd, z_lo), z_hi), inv_range, off); };
    float osum = 0.f;
    for (int i = threadIdx.x; i < n4; i += kNormThreads) {
        const float4 f = __ldg(reinterpret_cast<const float4*>(src) + i);
        const float4 o = make_float4(map(f.x), map(f.y), map(f.z), map(f.w));
        osum += (o.x + o.y) + (o.z + o.w);
        __stcs(reinterpret_cast<float4*>(dst) + i, o);
    }
    for (int i = n4 * 4 + threadIdx.x; i < n; i += kNormThreads) {
        const float o = map(src[i]);
        osum += o;
        dst[i] = o;
    }
    if (plane_mean != nullptr) {
        const double om = block_sum<double>(static_cast<double>(osum), scratch);
        if (threadIdx.x == 0) plane_mean[plane] = static_cast<float>(om / n);
    }
}

// ----------------------------------------------------------------- Nyul ----
constexpr int kMaxLandmarks = 16;
constexpr int kNyulThreads = 512;

// numpy.interp for one sample: xp ascending (ties allowed), float64 throughout, no FMA
// contraction (matches the C loop in numpy's compiled_base.c).
__device__ __forceinline__ double np_interp(double xv, const double* xp, const float* xpf, const double* fp,
                                            const double* slope, int L, int hint, int& j_out) {
    if (xv != xv) {
        j_out = 0;
        return xv;
    }
    // Segment j = largest index with xp[j] <= xv (0 when xv < xp[0]).  First guess: the caller's hint (the second
    // interpolation of a sample almost always lands in the segment of the first), else a 4-step binary search on
    // fp32 copies of the landmarks (L <= 16); then an exact fp64 fix-up, normally two compares that change nothing.
    int j = hint;
    if (hint < 0) {
        const float xf = static_cast<float>(xv);
        j = 0;
#pragma unroll
        for (int step = 8; step >= 1; step >>= 1) {
            const int t = j + step;
            if (t < L && xpf[t] <= xf) j = t;
        }
    }
    while (j > 0 && xp[j] > xv) --j;
    while (j + 1 < L && xp[j + 1] <= xv) ++j;
    j_out = j;
    // numpy.interp: left / right fill, exact hits, then slope * (x - xp[j]) + fp[j] with its NaN fallbacks
    if (j == L - 1) return fp[j];            // xv >= xp[L-1]
    const double x0 = xp[j];
    if (!(xv > x0)) return fp[j];            // xv == xp[j], or xv < xp[0] (j == 0)
    double r = __dadd_rn(__dmul_rn(slope[j], __dadd_rn(xv, -x0)), fp[j]);
    if (r != r) {
        r = __dadd_rn(__dmul_rn(slope[j], __dadd_rn(xv, -xp[j + 1])), fp[j + 1]);
        if (r != r && fp[j] == fp[j + 1]) r = fp[j];
    }
    return r;
}

constexpr int kNyulBins = 4096;   // linear bins over [min, max] of the plane
constexpr int kNyulListCap = 64;   // candidates kept per landmark rank
constexpr int kNyulMaxRanks = 2 * kMaxLandmarks;

// Tail shared by both Nyul kernels: the L percentiles from the 2L selected order statistics (numpy's "linear"
// rule: float32 difference, fp64 lerp, switched at gamma >= 0.5), the two interpolation tables, then
// out = interp(interp(x, orig, avg), avg, std) over the plane.  `s_val` holds the order statistics (shared).
//
// EXACT = false (the default product path): the two chained interpolations are composed ONCE per plane into one
// piece-wise linear table.  Within segment j of the image's own landmarks (orig[j] <= x < orig[j+1]) the first
// np.interp lands in [avg[j], avg[j+1]] and the second maps that interval linearly onto [std[j], std[j+1]], so
//     out = c_j + m_j * max(x - orig[j], 0),   m_j = (std[j+1] - std[j]) / (orig[j+1] - orig[j])
// with np.interp's own tie semantics folded into the table: c_j = std[last k with avg[k] == avg[j]] (an exact hit on
// a run of equal xp returns the run's last fp), m_j = 0 where avg or orig does not increase, left / right fill =
// c_0 / c_{L-1}.  The table is built in fp64; per sample the segment comes from fp32 compares against the landmarks
// rounded UP to float (x >= orig[j] in fp64  <=>  x >= ru(orig[j]) for a float x: exact), and the value from one
// fp64 subtract + fma.  ~35 instructions per sample instead of ~200; equal to the exact path to <= 1 fp32 ulp (the
// contract is 1e-5 relative).  EXACT = true keeps numpy's operation order bit for bit (tests; `exact=True`).
template <bool EXACT, int NREG = 0, typename Load>
__device__ __forceinline__ void nyul_apply(const float* s_val, int L, int c, int n, int plane,
                                           const double* __restrict__ avg_landmarks,
                                           const double* __restrict__ standard_scale,
                                           const double* __restrict__ gamma, Load load, float* __restrict__ dst,
                                           float* __restrict__ plane_mean, const float* __restrict__ gsrc = nullptr,
                                           double* __restrict__ table_out = nullptr, const float* vreg = nullptr) {
    __shared__ double s_orig[kMaxLandmarks], s_avg[kMaxLandmarks], s_std[kMaxLandmarks];
    __shared__ double s_slope1[kMaxLandmarks], s_slope2[kMaxLandmarks];
    __shared__ float s_origf[kMaxLandmarks], s_avgf[kMaxLandmarks];
    __shared__ double scratch[33];
    const int tid = threadIdx.x;
    if (tid < L) {
        const int t = tid;
        const float a = s_val[2 * t], b2 = s_val[2 * t + 1];
        const float diff = b2 - a;  // numpy subtracts in the array dtype (float32) first
        const double g = gamma[t];
        double pv;
        if (g >= 0.5) pv = __dadd_rn(static_cast<double>(b2), -__dmul_rn(static_cast<double>(diff), __dadd_rn(1.0, -g)));
        else pv = __dadd_rn(static_cast<double>(a), __dmul_rn(static_cast<double>(diff), g));
        s_orig[t] = pv;
        s_avg[t] = avg_landmarks[c * L + t];
        s_std[t] = standard_scale[t];
        s_origf[t] = static_cast<float>(pv);
        s_avgf[t] = static_cast<float>(s_avg[t]);
    }
    __syncthreads();
    if (tid < L - 1) {
        const int t = tid;
        s_slope1[t] = __ddiv_rn(__dadd_rn(s_avg[t + 1], -s_avg[t]), __dadd_rn(s_orig[t + 1], -s_orig[t]));
        s_slope2[t] = __ddiv_rn(__dadd_rn(s_std[t + 1], -s_std[t]), __dadd_rn(s_avg[t + 1], -s_avg[t]));
    }
    __syncthreads();
    // composed table (fast path)
    __shared__ double s_tc[kMaxLandmarks], s_tm[kMaxLandmarks];
    __shared__ float s_up[kMaxLandmarks];
    if (!EXACT) {
        if (tid < L) {
            const int t = tid;
            int k = t;
            while (k + 1 < L && s_avg[k + 1] == s_avg[t]) ++k;
            s_tc[t] = s_std[k];
            double m = 0.0;
            if (t + 1 < L && s_avg[t + 1] > s_avg[t] && s_orig[t + 1] > s_orig[t])
                m = __ddiv_rn(__dadd_rn(s_std[t + 1], -s_std[t]), __dadd_rn(s_orig[t + 1], -s_orig[t]));
            s_tm[t] = m;
            s_up[t] = __double2float_ru(s_orig[t]);
            if (table_out != nullptr) {  // per plane: orig[16] | slope[16] | value[16] (fp64) | up[16] (fp32, in 8 doubles)
                double* tb = table_out + static_cast<size_t>(plane) * (3 * kMaxLandmarks + kMaxLandmarks / 2);
                tb[t] = s_orig[t];
                tb[kMaxLandmarks + t] = m;
                tb[2 * kMaxLandmarks + t] = s_tc[t];
                reinterpret_cast<float*>(tb + 3 * kMaxLandmarks)[t] = s_up[t];
            }
        }
        __syncthreads();
    }
    float up[kMaxLandmarks];  // landmarks 1 .. L-1 in registers (unused slots never compare true)
    if (!EXACT) {
#pragma unroll
        for (int t = 1; t < kMaxLandmarks; ++t) up[t] = t < L ? s_up[t] : __int_as_float(0x7f800000);
    }
    double osum = 0.0;
    auto map = [&](float v) {
        if (EXACT) {
            int j1, j2;
            const double mid = np_interp(static_cast<double>(v), s_orig, s_origf, s_avg, s_slope1, L, -1, j1);
            return static_cast<float>(np_interp(mid, s_avg, s_avgf, s_std, s_slope2, L, j1, j2));
        }
        int j = 0;  // largest j with orig[j] <= v (0 below the first landmark)
#pragma unroll
        for (int t = 1; t < kMaxLandmarks; ++t) j += (v >= up[t]) ? 1 : 0;
        const double d = static_cast<double>(v) - s_orig[j];
        const float o = static_cast<float>(fma(s_tm[j], d > 0.0 ? d : 0.0, s_tc[j]));
        return v != v ? v : o;
    };
    if (plane_mean == nullptr && dst == nullptr) return;  // tables only
    if (NREG > 0) {  // the plane sits in the caller's registers: sample tid + k * blockDim.x is vreg[k]
#pragma unroll
        for (int k = 0; k < NREG; ++k) {
            const int i = tid + k * static_cast<int>(blockDim.x);
            if (i < n) {
                const float o = map(vreg[k]);
                osum += static_cast<double>(o);
                if (dst != nullptr) __stcs(dst + i, o);
            }
        }
    } else if (gsrc != nullptr && (n & 3) == 0 && ((reinterpret_cast<uintptr_t>(gsrc) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0) {
        // plane read straight from global / L2: 16-byte loads and stores, four independent interpolations per trip
        for (int i = tid; i < (n >> 2); i += blockDim.x) {
            const float4 q4 = __ldg(reinterpret_cast<const float4*>(gsrc) + i);
            const float4 o = make_float4(map(q4.x), map(q4.y), map(q4.z), map(q4.w));
            osum += (static_cast<double>(o.x) + static_cast<double>(o.y)) + (static_cast<double>(o.z) + static_cast<double>(o.w));
            if (dst != nullptr) __stcs(reinterpret_cast<float4*>(dst) + i, o);
        }
    } else {
        for (int i = tid; i < n; i += blockDim.x) {
            const float o = map(load(i));
            osum += static_cast<double>(o);
            if (dst != nullptr) __stcs(dst + i, o);
        }
    }
    if (plane_mean != nullptr) {
        const double om = block_sum<double>(osum, scratch);
        if (tid == 0) plane_mean[plane] = static_cast<float>(om / n);
    }
}

// One CTA per (case, channel) plane.  The 2L order statistics numpy's "linear" percentile rule needs are
// found WITHOUT sorting the plane: a monotone linear binning of [min, max] into 4096 bins, an exclusive
// scan, then for each wanted rank the (typically 1-3) samples of its bin are gathered and the in-bin rank
// is resolved by counting.  Monotone binning preserves order, so the selected values are exactly the
// sorted array's entries.  A bin holding more than 64 samples (heavy ties) falls back to a full in-shared-
// memory bitonic sort of the plane.  Interpolation then runs from the shared-memory copy, so the plane is
// read from HBM once and written once.
template <bool EXACT>
__global__ void __launch_bounds__(kNyulThreads)
nyul_transform_kernel(const float* __restrict__ x, float* __restrict__ out, int C, int n, int npad, int L,
                      const double* __restrict__ avg_landmarks,  // [C, L]
                      const double* __restrict__ standard_scale,  // [L]
                      const int* __restrict__ prev_index,         // [L] floor(q*(n-1))
                      const double* __restrict__ gamma,           // [L] fractional part
                      float* __restrict__ plane_mean, double* __restrict__ table_out) {
    extern __shared__ float s_x[];  // npad floats: the plane (later sorted in place on the fallback path)
    __shared__ int s_hist[kNyulBins];
    __shared__ unsigned char s_mark[kNyulBins];
    __shared__ float s_list[kNyulMaxRanks][kNyulListCap];
    __shared__ int s_cnt[kNyulMaxRanks];
    __shared__ int s_rank[kNyulMaxRanks], s_bin[kNyulMaxRanks], s_inbin[kNyulMaxRanks], s_lid[kNyulMaxRanks];
    __shared__ float s_val[kNyulMaxRanks];
    __shared__ int s_flags[2];  // [0] overflow -> sort fallback, [1] number of distinct target bins
    __shared__ float s_red[2 * (kNyulThreads / 32)];
    __shared__ int s_scan[kNyulThreads / 32];
    const int plane = blockIdx.x;
    const int c = plane % C;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float* src = x + static_cast<size_t>(plane) * n;
    float* dst = out != nullptr ? out + static_cast<size_t>(plane) * n : nullptr;
    const int R = 2 * L;

    // ---- load, min / max ----
    float mn = FLT_MAX, mx = -FLT_MAX;
    for (int i = tid; i < npad; i += kNyulThreads) {
        const float v = i < n ? __ldcs(src + i) : FLT_MAX;
        s_x[i] = v;
        if (i < n) {
            mn = fminf(mn, v);
            mx = fmaxf(mx, v);
        }
    }
    for (int i = tid; i < kNyulBins; i += kNyulThreads) {
        s_hist[i] = 0;
        s_mark[i] = 0;
    }
    if (tid < kNyulMaxRanks) s_cnt[tid] = 0;
    if (tid < 2) s_flags[tid] = 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if (lane == 0) {
        s_red[warp] = mn;
        s_red[kNyulThreads / 32 + warp] = mx;
    }
    __syncthreads();
    mn = s_red[0];
    mx = s_red[kNyulThreads / 32];
    for (int w = 1; w < kNyulThreads / 32; ++w) {
        mn = fminf(mn, s_red[w]);
        mx = fmaxf(mx, s_red[kNyulThreads / 32 + w]);
    }
    const float range = mx - mn;
    const float inv = range > 0.f ? static_cast<float>(kNyulBins) / range : 0.f;
    auto bin_of = [&](float v) { return min(kNyulBins - 1, static_cast<int>((v - mn) * inv)); };

    // ---- histogram + exclusive scan (s_hist becomes the count of samples in lower bins) ----
    for (int i = tid; i < n; i += kNyulThreads) atomicAdd(&s_hist[bin_of(s_x[i])], 1);
    __syncthreads();
    {
        constexpr int kPer = kNyulBins / kNyulThreads;  // 8 consecutive bins per thread
        int local[kPer], sum = 0;
#pragma unroll
        for (int k = 0; k < kPer; ++k) {
            local[k] = s_hist[tid * kPer + k];
            sum += local[k];
        }
        int incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) s_scan[warp] = incl;
        __syncthreads();
        int base = 0;
        for (int w = 0; w < warp; ++w) base += s_scan[w];
        int run = base + incl - sum;
#pragma unroll
        for (int k = 0; k < kPer; ++k) {
            s_hist[tid * kPer + k] = run;
            run += local[k];
        }
    }
    __syncthreads();
    // ---- locate the bin of every wanted rank ----
    if (tid < R) {
        const int l = tid >> 1;
        const int lo = prev_index[l];
        const int rank = (tid & 1) ? min(lo + 1, n - 1) : lo;
        int a = 0, bnd = kNyulBins - 1;  // last bin whose exclusive prefix is <= rank
        while (a < bnd) {
            const int mid = (a + bnd + 1) >> 1;
            if (s_hist[mid] <= rank) a = mid;
            else bnd = mid - 1;
        }
        s_rank[tid] = rank;
        s_bin[tid] = a;
        s_inbin[tid] = rank - s_hist[a];
    }
    __syncthreads();
    if (warp == 0) {  // distinct target bins -> candidate lists (one lane per target)
        const bool on = lane < R;
        const int mybin = on ? s_bin[lane] : -1 - lane;
        int first = lane;
        for (int u = 0; u < R; ++u) {
            const int bu = __shfl_sync(0xffffffffu, mybin, u);
            if (on && u < first && bu == mybin) first = u;
        }
        const unsigned leaders = __ballot_sync(0xffffffffu, on && first == lane);
        const int id = __popc(leaders & ((1u << first) - 1u));
        if (on) s_lid[lane] = id;
        if (on && first == lane) s_mark[mybin] = static_cast<unsigned char>(id + 1);
        if (lane == 0) s_flags[1] = __popc(leaders);
    }
    __syncthreads();
    for (int i = tid; i < n; i += kNyulThreads) {
        const float v = s_x[i];
        const int m = s_mark[bin_of(v)];
        if (m != 0) {
            const int pos = atomicAdd(&s_cnt[m - 1], 1);
            if (pos < kNyulListCap) s_list[m - 1][pos] = v;
            else s_flags[0] = 1;
        }
    }
    __syncthreads();
    const bool fallback = s_flags[0] != 0;
    if (!fallback) {
        // in-bin rank by counting: the wanted value e has (#smaller) <= r < (#smaller + #equal)
        for (int t = warp; t < R; t += kNyulThreads / 32) {
            const int id = s_lid[t], m = s_cnt[id], r = s_inbin[t];
            for (int j = lane; j < m; j += 32) {
                const float e = s_list[id][j];
                int less = 0, eq = 0;
                for (int k = 0; k < m; ++k) {
                    const float f = s_list[id][k];
                    less += f < e;
                    eq += f == e;
                }
                if (less <= r && r < less + eq) s_val[t] = e;
            }
        }
    } else {
        // Bitonic sort of the padded plane, ascending (padding = FLT_MAX sorts to the end).
        for (int k = 2; k <= npad; k <<= 1) {
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int t = tid; t < (npad >> 1); t += kNyulThreads) {
                    const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));  // index with bit j clear
                    const int l2 = i | j;
                    const bool up = (i & k) == 0;
                    const float a = s_x[i], b2 = s_x[l2];
                    if ((a > b2) == up) {
                        s_x[i] = b2;
                        s_x[l2] = a;
                    }
                }
                __syncthreads();
            }
        }
        if (tid < R) s_val[tid] = s_x[s_rank[tid]];
    }
    __syncthreads();
    // the sort fallback permuted the shared copy: re-read the plane (an L2 hit) on that path only
    nyul_apply<EXACT>(s_val, L, c, n, plane, avg_landmarks, standard_scale, gamma,
                      [&](int i) { return fallback ? src[i] : s_x[i]; }, dst, plane_mean, nullptr, table_out);
}

// Planes too large to stage in shared memory (224 x 224 after the C4 resize = 50 176 samples): the 2L order
// statistics come from an exact radix select on the order-preserving integer image of the floats - four passes
// of 8 bits over the plane (L2-resident after the first), one 256-bin histogram per distinct key prefix still
// alive (at most 2L), warp-aggregated shared-memory atomics so that heavy ties (a zero background) cost one
// atomic per warp.  Bitwise exact by construction, no distribution assumptions, no fallback.
__device__ __forceinline__ uint32_t nyul_ordkey(float v) {
    const uint32_t u = __float_as_uint(v);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float nyul_ordkey_inv(uint32_t k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

template <bool EXACT>
__global__ void __launch_bounds__(kNyulThreads)
nyul_transform_large_kernel(const float* __restrict__ x, float* __restrict__ out, int C, int n, int L,
                            const double* __restrict__ avg_landmarks, const double* __restrict__ standard_scale,
                            const int* __restrict__ prev_index, const double* __restrict__ gamma,
                            float* __restrict__ plane_mean, double* __restrict__ table_out) {
    __shared__ int s_hist[kNyulMaxRanks][256];
    __shared__ uint32_t s_prefix[kNyulMaxRanks], s_uprefix[kNyulMaxRanks];
    __shared__ int s_rem[kNyulMaxRanks], s_uid[kNyulMaxRanks];
    __shared__ int s_nu;
    __shared__ float s_val[kNyulMaxRanks];
    // alive-prefix lookup of the current pass: last digit of a prefix -> first alive prefix id carrying it, then a
    // chain through the ids that share that digit (one LDS for the samples that match nothing, i.e. most of them
    // from the third pass on, instead of a scan over all <= 2L prefixes)
    __shared__ int s_lut[256], s_chain[kNyulMaxRanks];
    const int plane = blockIdx.x;
    const int c = plane % C;
    const int tid = threadIdx.x, lane = tid & 31;
    const float* src = x + static_cast<size_t>(plane) * n;
    float* dst = out != nullptr ? out + static_cast<size_t>(plane) * n : nullptr;
    const int R = 2 * L;
    if (tid < R) {
        const int lo = prev_index[tid >> 1];
        s_rem[tid] = (tid & 1) ? min(lo + 1, n - 1) : lo;
        s_prefix[tid] = 0u;
        s_uid[tid] = 0;
    }
    if (tid == 0) {
        s_nu = 1;
        s_uprefix[0] = 0u;
    }
    __syncthreads();
    for (int pass = 0; pass < 4; ++pass) {
        const int shift = 24 - 8 * pass;
        const int nu = s_nu;
        for (int i = tid; i < nu * 256; i += kNyulThreads) (&s_hist[0][0])[i] = 0;
        if (tid < 256) s_lut[tid] = -1;
        __syncthreads();
        if (pass != 0) {
            if (tid == 0) {
                for (int q = nu - 1; q >= 0; --q) {
                    const int d = static_cast<int>(s_uprefix[q] & 255u);
                    s_chain[q] = s_lut[d];
                    s_lut[d] = q;
                }
            }
            __syncthreads();
        }
        // four samples per thread and trip (one 16-byte load when the plane allows it): the passes are bound by the
        // L2 round trip of the load, not by arithmetic
        const bool vec = (n & 3) == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0;
        const int n_trip = (n + 4 * kNyulThreads - 1) / (4 * kNyulThreads);  // whole warps stay converged
        for (int t = 0; t < n_trip; ++t) {
            const int i0 = (t * kNyulThreads + tid) * 4;
            float f[4];
            if (vec && i0 + 3 < n) {
                const float4 q4 = __ldg(reinterpret_cast<const float4*>(src + i0));
                f[0] = q4.x; f[1] = q4.y; f[2] = q4.z; f[3] = q4.w;
            } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) f[e] = i0 + e < n ? __ldg(src + i0 + e) : 0.f;
            }
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                int slot = -1;
                if (i0 + e < n) {
                    const uint32_t key = nyul_ordkey(f[e]);
                    int u = 0;
                    if (pass != 0) {
                        const uint32_t hi = key >> (shift + 8);
                        u = s_lut[hi & 255u];
                        while (u >= 0 && s_uprefix[u] != hi) u = s_chain[u];
                    }
                    if (u >= 0) slot = u * 256 + static_cast<int>((key >> shift) & 255u);
                }
                // Histogram update.  Two rounds of warp aggregation (the lowest active lane's slot, everybody who
                // shares it, one atomic for the group) catch the heavy ties - a zero background puts most of a warp
                // on one slot - and whoever is left adds individually: distinct slots do not contend.
                uint32_t active = __ballot_sync(0xffffffffu, slot >= 0);
#pragma unroll
                for (int round = 0; round < 2; ++round) {
                    if (active == 0u) break;  // warp-uniform
                    const int leader = __ffs(active) - 1;
                    const int s0 = __shfl_sync(0xffffffffu, slot, leader);
                    const uint32_t same = __ballot_sync(0xffffffffu, slot == s0) & active;
                    if (lane == leader) atomicAdd(&(&s_hist[0][0])[s0], __popc(same));
                    active &= ~same;
                }
                if ((active >> lane) & 1u) atomicAdd(&(&s_hist[0][0])[slot], 1);
            }
        }
        __syncthreads();
        if (tid < R) {
            const int* h = s_hist[s_uid[tid]];
            int rem = s_rem[tid], d = 0;
            for (; d < 255; ++d) {
                const int cnt = h[d];
                if (rem < cnt) break;
                rem -= cnt;
            }
            s_rem[tid] = rem;
            s_prefix[tid] = (s_prefix[tid] << 8) | static_cast<uint32_t>(d);
        }
        __syncthreads();
        if (tid < 32) {  // distinct prefixes still alive -> one histogram each in the next pass (one lane per rank)
            const bool on = lane < R;
            const uint32_t mine = on ? s_prefix[lane] : 0u;
            int first = lane;
            for (int u = 0; u < R; ++u) {
                const uint32_t pu = __shfl_sync(0xffffffffu, mine, u);
                if (on && u < first && pu == mine) first = u;
            }
            const unsigned leaders = __ballot_sync(0xffffffffu, on && first == lane);
            const int id = __popc(leaders & ((1u << first) - 1u));
            if (on) s_uid[lane] = id;
            if (on && first == lane) s_uprefix[id] = mine;
            if (lane == 0) s_nu = __popc(leaders);
        }
        __syncthreads();
    }
    if (tid < R) s_val[tid] = nyul_ordkey_inv(s_prefix[tid]);
    __syncthreads();
    nyul_apply<EXACT>(s_val, L, c, n, plane, avg_landmarks, standard_scale, gamma, [&](int i) { return __ldg(src + i); },
                      dst, plane_mean, src, table_out);
}

// ADC map (reference preprocess_helpers.py:133-167): per pixel, minus the least-squares slope of log(max(S, eps))
// over the b-values: adc = -sum_c (b_c - mean b)(log S_c - mean log S) / (sum_c (b_c - mean b)^2 + eps).
// One thread per pixel, the C planes read with unit stride across threads; C <= 32.
__global__ void __launch_bounds__(kNormThreads)
adc_map_kernel(const float* __restrict__ x, const float* __restrict__ bvals, int C, int n, float eps,
               float* __restrict__ out, size_t total) {
    __shared__ float s_db[32];
    __shared__ float s_inv_var;
    if (threadIdx.x == 0) {
        float mb = 0.f;
        for (int c = 0; c < C; ++c) mb += bvals[c];
        mb /= C;
        float var = 0.f;
        for (int c = 0; c < C; ++c) {
            s_db[c] = bvals[c] - mb;
            var += s_db[c] * s_db[c];
        }
        s_inv_var = 1.0f / (var + eps);
    }
    __syncthreads();
    const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
    if (i >= total) return;
    const size_t b = i / n;
    const int pix = static_cast<int>(i - b * n);
    const float* src = x + b * static_cast<size_t>(C) * n + pix;
    float ls[32];
    float mean = 0.f;
#pragma unroll 8
    for (int c = 0; c < C; ++c) {
        ls[c] = logf(fmaxf(__ldg(src + static_cast<size_t>(c) * n), eps));
        mean += ls[c];
    }
    mean /= C;
    float cov = 0.f;
    for (int c = 0; c < C; ++c) cov += s_db[c] * (ls[c] - mean);
    out[i] = -(cov * s_inv_var);
}

__global__ void __launch_bounds__(kNormThreads)
plane_mean_kernel(const float* __restrict__ x, int n, float* __restrict__ plane_mean) {
    __shared__ double scratch[33];
    const float* src = x + static_cast<size_t>(blockIdx.x) * n;
    double s = 0.0;
    for (int i = threadIdx.x; i < n; i += kNormThreads) s += static_cast<double>(src[i]);
    const double t = block_sum<double>(s, scratch);
    if (threadIdx.x == 0) plane_mean[blockIdx.x] = static_cast<float>(t / n);
}

}  // namespace b200

extern "C" int b200_dwi_normalize_ex(const float* x, float* out, int planes, int C, int n, int skip_last, float z_lo,
                                     float z_hi, float* plane_mean, float* stats_out, void* stream) {
    using namespace b200;
    if (planes < 0 || C <= 0 || n <= 0 || planes % C != 0) return -1;
    if (planes == 0) return 0;
    if (x == nullptr || (out == nullptr && stats_out == nullptr)) return -2;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const bool aligned = (n % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0) &&
                         ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
    if ((out == nullptr || stats_out != nullptr) && !(aligned && n <= kNormThreads * 4 * 8)) return -3;  // statistics-only
    // mode exists for register-resident planes (<= 8 192 samples, 16-byte aligned): the ROI sizes of the CNN encoders
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
    }
    // persistent grid = resident CTAs (64 / 114 registers per thread -> 4 / 2 CTAs of 256 threads per SM)
    // With skip_last every C-th plane is a zero fill (half the traffic, no read).  Planes are dealt round-robin, so a
    // grid sharing a factor with C (592 = 16 * 37) would hand some CTAs nothing but cheap planes and leave the rest
    // 4-5 % more work than the average: make the grid coprime with C.
    auto coprime_grid = [&](int g) {
        if (!skip_last || g >= planes) return g < planes ? g : planes;
        auto gcd = [](int a, int b) { while (b) { const int t = a % b; a = b; b = t; } return a; };
        while (g > 1 && gcd(g, C) != 1) --g;
        return g;
    };
    int grid = coprime_grid(sms * 4);
    if (aligned && n <= kNormThreads * 4 * 4)
        dwi_normalize_reg_kernel<4><<<grid, kNormThreads, 0, s>>>(x, out, planes, C, n, skip_last, z_lo, z_hi,
                                                                  plane_mean, stats_out);
    else if (aligned && n <= kNormThreads * 4 * 8)
        dwi_normalize_reg_kernel<8><<<(grid = coprime_grid(sms * 2)), kNormThreads, 0, s>>>(x, out, planes, C, n, skip_last, z_lo, z_hi,
                                                                  plane_mean, stats_out);
    else
        dwi_normalize_stream_kernel<<<planes, kNormThreads, 0, s>>>(x, out, C, n, skip_last, z_lo, z_hi, plane_mean);
    return launch_status();
}

extern "C" int b200_dwi_normalize(const float* x, float* out, int planes, int C, int n, int skip_last, float z_lo,
                                  float z_hi, float* plane_mean, void* stream) {
    if (out == nullptr && planes > 0) return -2;
    return b200_dwi_normalize_ex(x, out, planes, C, n, skip_last, z_lo, z_hi, plane_mean, nullptr, stream);
}

namespace b200 {
template <bool EXACT>
static int nyul_launch(const float* x, float* out, int planes, int C, int n, int L, const double* avg_landmarks,
                       const double* standard_scale, const int* prev_index, const double* gamma, float* plane_mean,
                       double* table_out, cudaStream_t stream) {
    int npad = 2;
    while (npad < n) npad <<= 1;
    const size_t smem = static_cast<size_t>(npad) * sizeof(float);
    static const bool force_large = std::getenv("B200_NYUL_LARGE") != nullptr;  // test hook
    if (smem > 128 * 1024 || force_large) {  // > 32 768 samples: radix select straight from global / L2
        nyul_transform_large_kernel<EXACT><<<planes, kNyulThreads, 0, stream>>>(
            x, out, C, n, L, avg_landmarks, standard_scale, prev_index, gamma, plane_mean, table_out);
        return launch_status();
    }
    static size_t configured = 0;
    if (smem > 48 * 1024 && smem > configured) {
        cudaError_t e = cudaFuncSetAttribute(nyul_transform_kernel<EXACT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             static_cast<int>(smem));
        if (e != cudaSuccess) return static_cast<int>(e);
        configured = smem;
    }
    nyul_transform_kernel<EXACT><<<planes, kNyulThreads, smem, stream>>>(
        x, out, C, n, npad, L, avg_landmarks, standard_scale, prev_index, gamma, plane_mean, table_out);
    return launch_status();
}
}  // namespace b200

extern "C" int b200_nyul_transform_ex2(const float* x, float* out, int planes, int C, int n, int L,
                                       const double* avg_landmarks, const double* standard_scale, const int* prev_index,
                                       const double* gamma, float* plane_mean, int exact, double* table_out, void* stream) {
    using namespace b200;
    if (planes < 0 || C <= 0 || n <= 0 || planes % C != 0 || L < 2 || L > kMaxLandmarks) return -1;
    if (planes == 0) return 0;
    if (x == nullptr || avg_landmarks == nullptr || standard_scale == nullptr || prev_index == nullptr || gamma == nullptr)
        return -2;
    if (out == nullptr && table_out == nullptr) return -2;
    if (table_out != nullptr && exact) return -3;  // the per-plane table IS the composed (fast) form
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    return exact ? nyul_launch<true>(x, out, planes, C, n, L, avg_landmarks, standard_scale, prev_index, gamma, plane_mean,
                                     nullptr, s)
                 : nyul_launch<false>(x, out, planes, C, n, L, avg_landmarks, standard_scale, prev_index, gamma,
                                      plane_mean, table_out, s);
}

extern "C" int b200_nyul_transform_ex(const float* x, float* out, int planes, int C, int n, int L,
                                      const double* avg_landmarks, const double* standard_scale, const int* prev_index,
                                      const double* gamma, float* plane_mean, int exact, void* stream) {
    if (out == nullptr) return -2;
    return b200_nyul_transform_ex2(x, out, planes, C, n, L, avg_landmarks, standard_scale, prev_index, gamma, plane_mean,
                                   exact, nullptr, stream);
}

extern "C" int b200_plane_mean(const float* x, int planes, int n, float* plane_mean, void* stream) {
    using namespace b200;
    if (planes < 0 || n <= 0) return -1;
    if (planes == 0) return 0;
    if (x == nullptr || plane_mean == nullptr) return -2;
    plane_mean_kernel<<<planes, kNormThreads, 0, static_cast<cudaStream_t>(stream)>>>(x, n, plane_mean);
    return launch_status();
}

extern "C" int b200_adc_map(const float* x, int B, int C, int n, const float* bvals, float eps, float* out, void* stream) {
    using namespace b200;
    if (B < 0 || C <= 0 || C > 32 || n <= 0) return -1;
    if (B == 0) return 0;
    if (x == nullptr || bvals == nullptr || out == nullptr) return -2;
    const size_t total = static_cast<size_t>(B) * n;
    adc_map_kernel<<<static_cast<unsigned>((total + kNormThreads - 1) / kNormThreads), kNormThreads, 0,
                     static_cast<cudaStream_t>(stream)>>>(x, bvals, C, n, eps, out, total);
    return launch_status();
}

// DCE pre-scale of prep_data_by_mod (reference prepare_single_model.py:337-343): every case divided by its maximum over
// all channels and pixels.  One CTA per case: a max reduction over the case (which then sits in L2), then the IEEE
// division per element, exactly what torch's `imgs / imgs_max` computes.
namespace b200 {
__global__ void __launch_bounds__(kNormThreads)
case_max_scale_kernel(const float* __restrict__ x, long long n, float* __restrict__ out) {
    __shared__ float s_red[kNormThreads / 32];
    const float* src = x + static_cast<long long>(blockIdx.x) * n;
    float* dst = out + static_cast<long long>(blockIdx.x) * n;
    const bool vec = (n & 3) == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0;
    float m = -FLT_MAX;
    if (vec) {
        for (long long i = threadIdx.x; i < (n >> 2); i += kNormThreads) {
            const float4 q = __ldg(reinterpret_cast<const float4*>(src) + i);
            m = fmaxf(m, fmaxf(fmaxf(q.x, q.y), fmaxf(q.z, q.w)));
        }
    } else {
        for (long long i = threadIdx.x; i < n; i += kNormThreads) m = fmaxf(m, __ldg(src + i));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = m;
    __syncthreads();
    m = s_red[0];
    for (int w = 1; w < kNormThreads / 32; ++w) m = fmaxf(m, s_red[w]);
    if (vec) {
        for (long long i = threadIdx.x; i < (n >> 2); i += kNormThreads) {
            const float4 q = __ldg(reinterpret_cast<const float4*>(src) + i);
            __stcs(reinterpret_cast<float4*>(dst) + i, make_float4(__fdiv_rn(q.x, m), __fdiv_rn(q.y, m), __fdiv_rn(q.z, m), __fdiv_rn(q.w, m)));
        }
    } else {
        for (long long i = threadIdx.x; i < n; i += kNormThreads) dst[i] = __fdiv_rn(__ldg(src + i), m);
    }
}
}  // namespace b200

extern "C" int b200_case_max_scale(const float* x, int B, long long n, float* out, void* stream) {
    using namespace b200;
    if (B < 0 || n <= 0) return -1;
    if (B == 0) return 0;
    if (x == nullptr || out == nullptr) return -2;
    case_max_scale_kernel<<<B, kNormThreads, 0, static_cast<cudaStream_t>(stream)>>>(x, n, out);
    return launch_status();
}
