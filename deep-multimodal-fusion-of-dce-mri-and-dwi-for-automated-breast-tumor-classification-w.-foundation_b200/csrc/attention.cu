// Fused multi-head self-attention for sm_100a: softmax(q k^T / sqrt(d)) v in ONE launch, nothing but the packed qkv
// rows read and the head outputs written (no score / probability buffer, no transposed V in HBM).
//
// Reference: MultiHeadSelfAttention.forward, transformer_model.py:98-116 (hybrid stage: 256 tokens, 4 heads x 128) and
// the timm ViT-B/16 attention the backbone runs (foundation_model.py:371-431: 197 tokens, 12 heads x 64).  Both feed
// `qkv = Linear(E, 3E)(x).reshape(B, N, 3, heads, d)`, i.e. row (b, n) of the qkv buffer holds q | k | v, each
// [heads, d] - exactly what the TMA boxes below pick apart.
//
// This kernel (attn_fused_kernel) serves N <= 256; attn_long_kernel below streams the keys for 256 < N <= 16384.
// One work item = (case, head, 128-query tile); persistent CTAs, 160 threads:
//   warp 4 (one elected lane)  TMA: Q box {64, 128} and K box {64, 256} per 64-wide slice of d (128-byte swizzle,
//                              K-major operands), V box {64, 256} (the same rows, used MN-major: keys are the MMA's
//                              K dimension, d its N); rows past the case's N tokens arrive as zeros (OOB fill).
//                              MMA 1: S[128, 256] = Q K^T into 256 TMEM columns.  MMA 2: O[128, d] = P V over the
//                              ceil(N / 16) key steps that hold real keys, into the first d columns of the same TMEM
//                              allocation (S is dead once P is written).
//   warps 0-3                  one query row per thread (TMEM lane = row): p = 2^((s - ref) * scale * log2 e) -> bf16
//                              -> shared memory in the swizzled K-major layout MMA 2 reads (P overwrites the Q / K
//                              staging area, free since MMA 1 retired), fp32 row sum; then O * (1 / sum) -> bf16 ->
//                              global.  Scores are read out of TMEM once (see softmax_rows).
// d = 64: 96 KB of shared memory and 256 TMEM columns per CTA, two CTAs per SM so one CTA's softmax overlaps the
// other's loads and MMAs.  d = 128: 160 KB, one CTA per SM.
//
// Measured (B = 256 cases of ViT-B/16: 197 tokens, 12 heads x 64): 126 us per launch = 243 TFLOP/s of 4 N^2 d flops,
// 2.46 TB/s of algorithmic bytes.  The stall samples put the softmax warps 40 % of the time on the two MMA barriers:
// with 512 TMEM columns per SM only two such CTAs fit, so the chain load -> MMA 1 -> softmax -> MMA 2 -> store of a
// work item is covered by one other CTA only.  (A one-CTA-per-SM variant holding both query tiles of a head with K / V
// loaded once and the scores split over 8 warps was measured slower: 203 us.)
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cstdint>

#include "b200_fusion.h"
#include "common.cuh"
#include "ptx.cuh"

namespace b200 {

constexpr int kAtThreads = 160;
constexpr int kAtQBox = 128 * 128;   // Q box: 128 rows x 128 B
constexpr int kAtKBox = 256 * 128;   // K / V box: 256 rows x 128 B
constexpr int kAtPBytes = 4 * kAtQBox;  // P: four 64-key slices of [128 rows x 128 B]

struct AttnParams {
    int N, heads, B, q_tiles, n_items;
    int n_chunks;  // ceil(N / 32): 32-column score chunks holding real keys
    int k_steps;   // ceil(N / 16): MMA 2 key steps
    int out_ld;
    float scale_log2;  // scale * log2(e)
    __nv_bfloat16* out;
    // attention dropout (DROP = true only): probability (case b, head h, query row, key j) is dropped when word j % 4
    // of Philox4x32-7(seed; ((b * heads + h) * N + row) * 64 * ceil(N / 256) + j / 4) < drop_thresh (a 64-bit counter;
    // the row stride is 64 for every N <= 256, so each row owns counters of its own at any N)
    unsigned int drop_thresh;
    float drop_scale;  // 1 / (1 - p), folded into the row's 1 / sum
    unsigned int drop_seed_lo, drop_seed_hi;
};

__device__ __forceinline__ uint64_t at_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
    d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;  // next 64-wide group of the MN dimension
    d |= static_cast<uint64_t>(1024 >> 4) << 32;                   // next 8 rows of the K dimension
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(2) << 61;
    return d;
}

// 32 scores of one row -> probabilities (unnormalised), stored as bf16 in the row's four 16-byte pieces of the
// swizzled [128 x 128 B] slice; returns their fp32 sum.  MASK: columns >= valid are past the case's last key -> 0.
// DROP: the sum is that of the undropped probabilities (the softmax denominator); dropped ones are stored as 0.
// `ctr` is the Philox counter of the chunk's first four keys (see AttnParams).
template <bool MASK, bool DROP>
__device__ __forceinline__ float softmax_chunk(const uint32_t (&v)[32], float scale_log2, float mneg, int valid,
                                               uint8_t* dst, int j0, int swz, const AttnParams& p,
                                               unsigned long long ctr) {
    uint32_t pk[16];
    float s4[4] = {0.f, 0.f, 0.f, 0.f};
    uint4 rnd = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
    for (int i = 0; i < 32; i += 2) {
        float e0 = ex2_approx(fmaf(__uint_as_float(v[i]), scale_log2, mneg));
        float e1 = ex2_approx(fmaf(__uint_as_float(v[i + 1]), scale_log2, mneg));
        if (MASK) {
            if (i >= valid) e0 = 0.f;
            if (i + 1 >= valid) e1 = 0.f;
        }
        s4[(i >> 1) & 3] += e0 + e1;
        if (DROP) {
            if ((i & 3) == 0) rnd = philox4x32_7(ctr + (i >> 2), p.drop_seed_lo, p.drop_seed_hi);
            const uint32_t r0 = (i & 3) == 0 ? rnd.x : rnd.z, r1 = (i & 3) == 0 ? rnd.y : rnd.w;
            if (r0 < p.drop_thresh) e0 = 0.f;
            if (r1 < p.drop_thresh) e1 = 0.f;
        }
        const __nv_bfloat162 t = __floats2bfloat162_rn(e0, e1);
        pk[i >> 1] = *reinterpret_cast<const uint32_t*>(&t);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
        *reinterpret_cast<uint4*>(dst + (((j0 + j) ^ swz) << 4)) =
            make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
    return (s4[0] + s4[1]) + (s4[2] + s4[3]);
}

// One query row per thread: scores S[row, 0:N] in TMEM (lane = row) -> unnormalised probabilities as bf16 into the
// swizzled K-major slices of `s_p`; returns 1 / (fp32 row sum), times 1 / (1 - p) with DROP.  `ctr` = Philox counter
// of the row's keys 0-3 (DROP only).
//
// Reading the scores back out of TMEM (64 B/clk per SM) is what bounds this kernel, so the common case reads them
// ONCE: the reference point of the exponent is the max of the row's first 32 scores, not the row max.  Softmax is
// invariant to that choice (numerator and denominator carry the same factor, and bf16 / fp32 keep their relative
// precision at any exponent); the true max is >= the reference, so nothing underflows, and overflow shows up as a
// row sum that is not < 1e30 - any such row (scores rising by more than ~100 * ln 2 past the first chunk; not seen
// on trained or random weights) sends its warp through the classic two-pass softmax instead.
template <bool DROP>
__device__ __forceinline__ float softmax_rows(uint32_t taddr, uint8_t* s_p, int r, const AttnParams& p,
                                              unsigned long long ctr) {
    const int swz = r & 7;
    float sum = 0.f;
    {
        uint32_t v[32];
        tmem_ld_32x32(taddr, v);
        tmem_ld_wait32(v);
        float m4[4] = {-3.0e38f, -3.0e38f, -3.0e38f, -3.0e38f};
        const int valid0 = p.N;
#pragma unroll
        for (int i = 0; i < 32; ++i)
            if (i < valid0) m4[i & 3] = fmaxf(m4[i & 3], __uint_as_float(v[i]));
        const float mneg = -fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3])) * p.scale_log2;
        for (int c = 0; c < p.n_chunks; ++c) {
            if (c != 0) {
                tmem_ld_32x32(taddr + c * 32, v);
                tmem_ld_wait32(v);
            }
            const int valid = p.N - c * 32;
            uint8_t* const dst = s_p + (c >> 1) * kAtQBox + r * 128;
            const int j0 = (c & 1) * 4;
            if (valid >= 32)
                sum += softmax_chunk<false, DROP>(v, p.scale_log2, mneg, valid, dst, j0, swz, p, ctr + c * 8);
            else
                sum += softmax_chunk<true, DROP>(v, p.scale_log2, mneg, valid, dst, j0, swz, p, ctr + c * 8);
        }
    }
    if (__any_sync(0xffffffffu, !(sum < 1.0e30f))) {  // overflow of the lazy reference somewhere in this warp
        float m4[4] = {-3.0e38f, -3.0e38f, -3.0e38f, -3.0e38f};
        for (int c = 0; c < p.n_chunks; ++c) {
            uint32_t v[32];
            tmem_ld_32x32(taddr + c * 32, v);
            tmem_ld_wait32(v);
            const int valid = p.N - c * 32;
#pragma unroll
            for (int i = 0; i < 32; ++i)
                if (i < valid) m4[i & 3] = fmaxf(m4[i & 3], __uint_as_float(v[i]));
        }
        const float mneg = -fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3])) * p.scale_log2;
        sum = 0.f;
        for (int c = 0; c < p.n_chunks; ++c) {
            uint32_t v[32];
            tmem_ld_32x32(taddr + c * 32, v);
            tmem_ld_wait32(v);
            const int valid = p.N - c * 32;
            uint8_t* const dst = s_p + (c >> 1) * kAtQBox + r * 128;
            sum += softmax_chunk<true, DROP>(v, p.scale_log2, mneg, valid, dst, (c & 1) * 4, swz, p, ctr + c * 8);
        }
    }
    return (DROP ? p.drop_scale : 1.0f) / sum;
}

// O[row, 0:DH] in TMEM -> * inv_sum -> bf16 -> dst (the row's DH contiguous outputs); `store` = the row is a real query.
template <int DH>
__device__ __forceinline__ void store_rows(uint32_t taddr, __nv_bfloat16* dst, bool store, float inv_sum) {
#pragma unroll
    for (int c = 0; c < DH / 32; ++c) {
        uint32_t v[32];
        tmem_ld_32x32(taddr + c * 32, v);
        tmem_ld_wait32(v);
        if (store) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                uint32_t w[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const __nv_bfloat162 t = __floats2bfloat162_rn(__uint_as_float(v[8 * j + 2 * i]) * inv_sum,
                                                                   __uint_as_float(v[8 * j + 2 * i + 1]) * inv_sum);
                    w[i] = *reinterpret_cast<const uint32_t*>(&t);
                }
                *reinterpret_cast<uint4*>(dst + c * 32 + j * 8) = make_uint4(w[0], w[1], w[2], w[3]);
            }
        }
    }
}

template <int DH, bool DROP>
__global__ void __launch_bounds__(kAtThreads, DH == 64 ? 2 : 1)
attn_fused_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmKV, const AttnParams p) {
    constexpr int KC = DH / 64;
    constexpr int kQKBytes = KC * (kAtQBox + kAtKBox);
    constexpr int kRegionA = kQKBytes > kAtPBytes ? kQKBytes : kAtPBytes;
    constexpr int kVBytes = KC * kAtKBox;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (static_cast<uint32_t>(__cvta_generic_to_shared(smem_raw)) & 1023u)) & 1023u);
    uint8_t* const s_q = smem;                    // KC x [128 x 128 B]
    uint8_t* const s_k = smem + KC * kAtQBox;     // KC x [256 x 128 B]
    uint8_t* const s_p = smem;                    // 4 x [128 x 128 B], aliases Q / K
    uint8_t* const s_v = smem + kRegionA;         // KC x [256 x 128 B]
    uint64_t* const bars = reinterpret_cast<uint64_t*>(smem + kRegionA + kVBytes);
    uint64_t* const bar_qk = bars + 0;
    uint64_t* const bar_v = bars + 1;
    uint64_t* const bar_s = bars + 2;
    uint64_t* const bar_p = bars + 3;
    uint64_t* const bar_o = bars + 4;
    uint64_t* const bar_done = bars + 5;
    uint32_t* const tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        mbar_init(bar_qk, 1);
        mbar_init(bar_v, 1);
        mbar_init(bar_s, 1);
        mbar_init(bar_p, 128);
        mbar_init(bar_o, 1);
        mbar_init(bar_done, 128);
        fence_mbar_init();
    }
    if (warp == 4) {
        if (lane == 0) {
            tma_prefetch_desc(&tmQ);
            tma_prefetch_desc(&tmKV);
        }
        tmem_alloc<256>(tmem_slot);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    uint32_t ph = 0;
    if (warp == 4) {
        if (lane == 0) {
            constexpr uint32_t idesc1 = umma_idesc_bf16(128, 256);
            constexpr uint32_t idesc2 = umma_idesc_bf16(128, DH) | (1u << 16);  // B (= V) is MN-major
            for (int item = blockIdx.x; item < p.n_items; item += gridDim.x, ph ^= 1u) {
                const int qt = item % p.q_tiles;
                const int h = (item / p.q_tiles) % p.heads;
                const int b = item / (p.q_tiles * p.heads);
                if (item != static_cast<int>(blockIdx.x)) {
                    mbar_wait(bar_o, ph ^ 1u);     // MMA 2 of the previous item has read P and V
                }
                const int E = p.heads * DH;
                mbar_arrive_expect_tx(bar_qk, kQKBytes);
#pragma unroll
                for (int kc = 0; kc < KC; ++kc) {
                    tma_load_4d(s_q + kc * kAtQBox, &tmQ, bar_qk, h * DH + kc * 64, qt * 128, b, 0);
                    tma_load_4d(s_k + kc * kAtKBox, &tmKV, bar_qk, E + h * DH + kc * 64, 0, b, 0);
                }
                mbar_arrive_expect_tx(bar_v, kVBytes);
#pragma unroll
                for (int kc = 0; kc < KC; ++kc)
                    tma_load_4d(s_v + kc * kAtKBox, &tmKV, bar_v, 2 * E + h * DH + kc * 64, 0, b, 0);
                if (item != static_cast<int>(blockIdx.x)) {
                    mbar_wait(bar_done, ph ^ 1u);  // the previous item's rows have left TMEM
                }
                mbar_wait(bar_qk, ph);
                tc_fence_after();
#pragma unroll
                for (int kc = 0; kc < KC; ++kc) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const uint64_t da = umma_desc_sw128(smem_u32(s_q + kc * kAtQBox) + k * 32);
                        const uint64_t db = umma_desc_sw128(smem_u32(s_k + kc * kAtKBox) + k * 32);
                        umma_bf16(tmem_base, da, db, idesc1, (kc | k) != 0 ? 1u : 0u);
                    }
                }
                umma_commit(bar_s);
                mbar_wait(bar_v, ph);
                mbar_wait(bar_p, ph);
                tc_fence_after();
                for (int ks = 0; ks < p.k_steps; ++ks) {
                    const uint64_t da = umma_desc_sw128(smem_u32(s_p + (ks >> 2) * kAtQBox) + (ks & 3) * 32);
                    const uint64_t db = at_desc_mn_sw128(smem_u32(s_v) + ks * 2048, kAtKBox);
                    umma_bf16(tmem_base, da, db, idesc2, ks != 0 ? 1u : 0u);
                }
                umma_commit(bar_o);
            }
        }
    } else {
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);
        const int r = warp * 32 + lane;  // row inside the query tile
        for (int item = blockIdx.x; item < p.n_items; item += gridDim.x, ph ^= 1u) {
            const int qt = item % p.q_tiles;
            const int h = (item / p.q_tiles) % p.heads;
            const int b = item / (p.q_tiles * p.heads);
            const int row = qt * 128 + r;
            const bool warp_live = qt * 128 + warp * 32 < p.N;  // some row of this warp is a real query
            mbar_wait(bar_s, ph);
            tc_fence_after();
            unsigned long long ctr = 0;
            if (DROP) ctr = ((static_cast<unsigned long long>(b) * p.heads + h) * p.N + row) * 64;
            const float inv_sum = warp_live ? softmax_rows<DROP>(taddr, s_p, r, p, ctr) : 0.f;
            fence_proxy_async_smem();  // P (generic-proxy stores) -> visible to the MMA's async-proxy reads
            tc_fence_before();
            mbar_arrive(bar_p);
            mbar_wait(bar_o, ph);
            tc_fence_after();
            if (warp_live) store_rows<DH>(taddr, p.out + (static_cast<long long>(b) * p.N + row) * p.out_ld + h * DH,
                                          row < p.N, inv_sum);
            tc_fence_before();
            mbar_arrive(bar_done);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4) {
        tc_fence_after();
        tmem_dealloc<256>(tmem_base);
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// attn_long_kernel<DH, DROP>: the same contract for 256 < N <= kAtLongMaxN, with the keys streamed in 128-key tiles
// through an online softmax.  One work item = (case, head, 128-query tile); persistent CTAs, one per SM, 192 threads:
//   warp 4 (one lane)  TMA: Q box {64, 128} once per item; K and V of key tile j (rows j*128 .. j*128+127 of the case,
//                      the same {64, 128} box) into ring stage j % 2.  Rows past N arrive as zeros (OOB fill).
//   warp 5 (one lane)  allocates 512 TMEM columns: S buffers at columns 0 and 128, O at 256 .. 256+DH.
//                      MMA 1: S[j % 2] = Q K_j^T, issued one tile ahead, so S_{j+1} is computed while the softmax
//                      reads S_j.  MMA 2: O (+)= P_j V_j (V MN-major from its natural layout, as above).
//   warps 0-3          one query row per thread: S_j -> 128 registers (read out of TMEM once), then P_j -> the one
//                      swizzled K-major P buffer, fp32 row sum l; at the end of the item O * (1 / l) -> bf16 -> global.
//
// Ordering (mbarriers; "commit" = tcgen05.commit, which arrives once every earlier MMA of the issuing thread retired):
//   q_full   TMA -> MMA (tx bytes)        q_empty   commit after the item's last MMA 1 -> TMA may load the next Q
//   kv_full  TMA -> MMA (tx bytes)        kv_empty  commit after MMA 2 of the tile -> TMA may refill the stage
//   s_full   commit after MMA 1 -> softmax            s_empty   128 arrivals once S_j is in registers -> MMA 1 of j+2
//   p_full   128 arrivals: P_j stored (fence.proxy.async) and O rescaled (tcgen05.wait::st) -> MMA 2 of tile j
//   o_full   commit after MMA 2 of tile j -> softmax: P free for P_{j+1}, O may be rescaled / read
//   o_empty  128 arrivals once the item's O left TMEM -> first MMA 2 of the next item (which overwrites O)
// Every softmax thread passes every wait, live rows or not, so no thread arrives on a barrier's next phase early.
//
// Online softmax with a lazy, conditionally moved reference m (log2 units, per row): m starts at the max of the first
// key tile; a later tile moves it only when its max exceeds m by more than kAtRescaleLog2 (tau), and then l and the
// row of O are scaled by 2^(m_old - m_new) (O through tcgen05.ld / st, after o_full of the previous tile).  Otherwise
// the exponents stay <= 2^tau: harmless in fp32 l and bf16 P.  Scores rising slowly never pay for a rescale.
//
// Shared memory: Q KC x 16 KB + 2 stages x (K + V) KC x 16 KB + P 32 KB = 192 KB at d = 128, 112 KB at d = 64.  At
// d = 64 one CTA per SM as well: two would need a single S buffer each (256 TMEM columns: S 128 + O 64), which
// serialises MMA 1 behind the softmax; the launch asks for at least 116 KB so that two CTAs never share an SM (each
// allocates 512 TMEM columns).
constexpr int kAtLongThreads = 192;
constexpr int kAtLongMaxN = 16384;   // a 128 x 128 token grid
constexpr float kAtRescaleLog2 = 8.0f;
constexpr int kAtLongMinSmem = 116 * 1024;

template <int DH>
struct AtLongSmem {
    static constexpr int KC = DH / 64;
    static constexpr int kTile = KC * kAtQBox;  // one 128-row box per 64-wide slice of d
    static constexpr int kQ = 0, kK = kTile, kV = 3 * kTile, kP = 5 * kTile, kBars = 5 * kTile + 2 * kAtQBox;
    static constexpr int kBytes = kBars + 128 /*barriers*/ + 1024 /*alignment slack*/;
    static constexpr int kLaunch = kBytes > kAtLongMinSmem ? kBytes : kAtLongMinSmem;
};

template <int DH, bool DROP>
__global__ void __launch_bounds__(kAtLongThreads, 1)
attn_long_kernel(const __grid_constant__ CUtensorMap tm, const AttnParams p) {
    using L = AtLongSmem<DH>;
    constexpr int KC = L::KC;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (static_cast<uint32_t>(__cvta_generic_to_shared(smem_raw)) & 1023u)) & 1023u);
    uint8_t* const s_q = smem + L::kQ;
    uint8_t* const s_k = smem + L::kK;  // stage s at s * kTile
    uint8_t* const s_v = smem + L::kV;
    uint8_t* const s_p = smem + L::kP;  // 2 x [128 rows x 128 B]: keys 0-63 | 64-127 of the tile
    uint64_t* const bars = reinterpret_cast<uint64_t*>(smem + L::kBars);
    uint64_t* const q_full = bars + 0;
    uint64_t* const q_empty = bars + 1;
    uint64_t* const kv_full = bars + 2;   // [2]
    uint64_t* const kv_empty = bars + 4;  // [2]
    uint64_t* const s_full = bars + 6;    // [2]
    uint64_t* const s_empty = bars + 8;   // [2]
    uint64_t* const p_full = bars + 10;
    uint64_t* const o_full = bars + 11;
    uint64_t* const o_empty = bars + 12;
    uint32_t* const tmem_slot = reinterpret_cast<uint32_t*>(bars + 14);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_kt = (p.N + 127) >> 7;  // key tiles
    if (threadIdx.x == 0) {
        mbar_init(q_full, 1);
        mbar_init(q_empty, 1);
        for (int s = 0; s < 2; ++s) {
            mbar_init(kv_full + s, 1);
            mbar_init(kv_empty + s, 1);
            mbar_init(s_full + s, 1);
            mbar_init(s_empty + s, 128);
        }
        mbar_init(p_full, 128);
        mbar_init(o_full, 1);
        mbar_init(o_empty, 128);
        fence_mbar_init();
    }
    if (warp == 5) tmem_alloc<512>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t tmem_o = tmem_base + 256;
    const int E = p.heads * DH;

    if (warp == 4) {
        if (lane == 0) {
            tma_prefetch_desc(&tm);
            uint32_t t = 0, it = 0;
            for (int item = blockIdx.x; item < p.n_items; item += gridDim.x, ++it) {
                const int qt = item % p.q_tiles;
                const int h = (item / p.q_tiles) % p.heads;
                const int b = item / (p.q_tiles * p.heads);
                mbar_wait(q_empty, (it & 1u) ^ 1u);
                mbar_arrive_expect_tx(q_full, L::kTile);
#pragma unroll
                for (int kc = 0; kc < KC; ++kc)
                    tma_load_4d(s_q + kc * kAtQBox, &tm, q_full, h * DH + kc * 64, qt * 128, b, 0);
                for (int j = 0; j < n_kt; ++j, ++t) {
                    const int s = t & 1;
                    mbar_wait(kv_empty + s, ((t >> 1) & 1u) ^ 1u);
                    mbar_arrive_expect_tx(kv_full + s, 2 * L::kTile);
#pragma unroll
                    for (int kc = 0; kc < KC; ++kc) {
                        tma_load_4d(s_k + s * L::kTile + kc * kAtQBox, &tm, kv_full + s, E + h * DH + kc * 64, j * 128, b, 0);
                        tma_load_4d(s_v + s * L::kTile + kc * kAtQBox, &tm, kv_full + s, 2 * E + h * DH + kc * 64, j * 128,
                                    b, 0);
                    }
                }
            }
        }
    } else if (warp == 5) {
        if (lane == 0) {
            constexpr uint32_t idesc1 = umma_idesc_bf16(128, 128);
            constexpr uint32_t idesc2 = umma_idesc_bf16(128, DH) | (1u << 16);  // B (= V) is MN-major
            uint32_t t = 0, it = 0;
            // MMA 1 of key tile j of the current item, the CTA's tile number tt
            auto issue_s = [&](int j, uint32_t tt) {
                const int s = tt & 1;
                mbar_wait(kv_full + s, (tt >> 1) & 1u);
                mbar_wait(s_empty + s, ((tt >> 1) & 1u) ^ 1u);
                tc_fence_after();
#pragma unroll
                for (int kc = 0; kc < KC; ++kc) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const uint64_t da = umma_desc_sw128(smem_u32(s_q + kc * kAtQBox) + k * 32);
                        const uint64_t db = umma_desc_sw128(smem_u32(s_k + s * L::kTile + kc * kAtQBox) + k * 32);
                        umma_bf16(tmem_base + s * 128, da, db, idesc1, (kc | k) != 0 ? 1u : 0u);
                    }
                }
                umma_commit(s_full + s);
                if (j == n_kt - 1) umma_commit(q_empty);
            };
            for (int item = blockIdx.x; item < p.n_items; item += gridDim.x, ++it) {
                mbar_wait(q_full, it & 1u);
                tc_fence_after();
                issue_s(0, t);
                for (int j = 0; j < n_kt; ++j, ++t) {
                    if (j + 1 < n_kt) issue_s(j + 1, t + 1);
                    if (j == 0) mbar_wait(o_empty, (it & 1u) ^ 1u);  // the previous item's O has left TMEM
                    mbar_wait(p_full, t & 1u);
                    tc_fence_after();
                    const int s = t & 1;
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks) {
                        const uint64_t da = umma_desc_sw128(smem_u32(s_p + (ks >> 2) * kAtQBox) + (ks & 3) * 32);
                        const uint64_t db = at_desc_mn_sw128(smem_u32(s_v + s * L::kTile) + ks * 2048, kAtQBox);
                        umma_bf16(tmem_o, da, db, idesc2, (j | ks) != 0 ? 1u : 0u);
                    }
                    umma_commit(kv_empty + s);
                    umma_commit(o_full);
                }
            }
        }
    } else {
        const uint32_t lane_off = static_cast<uint32_t>(warp * 32) << 16;
        const int r = warp * 32 + lane;  // row inside the query tile
        const int swz = r & 7;
        const unsigned long long ctr_stride = 64ull * ((p.N + 255) >> 8);
        uint32_t t = 0, it = 0;
        for (int item = blockIdx.x; item < p.n_items; item += gridDim.x, ++it) {
            const int qt = item % p.q_tiles;
            const int h = (item / p.q_tiles) % p.heads;
            const int b = item / (p.q_tiles * p.heads);
            const int row = qt * 128 + r;
            const bool warp_live = qt * 128 + warp * 32 < p.N;  // some row of this warp is a real query
            unsigned long long ctr = 0;
            if (DROP) ctr = ((static_cast<unsigned long long>(b) * p.heads + h) * p.N + row) * ctr_stride;
            float m = 0.f, l = 0.f;
            for (int j = 0; j < n_kt; ++j, ++t) {
                const int s = t & 1;
                uint32_t v[128];
                mbar_wait(s_full + s, (t >> 1) & 1u);
                tc_fence_after();
                if (warp_live) {
#pragma unroll
                    for (int c = 0; c < 4; ++c)
                        tmem_ld_32x32(tmem_base + lane_off + s * 128 + c * 32, *reinterpret_cast<uint32_t(*)[32]>(v + 32 * c));
#pragma unroll
                    for (int c = 0; c < 4; ++c) tmem_ld_wait32(*reinterpret_cast<uint32_t(*)[32]>(v + 32 * c));
                }
                tc_fence_before();
                mbar_arrive(s_empty + s);
                const int valid = p.N - j * 128;
                float mx = -3.0e38f;
                if (warp_live) {
                    float m4[4] = {-3.0e38f, -3.0e38f, -3.0e38f, -3.0e38f};
#pragma unroll
                    for (int i = 0; i < 128; ++i)
                        if (i < valid) m4[i & 3] = fmaxf(m4[i & 3], __uint_as_float(v[i]));
                    mx = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3])) * p.scale_log2;
                }
                if (j != 0) {
                    mbar_wait(o_full, (t - 1) & 1u);  // MMA 2 of tile j-1 retired: P is free, O is final for j-1
                    tc_fence_after();
                }
                if (warp_live) {
                    if (j == 0) m = mx;
                    const bool move = mx > m + kAtRescaleLog2;
                    if (__any_sync(0xffffffffu, move)) {
                        const float alpha = move ? ex2_approx(m - mx) : 1.0f;
                        if (move) m = mx;
                        l *= alpha;
#pragma unroll
                        for (int c = 0; c < DH / 32; ++c) {
                            uint32_t o[32];
                            tmem_ld_32x32(tmem_o + lane_off + c * 32, o);
                            tmem_ld_wait32(o);
#pragma unroll
                            for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
                            tmem_st_32x32(tmem_o + lane_off + c * 32, o);
                        }
                        tmem_st_wait();
                    }
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        uint8_t* const dst = s_p + (c >> 1) * kAtQBox + r * 128;
                        const uint32_t(&vc)[32] = *reinterpret_cast<const uint32_t(*)[32]>(v + 32 * c);
                        const unsigned long long cc = ctr + j * 32 + c * 8;
                        if (valid >= 128)
                            l += softmax_chunk<false, DROP>(vc, p.scale_log2, -m, 32, dst, (c & 1) * 4, swz, p, cc);
                        else
                            l += softmax_chunk<true, DROP>(vc, p.scale_log2, -m, valid - c * 32, dst, (c & 1) * 4, swz, p,
                                                           cc);
                    }
                }
                fence_proxy_async_smem();  // P (generic-proxy stores) -> visible to the MMA's async-proxy reads
                tc_fence_before();
                mbar_arrive(p_full);
            }
            mbar_wait(o_full, (t - 1) & 1u);  // the item's last MMA 2 retired
            tc_fence_after();
            if (warp_live)
                store_rows<DH>(tmem_o + lane_off, p.out + (static_cast<long long>(b) * p.N + row) * p.out_ld + h * DH,
                               row < p.N, (DROP ? p.drop_scale : 1.0f) / l);
            tc_fence_before();
            mbar_arrive(o_empty);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 5) {
        tc_fence_after();
        tmem_dealloc<512>(tmem_base);
    }
}


typedef CUresult (*AtEncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static AtEncodeTiledFn at_encode_fn() {
    static AtEncodeTiledFn fn = nullptr;
    if (fn == nullptr) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
            qres != cudaDriverEntryPointSuccess)
            return nullptr;
        fn = reinterpret_cast<AtEncodeTiledFn>(ptr);
    }
    return fn;
}

// qkv viewed as [1][B][N][cols]: a box is {64 columns, rows, 1, 1}; rows >= N of a case are out of bounds -> zeros
static int at_encode_map(AtEncodeTiledFn enc, CUtensorMap* tm, const void* base, int cols, int ld, int N, int B, int rows) {
    const cuuint64_t dims[4] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(N), static_cast<cuuint64_t>(B), 1};
    const cuuint64_t strides[3] = {static_cast<cuuint64_t>(ld) * 2, static_cast<cuuint64_t>(ld) * N * 2,
                                   static_cast<cuuint64_t>(ld) * N * B * 2};
    const cuuint32_t box[4] = {64, static_cast<cuuint32_t>(rows), 1, 1};
    const cuuint32_t es[4] = {1, 1, 1, 1};
    CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : -300 - static_cast<int>(r);
}

template <int DH, bool DROP>
static int at_launch(const CUtensorMap& tmQ, const CUtensorMap& tmKV, const AttnParams& p, int num_sms, cudaStream_t s) {
    constexpr int KC = DH / 64;
    constexpr int kQKBytes = KC * (kAtQBox + kAtKBox);
    constexpr int kRegionA = kQKBytes > kAtPBytes ? kQKBytes : kAtPBytes;
    constexpr int smem = kRegionA + KC * kAtKBox + 128 /*barriers*/ + 1024 /*alignment slack*/;
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(attn_fused_kernel<DH, DROP>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return static_cast<int>(e);
        configured = true;
    }
    int grid = num_sms * (DH == 64 ? 2 : 1);
    if (grid > p.n_items) grid = p.n_items;
    attn_fused_kernel<DH, DROP><<<grid, kAtThreads, smem, s>>>(tmQ, tmKV, p);
    return static_cast<int>(cudaGetLastError());
}

template <int DH, bool DROP>
static int at_long_launch(const CUtensorMap& tm, const AttnParams& p, int num_sms, cudaStream_t s) {
    constexpr int smem = AtLongSmem<DH>::kLaunch;
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(attn_long_kernel<DH, DROP>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return static_cast<int>(e);
        configured = true;
    }
    const int grid = num_sms < p.n_items ? num_sms : p.n_items;
    attn_long_kernel<DH, DROP><<<grid, kAtLongThreads, smem, s>>>(tm, p);
    return static_cast<int>(cudaGetLastError());
}

// Argument checks, tensor maps and launch of b200_attention / b200_attention_mc (drop_p in [0, 1); 0 = no dropout).
// N <= 256 runs attn_fused_kernel (one score tile per item), 256 < N <= kAtLongMaxN attn_long_kernel.
static int attention_run(const void* qkv, int qkv_ld, void* out, int out_ld, int B, int N, int heads, int dh, float scale,
                         float drop_p, unsigned long long drop_seed, void* stream) {
    if (B < 0 || N <= 0 || N > kAtLongMaxN || heads <= 0 || (dh != 64 && dh != 128)) return -1;
    if (N > 256 && static_cast<long long>(B) * heads * ((N + 127) / 128) > 0x7fffffffLL) return -1;  // items are ints
    if (B == 0) return 0;
    if (qkv == nullptr || out == nullptr) return -2;
    const int E = heads * dh;
    if (qkv_ld < 3 * E || qkv_ld % 8 != 0 || out_ld < E || out_ld % 8 != 0) return -3;
    if ((reinterpret_cast<uintptr_t>(qkv) & 15) || (reinterpret_cast<uintptr_t>(out) & 15)) return -5;
    static int num_sms = 0;
    if (num_sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
        if (num_sms <= 0) return -9;
    }
    AtEncodeTiledFn enc = at_encode_fn();
    if (enc == nullptr) return -8;
    CUtensorMap tmQ, tmKV;
    int rc;
    if ((rc = at_encode_map(enc, &tmQ, qkv, 3 * E, qkv_ld, N, B, 128)) != 0) return rc - 1000;
    if (N <= 256 && (rc = at_encode_map(enc, &tmKV, qkv, 3 * E, qkv_ld, N, B, 256)) != 0) return rc - 2000;
    AttnParams p{};
    p.N = N;
    p.heads = heads;
    p.B = B;
    p.q_tiles = (N + 127) / 128;
    p.n_items = B * heads * p.q_tiles;
    p.n_chunks = (N + 31) / 32;
    p.k_steps = (N + 15) / 16;
    p.out_ld = out_ld;
    p.scale_log2 = scale * 1.4426950408889634f;
    p.out = static_cast<__nv_bfloat16*>(out);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (drop_p > 0.f) {
        p.drop_thresh = dropout_threshold(drop_p);
        p.drop_scale = 1.0f / (1.0f - drop_p);
        p.drop_seed_lo = static_cast<unsigned int>(drop_seed);
        p.drop_seed_hi = static_cast<unsigned int>(drop_seed >> 32);
        if (N > 256)
            return dh == 64 ? at_long_launch<64, true>(tmQ, p, num_sms, s) : at_long_launch<128, true>(tmQ, p, num_sms, s);
        return dh == 64 ? at_launch<64, true>(tmQ, tmKV, p, num_sms, s) : at_launch<128, true>(tmQ, tmKV, p, num_sms, s);
    }
    if (N > 256)
        return dh == 64 ? at_long_launch<64, false>(tmQ, p, num_sms, s) : at_long_launch<128, false>(tmQ, p, num_sms, s);
    return dh == 64 ? at_launch<64, false>(tmQ, tmKV, p, num_sms, s) : at_launch<128, false>(tmQ, tmKV, p, num_sms, s);
}

}  // namespace b200

extern "C" int b200_attention(const void* qkv, int qkv_ld, void* out, int out_ld, int B, int N, int heads, int dh,
                              float scale, void* stream) {
    return b200::attention_run(qkv, qkv_ld, out, out_ld, B, N, heads, dh, scale, 0.f, 0, stream);
}

// b200_attention with nn.Dropout(drop_p) on the softmax probabilities (MC-dropout inference): the row sums stay those
// of the undropped softmax, kept probabilities are scaled by 1 / (1 - drop_p).  drop_p == 0 runs b200_attention.
extern "C" int b200_attention_mc(const void* qkv, int qkv_ld, void* out, int out_ld, int B, int N, int heads, int dh,
                                 float scale, float drop_p, unsigned long long drop_seed, void* stream) {
    if (!(drop_p >= 0.f && drop_p < 1.f)) return -19;  // NaN fails both comparisons
    return b200::attention_run(qkv, qkv_ld, out, out_ld, B, N, heads, dh, scale, drop_p, drop_seed, stream);
}
