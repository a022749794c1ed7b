// Implicit-GEMM convolution / linear layer for sm_100a.
//
//   out[pixel, n] = epilogue( sum_{tap, c} x[pixel + offset(tap), c] * w[n, tap*Cin + c] )
//
// Activations are NHWC bf16, weights are [Cout, taps*Cin] bf16 (K-major), the accumulator lives in
// TMEM (fp32).  One persistent CTA per SM, warp-specialised, 384 threads (kThreads):
//   warp 0      TMA producer: one 4-D box {64 ch, BW, BH, 1} of the input per (tap, 64-channel slice) -
//               the tap shift is a coordinate offset, the zero padding is the TMA out-of-bounds fill -
//               plus one 2-D box {64, BLOCK_N} of the weights, both written with the 128-byte swizzle.
//               PAIR (BLOCK_N = 128 layers, plain and tap-dot epilogues, and 3x3 BLOCK_N = 64 layers, with
//               >= 2 x 148 M tiles): a second input box per stage, so one weight slab feeds two M tiles.
//   warp 1      tcgen05.mma issuer (single thread), M=128, N=BLOCK_N, K=16 per instruction; PAIR issues
//               the second tile's MMAs into the next BLOCK_N TMEM columns off the same B descriptor
//   warp 2      TMEM allocation / release: 2 accumulator stages (4 with PAIR) - the epilogue of tile i
//               overlaps the MMAs of tile i+1
//   warp 3      idle (keeps the epilogue warps aligned to TMEM lane quadrants: quadrant = warp % 4)
//   warps 4-11  epilogue (kNumEpiWarps = 8, two per TMEM lane quadrant): each warp owns 32 accumulator
//               rows x BLOCK_N/2 columns and walks them in 32-column chunks (tcgen05.ld.32x32b.x32):
//               folded-BN FMA -> residual (its own TMA-loaded box, prefetched one tile ahead) -> GELU ->
//               (Philox dropout) -> bf16 -> swizzled shared-memory box -> TMA store.  Optional fused products: per-case channel
//               sums, a second output segment with its own activation, the 9 per-tap dot products of a
//               following 3x3 C->1 convolution, 2x2-replicated (strided TMA) stores.
//
// Covers the reference's conv/BN/GELU stacks (model_module.py:259-269, :113-118, :150, :337-345,
// :386-390, :857-858) and nn.Linear layers (transformer_model.py:93-125).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdlib>

#include "b200_fusion.h"
#include "common.cuh"
#include "ptx.cuh"

namespace b200 {

struct ConvGemmParams {
    int H, W, Cout;
    int BH, BW;            // TMA box over (h, w); BH*BW == 128
    // exact division by launch constants without the 25-instruction software divide (the tile -> coordinate maps run per
    // tile in every role; they were 14 % of the instructions the block-tail kernels issued): q = umulhi(n, m) [+ n when
    // d == 1], m = floor(2^32 / d) + 1, exact while n * d < 2^32
    struct FastDiv {
        uint32_t d, m;
    };
    FastDiv fd_ntiles, fd_tw, fd_th, fd_twth;
    int BB, B;             // cases per M tile (box extent over the batch dimension; 1 unless the planner packs several
                           // cases of a small map into one tile) and the number of cases
    int tiles_w, tiles_h;  // tiles per image row / column
    int n_tiles, m_tiles;
    int kc;                // Cin / 64
    int k_blocks;          // taps * kc
    int taps;
    const float* scale;    // [Cout] or nullptr (=1)
    const float* bias;     // [Cout] or nullptr (=0)
    const __nv_bfloat16* res;
    int res_ld;
    int res_mode;          // 0 none, 1 add before activation, 2 add after activation
    int act;               // 0 none, 1 GELU (gelu_fast2), 2 ReLU
    __nv_bfloat16* out;
    int out_ld;
    int up2;               // replicate every output pixel into a 2x2 block of a [B,2H,2W,ld] map
    int tma_epi;           // outputs / residual go through shared memory + TMA (coalesced); else direct
    int share_box;         // BN = 256: a warp's two 64-column output boxes share one 4 KB staging slot (one more ring stage)
    // MC-dropout (mode 3): element (pixel, channel) of the segments selected by drop_seg (bit 0 = first output,
    // bit 1 = second) is zeroed when Philox4x32-7(seed; pixel * Cout + channel) < drop_thresh, else scaled by
    // drop_scale = 1 / (1 - p).  Applied after the activation, before the store / channel sums.  Mode 4 (the fp32
    // epilogue of b200_linear_mc) applies the same rule before the residual add.
    unsigned int drop_thresh;
    float drop_scale;
    unsigned int drop_seed_lo, drop_seed_hi;
    int drop_seg;
    float* gap;            // [B, Cout] fp32 sums over the pixels of each case, or nullptr
    int n_split;           // channels [n_split, Cout) are a second output segment (== Cout when unused)
    __nv_bfloat16* out2;
    int out2_ld;
    int act2;
    const float* dot_w;    // [ndot, Cout] fp32 or nullptr: fused per-pixel projection of the epilogue result
    float* dot_out;        // [pixels, ndot] fp32 (+ dot_bias)
    float dot_bias;
    int ndot;
    int a_box_bytes;       // bytes one A box really delivers (BW*BH rows x 128 B; < 16 KB when BW*BH < 128)
    int cstride;           // convolution stride
    int dil;               // dilation of the 3x3 taps (1 = dense) (1, or 2 for the 2x2 / stride-2 patch embedding: taps == 4)
    int res_f32, out_f32;  // residual / output are fp32 row-major (transformer residual stream); direct path
    int stages;            // operand ring depth
    int obuf2;             // output staging double-buffered per epilogue warp (tile i+1 is staged while the TMA store of
                           // tile i still reads its boxes); 0: one set of boxes, the store is waited for at the next tile
    int pair;              // BN = 128: two M tiles per CTA iteration share one weight slab (conv_gemm_kernel<..., PAIR>)
    int off_bar, off_union, off_rbox;  // shared-memory plan (bytes from the 1 KB-aligned base)
    int off_aff;           // >= 0: [scale Cout | bias Cout] parked in shared memory once per CTA (BN <= 128 launches);
                           // -1: they are read from global memory per chunk
};

__device__ __forceinline__ int fd_div(const ConvGemmParams::FastDiv& f, int n) {
    return static_cast<int>(__umulhi(static_cast<uint32_t>(n), f.m) + (f.d == 1 ? static_cast<uint32_t>(n) : 0u));
}
__device__ __forceinline__ int fd_mod(const ConvGemmParams::FastDiv& f, int n) {
    return n - fd_div(f, n) * static_cast<int>(f.d);
}
// M tile index -> (w0 tile, h0 tile, case group) indices
__device__ __forceinline__ void tile_whb(const ConvGemmParams& p, int mt, int& tw, int& th, int& tb) {
    const int a = fd_div(p.fd_tw, mt);
    tw = mt - a * static_cast<int>(p.fd_tw.d);
    tb = fd_div(p.fd_twth, mt);
    th = a - tb * static_cast<int>(p.fd_th.d);
}


constexpr int kBlockM = 128;
constexpr int kF32BlockBytes = 32 * 33 * 4;  // one warp's padded 32 x 32 fp32 transposition block (fp32 epilogue)
constexpr int kBlockK = 64;
constexpr int kABytes = kBlockM * kBlockK * 2;
constexpr int kEpiWarp0 = 4;
constexpr int kNumEpiWarps = 8;
constexpr int kThreads = (kEpiWarp0 + kNumEpiWarps) * 32;
constexpr int kChunk = 32;  // accumulator columns per epilogue step (one tcgen05.ld.32x32b.x32)
constexpr int kMaxStages = 12;
constexpr int kBarBytes = 512;

// Shared-memory plan, computed on the host (plan_smem) and passed in ConvGemmParams:
//   [ operand ring | barriers | union{output boxes, tap-dot buffers} | residual boxes ]
template <int BN>
struct Tile {
    static constexpr int kBBytes = BN * kBlockK * 2;
    static constexpr int kTmemCols = 2 * BN;             // two accumulator stages: 128 / 256 / 512 columns
    static constexpr int kTmemColsPair = 4 * BN;         // PAIR (BN = 128): four stages = 512 columns
    static constexpr int kColsPerWarp = BN / 2;           // each epilogue warp: 32 rows x BN/2 columns
    static constexpr int kChunksPerWarp = kColsPerWarp / kChunk;
    static constexpr int kBoxCols = kColsPerWarp < 64 ? kColsPerWarp : 64;  // TMA box width (<= 128 B rows)
    static constexpr int kBoxesPerWarp = kColsPerWarp / kBoxCols;
    static constexpr int kRowBytes = kBoxCols * 2;
    static constexpr int kBoxBytes = 32 * kRowBytes;      // 2 KB (64-byte swizzle) or 4 KB (128-byte swizzle)
    static constexpr int kWarpBoxBytes = kBoxesPerWarp * kBoxBytes;
    static constexpr int kDotBytes = 9 * BN * 4 + 2 * kBlockM * 9 * 4;
};

// The epilogue GELU is common.cuh's gelu_fast2 (tanh form on MUFU.TANH, two elements per packed instruction).

// nn.Dropout in MC-dropout inference (reference train_fusion.py:478-481: dropout modules in train mode, BatchNorm
// frozen) on the 32 columns [n0, n0 + 32) of row `pix`: one Philox call yields the keep decisions of 4 consecutive
// channels
__device__ __forceinline__ void dropout_chunk(float (&v)[kChunk], long long pix, int n0, const ConvGemmParams& p) {
    const unsigned long long e0 = static_cast<unsigned long long>(pix) * p.Cout + n0;
#pragma unroll
    for (int j = 0; j < kChunk / 4; ++j) {
        const uint4 rnd = philox4x32_7(e0 / 4 + j, p.drop_seed_lo, p.drop_seed_hi);
        v[4 * j + 0] = rnd.x < p.drop_thresh ? 0.f : v[4 * j + 0] * p.drop_scale;
        v[4 * j + 1] = rnd.y < p.drop_thresh ? 0.f : v[4 * j + 1] * p.drop_scale;
        v[4 * j + 2] = rnd.z < p.drop_thresh ? 0.f : v[4 * j + 2] * p.drop_scale;
        v[4 * j + 3] = rnd.w < p.drop_thresh ? 0.f : v[4 * j + 3] * p.drop_scale;
    }
}

// Epilogue features are compile-time so that the per-element instruction stream carries no flag tests:
//   RES  0 none, 1 residual added before the activation, 2 after it
//   GAP  per-case channel sums          NDOT 0, or 1 / 9 fused per-pixel dot products (no map store)
//   MODE 0 standard; 2 fp32 residual / output (b200_linear); 3 MC dropout after the activation; 4 = 2 with MC
//        dropout before the residual add (b200_linear_mc)
//   PAIR (BN = 128 only): a CTA works on TWO consecutive M tiles of the same N tile at once - 256 x 128 outputs: per
//        64-deep k-block the weight slab is loaded once and feeds two MMAs (one per M tile, each with its own TMEM
//        accumulator), so a stage moves 48 KB for 2 x (128 x 128 x 64) MACs instead of 64 KB.  128 x 128 tiles were
//        shared-memory-feed bound (0.64 PFLOP/s on 3x3 128->128 against 1.24 for the 128 x 256 tiles); four accumulator
//        stages (512 TMEM columns) keep the epilogue of one pair overlapped with the MMAs of the next.
template <int BN, int RES, bool GAP, int NDOT, int MODE, bool PAIR = false>
__global__ void __launch_bounds__(kThreads, 1)
conv_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const __grid_constant__ CUtensorMap tmOut, const __grid_constant__ CUtensorMap tmOut2,
                 const __grid_constant__ CUtensorMap tmRes, const ConvGemmParams p) {
    using T = Tile<BN>;
    constexpr bool DOT = NDOT > 0;
    extern __shared__ uint8_t smem_raw[];
    // 1 KB alignment by OFFSET (not by rounding the generic address): the compiler keeps the shared state space
    // and emits STS / LDS for the staging traffic instead of generic ST / LD
    uint8_t* smem = smem_raw + ((1024u - (static_cast<uint32_t>(__cvta_generic_to_shared(smem_raw)) & 1023u)) & 1023u);
    uint8_t* sRing = smem;
    static_assert(!PAIR || ((BN == 128 || BN == 64) && MODE == 0), "PAIR: BN = 128 / 64, standard epilogue");
    constexpr int kStageBytes = (PAIR ? 2 * kABytes : kABytes) + T::kBBytes;
    constexpr int kAcc = PAIR ? 4 : 2;             // accumulator stages in TMEM
    constexpr int kTmemCols = PAIR ? T::kTmemColsPair : T::kTmemCols;
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + p.off_bar);
    uint64_t* empty = full + kMaxStages;
    uint64_t* tfull = empty + kMaxStages;
    uint64_t* tempty = tfull + 4;
    uint64_t* resbar = tempty + 4;  // [kNumEpiWarps][2] residual-box arrival, one per epilogue warp and box
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(resbar + 2 * kNumEpiWarps);
    uint8_t* s_union = smem + p.off_union;
    float* s_dotw = reinterpret_cast<float*>(s_union);  // [NDOT][BN]       (dot mode)
    float* s_dots = s_dotw + NDOT * BN;                 // [2][128][NDOT]   (dot mode)

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int stages = p.stages;
    // tile walk: tiles are dealt round-robin, N fastest
    const int total_tiles = PAIR ? ((p.m_tiles + 1) / 2) * p.n_tiles : p.m_tiles * p.n_tiles;  // PAIR: super-tiles
    const int n_iters = total_tiles > static_cast<int>(blockIdx.x)
                            ? (total_tiles - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) /
                                  static_cast<int>(gridDim.x)
                            : 0;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        if (p.tma_epi) {
            if (p.out != nullptr) tma_prefetch_desc(&tmOut);
            if (p.n_split < p.Cout) tma_prefetch_desc(&tmOut2);
            if (RES != 0) tma_prefetch_desc(&tmRes);
        }
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < stages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        for (int s = 0; s < kAcc; ++s) {
            mbar_init(&tfull[s], 1);
            mbar_init(&tempty[s], kNumEpiWarps);
        }
        for (int s = 0; s < 2 * kNumEpiWarps; ++s) mbar_init(&resbar[s], 1);
        fence_mbar_init();
    }
    if (warp == 2) tmem_alloc<kTmemCols>(tmem_slot);
    if (DOT && warp >= kEpiWarp0) {
        for (int i = threadIdx.x - kEpiWarp0 * 32; i < NDOT * BN; i += kNumEpiWarps * 32) s_dotw[i] = p.dot_w[i];
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0 && n_iters > 0) {
            int stage = 0;
            uint32_t phase = 0;
            int tile = blockIdx.x;
            for (int it = 0; it < n_iters; ++it, tile += gridDim.x) {
                const int tq = fd_div(p.fd_ntiles, tile);
                const int n_tile = tile - tq * p.n_tiles;
                const int mt = PAIR ? 2 * tq : tq;
                int tw0, th0, tb0, tw1 = 0, th1 = 0, tb1 = 0;
                tile_whb(p, mt, tw0, th0, tb0);
                const int w0 = tw0 * p.BW, h0 = th0 * p.BH, b = tb0 * p.BB;
                // PAIR: the second M tile of the pair (absent only for the last tile of an odd count)
                const bool has2 = PAIR && mt + 1 < p.m_tiles;
                if (PAIR) tile_whb(p, mt + 1, tw1, th1, tb1);
                const int w1 = tw1 * p.BW, h1 = th1 * p.BH, b1 = tb1 * p.BB;
                for (int kb = 0; kb < p.k_blocks; ++kb) {
                    const int tap = kb / p.kc;
                    const int c0 = (kb - tap * p.kc) * kBlockK;
                    int dy = 0, dx = 0;
                    if (p.taps == 9) {
                        dy = (tap / 3 - 1) * p.dil;
                        dx = (tap % 3 - 1) * p.dil;
                    } else if (p.taps == 4) {
                        dy = tap >> 1;
                        dx = tap & 1;
                    }
                    mbar_wait(&empty[stage], phase ^ 1);
                    mbar_arrive_expect_tx(&full[stage], p.a_box_bytes * (has2 ? 2 : 1) + T::kBBytes);
                    uint8_t* dst = sRing + stage * kStageBytes;
                    tma_load_4d(dst, &tmA, &full[stage], c0, p.cstride * w0 + dx, p.cstride * h0 + dy, b);
                    if (has2) tma_load_4d(dst + kABytes, &tmA, &full[stage], c0, p.cstride * w1 + dx, p.cstride * h1 + dy, b1);
                    constexpr int kBOff = PAIR ? 2 * kABytes : kABytes;
                    tma_load_2d(dst + kBOff, &tmB, &full[stage], kb * kBlockK, n_tile * BN);
                    if (++stage == stages) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0 && n_iters > 0) {
            constexpr uint32_t idesc = umma_idesc_bf16(kBlockM, BN);
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            int tile = blockIdx.x;
            for (int it = 0; it < n_iters; ++it, tile += gridDim.x) {
                const bool has2 = PAIR && 2 * fd_div(p.fd_ntiles, tile) + 1 < p.m_tiles;
                mbar_wait(&tempty[acc], acc_phase ^ 1);
                if (has2) mbar_wait(&tempty[acc + 1], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * BN;
                for (int kb = 0; kb < p.k_blocks; ++kb) {
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    const uint8_t* a_src = sRing + stage * kStageBytes;
                    const uint64_t da = umma_desc_sw128(smem_u32(a_src));
                    const uint64_t db = umma_desc_sw128(smem_u32(a_src + (PAIR ? 2 * kABytes : kABytes)));
#pragma unroll
                    for (int k = 0; k < kBlockK / 16; ++k) {
                        // 16 bf16 = 32 bytes along K inside the 128-byte swizzle row -> +2 in 16-byte units
                        umma_bf16(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
                    }
                    if (has2) {  // the pair's second M tile: its own A box and accumulator, the SAME weight slab
                        const uint64_t da1 = umma_desc_sw128(smem_u32(a_src + kABytes));
#pragma unroll
                        for (int k = 0; k < kBlockK / 16; ++k)
                            umma_bf16(d_tmem + BN, da1 + 2 * k, db + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
                    }
                    umma_commit(&empty[stage]);
                    if (++stage == stages) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
                umma_commit(&tfull[acc]);
                if (has2) umma_commit(&tfull[acc + 1]);
                acc += PAIR ? 2 : 1;
                if (acc == kAcc) {
                    acc = 0;
                    acc_phase ^= 1;
                }
            }
        }
    } else if (warp >= kEpiWarp0) {
        const int ew = warp - kEpiWarp0;
        const int q = warp & 3;    // TMEM lane quadrant this warp may read (rows q*32 .. q*32+31 of the tile)
        const int half = ew >> 2;  // column half: columns [half*BN/2, (half+1)*BN/2)
        const int colw0 = half * T::kColsPerWarp;
        const bool share = p.share_box != 0;  // warp-uniform; set by the host for BN = 256 plain-output launches only
        uint8_t* const obuf0 = s_union + ew * ((MODE == 2 || MODE == 4) ? kF32BlockBytes : (share ? T::kBoxBytes : T::kWarpBoxBytes));
        const int obuf_flip = p.obuf2 ? 8 * T::kWarpBoxBytes : 0;  // second set of boxes (all 8 warps') behind the first
        int obuf_sel = 0;
        uint8_t* const rbuf = smem + p.off_rbox + ew * T::kWarpBoxBytes;
        uint64_t* const rbar = &resbar[2 * ew];  // one barrier per staged residual box
        uint32_t rphase = 0;                     // bit bx = phase of box bx
        // A staged box is 32 rows x kBoxCols bf16 under the TMA swizzle of its row width (64 or 128 B):
        // 16-byte chunk c of row r sits at chunk c ^ (((r * rowBytes) >> 7) & (rowBytes/16 - 1)).
        const int swz = ((lane * T::kRowBytes) >> 7) & (T::kRowBytes / 16 - 1);
        const int row_off = lane * T::kRowBytes;
        const bool tma_epi = p.tma_epi != 0;
        // fp32 residual / output (never TMA-staged): transpose through the warp's staging box when it is large enough
        constexpr bool kF32 = MODE == 2 || MODE == 4;  // the fp32 code exists only in the instantiations b200_linear uses
        constexpr bool kTransposeF32 = true;  // the host plans 8 transposition blocks for mode 2
        int acc = 0;
        uint32_t acc_phase = 0;
        int tile = blockIdx.x;
        // tile-invariant pieces of the row -> pixel map (the TMA box is {64 ch, BW, BH, BB}, rows in that order)
        const int trow = q * 32 + lane;
        const int r_w = trow % p.BW, r_h = (trow / p.BW) % p.BH, r_b = trow / (p.BW * p.BH);
        const int q_w = (q * 32) % p.BW, q_h = (q * 32) / p.BW;
        const bool row_in_box = trow < p.BW * p.BH * p.BB;
        // Folded-BN scale | bias of ALL output channels, parked in shared memory once per CTA by the epilogue warps
        // ([scale Cout | bias Cout] fp32): per 32-column chunk every lane needs the same 32 + 32 floats, which cost 16
        // LDG.128 + 32 descriptor moves (R2UR) per chunk and lane when read from global memory - 15 % of the instructions
        // of a BN = 64 tile (profiles/r2_ncu_full.csv, capture r2_k64).  BN <= 128 launches only (the host plans it).
        float* const s_aff = p.off_aff >= 0 ? reinterpret_cast<float*>(smem + p.off_aff) : nullptr;
        if (s_aff != nullptr) {
            const int et = threadIdx.x - kEpiWarp0 * 32;  // 0 .. 255 over the epilogue warps
            for (int i = et; i < p.Cout / 4; i += kNumEpiWarps * 32) {
                reinterpret_cast<float4*>(s_aff)[i] = __ldg(reinterpret_cast<const float4*>(p.scale) + i);
                reinterpret_cast<float4*>(s_aff + p.Cout)[i] = __ldg(reinterpret_cast<const float4*>(p.bias) + i);
            }
            asm volatile("bar.sync 1, 256;" ::: "memory");
        }
        // Residual boxes are fetched one tile ahead: box bx of tile i+1 is requested as soon as the last lane
        // has read box bx of tile i, so its DRAM latency hides behind the rest of tile i's epilogue.
        auto res_fetch = [&](int nt, int mt, int bx) {
            int ftw, fth, fb;
            tile_whb(p, mt, ftw, fth, fb);
            const int fw = ftw * p.BW + q_w, fh = fth * p.BH + q_h;
            mbar_arrive_expect_tx(&rbar[bx], T::kBoxBytes);
            tma_load_4d(rbuf + bx * T::kBoxBytes, &tmRes, &rbar[bx], nt * BN + colw0 + bx * T::kBoxCols, fw, fh, fb);
        };
        // the CTA's tile sequence: (tile index, sub) -> (N tile, M tile); PAIR walks super-tiles of two M tiles
        auto tile_nm = [&](int t_idx, int sub, int& nt, int& mt) {
            const int tq = fd_div(p.fd_ntiles, t_idx);
            nt = t_idx - tq * p.n_tiles;
            mt = PAIR ? 2 * tq + sub : tq;
            return mt < p.m_tiles;
        };
        if (RES != 0 && tma_epi && lane == 0 && n_iters > 0) {
            int nt0, mt0;
            tile_nm(tile, 0, nt0, mt0);
#pragma unroll
            for (int bx = 0; bx < T::kBoxesPerWarp; ++bx) res_fetch(nt0, mt0, bx);
        }
        for (int it = 0; it < n_iters; ++it, tile += gridDim.x) {
          for (int sub = 0; sub < (PAIR ? 2 : 1); ++sub) {
            int n_tile, m_tile;
            if (!tile_nm(tile, sub, n_tile, m_tile)) {  // (PAIR) the absent second tile of an odd count
                if (++acc == kAcc) {
                    acc = 0;
                    acc_phase ^= 1;
                }
                continue;
            }
            // the tile this warp handles next (its residual boxes are prefetched while this one is in flight)
            int n_next = 0, m_next = 0;
            bool have_next = false;
            if (PAIR && sub == 0) have_next = tile_nm(tile, 1, n_next, m_next);
            if (!have_next && it + 1 < n_iters) have_next = tile_nm(tile + gridDim.x, 0, n_next, m_next);
            // tile -> (w0, h0, b); this warp's slab = 32 consecutive rows of the tile = a {bw, bh} box in (w, h)
            int tw0, th0, tb0;
            tile_whb(p, m_tile, tw0, th0, tb0);
            const int w0 = tw0 * p.BW, h0 = th0 * p.BH, b = tb0 * p.BB;
            const int slab_w = w0 + q_w, slab_h = h0 + q_h;  // (staged epilogue: BB = 1)
            const int pw = w0 + r_w, ph = h0 + r_h, pb = b + r_b;
            const bool valid = row_in_box && pw < p.W && ph < p.H && pb < p.B;
            const long long pix = (static_cast<long long>(pb) * p.H + ph) * p.W + pw;
            // pixel index of tile row r, or -1 when that row does not exist (ragged tiles / tails)
            // (used by the fp32 epilogue, i.e. b200_linear only: H = 1 and a tile is 128 consecutive rows)
            auto row_pix = [&](int r) -> long long { return w0 + r < p.W ? static_cast<long long>(w0 + r) : -1; };

            const bool seg2 = n_tile * BN >= p.n_split;
            __nv_bfloat16* const out_ptr = seg2 ? p.out2 : p.out;
            const int act = seg2 ? p.act2 : p.act;
            constexpr bool use_res = RES != 0;  // (the host rejects a residual together with two segments)
            const int out_col0 = (seg2 ? n_tile * BN - p.n_split : n_tile * BN) + colw0;
            const CUtensorMap* const tm_out = seg2 ? &tmOut2 : &tmOut;
            const int nbase = n_tile * BN + colw0;
            float dsum[DOT ? NDOT : 1];
            if (DOT) {
#pragma unroll
                for (int k = 0; k < NDOT; ++k) dsum[k] = 0.f;
            }
            uint8_t* const obuf = obuf0 + obuf_sel * obuf_flip;
            obuf_sel ^= 1;
            if (!DOT && tma_epi && out_ptr != nullptr) {
                // the store that last read THESE boxes has finished reading them: the previous tile's with one set of
                // boxes, the one before it with two (the previous tile's store may still be in flight)
                if (lane == 0) {
                    if (p.obuf2) tma_store_wait_read<1>();
                    else tma_store_wait_read<0>();
                }
                __syncwarp();
            }
            if (kF32 && RES != 0 && p.res_f32) {
                // fp32 residual: pull this warp's 32 x kColsPerWarp block towards L2 while the accumulator is
                // still being produced (the residual does not depend on it); no registers are held
                constexpr int kLinesPerRow = T::kColsPerWarp * 4 / 128;
#pragma unroll
                for (int i = 0; i < kLinesPerRow; ++i) {
                    const int line = lane + 32 * i;
                    const long long rp = row_pix(q * 32 + line / kLinesPerRow);
                    if (rp >= 0)
                        prefetch_l2(reinterpret_cast<const float*>(p.res) + rp * p.res_ld + nbase +
                                    (line % kLinesPerRow) * 32);
                }
            }
            mbar_wait(&tfull[acc], acc_phase);
            tc_fence_after();
            const uint32_t tm_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BN + colw0;
#pragma unroll
            for (int ch = 0; ch < T::kChunksPerWarp; ++ch) {
                const int n0 = nbase + ch * kChunk;
                // fp32 residual (mode 2): its coalesced global loads are issued before the TMEM load so that the
                // DRAM latency overlaps the TMEM round trip and the affine math of the same chunk
                float4 rf[kF32 ? 8 : 1];
                if (kF32 && RES != 0 && p.res_f32) {
                    const float* const rbase = reinterpret_cast<const float*>(p.res) + n0 + (lane & 7) * 4;
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        const long long rp = row_pix(q * 32 + 4 * k + (lane >> 3));
                        rf[k] = rp >= 0 ? __ldg(reinterpret_cast<const float4*>(rbase + rp * p.res_ld))
                                        : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                }
                uint32_t r[kChunk];
                tmem_ld_32x32(tm_row + ch * kChunk, r);
                tmem_ld_wait();
                float v[kChunk];
                float2* const v2 = reinterpret_cast<float2*>(v);
                if (s_aff != nullptr) {
                    const float4* s4 = reinterpret_cast<const float4*>(s_aff + n0);
                    const float4* b4 = reinterpret_cast<const float4*>(s_aff + p.Cout + n0);
#pragma unroll
                    for (int j = 0; j < kChunk / 4; ++j) {
                        const float4 s = s4[j], t = b4[j];
                        v2[2 * j + 0] = __ffma2_rn(make_float2(__uint_as_float(r[4 * j + 0]), __uint_as_float(r[4 * j + 1])),
                                                   make_float2(s.x, s.y), make_float2(t.x, t.y));
                        v2[2 * j + 1] = __ffma2_rn(make_float2(__uint_as_float(r[4 * j + 2]), __uint_as_float(r[4 * j + 3])),
                                                   make_float2(s.z, s.w), make_float2(t.z, t.w));
                    }
                } else {
                    const float4* s4 = reinterpret_cast<const float4*>(p.scale + n0);
                    const float4* b4 = reinterpret_cast<const float4*>(p.bias + n0);
#pragma unroll
                    for (int j = 0; j < kChunk / 4; ++j) {
                        const float4 s = __ldg(s4 + j), t = __ldg(b4 + j);
                        v2[2 * j + 0] = __ffma2_rn(make_float2(__uint_as_float(r[4 * j + 0]), __uint_as_float(r[4 * j + 1])),
                                                   make_float2(s.x, s.y), make_float2(t.x, t.y));
                        v2[2 * j + 1] = __ffma2_rn(make_float2(__uint_as_float(r[4 * j + 2]), __uint_as_float(r[4 * j + 3])),
                                                   make_float2(s.z, s.w), make_float2(t.z, t.w));
                    }
                }
                // box / chunk position of these 32 columns inside the warp's staged boxes
                const int bx = (ch * kChunk) / T::kBoxCols;
                const int c16 = ((ch * kChunk) % T::kBoxCols) / 8;  // first 16-byte chunk inside the box row
                if (RES != 0) {
                    if (kF32 && use_res && p.res_f32) {
                        // fp32 residual stream: every thread owns one 128-byte row segment per chunk
                        if (RES == 2 && act != 0) {

                            if (act == 1) {
#pragma unroll

                                for (int j = 0; j < kChunk / 2; ++j) v2[j] = gelu_fast2(v2[j]);

                            } else {  // act == 2: ReLU (ResNet backbones)
#pragma unroll

                                for (int j = 0; j < kChunk; ++j) v[j] = fmaxf(v[j], 0.f);

                            }
                        }
                        if (MODE == 4) dropout_chunk(v, pix, n0, p);  // res + drop(act(acc * scale + bias))
                        if (kTransposeF32) {
                            // Coalesced: one warp instruction reads 4 rows x 128 B (8 lanes x 16 B per row), the
                            // 32 x 32 block goes through this warp's (otherwise unused) staging box so that every
                            // thread ends up with its own row.  Rows are 33 words apart: the transposed writes and
                            // the row reads are both bank-conflict free, with constant offsets from one base.
                            float* const tb = reinterpret_cast<float*>(obuf);
                            float* const tq = tb + (lane >> 3) * 33 + (lane & 7) * 4;
                            __syncwarp();
#pragma unroll
                            for (int k = 0; k < 8; ++k) {
                                const float4 f = rf[k];
                                tq[k * 132 + 0] = f.x;
                                tq[k * 132 + 1] = f.y;
                                tq[k * 132 + 2] = f.z;
                                tq[k * 132 + 3] = f.w;
                            }
                            __syncwarp();
#pragma unroll
                            for (int j = 0; j < kChunk / 2; ++j)
                                v2[j] = __fadd2_rn(v2[j], make_float2(tb[lane * 33 + 2 * j], tb[lane * 33 + 2 * j + 1]));
                        } else if (valid) {
                            const float4* r4 = reinterpret_cast<const float4*>(
                                reinterpret_cast<const float*>(p.res) + pix * p.res_ld + n0);
#pragma unroll
                            for (int j = 0; j < kChunk / 4; ++j) {
                                const float4 f = __ldg(r4 + j);
                                v2[2 * j + 0] = __fadd2_rn(v2[2 * j + 0], make_float2(f.x, f.y));
                                v2[2 * j + 1] = __fadd2_rn(v2[2 * j + 1], make_float2(f.z, f.w));
                            }
                        }
                        if (RES == 1 && act != 0) {

                            if (act == 1) {
#pragma unroll

                                for (int j = 0; j < kChunk / 2; ++j) v2[j] = gelu_fast2(v2[j]);

                            } else {  // act == 2: ReLU (ResNet backbones)
#pragma unroll

                                for (int j = 0; j < kChunk; ++j) v[j] = fmaxf(v[j], 0.f);

                            }
                        }
                    } else if (use_res) {
                        uint4 u[4];
                        if (tma_epi) {
                            constexpr int kChunksPerBox = T::kBoxCols / kChunk;
                            if (ch % kChunksPerBox == 0) {  // first use of this box in this tile
                                mbar_wait(&rbar[bx], (rphase >> bx) & 1u);
                                rphase ^= 1u << bx;
                            }
#pragma unroll
                            for (int j = 0; j < 4; ++j)
                                u[j] = *reinterpret_cast<const uint4*>(rbuf + bx * T::kBoxBytes + row_off +
                                                                       (((c16 + j) ^ swz) << 4));
                            if (ch % kChunksPerBox == kChunksPerBox - 1) {  // last use: refill it for the next tile
                                __syncwarp();
                                if (lane == 0 && have_next) res_fetch(n_next, m_next, bx);
                            }
                        } else if (valid) {
                            const uint4* r4 = reinterpret_cast<const uint4*>(p.res + static_cast<long long>(pix) * p.res_ld + n0);
#pragma unroll
                            for (int j = 0; j < 4; ++j) u[j] = __ldg(r4 + j);
                        } else {
#pragma unroll
                            for (int j = 0; j < 4; ++j) u[j] = make_uint4(0u, 0u, 0u, 0u);
                        }
                        if (RES == 2 && act != 0) {

                            if (act == 1) {
#pragma unroll

                                for (int j = 0; j < kChunk / 2; ++j) v2[j] = gelu_fast2(v2[j]);

                            } else {  // act == 2: ReLU (ResNet backbones)
#pragma unroll

                                for (int j = 0; j < kChunk; ++j) v[j] = fmaxf(v[j], 0.f);

                            }
                        }
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const uint32_t uu[4] = {u[j].x, u[j].y, u[j].z, u[j].w};
#pragma unroll
                            for (int t = 0; t < 4; ++t)  // bf16 pair -> fp32 pair, packed add
                                v2[4 * j + t] = __fadd2_rn(v2[4 * j + t], make_float2(__uint_as_float(uu[t] << 16),
                                                                                     __uint_as_float(uu[t] & 0xffff0000u)));
                        }
                        if (RES == 1 && act != 0) {

                            if (act == 1) {
#pragma unroll

                                for (int j = 0; j < kChunk / 2; ++j) v2[j] = gelu_fast2(v2[j]);

                            } else {  // act == 2: ReLU (ResNet backbones)
#pragma unroll

                                for (int j = 0; j < kChunk; ++j) v[j] = fmaxf(v[j], 0.f);

                            }
                        }
                    } else if (act != 0) {

                        if (act == 1) {
#pragma unroll

                            for (int j = 0; j < kChunk / 2; ++j) v2[j] = gelu_fast2(v2[j]);

                        } else {  // act == 2: ReLU (ResNet backbones)
#pragma unroll

                            for (int j = 0; j < kChunk; ++j) v[j] = fmaxf(v[j], 0.f);

                        }
                    }
                } else if (act != 0) {

                    if (act == 1) {
#pragma unroll

                        for (int j = 0; j < kChunk / 2; ++j) v2[j] = gelu_fast2(v2[j]);

                    } else {  // act == 2: ReLU (ResNet backbones)
#pragma unroll

                        for (int j = 0; j < kChunk; ++j) v[j] = fmaxf(v[j], 0.f);

                    }
                }
                if ((MODE == 3 && (p.drop_seg & (seg2 ? 2 : 1))) || (MODE == 4 && RES == 0)) dropout_chunk(v, pix, n0, p);
                if (DOT) {
#pragma unroll
                    for (int k = 0; k < NDOT; ++k) {
                        const float4* w4 = reinterpret_cast<const float4*>(s_dotw + k * BN + colw0 + ch * kChunk);
#pragma unroll
                        for (int j = 0; j < kChunk / 4; ++j) {
                            const float4 wv = w4[j];
                            dsum[k] = fmaf(v[4 * j + 0], wv.x, dsum[k]);
                            dsum[k] = fmaf(v[4 * j + 1], wv.y, dsum[k]);
                            dsum[k] = fmaf(v[4 * j + 2], wv.z, dsum[k]);
                            dsum[k] = fmaf(v[4 * j + 3], wv.w, dsum[k]);
                        }
                    }
                } else if (kF32 && out_ptr != nullptr && p.out_f32 && kTransposeF32) {
                    float* const tb = reinterpret_cast<float*>(obuf);
                    float* const tq = tb + (lane >> 3) * 33 + (lane & 7) * 4;
                    __syncwarp();  // the residual pass (if any) has finished reading the block
#pragma unroll
                    for (int j = 0; j < kChunk; ++j) tb[lane * 33 + j] = v[j];
                    __syncwarp();
                    float* const obase = reinterpret_cast<float*>(out_ptr) + out_col0 + ch * kChunk + (lane & 7) * 4;
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        const long long rp = row_pix(q * 32 + 4 * k + (lane >> 3));
                        const float4 f = make_float4(tq[k * 132 + 0], tq[k * 132 + 1], tq[k * 132 + 2], tq[k * 132 + 3]);
                        if (rp >= 0) *reinterpret_cast<float4*>(obase + rp * p.out_ld) = f;
                    }
                } else if (kF32 && out_ptr != nullptr && p.out_f32) {
                    if (valid) {
                        float4* dst = reinterpret_cast<float4*>(reinterpret_cast<float*>(out_ptr) + pix * p.out_ld +
                                                                out_col0 + ch * kChunk);
#pragma unroll
                        for (int j = 0; j < kChunk / 4; ++j)
                            dst[j] = make_float4(v[4 * j + 0], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                    }
                } else if (out_ptr != nullptr) {
                    uint4 o[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        uint32_t w32[4];
#pragma unroll
                        for (int t = 0; t < 4; ++t) {
                            const __nv_bfloat162 h2 = __floats2bfloat162_rn(v[8 * j + 2 * t], v[8 * j + 2 * t + 1]);
                            w32[t] = *reinterpret_cast<const uint32_t*>(&h2);
                        }
                        o[j] = make_uint4(w32[0], w32[1], w32[2], w32[3]);
                    }
                    if (tma_epi) {
                        constexpr int kChunksPerBoxO = T::kBoxCols / kChunk;
                        if (share && ch != 0 && ch % kChunksPerBoxO == 0) {
                            // the previous box is complete: store it, and wait until the TMA has read the slot
                            // before this chunk overwrites it (this chunk's TMEM load and math are already done)
                            fence_proxy_async_smem();
                            __syncwarp();
                            if (lane == 0) {
                                tma_store_4d(tm_out, obuf, out_col0 + (bx - 1) * T::kBoxCols, slab_w, slab_h, b);
                                tma_store_commit();
                                tma_store_wait_read<0>();
                            }
                            __syncwarp();
                        }
                        uint8_t* const slot = obuf + (share ? 0 : bx * T::kBoxBytes);
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            *reinterpret_cast<uint4*>(slot + row_off + (((c16 + j) ^ swz) << 4)) = o[j];
                    } else if (valid) {  // direct 2x2-replicated store (only when the strided TMA form does not apply)
                        const int h = ph, w = pw;
                        const int out_ld = seg2 ? p.out2_ld : p.out_ld;
#pragma unroll
                        for (int rep = 0; rep < 4; ++rep) {
                            const long long opix = p.up2 ? (static_cast<long long>(b) * (2 * p.H) + 2 * h + (rep >> 1)) *
                                                                   (2 * p.W) + 2 * w + (rep & 1)
                                                         : static_cast<long long>(pix);
                            if (p.up2 || rep == 0) {
                                uint4* dst = reinterpret_cast<uint4*>(out_ptr + opix * out_ld + out_col0 + ch * kChunk);
#pragma unroll
                                for (int j = 0; j < 4; ++j) dst[j] = o[j];
                            }
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[acc]);
            if (!DOT && tma_epi && out_ptr != nullptr) {
                // one TMA store per staged box: full 64/128-byte row segments, rows past the end are clipped
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) {
                    if (share) {  // the last box; the earlier one went out when its slot was recycled
                        tma_store_4d(tm_out, obuf, out_col0 + (T::kBoxesPerWarp - 1) * T::kBoxCols, slab_w, slab_h, b);
                    } else if (!p.up2) {
#pragma unroll
                        for (int bx = 0; bx < T::kBoxesPerWarp; ++bx)
                            tma_store_4d(tm_out, obuf + bx * T::kBoxBytes, out_col0 + bx * T::kBoxCols, slab_w, slab_h, b);
                    } else {
                        // [B, 2H, 2W, C] map walked with traversal stride 2 along w and h: the slab's pixels
                        // land on (2h+i, 2w+j) for the four (i, j)
#pragma unroll
                        for (int rep = 0; rep < 4; ++rep) {
#pragma unroll
                            for (int bx = 0; bx < T::kBoxesPerWarp; ++bx)
                                tma_store_4d(tm_out, obuf + bx * T::kBoxBytes, out_col0 + bx * T::kBoxCols,
                                             2 * slab_w + (rep & 1), 2 * slab_h + (rep >> 1), b);
                        }
                    }
                    tma_store_commit();
                }
            }
            if (GAP) {
                // Per-case channel sums from the staged bf16 boxes (exactly the values the map holds): lane L
                // adds columns 2L, 2L+1 of each box over the slab's valid rows; one atomic per column and warp.
                const int n_valid = __popc(__ballot_sync(0xffffffffu, valid));  // valid rows are a prefix of the slab
                constexpr int kLanes = T::kBoxCols / 2;
                if (lane < kLanes) {
#pragma unroll
                    for (int bx = 0; bx < T::kBoxesPerWarp; ++bx) {
                        float s0 = 0.f, s1 = 0.f;
                        const uint8_t* base = obuf + bx * T::kBoxBytes + (lane & 3) * 4;
#pragma unroll 8
                        for (int rr = 0; rr < n_valid; ++rr) {
                            const int phys = (lane >> 2) ^ (((rr * T::kRowBytes) >> 7) & (T::kRowBytes / 16 - 1));
                            const uint32_t wv = *reinterpret_cast<const uint32_t*>(base + rr * T::kRowBytes + (phys << 4));
                            s0 += __uint_as_float(wv << 16);
                            s1 += __uint_as_float(wv & 0xffff0000u);
                        }
                        float* g = p.gap + static_cast<long long>(b) * p.Cout + nbase + bx * T::kBoxCols + 2 * lane;
                        atomicAdd(g, s0);
                        atomicAdd(g + 1, s1);
                    }
                }
            }
            if (DOT) {
                // The two column halves of a row live in different warps: half 1 parks its 9 partial sums in
                // shared memory (double buffered by accumulator stage), one named barrier over the 8 epilogue
                // warps, half 0 adds its own and writes the row.  Deterministic, no atomics.
                float* buf = s_dots + ((acc & 1) * kBlockM + q * 32 + lane) * NDOT;
                if (half == 1) {
#pragma unroll
                    for (int k = 0; k < NDOT; ++k) buf[k] = dsum[k];
                }
                asm volatile("bar.sync 1, 256;" ::: "memory");
                if (half == 0 && valid) {
                    float* dst = p.dot_out + static_cast<long long>(pix) * NDOT;
#pragma unroll
                    for (int k = 0; k < NDOT; ++k) dst[k] = dsum[k] + buf[k] + p.dot_bias;
                }
            }
            if (++acc == kAcc) {
                acc = 0;
                acc_phase ^= 1;
            }
          }
        }
        if (tma_epi && lane == 0) tma_store_wait_all<0>();  // global writes done before the CTA retires
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc<kTmemCols>(tmem_base);
    }
}

// ------------------------------------------------------------------- host --
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (fn == nullptr) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
            qres != cudaDriverEntryPointSuccess)
            return nullptr;
        fn = reinterpret_cast<EncodeTiledFn>(ptr);
    }
    return fn;
}

static int g_num_sms = 0;
constexpr int kSmemLimit = 227 * 1024;

template <int BN, int RES, bool GAP, int NDOT, int MODE, bool PAIR = false>
static int launch(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmOut, const CUtensorMap& tmOut2,
                  const CUtensorMap& tmRes, const ConvGemmParams& p, int smem_bytes, int grid, cudaStream_t stream) {
    static int configured = 0;
    if (smem_bytes > configured) {
        cudaError_t e = cudaFuncSetAttribute(conv_gemm_kernel<BN, RES, GAP, NDOT, MODE, PAIR>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
        if (e != cudaSuccess) return static_cast<int>(e);
        configured = smem_bytes;
    }
    conv_gemm_kernel<BN, RES, GAP, NDOT, MODE, PAIR>
        <<<grid, kThreads, static_cast<size_t>(smem_bytes), stream>>>(tmA, tmB, tmOut, tmOut2, tmRes, p);
    return static_cast<int>(cudaGetLastError());
}

template <int BN>
static int dispatch(int res_mode, bool gap, int ndot, int mode, const CUtensorMap& tmA, const CUtensorMap& tmB,
                    const CUtensorMap& tmOut, const CUtensorMap& tmOut2, const CUtensorMap& tmRes,
                    const ConvGemmParams& p, int smem_bytes, int grid, cudaStream_t s) {
#define B200_GO(RES, GAP, DOT, MODE) \
    return launch<BN, RES, GAP, DOT, MODE>(tmA, tmB, tmOut, tmOut2, tmRes, p, smem_bytes, grid, s)
    if (mode == 3) {  // MC-dropout epilogue (plain / residual, with or without channel sums)
        if (ndot == 0) {
            if (res_mode == 0 && gap) B200_GO(0, true, 0, 3);
            if (res_mode == 0) B200_GO(0, false, 0, 3);
            if (res_mode == 1 && gap) B200_GO(1, true, 0, 3);
            if (res_mode == 1) B200_GO(1, false, 0, 3);
        }
        return -14;
    }
    if (mode == 2) {  // fp32 residual stream and / or fp32 output (b200_linear)
        if (!gap && ndot == 0 && p.H == 1 && p.BW == kBlockM && p.drop_seg != 0) {  // b200_linear_mc
            if (res_mode == 0) B200_GO(0, false, 0, 4);
            if (res_mode == 2) B200_GO(2, false, 0, 4);
            return -14;
        }
        if (!gap && ndot == 0 && p.H == 1 && p.BW == kBlockM) {
            if (res_mode == 0) B200_GO(0, false, 0, 2);
            if (res_mode == 1) B200_GO(1, false, 0, 2);
            if (res_mode == 2) B200_GO(2, false, 0, 2);
        }
        return -14;
    }
    if (ndot != 0) {
        if constexpr (BN == 128) {
            // paired M tiles for the N = 128 tap-dot layers too (3x3 128->128 + GELU + nine dots, the reconstruction
            // heads): the unpaired 128 x 128 tiles were shared-memory-feed bound like the plain ones
            if (p.pair && res_mode == 0 && !gap && ndot == 9)
                return launch<BN, 0, false, 9, 0, true>(tmA, tmB, tmOut, tmOut2, tmRes, p, smem_bytes, grid, s);
            if (p.pair) return -14;
        }
        if (res_mode == 0 && !gap && ndot == 9) B200_GO(0, false, 9, 0);
        if (res_mode == 0 && !gap && ndot == 1) B200_GO(0, false, 1, 0);
        return -14;
    }
    if constexpr (BN == 128 || BN == 64) {
        if (p.pair) {
#define B200_GO_PAIR(RES, GAP) \
    return launch<BN, RES, GAP, 0, 0, true>(tmA, tmB, tmOut, tmOut2, tmRes, p, smem_bytes, grid, s)
            if (res_mode == 0 && gap) B200_GO_PAIR(0, true);
            if (res_mode == 0) B200_GO_PAIR(0, false);
            if (res_mode == 1 && gap) B200_GO_PAIR(1, true);
            if (res_mode == 1) B200_GO_PAIR(1, false);
            if (res_mode == 2 && !gap) B200_GO_PAIR(2, false);
#undef B200_GO_PAIR
            return -14;
        }
    }
    if (res_mode == 0) {
        if (gap) B200_GO(0, true, 0, 0);
        B200_GO(0, false, 0, 0);
    }
    if (res_mode == 1) {
        if (gap) B200_GO(1, true, 0, 0);
        B200_GO(1, false, 0, 0);
    }
    if (res_mode == 2 && !gap) B200_GO(2, false, 0, 0);
    return -14;
#undef B200_GO
}

// Identity scale / zero bias for callers that pass NULL (immutable, allocated once per process).
static const float* identity_affine(bool ones) {
    static float* buf = nullptr;
    constexpr int kN = 8192;
    if (buf == nullptr) {
        float* d = nullptr;
        if (cudaMalloc(&d, 2 * kN * sizeof(float)) != cudaSuccess) return nullptr;
        float* h = static_cast<float*>(std::malloc(2 * kN * sizeof(float)));
        for (int i = 0; i < kN; ++i) {
            h[i] = 1.f;
            h[kN + i] = 0.f;
        }
        cudaMemcpy(d, h, 2 * kN * sizeof(float), cudaMemcpyHostToDevice);
        std::free(h);
        buf = d;
    }
    return ones ? buf : buf + kN;
}

static inline int align1k(int v) { return (v + 1023) & ~1023; }

// Lays out shared memory for BN and returns the total dynamic size, or -1 if the configuration does not fit / leaves
// fewer than 3 ring stages.
static int plan_smem(ConvGemmParams& p, int BN, bool has_out, bool has_res, int ndot, int mode, bool share_box,
                     bool pair) {
    const int b_bytes = BN * kBlockK * 2;
    const int stage_bytes = (pair ? 2 * kABytes : kABytes) + b_bytes;
    const int box_all = kBlockM * BN * 2;  // 8 warps x (32 rows x BN/2 columns) of bf16
    const int dot_bytes = ndot * BN * 4 + 2 * kBlockM * ndot * 4;
    // mode 2 (fp32 epilogue) needs only the eight 32 x 33-word transposition blocks
    // One-k-block-deep layers (1x1, Cin <= 256) are epilogue bound, and with one set of staging boxes every tile's
    // epilogue starts by waiting for the previous tile's TMA store to finish reading them: a second set hides that.
    const bool want2 = BN <= 128 && (mode == 0 || mode == 3) && has_out && !share_box && ndot == 0 && p.tma_epi &&
                       p.k_blocks <= 4;
    int out_stage = mode == 2 ? 8 * kF32BlockBytes : (share_box ? box_all / 2 : box_all);
    p.obuf2 = 0;
    if (want2) {
        const int fixed2 = align1k(kBarBytes) + align1k(2 * box_all) + (has_res ? align1k(box_all) : 0) + 1024;
        if ((kSmemLimit - fixed2) / stage_bytes >= 4) {
            out_stage = 2 * box_all;
            p.obuf2 = 1;
        }
    }
    const int union_bytes = align1k(ndot ? dot_bytes : (has_out ? out_stage : 0));
    const int rbox_bytes = has_res ? align1k(box_all) : 0;
    const int aff_bytes = ((BN <= 128 || p.k_blocks <= 4) && p.Cout <= 2048) ? align1k(2 * p.Cout * 4) : 0;
    const int fixed = align1k(kBarBytes) + union_bytes + rbox_bytes + aff_bytes + 1024 /*alignment slack*/;
    int stages = (kSmemLimit - fixed) / stage_bytes;
    if (stages > kMaxStages) stages = kMaxStages;
    if (stages < 3) return -1;
    p.stages = stages;
    p.off_bar = stages * stage_bytes;
    p.off_union = p.off_bar + align1k(kBarBytes);
    p.off_rbox = p.off_union + union_bytes;
    p.off_aff = aff_bytes ? p.off_rbox + rbox_bytes : -1;
    return fixed + stages * stage_bytes;
}

// A 4-D bf16 view {cols, W, H, B} (element strides) for cuTensorMapEncodeTiled.
struct View4 {
    const void* base;
    long long dims[4];
    long long strides[3];  // elements: W-step, H-step, B-step (cols are contiguous)
};

static int encode_view(EncodeTiledFn encode, CUtensorMap* tm, const View4& v, const int box[4], const int estr[4],
                       CUtensorMapSwizzle swz, CUtensorMapL2promotion promo) {
    cuuint64_t dims[4], strides[3];
    cuuint32_t bx[4], es[4];
    for (int i = 0; i < 4; ++i) {
        dims[i] = static_cast<cuuint64_t>(v.dims[i] > 0 ? v.dims[i] : 1);
        bx[i] = static_cast<cuuint32_t>(box[i]);
        es[i] = static_cast<cuuint32_t>(estr[i]);
    }
    for (int i = 0; i < 3; ++i) {
        // a degenerate dimension still needs a legal (16-byte multiple, non-zero) stride
        long long st = v.strides[i] > 0 ? v.strides[i] : v.dims[0];
        strides[i] = static_cast<cuuint64_t>(st) * 2;
        if (strides[i] % 16 != 0) return -400;
    }
    if (reinterpret_cast<uintptr_t>(v.base) & 15) return -401;
    CUresult r = encode(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(v.base), dims, strides, bx, es,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, swz, promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : -300 - static_cast<int>(r);
}

// Everything the two C entry points hand to the common launcher.
struct GemmJob {
    View4 a;       // {K, W, H, B}: K-major rows of the A operand (the activations)
    const void* w; // 2-D weights [N, K]
    View4 out, out2, res;  // {cols, W', H', B}
    int K;         // reduction length = taps * Cin
};

static int run_job(ConvGemmParams& p, const GemmJob& j, int mode, cudaStream_t stream) {
    if (g_num_sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
        if (g_num_sms <= 0) return -9;
    }
    EncodeTiledFn encode = get_encode_fn();
    if (encode == nullptr) return -8;
    const int Cout = p.Cout, n_split = p.n_split;
    const bool two = n_split < Cout;
    const int seg2 = Cout - n_split;
    const bool has_out = p.out != nullptr;
    const bool has_res = p.res_mode != 0 && mode != 2;  // an fp32 residual is never staged by TMA
    const int ndot = p.dot_w != nullptr ? p.ndot : 0;
    auto divides = [&](int bn) { return Cout % bn == 0 && n_split % bn == 0 && (!two || seg2 % bn == 0); };
    int BN = 0, smem_bytes = -1;
    // TMA-staged epilogue?  Needs the warp's 32-row slab to be a {bw, bh} box and bf16 output / residual.
    const bool slab_is_box = p.BB == 1 && p.BW * p.BH == kBlockM && (p.BW % 32 == 0 || 32 % p.BW == 0) &&
                             (p.H == 1 || p.H % p.BH == 0);
    p.tma_epi = (p.res_f32 || p.out_f32 || !slab_is_box) ? 0 : 1;
    p.share_box = 0;
    for (int bn : {256, 128, 64}) {
        if (!divides(bn) || (ndot != 0 && bn != Cout)) continue;
        // BN = 256 with a plain staged output: one 4 KB slot per warp instead of two buys a 4th ring stage,
        // and the kernel is TMA-latency bound with three (measured: 2 -> 3 stages = +17..32 %)
        const bool share = bn == 256 && p.tma_epi && has_out && !has_res && p.gap == nullptr && ndot == 0 &&
                           mode == 0 && !p.up2;
        // staging boxes exist only for the TMA epilogue (mode 2 keeps its transposition blocks)
        const bool st_out = has_out && (p.tma_epi || mode == 2), st_res = has_res && p.tma_epi;
        // BN = 128: pair two M tiles per iteration when there is enough work to keep every SM busy with pairs
        // (N = 64: only the 3x3 layers gain - 64->64 0.211 -> 0.158 ms; the 1x1 layers lose 5-9 %)
        const bool pair = ((bn == 128 && (ndot == 0 || ndot == 9)) || (bn == 64 && ndot == 0 && p.k_blocks >= 8)) &&
                          mode == 0 && (p.m_tiles / 2) * (Cout / bn) >= g_num_sms;
        smem_bytes = plan_smem(p, bn, st_out, st_res, ndot, mode, share, pair);
        p.pair = (pair && smem_bytes > 0) ? 1 : 0;
        if (pair && smem_bytes <= 0) smem_bytes = plan_smem(p, bn, st_out, st_res, ndot, mode, share, false);
        if (smem_bytes > 0) {
            BN = bn;
            p.share_box = share ? 1 : 0;
            break;
        }
    }
    if (BN == 0) return -13;
    p.n_tiles = Cout / BN;
    {
        auto fd = [](int d) {
            ConvGemmParams::FastDiv f;
            f.d = static_cast<uint32_t>(d);
            f.m = d == 1 ? 0u : static_cast<uint32_t>((1ull << 32) / static_cast<uint32_t>(d)) + 1u;
            return f;
        };
        p.fd_ntiles = fd(p.n_tiles);
        p.fd_tw = fd(p.tiles_w);
        p.fd_th = fd(p.tiles_h);
        p.fd_twth = fd(p.tiles_w * p.tiles_h);
        // exactness bound of the multiply-high division: n * d < 2^32 for every n the kernel divides
        const unsigned long long n_max = static_cast<unsigned long long>(p.m_tiles + 2) * p.n_tiles + 2ull * g_num_sms;
        if (n_max * static_cast<unsigned long long>(p.tiles_w) * p.tiles_h >= (1ull << 32) ||
            n_max * p.n_tiles >= (1ull << 32))
            return -21;
    }
    if (Cout > 8192) return -15;
    if (p.scale == nullptr) p.scale = identity_affine(true);
    if (p.bias == nullptr) p.bias = identity_affine(false);
    if (p.scale == nullptr || p.bias == nullptr) return -16;

    CUtensorMap tmA, tmB, tmOut, tmOut2, tmRes;
    int rc;
    {
        const int s = p.cstride;
        const int box[4] = {64, p.BW * s, p.BH * s, p.BB};
        const int estr[4] = {1, s, s, 1};
        if ((rc = encode_view(encode, &tmA, j.a, box, estr, CU_TENSOR_MAP_SWIZZLE_128B,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_256B)) != 0)
            return rc - 1000;
    }
    {
        const cuuint64_t dims[2] = {static_cast<cuuint64_t>(j.K), static_cast<cuuint64_t>(Cout)};
        const cuuint64_t strides[1] = {static_cast<cuuint64_t>(j.K) * 2};
        const cuuint32_t box[2] = {64, static_cast<cuuint32_t>(BN)};
        const cuuint32_t estr[2] = {1, 1};
        CUresult r = encode(&tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(j.w), dims, strides, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                            CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return -200 - static_cast<int>(r);
    }
    // Staged (TMA) epilogue: per epilogue warp one {cw columns, bw, bh} box = its 32 rows x BN/2 columns
    // (two boxes when BN = 256), swizzled by the row width.  The 2x2-replicating store walks a
    // [B, 2H, 2W, ld] map with a traversal stride of 2 along w and h.
    tmOut = tmA;
    tmOut2 = tmA;
    tmRes = tmA;
    p.a_box_bytes = p.BW * p.BH * p.BB * kBlockK * 2;
    if (p.tma_epi) {
        const int cw = BN / 2 < 64 ? BN / 2 : 64;
        const CUtensorMapSwizzle swz = cw == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
        const int bw = p.BW < 32 ? p.BW : 32, bh = 32 / bw;
        const int us = p.up2 ? 2 : 1;
        const int obox[4] = {cw, bw * us, bh * us, 1};
        const int oestr[4] = {1, us, us, 1};
        const int rbox[4] = {cw, bw, bh, 1};
        const int one[4] = {1, 1, 1, 1};
        if (has_out && (rc = encode_view(encode, &tmOut, j.out, obox, oestr, swz, CU_TENSOR_MAP_L2_PROMOTION_NONE)) != 0)
            return rc - 3000;
        if (two && (rc = encode_view(encode, &tmOut2, j.out2, rbox, one, swz, CU_TENSOR_MAP_L2_PROMOTION_NONE)) != 0)
            return rc - 4000;
        if (has_res && (rc = encode_view(encode, &tmRes, j.res, rbox, one, swz, CU_TENSOR_MAP_L2_PROMOTION_NONE)) != 0)
            return rc - 5000;
    }
    const int total = p.pair ? ((p.m_tiles + 1) / 2) * p.n_tiles : p.m_tiles * p.n_tiles;
    const int grid = total < g_num_sms ? total : g_num_sms;
    const bool g = p.gap != nullptr;
    const int rm = p.res_mode;
    if (BN == 256) return dispatch<256>(rm, g, ndot, mode, tmA, tmB, tmOut, tmOut2, tmRes, p, smem_bytes, grid, stream);
    if (BN == 128) return dispatch<128>(rm, g, ndot, mode, tmA, tmB, tmOut, tmOut2, tmRes, p, smem_bytes, grid, stream);
    return dispatch<64>(rm, g, ndot, mode, tmA, tmB, tmOut, tmOut2, tmRes, p, smem_bytes, grid, stream);
}

}  // namespace b200

static int conv_gemm_launch(const void* x, int x_ld, const void* w, const float* scale, const float* bias,
                            const void* res, int res_ld, int res_mode, int act, void* out, int out_ld, int up2,
                            float* gap, int n_split, void* out2, int out2_ld, int act2, const float* dot_w, int ndot,
                            float dot_bias, float* dot_out, int B, int H, int W, int Cin, int Cout, int taps,
                            int stride, int dilation, b200::DropoutArgs drop, void* stream) {
    using namespace b200;
    if (dilation < 1 || dilation > 8 || (dilation != 1 && taps != 9)) return -6;
    if (dot_w == nullptr) ndot = 0;
    if (ndot != 0 && ndot != 1 && ndot != 9) return -18;
    if (x == nullptr || w == nullptr || B <= 0 || H <= 0 || W <= 0) return -1;
    if (Cin % 64 != 0 || Cout % 64 != 0 || (taps != 1 && taps != 9 && taps != 4)) return -2;
    if (x_ld % 8 != 0 || x_ld < Cin || (out != nullptr && out_ld % 8 != 0)) return -3;
    if (res_mode != 0 && (res == nullptr || res_ld % 8 != 0)) return -4;
    if ((reinterpret_cast<uintptr_t>(x) & 15) || (reinterpret_cast<uintptr_t>(w) & 15) ||
        (reinterpret_cast<uintptr_t>(out) & 15) || (reinterpret_cast<uintptr_t>(res) & 15))
        return -5;

    ConvGemmParams p{};
    p.BB = 1;
    p.B = B;
    if (stride != 1 && stride != 2) return -6;
    if (n_split <= 0 || n_split > Cout || n_split % 64 != 0) return -10;
    const bool two = n_split < Cout;
    // taps == 4: 2x2 kernel, stride 2, no padding (patch embedding); taps 1 / 9 with stride 2: the strided 1x1 and
    // 3x3 (padding 1) convolutions of down-sampling blocks and of the mask head (input pixel 2*o + tap - pad)
    const int cs = taps == 4 ? 2 : stride;
    if (cs == 2 && (H % 2 != 0 || W % 2 != 0 || up2 || H == 1)) return -6;
    const int Ho = H / cs, Wo = W / cs;  // output map
    if (H == 1) {  // plain GEMM over W rows: 128-row boxes, ragged tail handled by TMA OOB fill / clipping
        if (taps != 1 || up2) return -6;
        p.BW = 128;
        p.BH = 1;
        p.tiles_w = (W + 127) / 128;
        p.tiles_h = 1;
    } else {
        // A tile is BW x BH output pixels of one case with BW = W.  Maps whose width does not divide 128
        // (the 14 x 14 ViT grid: 14 x 9 = 126-row tiles, two per case) leave the last MMA rows unused and
        // take the direct (non-TMA) epilogue; rows past the map come back as zeros from the TMA OOB fill.
        if (Wo > 128) return -7;
        p.BW = Wo;
        p.BH = 128 / Wo;
        p.tiles_w = 1;
        p.tiles_h = (Ho + p.BH - 1) / p.BH;
        const bool ragged = p.BW * p.BH != 128 || Ho % p.BH != 0;
        if (ragged && (up2 || gap != nullptr)) return -7;
        // Small ragged maps: a tile may span several cases (the 4th box dimension).  14 x 14 (ViT grid) as 9-row tiles
        // fills 196 of every 256 MMA rows; one image row of 9 consecutive cases per tile fills 126 of 128.  Pick the
        // (rows, cases) box with the best fill; plain stride-1 convolutions with the direct epilogue only.
        if (ragged && cs == 1 && !two && dot_w == nullptr && B > 1) {
            double best = static_cast<double>(Ho) * Wo / (p.tiles_h * 128.0);
            int best_bh = p.BH, best_bb = 1;
            for (int bh = 1; bh <= Ho && bh * Wo <= 128; ++bh) {
                int bb = 128 / (bh * Wo);
                if (bb > B) bb = B;
                if (bb > 256) bb = 256;
                const int groups = (B + bb - 1) / bb;
                const double fill = static_cast<double>(B) * Ho * Wo / (static_cast<double>(groups) * ((Ho + bh - 1) / bh) * 128.0);
                if (fill > best + 0.02) {
                    best = fill;
                    best_bh = bh;
                    best_bb = bb;
                }
            }
            p.BH = best_bh;
            p.BB = best_bb;
            p.tiles_h = (Ho + p.BH - 1) / p.BH;
        }
    }
    p.H = Ho;
    p.W = Wo;
    p.Cout = Cout;
    if (two && (out2 == nullptr || out2_ld % 8 != 0 || (reinterpret_cast<uintptr_t>(out2) & 15) || gap != nullptr ||
                up2 || dot_w != nullptr || res_mode != 0))
        return -11;
    if (gap != nullptr && (out == nullptr || up2)) return -17;  // channel sums are taken from the staged output boxes
    if (dot_w != nullptr && (dot_out == nullptr || H == 1 || out != nullptr)) return -12;
    p.m_tiles = ((B + p.BB - 1) / p.BB) * p.tiles_w * p.tiles_h;
    p.kc = Cin / 64;
    p.taps = taps;
    p.k_blocks = taps * p.kc;
    p.cstride = cs;
    p.dil = dilation;
    p.scale = scale;
    p.bias = bias;
    p.res = static_cast<const __nv_bfloat16*>(res);
    p.res_ld = res_ld;
    p.res_mode = res_mode;
    p.act = act;
    p.out = static_cast<__nv_bfloat16*>(out);
    p.out_ld = out_ld;
    p.up2 = up2;
    p.gap = gap;
    p.n_split = n_split;
    p.out2 = static_cast<__nv_bfloat16*>(out2);
    p.out2_ld = out2_ld;
    p.act2 = act2;
    p.dot_w = dot_w;
    p.ndot = ndot;
    p.dot_out = dot_out;
    p.dot_bias = dot_bias;

    GemmJob j{};
    j.K = taps * Cin;
    j.w = w;
    j.a = View4{x, {Cin, W, H, B}, {x_ld, static_cast<long long>(x_ld) * W, static_cast<long long>(x_ld) * W * H}};
    const int us = up2 ? 2 : 1;
    j.out = View4{out, {n_split, static_cast<long long>(Wo) * us, static_cast<long long>(Ho) * us, B},
                  {out_ld, static_cast<long long>(out_ld) * Wo * us, static_cast<long long>(out_ld) * Wo * us * Ho * us}};
    j.out2 = View4{out2, {Cout - n_split, Wo, Ho, B},
                   {out2_ld, static_cast<long long>(out2_ld) * Wo, static_cast<long long>(out2_ld) * Wo * Ho}};
    j.res = View4{res, {n_split, Wo, Ho, B},
                  {res_ld, static_cast<long long>(res_ld) * Wo, static_cast<long long>(res_ld) * Wo * Ho}};
    int mode = 0;
    if (drop.seg != 0) {
        if (dot_w != nullptr || up2 || res_mode == 2) return -19;  // dropout variants: plain / residual (+ channel sums)
        mode = 3;
        p.drop_thresh = dropout_threshold(drop.p);
        p.drop_scale = 1.0f / (1.0f - drop.p);
        p.drop_seed_lo = static_cast<unsigned int>(drop.seed);
        p.drop_seed_hi = static_cast<unsigned int>(drop.seed >> 32);
        p.drop_seg = drop.seg;
    }
    return run_job(p, j, mode, static_cast<cudaStream_t>(stream));
}
extern "C" int b200_conv_gemm_ex(const void* x, int x_ld, const void* w, const float* scale, const float* bias,
                                 const void* res, int res_ld, int res_mode, int act, void* out, int out_ld, int up2,
                                 float* gap, int n_split, void* out2, int out2_ld, int act2, const float* dot_w,
                                 int ndot, float dot_bias, float* dot_out, int B, int H, int W, int Cin, int Cout,
                                 int taps, int stride, int dilation, void* stream) {
    return conv_gemm_launch(x, x_ld, w, scale, bias, res, res_ld, res_mode, act, out, out_ld, up2, gap, n_split, out2,
                            out2_ld, act2, dot_w, ndot, dot_bias, dot_out, B, H, W, Cin, Cout, taps, stride, dilation,
                            b200::DropoutArgs{}, stream);
}

// b200_conv_gemm_ex with the MC-dropout epilogue: elements of the selected output segments (bit 0: out, bit 1: out2)
// are zeroed with probability drop_p and the survivors scaled by 1 / (1 - drop_p) after the activation.
extern "C" int b200_conv_gemm_mc(const void* x, int x_ld, const void* w, const float* scale, const float* bias,
                                 const void* res, int res_ld, int res_mode, int act, void* out, int out_ld, int up2,
                                 float* gap, int n_split, void* out2, int out2_ld, int act2, const float* dot_w,
                                 int ndot, float dot_bias, float* dot_out, int B, int H, int W, int Cin, int Cout,
                                 int taps, int stride, int dilation, float drop_p, unsigned long long drop_seed,
                                 int drop_segments, void* stream) {
    if (!b200::dropout_args_valid(drop_p, drop_segments)) return -19;
    b200::DropoutArgs d;
    d.p = drop_p;
    d.seed = drop_seed;
    d.seg = drop_p > 0.f ? drop_segments : 0;
    return conv_gemm_launch(x, x_ld, w, scale, bias, res, res_ld, res_mode, act, out, out_ld, up2, gap, n_split, out2,
                            out2_ld, act2, dot_w, ndot, dot_bias, dot_out, B, H, W, Cin, Cout, taps, stride, dilation, d,
                            stream);
}

static int linear_launch(const void* x, long long M, int K, const void* w, int N, const float* scale, const float* bias,
                         const void* res, int res_f32, int res_mode, int act, void* out, int out_f32,
                         b200::DropoutArgs drop, void* stream) {
    using namespace b200;
    if (x == nullptr || w == nullptr || out == nullptr || M <= 0 || M > 0x7fffffffLL) return -1;
    if (K % 64 != 0 || N % 64 != 0) return -2;
    if (res_mode != 0 && res == nullptr) return -4;
    ConvGemmParams p{};
    p.BB = 1;
    p.B = 1;
    p.H = 1;
    p.W = static_cast<int>(M);
    p.BW = 128;
    p.BH = 1;
    p.tiles_w = static_cast<int>((M + 127) / 128);
    p.tiles_h = 1;
    p.Cout = N;
    p.n_split = N;
    p.m_tiles = p.tiles_w;
    p.kc = K / 64;
    p.taps = 1;
    p.k_blocks = p.kc;
    p.cstride = 1;
    p.scale = scale;
    p.bias = bias;
    p.res = static_cast<const __nv_bfloat16*>(res);
    p.res_ld = N;
    p.res_mode = res_mode;
    p.res_f32 = res_mode != 0 ? res_f32 : 0;
    p.act = act;
    p.out = static_cast<__nv_bfloat16*>(out);
    p.out_ld = N;
    p.out_f32 = out_f32;
    GemmJob j{};
    j.K = K;
    j.w = w;
    j.a = View4{x, {K, M, 1, 1}, {K, 0, 0}};
    j.out = View4{out, {N, M, 1, 1}, {N, 0, 0}};
    j.res = View4{res, {N, M, 1, 1}, {N, 0, 0}};
    int mode = (p.res_f32 || p.out_f32) ? 2 : 0;
    if (drop.seg != 0) {  // fp32 epilogue: mode 2 with the dropout instantiations (4); bf16 without residual: mode 3
        if (mode == 0) mode = 3;
        p.drop_thresh = dropout_threshold(drop.p);
        p.drop_scale = 1.0f / (1.0f - drop.p);
        p.drop_seed_lo = static_cast<unsigned int>(drop.seed);
        p.drop_seed_hi = static_cast<unsigned int>(drop.seed >> 32);
        p.drop_seg = drop.seg;
    }
    return run_job(p, j, mode, static_cast<cudaStream_t>(stream));
}

extern "C" int b200_linear(const void* x, long long M, int K, const void* w, int N, const float* scale, const float* bias,
                           const void* res, int res_f32, int res_mode, int act, void* out, int out_f32,
                           void* stream) {
    return linear_launch(x, M, K, w, N, scale, bias, res, res_f32, res_mode, act, out, out_f32, b200::DropoutArgs{},
                         stream);
}

// b200_linear with MC dropout before the residual add: out = res + drop(act(acc * scale + bias)).
extern "C" int b200_linear_mc(const void* x, long long M, int K, const void* w, int N, const float* scale,
                              const float* bias, const void* res, int res_f32, int res_mode, int act, void* out,
                              int out_f32, float drop_p, unsigned long long drop_seed, void* stream) {
    if (!b200::dropout_args_valid(drop_p, 1)) return -19;
    // the residual must be fp32 (a bf16 one goes through mode 3, whose dropout sits after the residual), and added
    // after the activation: res_mode 1 is accepted without one, where it is the same as 2
    if (res_mode != 0 && (res_f32 == 0 || (res_mode == 1 && act != 0))) return -19;
    if (drop_p == 0.f) return b200_linear(x, M, K, w, N, scale, bias, res, res_f32, res_mode, act, out, out_f32, stream);
    b200::DropoutArgs d;
    d.p = drop_p;
    d.seed = drop_seed;
    d.seg = 1;
    return linear_launch(x, M, K, w, N, scale, bias, res, res_f32, res_mode == 1 ? 2 : res_mode, act, out, out_f32, d,
                         stream);
}
