/*
 * C ABI of the B200-native DWI+DCE fusion-classifier hot path.
 *
 * The reference (simhelgithub/Deep-Multimodal-Fusion-of-DCE-MRI-and-DWI-...) has no FFI:
 * its boundary is the Python module surface (SURVEY.md section 8b).  Every entry point
 * below is therefore the native half of one reference Python function or nn.Module
 * forward; the Python mirror of that function (same name and arguments) lives in the
 * package directory and calls these through ctypes.  Each declaration cites the
 * reference code it replaces (paths relative to /root/reference/).
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name ends in _host;
 *   - the caller allocates every output and workspace; nothing is retained between calls
 *     except immutable cached launch attributes;
 *   - `stream` is a cudaStream_t passed as void*; every call is asynchronous on it;
 *   - return value: 0 = launched, <0 = invalid argument (nothing launched),
 *     >0 = cudaError_t from the launch;
 *   - activations ("maps") are NHWC bfloat16 unless stated; `*_ld` is the element
 *     stride between consecutive pixels (>= channels, multiple of 8).
 */
#ifndef B200_FUSION_H
#define B200_FUSION_H

#ifdef __cplusplus
extern "C" {
#endif

/* Library/ABI version; bumped whenever a signature changes. */
int b200_abi_version(void);

/*
 * Implicit-GEMM convolution (1x1, 3x3 / padding 1 or 2x2 / stride 2) or linear layer with fused
 * epilogue, tcgen05/TMEM + TMA.  Replaces nn.Conv2d+BatchNorm2d(eval)+GELU(+residual)
 * stacks: code/model_module.py:259-269 (bottleneck), :276-280 (skip), :113-118
 * (ReconHead), :150 (MaskHeadResize.pre), :337-345 (Projector), :386-390
 * (FeatureDownAlign), :857-858 (FusionModel.proj_in_*), and nn.Linear at
 * code/transformer_model.py:93,95,123,125.
 *   x      [B,H,W,x_ld] bf16, channels [0,Cin) are read; H==1 selects plain-GEMM mode
 *          (W = number of rows, any value)
 *   w      [Cout, taps*Cin] bf16, k = tap*Cin + c, tap = ky*3+kx
 *   scale, bias  fp32 [Cout] per-output-channel affine (folded BatchNorm or conv bias); NULL = 1 / 0
 *   res    optional residual map (bf16, res_ld); res_mode 0 none, 1 add before the
 *          activation, 2 add after it
 *   act    0 none, 1 GELU, 2 ReLU
 *   out    bf16 map (out_ld), or NULL to skip the store; up2 != 0 replicates every pixel
 *          into a 2x2 block of a [B,2H,2W,out_ld] map (AdaptiveAvgPool2d to twice the
 *          size, model_module.py:534,707-710, commuted past the 1x1 projector)
 *   gap    optional fp32 [B,Cout]; the per-case sum over pixels of the epilogue result is
 *          ACCUMULATED into it (caller zeroes it)
 *   n_split/out2/out2_ld/act2: output channels [n_split, Cout) are a second layer that reads the same
 *     input (e.g. a block's skip conv and first bottleneck conv, code/model_module.py:299 and :303) and
 *     go to out2 with their own activation flag (no residual / gap / up2 on either segment then);
 *     n_split == Cout disables it.
 *   dot_w [ndot,Cout] fp32 / dot_out [pixels,ndot] fp32, ndot in {1, 9}: instead of storing the map, emits
 *     per pixel the ndot dot products of the fp32 epilogue result with dot_w[k,:] (+ dot_bias).  ndot = 9:
 *     the per-tap partial sums of the ReconHead's final 3x3, C -> 1 convolution
 *     (code/model_module.py:117), finished by b200_tapsum.  ndot = 1: a following 1x1, C -> 1 convolution
 *     (MaskHeadResize.out, code/model_module.py:187).  Requires Cout in {64,128,256} (one N tile), H > 1
 *     and out == NULL: the C-channel map never reaches HBM and is never rounded to bf16.
 *     dot_w == NULL disables it.
 * taps may also be 4: a 2x2 kernel with stride 2 and no padding (PatchEmbed, code/transformer_model.py:18-23),
 * k = (ky*2+kx)*Cin + c; the output map is then [B,H/2,W/2,*].
 * `stride` (1 or 2) applies to taps 1 / 9: the strided 1x1 convs of a down-sampling ResNetLiteBlock
 * (code/model_module.py:259-262, :276-280) and the 3x3 / stride-2 / padding-1 stacks of MaskHeadResize (:153-181);
 * H and W are the INPUT size, the output map is H/stride x W/stride.  `dilation` (>= 1, taps 9 only; padding =
 * dilation) serves the dilated layer3 / layer4 of the ResNet-50 backbones built with output_stride 8
 * (code/foundation_model.py:243-250).
 * Requires Cin % 64 == 0, Cout % 64 == 0, and for convolutions Wout <= 128; up2 and gap also need
 * 128 % Wout == 0 and Hout % (128/Wout) == 0.
 */
int b200_conv_gemm_ex(const void* x, int x_ld, const void* w, const float* scale, const float* bias,
                      const void* res, int res_ld, int res_mode, int act, void* out, int out_ld, int up2,
                      float* gap, int n_split, void* out2, int out2_ld, int act2, const float* dot_w, int ndot,
                      float dot_bias, float* dot_out, int B, int H, int W, int Cin, int Cout, int taps,
                      int stride, int dilation, void* stream);

/*
 * b200_conv_gemm_ex with the MC-dropout epilogue (code/train_fusion.py:478-536: nn.Dropout modules in train mode,
 * BatchNorm frozen; the dropouts of ResNetLiteBlock_withRecon, code/model_module.py:260, :271, :306).  The request is
 * part of the argument list - there is no ambient or per-thread state: each element of the selected output segments
 * (drop_segments bit 0 = out, bit 1 = out2) is zeroed with probability drop_p and the survivors are scaled by
 * 1 / (1 - drop_p), after the activation and before the store / channel sums.  Decisions are
 * Philox4x32-7(drop_seed; pixel * Cout + channel): reproducible for a given seed, statistically (not bitwise)
 * comparable with torch's generator.  drop_p outside [0, 1) or drop_segments outside [0, 3] -> -19.
 */
int b200_conv_gemm_mc(const void* x, int x_ld, const void* w, const float* scale, const float* bias,
                      const void* res, int res_ld, int res_mode, int act, void* out, int out_ld, int up2,
                      float* gap, int n_split, void* out2, int out2_ld, int act2, const float* dot_w, int ndot,
                      float dot_bias, float* dot_out, int B, int H, int W, int Cin, int Cout, int taps,
                      int stride, int dilation, float drop_p, unsigned long long drop_seed, int drop_segments,
                      void* stream);

/*
 * Fused multi-head self-attention: out[b, n, h*dh : (h+1)*dh] = softmax(q k^T * scale) v for every case b and head h,
 * from the packed rows qkv[b*N + n, :] = q | k | v (each [heads, dh]) that `Linear(E, 3E)` produces - the reference's
 * MultiHeadSelfAttention.forward between its qkv and proj layers (code/transformer_model.py:101-112; attn_drop is
 * identity in eval mode) and the timm ViT-B/16 attention of the backbone (code/foundation_model.py:371-431).
 * One launch, no score / probability buffer in HBM: S in TMEM -> softmax in registers -> P in shared memory -> P V.
 * N <= 256 holds a query tile's whole score row in TMEM; 256 < N <= 16384 streams the keys in 128-key tiles through an
 * online softmax.  bf16 in / out, fp32 accumulation and softmax.  1 <= N <= 16384 tokens, dh in {64, 128}; qkv_ld >=
 * 3*heads*dh, out_ld >= heads*dh, both multiples of 8 elements, 16-byte aligned bases.  Returns 0 (also for B == 0,
 * nothing launched), -1 unsupported shape (N or dh out of range, B < 0, heads <= 0, or more than 2^31 - 1 work items
 * B * heads * ceil(N / 128) at N > 256), -2 null pointer, -3 leading dimensions, -5 alignment, -8 / -9 / <= -1000
 * driver or tensor-map errors, > 0 a CUDA error of the launch.  Nothing is launched when the result is < 0.
 */
int b200_attention(const void* qkv, int qkv_ld, void* out, int out_ld, int B, int N, int heads, int dh, float scale,
                   void* stream);

/*
 * b200_attention with the attention dropout of MC-dropout inference (nn.Dropout(drop_p) in train mode on the softmax
 * probabilities, code/transformer_model.py:109-116): probability (b, h, n, j) is kept when word j % 4 of
 * Philox4x32-7(drop_seed; ((b * heads + h) * N + n) * 64 * ceil(N / 256) + j / 4) >= drop_p * 2^32, else it is 0
 * (the counter is a 64-bit integer; for N <= 256 its row stride is 64); the row sums are
 * those of the undropped softmax and the kept probabilities are scaled by 1 / (1 - drop_p).  The decision depends
 * only on the seed and the indices.  drop_p == 0 runs b200_attention.  Returns -19 unless 0 <= drop_p < 1 (nothing
 * launched), else as b200_attention.
 */
int b200_attention_mc(const void* qkv, int qkv_ld, void* out, int out_ld, int B, int N, int heads, int dh, float scale,
                      float drop_p, unsigned long long drop_seed, void* stream);

/*
 * Batched GEMM on the same tcgen05 kernel: for every (batch, head)
 *     out[m, n] = epilogue( sum_k A[m, k] * B[n, k] ),   A, B bf16 K-major, fp32 accumulation.
 * This is how the transformer blocks run (code/transformer_model.py:98-116): Q.K^T per head
 * (mode 1: the epilogue writes exp(alpha*acc - rowmax) as bf16 and 1/rowsum to rowsum_inv - the softmax
 * numerator of :108; columns >= n_valid are masked), P.V^T per head (rowscale = that 1/rowsum, so the
 * division of the softmax is applied to the fp32 accumulator), and V^T = W_v X^T with the weights on the A
 * side (a_shared).  Strides are in elements; rows of A / B must be 16-byte aligned; K tails are zero-filled
 * and ragged M tails clipped by the TMA.  mode 1 needs N == 256 (one tile holds a whole row).
 * scale / bias are indexed n + head * vec_h_stride.
 */
typedef struct b200_gemm_desc {
    int M, N, K, heads, batch;
    const void* a;
    long long a_row_stride, a_head_stride, a_batch_stride;
    int a_shared;
    const void* b;
    long long b_row_stride, b_head_stride, b_batch_stride;
    void* out;
    long long out_row_stride, out_head_stride, out_batch_stride;
    const void* res;
    long long res_row_stride, res_head_stride, res_batch_stride;
    int res_mode, act;
    const float* scale;
    const float* bias;
    int vec_h_stride;
    const float* rowscale; /* [batch, heads, M] or NULL */
    int mode;              /* 0 standard, 1 softmax numerator */
    float alpha;
    int n_valid;
    float* rowsum_inv;     /* [batch, heads, M] (mode 1) */
    int b_rows;            /* valid rows of B per (head, batch); 0 = N.  Rows beyond are read as zeros */
} b200_gemm_desc;

int b200_gemm_batched(const b200_gemm_desc* d, void* stream);

/* nn.LayerNorm over the last dimension of a token matrix [rows, C] (code/transformer_model.py:16, :71, :73),
 * C a multiple of 256 up to 1024, fp32 statistics; x / y are bf16, or fp32 when x_f32 / y_f32 (the
 * transformer residual stream is kept in fp32). */
int b200_layernorm(const void* x, int x_f32, long long rows, int C, const float* w, const float* b, float eps,
                   void* y, int y_f32, void* stream);

/*
 * ViT-B/16 glue (timm VisionTransformer as used by code/foundation_model.py:371-431):
 *   b200_patchify    fp32 NCHW image -> bf16 patch matrix [B*gh*gw, C*P*P] in Conv2d-weight order, so the patch
 *                    embedding is one GEMM; `gate` (nullable, [B, C]) multiplies plane (b, c) - the modality
 *                    attention x * w of code/model_module.py:41-43, :649-650 applied on the way in
 *   b200_vit_tokens  prepend the cls token and add the position embedding -> fp32 stream [B, 1+n, E]
 *   b200_vit_feature one block's feature map: fp32 stream -> bf16 [B, n, E] with the cls token stripped; rows are
 *                    written `out_ld` elements apart, so a block's map can land directly in its slot of the
 *                    channel-concatenated neck input (torch.cat of code/model_module.py:471)
 */
int b200_patchify(const float* x, const float* gate, int B, int C, int H, int W, int P, void* out, void* stream);
int b200_vit_tokens(const void* patches, const float* cls, const float* pos, int B, int n_patch, int E, float* t,
                    void* stream);
int b200_vit_feature(const float* t, int B, int n_patch, int E, void* out, int out_ld, void* stream);

/*
 * nn.Linear on a token matrix (code/transformer_model.py:93, :95, :123, :125): out[M,N] = epilogue(x[M,K] w[N,K]^T)
 * with the b200_conv_gemm_ex epilogue (scale, bias, GELU, residual).  The residual and / or the output may be
 * fp32 row-major [M,N] (res_f32 / out_f32): x + gamma * (W y + b) then accumulates into an fp32 stream.
 */
int b200_linear(const void* x, long long M, int K, const void* w, int N, const float* scale, const float* bias,
                const void* res, int res_f32, int res_mode, int act, void* out, int out_f32, void* stream);

/*
 * b200_linear with nn.Dropout(drop_p) in train mode (MC-dropout inference) before the residual add:
 *     out = res + drop(act(acc * scale + bias))
 * Element (row, col) is dropped when Philox4x32-7(drop_seed; row * N + col) < drop_p * 2^32 (one call decides four
 * consecutive columns; the rule of b200_conv_gemm_mc), the kept ones are scaled by 1 / (1 - drop_p).  Supported:
 * an fp32 residual (res_mode 1 with act 0, or res_mode 2) with fp32 or bf16 output, and no residual.  Returns -19
 * unless 0 <= drop_p < 1, and for a bf16 residual or res_mode 1 with an activation (nothing launched); drop_p == 0
 * runs b200_linear.  Other returns as b200_linear.
 */
int b200_linear_mc(const void* x, long long M, int K, const void* w, int N, const float* scale, const float* bias,
                   const void* res, int res_f32, int res_mode, int act, void* out, int out_f32, float drop_p,
                   unsigned long long drop_seed, void* stream);

/* out[b,h,w] = bias + sum_k d[(b,h+ky-1,w+kx-1)][k], zero padded: finishes a 3x3 C->1 conv from tap dots. */
int b200_tapsum(const float* d, int B, int H, int W, const float* bias, float* out, void* stream);

/*
 * DWINormalize.__call__ (code/dataset.py:14-41), batched over `planes` = cases*C image
 * planes of n = H*W fp32 samples (NCHW): per plane z-score with unbiased std clamped at
 * 1e-6, clip to [z_lo, z_hi], map to [0,1]; when skip_last != 0 the last channel of every
 * case is written as zeros (adc=True).  plane_mean (optional, fp32 [planes]) receives the
 * mean of each OUTPUT plane - the pooled vector the modality SE block needs
 * (code/model_module.py:35, :649-650).
 */
int b200_dwi_normalize(const float* x, float* out, int planes, int C, int n, int skip_last, float z_lo,
                       float z_hi, float* plane_mean, void* stream);

/* b200_dwi_normalize with an optional statistics output stats_out [planes][4] = {mean, 1/std, scale, offset}; out may
 * then be NULL (statistics only: the consumer - b200_stem_ex - applies the map while loading the raw plane).
 * Statistics mode needs register-resident planes: n <= 8192 samples, n % 4 == 0, 16-byte aligned. */
int b200_dwi_normalize_ex(const float* x, float* out, int planes, int C, int n, int skip_last, float z_lo, float z_hi,
                          float* plane_mean, float* stats_out, void* stream);

/*
 * NyulStandardizer.transform (code/preprocess_helpers.py:85-120), batched like the above.
 *   avg_landmarks  fp64 [C, L]  fitted channel_landmarks (preprocess_helpers.py:77-80)
 *   standard_scale fp64 [L]     np.linspace(target_range) (:60)
 *   prev_index int32 [L], gamma fp64 [L]: floor and fractional part of q/100*(n-1), the
 *   "linear" percentile rule of np.percentile (:100), computed on the host in float64.
 * Planes above 32 768 samples (224 x 224) take the radix-select kernel.
 * exact selects the arithmetic.  exact = 0: the two chained np.interp maps are composed once per plane, in fp64, into
 * one <= L-segment piece-wise linear table (np.interp's tie / fill semantics folded in) and every sample costs an fp32
 * segment search plus one fp64 fma - equal to numpy within 1 fp32 ulp, i.e. far inside the 1e-5 contract.  exact = 1:
 * numpy's own operation order in fp64 without FMA contraction, bit-identical to the reference on > 99.9 % of the
 * samples, ~6x the instructions.
 */
int b200_nyul_transform_ex(const float* x, float* out, int planes, int C, int n, int L, const double* avg_landmarks,
                           const double* standard_scale, const int* prev_index, const double* gamma,
                           float* plane_mean, int exact, void* stream);
/* ... and with the per-plane composed table written to table_out [planes][56] fp64 (orig[16] | slope[16] | value[16] |
 * up[16] as fp32); out may then be NULL (tables + plane means only, for b200_stem_ex).  exact must be 0 with a table. */
int b200_nyul_transform_ex2(const float* x, float* out, int planes, int C, int n, int L, const double* avg_landmarks,
                            const double* standard_scale, const int* prev_index, const double* gamma,
                            float* plane_mean, int exact, double* table_out, void* stream);

/* DCE pre-scale of prep_data_by_mod (code/prepare_single_model.py:337-343): out[b] = x[b] / max(x[b]) over all the
 * channels and pixels of case b (n = C*H*W elements per case; IEEE division, as torch's `imgs / imgs_max`). */
int b200_case_max_scale(const float* x, int B, long long n, float* out, void* stream);

/* Mean of each fp32 plane (AdaptiveAvgPool2d(1) of SEBlock, code/model_module.py:35). */
int b200_plane_mean(const float* x, int planes, int n, float* plane_mean, void* stream);

/*
 * Encoder stem: modality SE gate (code/model_module.py:25-43, :649-650) applied to the fp32
 * NCHW input, then the two stride-`stride` 1x1 convolutions of block1 that read it - skip
 * conv + BN (:276-280) and first bottleneck conv + BN + GELU (:260-262).
 *   se_w1 [Cm,C], se_b1 [Cm], se_w2 [C,Cm], se_b2 [C] fp32, or se_w1 == NULL for no gate
 *   wcat [n_skip+n_mid, C] fp32, scale/bias [n_skip+n_mid] folded BatchNorm
 *   skip_out [B,H/s,W/s,n_skip] bf16, mid_out [B,H/s,W/s,n_mid] bf16, mod_attn [B,C] fp32
 * The per-channel normalisation can be FUSED INTO THE OPERAND LOAD (north_star (1); the reference normalises per
 * sample on the CPU in SingleInputDataset.__getitem__, code/dataset.py:70-98): x is then the RAW input and exactly
 * one of
 *   in_affine [B*C][4] {mean, 1/std, scale, offset} from b200_dwi_normalize_ex(out = NULL) - DWINormalize
 *             (code/dataset.py:14-41): y = fma(clamp((x - mean) * (1/std), z_lo, z_hi), scale, offset); a skipped
 *             (zeroed) channel carries {0,0,0,0};
 *   in_table  [B*C][56] fp64 from b200_nyul_transform_ex2(out = NULL) - the composed NyulStandardizer table
 *             (code/preprocess_helpers.py:85-120): orig[16] | slope[16] | value[16] | up[16] (fp32)
 * is given.  plane_mean must then be the per-plane mean of the NORMALISED values, which both statistics kernels emit.
 * The normalised tensor never exists in HBM: the raw input is read once by the statistics kernel and once (the
 * stride-s pixels only) here.  Both NULL: x is already normalised.
 */
int b200_stem_ex(const float* x, int B, int C, int H, int W, int stride, const float* plane_mean, const float* se_w1,
                 const float* se_b1, const float* se_w2, const float* se_b2, int Cm, const float* wcat,
                 const float* scale, const float* bias, int n_skip, int n_mid, void* skip_out, void* mid_out,
                 float* mod_attn, const float* in_affine, float z_lo, float z_hi, const double* in_table, int L,
                 void* stream);

/* b200_stem_ex with MC dropout on the bottleneck (`mid`) map, the reference's first nn.Dropout (code/model_module.py:260). */
int b200_stem_mc(const float* x, int B, int C, int H, int W, int stride, const float* plane_mean, const float* se_w1,
                 const float* se_b1, const float* se_w2, const float* se_b2, int Cm, const float* wcat,
                 const float* scale, const float* bias, int n_skip, int n_mid, void* skip_out, void* mid_out,
                 float* mod_attn, const float* in_affine, float z_lo, float z_hi, const double* in_table, int L,
                 float drop_p, unsigned long long drop_seed, void* stream);

/*
 * SEBlock.fc on pooled sums (code/model_module.py:34-40): gate[b,:] =
 * sigmoid(W2 gelu(W1 (gap_sum[b,:]/npix) + b1) + b2); w1t [C,Cm] and w2t [Cm,C] are the
 * conv weights transposed; `hidden` is caller-provided scratch [B, Cm] fp32 (the GELU layer's output).
 */
int b200_se_gate(const float* gap_sum, int B, int C, int Cm, int npix, const float* w1t, const float* b1,
                 const float* w2t, const float* b2, float* gate, float* hidden, void* stream);

/*
 * y = x * gate[b,c] * (1 + gamma * attn[b,p]) on a bf16 NHWC map (in place allowed).
 * SE rescale (code/model_module.py:43) and MaskGuidedSpatialAttention modulation (:96);
 * gate / attn may be NULL; gamma is a device scalar.
 */
int b200_scale_map(const void* x, void* y, int B, int npix, int C, const float* gate, const float* attn,
                   const float* gamma, void* stream);

/* ReconHead last conv (code/model_module.py:117): 3x3 pad 1, C -> 1, bias; w [9,C] fp32; out fp32 [B,H,W]. */
int b200_conv3x3_c1(const void* x, int B, int H, int W, int C, const float* w, const float* bias, float* out,
                    void* stream);

/*
 * MaskHeadResize.out (code/model_module.py:187) on the `pre` activations [B,npix,Cm] bf16
 * -> mask_pred fp32 [B,npix]; when attn != NULL also MaskGuidedSpatialAttention's
 * mask_processor (:67-73, :92-93) -> attention map fp32 [B,npix] in [1e-4, 1-1e-4].
 */
/*
 * MaskGuidedSpatialAttention.mask_processor (code/model_module.py:67-73, :92-93) on an fp32 1-channel map
 * mask [B,npix] -> attention map fp32 [B,npix] clamped to [1e-4, 1-1e-4].
 */
int b200_mask_attention(const float* mask, int B, int npix, int Hc, const float* wa, const float* gn_w,
                        const float* gn_b, const float* wb, const float* bb, float gn_eps, float* attn,
                        void* stream);

/* F.interpolate(bilinear, align_corners=False) of an fp32 1-channel map [B,h,w] -> [B,H,W]
 * (MaskHeadResize fallback, code/model_module.py:205-211, commuted past the 1x1 `out` conv). */
int b200_resize_bilinear_c1(const float* in, int B, int h, int w, float* out, int H, int W, void* stream);

/* torchvision `transforms.Resize(input_size)` = F.interpolate(bilinear, align_corners=False, antialias=True) of
 * fp32 planes [B,h,w] -> [B,H,W] where a side shrinks (code/prepare_single_model.py:112, :116, :120 with ROIs larger
 * than `input_size`; code/parameters_generate.py:68).  ATen's separable triangle filter of support max(in/out, 1),
 * horizontal pass then vertical, fp32.  Growing sides reduce to the plain bilinear taps. */
int b200_resize_aa_c1(const float* in, int B, int h, int w, float* out, int H, int W, void* stream);

int b200_mask_tail(const void* pre, int B, int npix, int Cm, const float* w_out, const float* b_out,
                   float* mask_pred, int Hc, const float* wa, const float* gn_w, const float* gn_b, const float* wb,
                   const float* bb, float gn_eps, float* attn, void* stream);

/* First Projector layer on a 1-channel map (code/model_module.py:338-340, :639-640). */
int b200_lift_c1(const float* r, long long total_pix, int N, const float* w, const float* scale, const float* bias,
                 void* y, void* stream);

/*
 * ClassificationHead.forward (code/model_module.py:364-369) from pooled sums:
 * v = gap_sum/npix * gate; v /= max(||v||,1e-12) if normalize; logits = fc_w v + fc_b.
 */
int b200_cls_head(const float* gap_sum, const float* gate, int B, int C, int npix, int K, const float* fc_w,
                  const float* fc_b, int normalize, float* logits, float* pooled_out, void* stream);

/*
 * Backbone-adapter helpers (the ViT-B/16 path, 14 x 14 maps; all maps NHWC bf16, C a multiple of 8):
 *   b200_channel_sums   per-case channel sums [B, C] fp32 of a map with row stride x_ld - the global average
 *                       pools of SEBlock / ClassificationHead (code/model_module.py:35, :364) for maps whose
 *                       width does not divide 128, where the GEMM epilogue cannot take them from staged tiles
 *   b200_mix_instnorm   GroupNorm(C, C)(alpha * f_b + (1 - alpha) * f), alpha = sigmoid(*weight_logit)
 *                       (code/model_module.py:592-597, :673-675, :688-690): per (case, channel) mean / biased
 *                       variance over the npix pixels, affine gn_w / gn_b
 *   b200_adaptive_pool  nn.AdaptiveAvgPool2d((Ho, Wo)) (code/model_module.py:531-534, :707-710); x_f32 = 1:
 *                       1-channel fp32 map -> fp32; else bf16 -> bf16 with an optional GELU (act = 1) applied
 *                       to the pooled value (the pool is moved behind the Projector's first 1x1 conv + BN,
 *                       with which it commutes)
 *   b200_add_maps       out = a + b element-wise (f2 + f1_aligned with an identity FeatureDownAlign, :682-683)
 */
int b200_channel_sums(const void* x, int x_ld, int B, int npix, int C, float* out, void* stream);
int b200_mix_instnorm(const void* fb, const void* f, int B, int npix, int C, const float* weight_logit,
                      const float* gn_w, const float* gn_b, float eps, void* out, void* stream);
int b200_adaptive_pool(const void* x, int x_f32, int B, int H, int W, int C, int Ho, int Wo, int act, void* out,
                       void* stream);
int b200_add_maps(const void* a, const void* b, long long n_elems, void* out, void* stream);

/*
 * ResNet-50 backbone stem (timm / torchvision `resnet50` as built by code/foundation_model.py:15-68, :220-312):
 *   b200_maxpool3x3_s2  nn.MaxPool2d(3, 2, 1) on an NHWC bf16 map
 *   b200_im2col7x7_s2   conv1 (7x7, stride 2, padding 3) as a GEMM operand: bf16 patch matrix [B * H/2 * W/2, Kp]
 *                       (column c*49 + ky*7 + kx, zero padded to Kp, a multiple of 64) of the fp32 NCHW input, scaled
 *                       per (case, channel) by the modality-attention gate (nullable); conv1 + folded bn1 + ReLU is
 *                       then one b200_linear call
 * The bottlenecks run on b200_conv_gemm_ex (act = 2, stride, dilation, residual).
 */
int b200_maxpool3x3_s2(const void* x, int B, int H, int W, int C, void* y, void* stream);
int b200_im2col7x7_s2(const float* x, const float* gate, int B, int C, int H, int W, int Kp, void* out, void* stream);

/* compute_adc_map (code/preprocess_helpers.py:133-167): x [B, C, n] fp32 DWI stacks (n = H*W), bvals [C] on the
 * device -> out [B, n]: minus the per-pixel least-squares slope of log(max(S, eps)) over b.  C <= 32. */
int b200_adc_map(const float* x, int B, int C, int n, const float* bvals, float eps, float* out, void* stream);

/* Test-time-augmentation flips (code/train.py:916-923, used by code/train_fusion.py:543-632): out = flip of every
 * [H, W] plane of x [planes, H, W] fp32 along W and / or H.  Out of place. */
int b200_flip_planes(const float* x, float* out, long long planes, int H, int W, int flip_w, int flip_h,
                     void* stream);

/* Training-time augmentation, batched (code/prepare_single_model.py:107-113: torchvision RandomAffine(degrees=90,
 * translate=(0.1,0.1), shear=(0.1,0.1)) -> RandomHorizontalFlip -> RandomVerticalFlip, per sample on the CPU in the
 * reference).  x, out [B,C,H,W] fp32 (out of place); theta [B,6] = torchvision's INVERSE affine matrix of each case
 * (output pixel -> input pixel, centred coordinates; identity = {1,0,0,0,1,0}); flips [B] or NULL: bit 0 = horizontal,
 * bit 1 = vertical flip applied after the affine map.  Nearest-neighbour sampling, `fill` outside the image. */
int b200_augment(const float* x, float* out, int B, int C, int H, int W, const float* theta, const int* flips,
                 float fill, void* stream);

/* FusionModel._to_tokens (code/model_module.py:903-917): adaptive average pool to Hp x Wp tokens, fp32 [B,Hp*Wp,C]. */
int b200_fusion_tokens(const void* p, int B, int H, int W, int C, int Hp, int Wp, float* tokens, void* stream);

/* Device pointers to the small fusion-head parameters (all fp32; *_wt are transposed [in,out]). */
typedef struct b200_fusion_weights {
    int C, T, heads, se_mid, num_classes;
    int use_cross_attention, use_mask_attention, use_se;
    float ln_eps;
    const float* gate_w;      /* GatingAttention.fc.weight [2, 2C(+2)]   model_module.py:755 */
    const float* gate_b;      /* [2] */
    const float* in_proj_wt;  /* MultiheadAttention.in_proj_weight^T [C,3C] model_module.py:806 */
    const float* in_proj_b;   /* [3C] */
    const float* out_proj_wt; /* out_proj.weight^T [C,C] */
    const float* out_proj_b;  /* [C] */
    const float* ln_w;        /* attn_ffn.0 LayerNorm model_module.py:808 */
    const float* ln_b;
    const float* ffn1_wt;     /* attn_ffn.1.weight^T [C,C] */
    const float* ffn1_b;
    const float* ffn2_wt;     /* attn_ffn.3.weight^T [C,C] */
    const float* ffn2_b;
    const float* up_coef;     /* [T] mean bilinear weight of each token cell (GAP of the upsample) */
    const float* se_w1t;      /* fusion_se.fc.1.weight^T [C,Cm] model_module.py:867 */
    const float* se_b1;
    const float* se_w2t;      /* fusion_se.fc.3.weight^T [Cm,C] */
    const float* se_b2;
    const float* cls_w;       /* classifier.2.weight [K,C] model_module.py:895-899 */
    const float* cls_b;
} b200_fusion_weights;

/*
 * Per-case part of FusionModel.forward (code/model_module.py:942-986): gating softmax,
 * cross-attention + FFN on pooled tokens, SE gate and classifier on the pooled fused map.
 * pvec_*_sum are per-case channel SUMS of p_dwi / p_dce over npix pixels.
 */
int b200_fusion_core(const b200_fusion_weights* wts, int B, const float* pvec_dwi_sum, const float* pvec_dce_sum,
                     int npix, const float* mask_dwi, const float* mask_dce, int npix_mask, const float* tok_dwi,
                     const float* tok_dce, float* gating_out, float* attn_out, float* lowres_out, float* gate_out,
                     float* logits_out, void* stream);

/* fused_refined = (a0*p_dwi + a1*p_dce + bilinear_up(lowres)) * gate (code/model_module.py:958-978). */
int b200_fusion_mix(const void* p_dwi, const void* p_dce, const float* gating, const float* lowres,
                    const float* gate, int B, int H, int W, int C, int Hp, int Wp, void* out, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Fusion-head fine-tuning step (BASELINE config C5, frozen-encoder phase of code/train_fusion.py:203-321 with
 * code/selector_helpers.py:356-520: the fusion head is the always-trainable parameter group).  All fp32.
 * ------------------------------------------------------------------------------------------------------------ */

/* C = op(A) op(B): op(A) is [M,K] (A is [M,K] with row stride lda, or [K,M] when trans_a), op(B) is [K,N] (B is
 * [K,N], or [N,K] when trans_b - an nn.Linear weight used as stored).  Epilogue (split_k == 1 only): + bias[N],
 * + res[(row / res_div) * ldres + col] (res_div > 1 broadcasts one residual row over res_div consecutive rows),
 * pre (optional, row stride ldc) receives the value before the activation, act 1 = exact GELU, beta 1 adds the
 * previous C.  split_k > 1 splits K over grid.z and ACCUMULATES into C atomically (beta must be 1; the caller
 * zeroes C for a plain product).  Serves nn.Linear forward / data gradient / weight gradient of
 * FusionModel.proj_in_* (code/model_module.py:857-858, 929-930, applied to pooled tokens),
 * nn.MultiheadAttention's projections (:806) and attn_ffn (:807-812). */
int b200_sgemm(const float* A, long long lda, int trans_a, const float* B, long long ldb, int trans_b, float* C,
               long long ldc, int M, int N, int K, const float* bias, const float* res, long long ldres, int res_div,
               float* pre, int act, int beta, int split_k, void* stream);

/* out[n] += sum over rows of X[R,N] (bias gradients; the caller zeroes out). */
int b200_colsum(const float* X, long long ld, int R, int N, float* out, void* stream);

/* nn.MultiheadAttention core (code/model_module.py:806, :816; no dropout, no mask) for Tq, Tk <= 32 tokens:
 * probs[B,heads,Tq,Tk] = softmax(q k^T / sqrt(DH)), ctx = probs v.  q [B*Tq, ldq], k / v [B*Tk, ldkv], head h in
 * columns [h*DH, (h+1)*DH).  The backward writes dq (layout of q) and dk / dv (layout of k / v). */
int b200_mha_fwd(const float* q, long long ldq, const float* k, const float* v, long long ldkv, int B, int heads,
                 int Tq, int Tk, int DH, float* probs, float* ctx, long long ldc, void* stream);
int b200_mha_bwd(const float* q, long long ldq, const float* k, const float* v, long long ldkv, const float* probs,
                 const float* dctx, long long ldc, int B, int heads, int Tq, int Tk, int DH, float* dq, float* dk,
                 float* dv, void* stream);

/* nn.LayerNorm of attn_ffn (code/model_module.py:808) on [R,C] rows with saved statistics, and its backward:
 * dx = dres (optional residual-path gradient) + LN'(dy); dyxhat = dy * xhat, whose column sums are the weight
 * gradient (dy's column sums are the bias gradient). */
int b200_ln_fwd(const float* x, int R, int C, const float* w, const float* b, float eps, float* y, float* mean,
                float* rstd, void* stream);
int b200_ln_bwd(const float* x, const float* dy, const float* dres, int R, int C, const float* w, const float* mean,
                const float* rstd, float* dx, float* dyxhat, void* stream);

/* out = dg * gelu'(pre), exact (erf) GELU (nn.GELU of attn_ffn, code/model_module.py:810). */
int b200_gelu_bwd(const float* pre, const float* dg, long long n, float* out, void* stream);

/* Per-case tail of the head's logits path and its backward.  Weights in their nn.Module layouts. */
typedef struct b200_head_train {
    int C, T, se_mid, num_classes;
    int use_mask_attention, use_se;
    int npix_mask;
    float smoothing;            /* LabelSmoothing alpha (code/loss.py:190-213) */
    float gamma;                /* focal exponent (code/loss.py:133-188) */
    float loss_scale;           /* 1 / batch: reduction "mean" */
    const float* class_weights; /* [K] or NULL (SoftWeightedFocalLoss) */
    const float* tok_dwi;       /* [B,T,C] projected pooled tokens */
    const float* tok_dce;
    const float* lowres;        /* [B,T,C] cross-attention block output, or NULL (use_cross_attention False) */
    const float* mask_dwi;      /* [B,npix_mask] encoder mask logits (GatingAttention confidences) */
    const float* mask_dce;
    const long long* labels;    /* [B] int64 */
    const float* gate_w;        /* gating.fc.weight [2, 2C(+2)] */
    const float* gate_b;
    const float* up_coef;       /* [T] mean bilinear weight of each token cell */
    const float* se_w1;         /* fusion_se.fc.1.weight [Cm,C] */
    const float* se_b1;
    const float* se_w2;         /* fusion_se.fc.3.weight [C,Cm] */
    const float* se_b2;
    const float* cls_w;         /* classifier.2.weight [K,C] */
    const float* cls_b;
    float* loss_out;            /* scalar, ACCUMULATED (caller zeroes) */
    float* logits_out;          /* [B,K] or NULL */
    float* gating_out;          /* [B,2] or NULL */
    float* dlogits_out;         /* [B,K]   -> classifier weight / bias gradients */
    float* z_out;               /* [B,C]   gated pooled vector (classifier input) */
    float* gf_out;              /* [B,C]   pooled fused vector (SE input) */
    float* h_out;               /* [B,Cm]  SE hidden activation */
    float* da1_out;             /* [B,Cm]  gradient at the SE hidden pre-activation */
    float* da2_out;             /* [B,C]   gradient at the SE output pre-activation */
    float* gx_out;              /* [B,2C(+2)] gating input */
    float* dgl_out;             /* [B,2]   gradient at the gating logits */
    float* dpd_out;             /* [B,C]   gradient of each DWI token coming through the pooled vector (already / T) */
    float* dpc_out;             /* [B,C]   same for DCE */
    float* dlowres_out;         /* [B,T,C] gradient of lowres, or NULL with lowres */
    /* --- fused-mask dice term (NULL / 0 when the term is off) --- */
    int forward_only;           /* 1: stop after the logits (writes gating_out, gate_out, u_out, logits_out only) */
    const float* mask_v;        /* [C] v = mask_head.pre.weight^T mask_head.out.weight: fused mask logit = v . fused_refined + c0 */
    const float* mk_tmpd;       /* [B,C] proj_in_dwi.weight s_dwi, s = sum_pixels dmask * f3 (b200_mask_wsum) */
    const float* mk_tmpc;       /* [B,C] same for DCE */
    const float* mk_q;          /* [B,T] transposed bilinear up-sample of dmask (b200_mask_dice) */
    float* gate_out;            /* [B,C] SE gate, or NULL */
    float* u_out;               /* [B,C] v * gate (forward_only) */
    float* dug_out;             /* [B,C] (gradient of u) * gate -> column sums = gradient of v */
    float* aud_out;             /* [B,C] alpha_dwi * u -> proj_in_dwi weight gradient with s_dwi */
    float* auc_out;             /* [B,C] alpha_dce * u */
    /* --- pooled vectors given explicitly (token bins that overlap / differ in size: GAP(p) is then NOT the mean of
     * the tokens).  NULL: pooled vector = mean of the tokens, and dpd / dpc come back divided by T. --- */
    const float* pvec_dwi;      /* [B,C] proj_in applied to the per-case channel SUMS of f3 */
    const float* pvec_dce;
    float pvec_scale;           /* 1 / pixels; dpd / dpc then come back multiplied by it (gradient w.r.t. the sums) */
} b200_head_train;

/* FusionModel.forward tail (code/model_module.py:942-986: gating :952-958, GAP of the fused map, fusion_se :977,
 * classifier :986) + LabelSmoothing and Soft(Weighted)FocalLoss with mean reduction (code/train_fusion.py:238-242)
 * + the backward of that chain, one CTA per case. */
int b200_head_loss(const b200_head_train* args, int B, void* stream);

/* Fused-mask dice term of the reference's training loss (code/train_fusion.py:245-255: lambda_mask * mean of three
 * SoftDiceLoss terms, code/loss.py:45-62) for maps of the mask size, where MaskHeadResize is pre (1x1) -> out (1x1)
 * with nothing in between (code/model_module.py:153-215, the `32: None` dispatch): the fused mask logit is LINEAR
 * in fused_refined, m = c0 + v . fused_refined, so with u = v * gate
 *   m[b,p] = c0 + a_dwi (W_dwi^T u_b) . f3_dwi[b,p] + a_dce (W_dce^T u_b) . f3_dce[b,p] + sum_t U[p,t] (u_b . lowres[b,t]).
 * b200_mask_dot: D[b,p] = omega[b] . f3[b,p,:] (f3 NHWC bf16 [B,npix,Cin], omega fp32 [B,Cin]).
 * b200_mask_dice: builds m, the dice losses of the fused mask and (for the reported loss value only) of the two
 *   encoder masks, ACCUMULATES scale * (sum of the (1 - dice_b)) into loss_out, and writes the fused logits, dm =
 *   dloss/dm, q[b,t] = sum_p U[p,t] dm[b,p] and ACCUMULATES sum dm into dc0_out.  scale = lambda_mask / (3 B).
 * b200_mask_wsum: s[b,:] = sum_p dm[b,p] f3[b,p,:].
 * b200_mask_head_grads: gradients of mask_head.pre / .out from dv [C] and dc0 (ACCUMULATED into the outputs). */
int b200_mask_dot(const void* f3, const float* omega, int B, int npix, int Cin, float* D, void* stream);
int b200_mask_dice(const float* D_dwi, const float* D_dce, const float* gating, const float* u, const float* lowres,
                   const float* pre_b, const float* out_w, const float* out_b, int mid, const float* target,
                   const float* enc_mask_dwi, const float* enc_mask_dce, int B, int H, int W, int Ho, int Wo, int Hp,
                   int Wp, int C, float scale, float eps, int loss_type, float* m_out, float* dm_out, float* q_out, float* dc0_out,
                   float* loss_out, void* stream);
int b200_mask_wsum(const void* f3, const float* dm, int B, int npix, int Cin, float* s, void* stream);
int b200_mask_head_grads(const float* dv, const float* dc0, const float* pre_w, const float* pre_b,
                         const float* out_w, int mid, int C, float* g_pre_w, float* g_pre_b, float* g_out_w,
                         float* g_out_b, void* stream);

/* torch.optim.AdamW step (code/selector_helpers.py:222-229) on flat fp32 buffers; g is multiplied by grad_scale
 * first (1 / world_size after the summing gradient all-reduce).  step >= 1 is the update count. */
int b200_adamw(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1, float beta2,
               float eps, float weight_decay, int step, float grad_scale, void* stream);


/* The same update with per-element hyper-parameters: lr_vec / wd_vec [n] fp32 (learning rate x lr_mult; 0 = skip the
 * element), step0 [n] int32 or NULL (the element's bias correction counts from step - step0).  Parameter groups of
 * LightningFusionOptimizerFactory (code/selector_helpers.py:456-518): discriminative learning rates / regularisation
 * by depth, and groups added later by gradual unfreezing (:523-620) that start their own Adam step count. */
int b200_adamw_groups(float* p, const float* g, float* m, float* v, long long n, const float* lr_vec, const float* wd_vec,
                      const int* step0, float lr_mult, float beta1, float beta2, float eps, int step, float grad_scale,
                      void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Training step of the encoders / the whole fusion objective (BASELINE configs C1 and C5 with the encoders
 * unfrozen): torch autograd over code/model_module.py in train mode, restated as explicit backward kernels.
 * Maps are NHWC bf16 [rows, ld]; gradients of maps bf16; parameter gradients fp32, ACCUMULATED into the given
 * buffers (the caller zeroes them once per step) in the parameter's own nn.Module layout.
 * ------------------------------------------------------------------------------------------------------------ */

/* Weight gradient of a stride-1 1x1 / 3x3 (padding 1) nn.Conv2d on the tensor cores (csrc/conv_wgrad.cu):
 * dw[co, ci, tap] += sum_pixels dy[p, co] * x[p + offset(tap), ci]; dw is the fp32 gradient in the nn.Conv2d layout
 * [Cout, Cin, kh, kw].  Both NHWC maps are consumed as MN-major tcgen05 operands straight from their TMA boxes.
 * W must divide 64 or be a multiple of 64, H a multiple of 64 / min(W, 64). */
int b200_conv_wgrad(const void* dy, int dy_ld, const void* x, int x_ld, float* dw, int B, int H, int W, int Cin,
                    int Cout, int taps, void* stream);

/* fp32 master weights [Cout, Cin, kh, kw] -> bf16 [Cout, taps*Cin] (forward operand of b200_conv_gemm_ex) and / or
 * bf16 [Cin, taps*Cout] with flipped taps (operand of the data gradient: dX = conv(dY, w_dgrad)).  Either may be NULL. */
int b200_pack_conv_weights(const float* w, int Cout, int Cin, int taps, void* w_fwd, void* w_dgrad, void* stream);

/* nn.BatchNorm2d in training mode on a conv output z [R, C]: per-channel sum / sum of squares (fp64, accumulated
 * into zeroed buffers), then mean / 1/sqrt(biased var + eps) and the momentum update of the running statistics
 * (unbiased variance), as torch does. */
int b200_bn_stats(const void* z, long long R, int C, int ld, double* sum, double* sumsq, void* stream);
int b200_bn_finalize(const double* sum, const double* sumsq, int C, double count, float eps, float momentum,
                     float* running_mean, float* running_var, float* mean_out, float* invstd_out, void* stream);

/* out = dropout(act((z - mean) * invstd * gamma + beta + res)): BatchNorm apply + residual + activation (0 none,
 * 1 exact GELU, 2 ReLU) + nn.Dropout(drop_p) with Philox4x32-7 keyed by (seed, element index).  Any of mean / invstd /
 * gamma / beta / res may be NULL (0, 1, 1, 0, none): a conv bias is `beta` alone.
 * (code/model_module.py:259-269, :298-306: conv -> BN -> GELU -> Dropout; GELU(out + identity) -> Dropout.) */
int b200_bn_act_fwd(const void* z, int ldz, const void* res, int ldres, const float* mean, const float* invstd,
                    const float* gamma, const float* beta, int act, float drop_p, unsigned long long seed, long long R,
                    int C, void* out, int ldo, void* stream);

/* Backward of the above from dA (gradient of `out`): dY = dA * dropout mask * act'(.);
 * batch_stats = 1: dz = gamma * invstd * (dY - mean(dY) - xhat * mean(dY * xhat)) (training-mode BatchNorm);
 * batch_stats = 0: dz = gamma * invstd * dY.  dres = dY (NULL when there is no residual branch); dgamma += sum dY*xhat,
 * dbeta += sum dY (NULL to skip).  scratch2C: 2*C doubles of workspace. */
int b200_bn_act_bwd(const void* z, int ldz, const void* res, int ldres, const float* mean, const float* invstd,
                    const float* gamma, const float* beta, int act, float drop_p, unsigned long long seed, long long R,
                    int C, const void* dA, int ldd, int batch_stats, double* scratch2C, void* dz, int lddz, void* dres,
                    int lddres, float* dgamma, float* dbeta, void* stream);

/* out[b, c] = sum_p a[b,p,c] * b[b,p,c] (b NULL: channel sums) - SE gate gradient / global average pools. */
int b200_map_dot(const void* a, int lda, const void* b, int ldb, int B, int npix, int C, float* out, void* stream);
/* out[b,p,c] (+)= x[b,p,c] * gate[b,c] + add[b,c] (x NULL: 1; gate / add NULL: 1 / 0): SE rescale and its backward,
 * broadcast of a pooled-vector gradient over the pixels. */
int b200_map_scale_add(const void* x, int ldx, const float* gate, const float* add, int B, int npix, int C, void* out,
                       int ldo, int accumulate, void* stream);
/* y = alpha * a + beta * b on bf16 maps (b NULL: y = alpha * a): gradient accumulation, feature-norm gradient. */
int b200_map_axpby(const void* a, int lda, float alpha, const void* b, int ldb, float beta, long long R, int C, void* y,
                   int ldy, void* stream);
/* *out += sum of squares of a bf16 map (fp64): compute_feat_norm_loss, code/train.py:1021-1030. */
int b200_map_sumsq(const void* a, int lda, long long R, int C, double* out, void* stream);

/* SEBlock (code/model_module.py:25-43) with the weights in their nn.Conv2d layouts w1 [M,C], w2 [C,M]:
 * forward from per-case channel SUMS (pooled = sums / npix is written too); backward from dgate [B,C] through the
 * MLP: dpooled, and da2 [B,C], da1 [B,M], h [B,M] whose outer products with h / pooled are the weight gradients. */
int b200_se_fwd(const float* sums, int B, int C, int M, int npix, const float* w1, const float* b1, const float* w2,
                const float* b2, float* pooled, float* gate, void* stream);
int b200_se_bwd(const float* pooled, const float* w1, const float* b1, const float* w2, const float* b2,
                const float* dgate, int B, int C, int M, float* dpooled, float* da2, float* da1, float* h, void* stream);

/* C -> 1 convolutions, 1x1 or 3x3 padding 1 (ReconHead.conv[3], MaskHeadResize.out; code/model_module.py:117, :187):
 * w fp32 in the nn.Conv2d layout [1, C, kh, kw]; out / dout fp32 [B,H,W]; dx bf16 (optionally accumulated). */
int b200_convc1_fwd(const void* x, int ldx, int B, int H, int W, int C, int taps, const float* w, const float* bias,
                    float* out, void* stream);
int b200_convc1_bwd(const void* x, int ldx, const float* dout, int B, int H, int W, int C, int taps, const float* w,
                    void* dx, int lddx, int accumulate_dx, float* dw, float* dbias, void* stream);

/* 1 -> N convolution of a 1-channel fp32 map (Projector.proj[0] on a reconstruction, code/model_module.py:338):
 * z[p, n] = r[p] * w[n]; backward dw[n] += sum_p dz r, dr[p] = sum_n dz w (dr NULL to skip). */
int b200_lift_fwd(const float* r, long long P, int N, const float* w, void* z, void* stream);
int b200_lift_bwd(const void* dz, const float* r, long long P, int N, const float* w, float* dw, float* dr, void* stream);

/* MaskGuidedSpatialAttention (code/model_module.py:49-97) backward.  b200_modulate_bwd: y = f * (1 + gamma * A):
 * df = dy * (1 + gamma A), dA[b,p] = gamma * sum_c dy f, dgamma += sum dy f A.  b200_mask_attn_bwd: through
 * clamp(sigmoid(conv(gelu(GroupNorm(1,K)(conv(mask)))))) to dmask and the five small parameter gradients. */
int b200_modulate_bwd(const void* dy, int lddy, const void* f, int ldf, const float* A, const float* gamma, long long P,
                      int C, void* df, int lddf, float* dA, float* dgamma, void* stream);
int b200_mask_attn_bwd(const float* mask, const float* dA, int B, int npix, int K, const float* wa, const float* gnw,
                       const float* gnb, const float* wb, const float* bb, float eps, float* dm, float* dwa, float* dgnw,
                       float* dgnb, float* dwb, float* dbb, void* stream);

/* Backward of b200_stem_ex run with every output channel un-activated (training: BatchNorm follows): from dz
 * [B, npix, N] bf16 to dwcat [N, C] and the modality-attention gate gradient dgate [B, C]. */
int b200_stem_bwd(const float* x, int B, int C, int H, int W, int stride, const float* gate, const void* dz, int N,
                  const float* wcat, float* dwcat, float* dgate, void* stream);

/* ClassificationHead backward (code/model_module.py:355-369): pooled [B,C] = GAP mean; dfcw / dfcb accumulated. */
int b200_cls_head_bwd(const float* pooled, const float* dlogits, const float* fcw, int B, int C, int K, int normalize,
                      float* dfcw, float* dfcb, float* dpooled, void* stream);

/* Loss terms with their gradients; each ACCUMULATES scale * (sum over cases) into *loss.
 *   b200_focal_loss  LabelSmoothing + Soft(Weighted)FocalLoss (code/loss.py:133-213), scale = 1 / B
 *   b200_dice_loss   SoftDiceLoss (code/loss.py:45-62) on logits [B,n], scale = weight / B
 *   b200_recon_loss  bilinear up-sample -> sigmoid -> Charbonnier against the clamped channel mean of the input
 *                    (code/train.py:1041-1048, :446-454), scale = weight / (B*H*W); x2 / C2: a second input tensor
 *                    whose channels join the mean (the fusion step's cat([dwi, dce]), code/train_fusion.py:276-285)
 *   b200_mimic_loss  1 - cos(student, detached teacher) per case (code/train.py:1033-1038), scale = weight / B */
int b200_focal_loss(const float* logits, const long long* labels, int B, int K, float smoothing, float gamma,
                    const float* class_weights, float scale, float* loss, float* dlogits, void* stream);
int b200_dice_loss(const float* logits, const float* target, int B, int n, float eps, float scale, float* loss,
                   float* dlogits, void* stream);
int b200_recon_loss(const float* r, int B, int h, int w, const float* x, int C, const float* x2, int C2, int H, int W,
                    float eps, float scale, float* loss, float* dr, void* stream);
int b200_mimic_loss(const void* s, const void* t, int B, long long n, float scale, float* loss, void* ds, void* stream);

/* Full-resolution training of FusionModel (code/model_module.py:919-1000) - the pieces between the tensor-core layers:
 *   b200_gating_fwd     GatingAttention (:745-780) from per-case channel SUMS of p_dwi / p_dce (+ encoder mask logits):
 *                       gx [B, 2C(+2)] (the Linear's input, kept for its weight gradient), alpha [B,2] = softmax
 *   b200_gating_bwd     dalpha -> dgl [B,2] (logit gradients), dgx [B, 2C(+2)] = dgl W, and dpv_* [B,C] = the pooled
 *                       vectors' share of dgx / npix (what every pixel of p_dwi / p_dce receives)
 *   b200_fused_pool     GAP of the fused map, analytically: alpha0 pvec_dwi + alpha1 pvec_dce + sum_t up[t] lowres[:,t]
 *   b200_fusion_mix_bwd backward of fused = alpha0 p_dwi + alpha1 p_dce + bilinear_up(lowres): phase 0 accumulates
 *                       dalpha [B,2] and dlowres [B,T,C]; phase 1 writes dp_m = alpha_m dfused + dtok_m (token-pool
 *                       backward, already / bin size) + dpvec_m (already / npix)
 *   b200_mimic_pairs    the fusion step's mimic term over `proj_fused[:4]` exactly as the reference unpacks it
 *                       (code/train_fusion.py:287-296: the first four CASES; per-channel cosines) */
int b200_gating_fwd(const float* sum_d, const float* sum_c, int B, int C, int npix, const float* mask_d,
                    const float* mask_c, int npix_mask, const float* w, const float* bias, float* gx, float* alpha,
                    void* stream);
int b200_gating_bwd(const float* alpha, const float* dalpha, const float* w, int B, int C, int D, int npix, float* dgl,
                    float* dgx, float* dpv_d, float* dpv_c, void* stream);
int b200_fused_pool(const float* sum_d, const float* sum_c, int B, int C, int npix, const float* alpha,
                    const float* lowres, const float* up, int T, float* out, void* stream);
int b200_fusion_mix_bwd(const void* dfused, const void* p_dwi, const void* p_dce, const float* alpha, int B, int H, int W,
                        int C, int Hp, int Wp, float* dalpha, float* dlowres, const float* dtok_d, const float* dtok_c,
                        const float* dpv_d, const float* dpv_c, void* dp_dwi, void* dp_dce, int phase, void* stream);
int b200_mimic_pairs(const void* map, int B, int npix, int C, float scale, float* loss, void* dmap, void* stream);

/* din = sum of the four 2x2 replicas of dout [B,2H,2W,C] (backward of AdaptiveAvgPool2d to twice the size). */
int b200_up2_bwd(const void* dout, int B, int H, int W, int C, void* din, void* stream);
/* out[b, 0..n) = v[b * v_stride] * scale (gradient of the per-case mean of an fp32 map). */
int b200_row_bcast(const float* v, int v_stride, float scale, int B, int n, float* out, void* stream);
/* y = alpha * a + beta * y on fp32 vectors. */
int b200_vec_axpby(const float* a, float alpha, float beta, long long n, float* y, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200_FUSION_H */
