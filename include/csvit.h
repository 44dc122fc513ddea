/* csvit.h - C ABI of libcsvit_sm100.so, the B200 (sm_100a) kernels behind cs_vit.net.
 *
 * The reference (Mine268/CS-ViT) has no FFI: its hot path is PyTorch eager code that delegates the backbone
 * to HuggingFace `transformers` (ref:cs_vit/net/ti_poser.py:246,426).  The drop-in boundary is therefore the
 * Python surface of `cs_vit.net` (SURVEY.md section 8b); this header is the seam one level below it, the set
 * of entry points a maintainer binds (ctypes stub in INTEGRATION.md) to replace the ATen op sequences listed
 * per function.  "HF:" = transformers/models/swin/modeling_swin.py, "ref:" = the reference repository.
 *
 * Conventions
 *   - Plain C types only.  Pointers are CUDA device pointers owned by the caller (PyTorch); the library
 *     never allocates, frees or retains device memory.  `stream` is a cudaStream_t passed as void*.
 *   - Every function is asynchronous on `stream`, re-entrant, and returns 0 on success.  On failure it
 *     returns non-zero and csvit_last_error() (thread-local) describes why.  Nothing throws.
 *   - dtype codes: CSVIT_F32 = 0, CSVIT_BF16 = 1, CSVIT_F16 = 2 (the two 16-bit formats are interchangeable
 *     tensor-core operand formats: same MMA rate, fp16 carries 3 more mantissa bits).  Row-major; `ld*` are row pitches in ELEMENTS.
 *   - There is no CPU path: a missing GPU or a non-sm_100 device surfaces as a CUDA error code.
 */
#ifndef CSVIT_H_
#define CSVIT_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CSVIT_ABI_VERSION 11

#if defined(__GNUC__)
#define CSVIT_API __attribute__((visibility("default")))
#else
#define CSVIT_API
#endif

enum { CSVIT_F32 = 0, CSVIT_BF16 = 1, CSVIT_F16 = 2 };
enum { CSVIT_ACT_NONE = 0, CSVIT_ACT_GELU = 1, CSVIT_ACT_RELU = 2 };
enum { CSVIT_LN_IDENTITY = 0, CSVIT_LN_WINDOW = 1, CSVIT_LN_MERGE2X2 = 2 };
enum { CSVIT_GEMM_TENSORCORE = 0, CSVIT_GEMM_SIMT_FP32 = 1 };

CSVIT_API int csvit_abi_version(void);
CSVIT_API const char* csvit_last_error(void);

/* ---- integer maps (bit-exact contract, SURVEY.md section 8a) -------------------------------------------
 * Dumps of the closed-form maps the kernels use internally, for tests.
 * window_index_map: out[w*ws*ws + i] = flat token id that window w / slot i reads and writes
 *     = LN -> pad -> torch.roll(-shift) -> window_partition           HF:141-150, 608-622
 *     (same address for window_reverse -> roll(+shift)                 HF:153-160, 631-636)
 * shift_mask: out[nW, L, L] in {0, -100}                                HF:556-582 get_attn_mask
 * rel_pos_index: out[L, L]                                              HF:461-473 create_relative_position_index
 * merge_index_map: out[(H/2)*(W/2), 4] source tokens in concat order    HF:338-345 SwinPatchMerging.forward
 */
CSVIT_API int csvit_window_index_map(int H, int W, int ws, int shift, int32_t* out, void* stream);
CSVIT_API int csvit_shift_mask(int H, int W, int ws, int shift, float* out, void* stream);
CSVIT_API int csvit_rel_pos_index(int ws, int32_t* out, void* stream);
CSVIT_API int csvit_merge_index_map(int H, int W, int32_t* out, void* stream);

/* Host evaluation of the very same inline functions (HOST output pointers, no GPU needed): lets the CPU test
 * suite pin the integer logic that the kernels compile in. */
CSVIT_API int csvit_host_window_index_map(int H, int W, int ws, int shift, int32_t* out);
CSVIT_API int csvit_host_shift_mask(int H, int W, int ws, int shift, float* out);
CSVIT_API int csvit_host_rel_pos_index(int ws, int32_t* out);
CSVIT_API int csvit_host_merge_index_map(int H, int W, int32_t* out);

/* bias[h, i, j] = table[rel_pos_index(i, j), h]; table is [(2ws-1)^2, heads] fp32.      HF:428-434 */
CSVIT_API int csvit_expand_rel_bias(const float* table, float* out, int heads, int ws, void* stream);

/* ---- row kernels (HBM-bound) ----------------------------------------------------------------------------
 * LayerNorm over the last dim of fp32 x[B, H*W, C], eps inside the sqrt, output fp32 or bf16.
 *   CSVIT_LN_IDENTITY : out row r <- x row r                            HF:606/648 layernorm_*, HF:882 final norm
 *   CSVIT_LN_WINDOW   : out rows in window order (shift + partition folded into the read address)
 *                       replaces layernorm_before + F.pad + torch.roll + window_partition   HF:606-622
 *   CSVIT_LN_MERGE2X2 : out row (b,Y,X) = LN over the 4C concat of the 2x2 neighbourhood    HF:338-346
 * rows = number of OUTPUT rows (B*H*W, or B*(H/2)*(W/2) for MERGE2X2).  gamma/beta have the output width. */
CSVIT_API int csvit_layernorm(const float* x, const float* gamma, const float* beta, float eps, void* out, int out_dtype,
                    long long ldo, int rows, int C, int mode, int H, int W, int ws, int shift, void* stream);

/* y[r, c] = x[r, c] * scale[c] + shift[c]: eval-mode BatchNorm1d folded to an affine map.
 * Replaces norm(x.transpose(-1,-2)).transpose(-1,-2)   ref:cs_vit/net/transformer_module.py:312,316,341,345,349 */
CSVIT_API int csvit_affine_rows(const float* x, const float* scale, const float* shift, void* out, int out_dtype,
                      long long rows, int C, void* stream);

/* out[(b,py,px), c*16+ky*4+kx] = (img[b,c,4py+ky,4px+kx] - mean[c]) / std[c]; img fp32 NCHW [B,3,S,S].
 * Replaces transforms.Normalize + the unfold half of the 4x4/stride-4 conv.
 * ref:cs_vit/net/ti_poser.py:239-243,425   HF:286-295.   mean/std are HOST pointers to 3 floats. */
CSVIT_API int csvit_patch_im2col(const float* img, void* out, int out_dtype, int B, int S, const float* mean3,
                       const float* std3, void* stream);

/* On-device crop-and-resize of the hand region: out[n] = bilinear S x S resample of frames[n] over the box of image n, zeros outside
 * the frame, endpoints inclusive (align_corners) - what ref:cs_vit/utils/img.py:339-390 crop_tensor_with_square_box computes per
 * sample on the CPU with kornia.  frames: fp32 [N,3,H,W] in [0,1] (frames_u8 = 0) or uint8 [N,H,W,3] as decoded (frames_u8 = 1,
 * scaled by 1/255).  boxes [N,4] xyxy pixels: with expansion_ratio > 0 they are TIGHT boxes and the kernel first makes them square
 * on the longer side and scales them about the centre (ref :358-370), writing the boxes it cropped to square_boxes_out [N,4]
 * (may be NULL) - the `square_bboxes` Poser.predict_batch needs; with expansion_ratio <= 0 they are cropped as given.
 * out: fp32 [N,3,S,S]. */
CSVIT_API int csvit_crop_resize(const void* frames, int frames_u8, int N, int H, int W, const float* boxes, float expansion_ratio,
                                float* square_boxes_out, float* out, int S, void* stream);

/* ---- GEMM engine (tcgen05 + TMEM + TMA) ----------------------------------------------------------------
 * out[orow, :N] = act(A[M,K] @ W[N,K]^T + bias) + resid[orow, :N]
 *   in_dtype CSVIT_BF16 / CSVIT_F16: A and W in that format, kind::f16 MMA;  CSVIT_F32: A and W fp32, kind::tf32 MMA
 *   (or exact fp32 FMA with impl = CSVIT_GEMM_SIMT_FP32).  fp32 accumulation in all cases.
 *   bias, resid may be NULL.  resid is fp32 with pitch ldr and may alias out (in-place residual add: with the same pitch the tile then
 *   leaves as ONE fp32 reduction per element into out - TMA reduce-add / red.global.add.v4.f32 - instead of load + add + store; the
 *   result is the same single rounding fl(resid + fl(acc + bias)) and is reproducible run to run).
 *   scatter_ws > 0: GEMM rows are window-ordered tokens; orow = window_index_map(row) per image of
 *   scatter_H x scatter_W tokens (window_reverse + roll(+shift) folded into the store).  Else orow = row.
 * Replaces nn.Linear / addmm call sites: HF:404-406 (Q,K,V as one N=3C GEMM), HF:479, HF:514, HF:527,
 * HF:347 (reduction), HF:286 (projection as GEMM over csvit_patch_im2col), the residual adds HF:646,650,
 * and ref:cs_vit/net/transformer_module.py:262-264,282,290-294. */
CSVIT_API int csvit_linear(const void* A, long long lda, const void* W, long long ldw, int in_dtype, int M, int N, int K,
                 const float* bias, int act, const float* resid, long long ldr, void* out, long long ldo,
                 int out_dtype, int scatter_H, int scatter_W, int scatter_ws, int scatter_shift, int impl,
                 void* stream);

/* Fused MLP half-block for C in {128, 256}:  x[M,C] += GELU(xn[M,C] @ W1[4C,C]^T + b1) @ W2[C,4C]^T + b2, x fp32 in place,
 * xn / W1 / W2 16-bit (dtype).  The [M,4C] hidden tensor never reaches HBM (128x128 chunks: TMEM -> GELU -> smem ->
 * second tcgen05 GEMM).  Replaces intermediate.dense + GELU + output.dense + residual add   (HF:510-531, 650). */
CSVIT_API int csvit_mlp_fused(const void* xn, long long ldxn, const void* W1, long long ldw1, const float* b1, const void* W2,
                              long long ldw2, const float* b2, float* x, long long ldx, int dtype, int M, int C, void* stream);

/* Which kernel the calling thread's last csvit_linear launched: 1 = gemm_pair_kernel (CTA pairs, cta_group::2), 2 = gemm_tc_kernel
 * (single CTA), 3 = gemm_simt_f32_kernel (exact fp32), 0 = nothing.  Measurement aid: bench.py attributes launch times per kernel. */
CSVIT_API int csvit_last_gemm_kernel(void);

/* Process-wide tuning knobs of the GEMM engine (benchmarking / ablation; defaults are automatic):
 *   cluster   0 = auto, 1 / 2 / 4 = CTAs per cluster sharing the weight tile by TMA multicast
 *   tma_store -1 = auto, 0 = direct register stores, 1 = smem-staged TMA stores where legal
 *   max_ctas  0 = one CTA per SM
 *   pair      -1 = auto, 0 = never, 1 = CTA-pair (cta_group::2, 256-row MMA) kernel where legal */
CSVIT_API int csvit_set_gemm_tuning(int cluster, int tma_store, int max_ctas, int pair);

/* ---- attention cores -------------------------------------------------------------------------------------
 * Swin window attention on window-ordered fp32 qkv[B*H*W, 3C] (Q|K|V column blocks, head h at columns 32h..):
 *   out[B*H*W, C] = softmax(Q K^T / sqrt(32) + bias[h] + shift_mask) V, heads merged.       HF:410-459
 * Exact fp32 kernel of the validation mode (dtype must be CSVIT_F32); `bias` = the [heads, L, L] table of csvit_expand_rel_bias.
 * 16-bit operands take csvit_swin_attn_core / csvit_swin_attn_fused (tcgen05) below. */
CSVIT_API int csvit_window_attention(const void* qkv, const float* bias, void* out, int dtype, int B, int H, int W, int C,
                                     int heads, int ws, int shift, void* stream);

/* Fused shifted-window attention (north-star kernel; tcgen05 / TMEM, C in {128, 256}, window 7, head_dim 32): one launch from the
 * fp32 residual stream x[B*H*W, C] to the TOKEN-ordered 16-bit attention context ctx[B*H*W, C],
 *   ctx = window_reverse(roll(+s)( softmax(Q K^T / sqrt(32) + bias + shift_mask) V )),  Q|K|V = LN(x gathered by roll(-s) + window_partition) Wqkv^T + b
 * replacing layernorm_before, pad / roll / window_partition, query / key / value, the attention core and window_reverse / roll
 * (HF:swin/modeling_swin.py:404-459, 556-582, 604-636).  LN output, Q, K, V, logits and probabilities stay in SMEM / TMEM: 4C bytes
 * read + 2C written per token.  Two 49-token windows share a 128-row MMA tile (block structure in the operands, see attn_fused.cu).
 *   wqkv_h  [3C, C] 16-bit (dtype), rows re-ordered PER HEAD: head h owns rows 96h..96h+95 = Wq[32h..] | Wk[32h..] | Wv[32h..],
 *           with layernorm_before's gamma folded into the columns: W' = W diag(gamma) (the kernel normalises without gamma / beta)
 *   bqkv_h  [3C] fp32 in the same order, b' = b + W beta; the q part multiplied by log2(e)/sqrt(32) (the softmax runs in the log2
 *           domain).  The k part is not read: a key bias adds the same q.bk to every logit of a row and cancels in the softmax.
 *   bias_op [heads*49, 56] fp16: bias_op[49h + i, j] = log2(e) * table[rel_pos_index(i, j), h] for j < 49, 0 for j >= 49:
 *           one head's rows are one contiguous bulk copy; the softmax thread of query slot i adds row i to its logits.
 * The output projection + residual (csvit_linear with resid) follows on plain rows. */
CSVIT_API int csvit_swin_attn_fused(const float* x, float eps, const void* wqkv_h, const float* bqkv_h,
                                    const void* bias_op, void* ctx, int dtype, int B, int H, int W, int C,
                                    int heads, int ws, int shift, void* stream);

/* Window-attention core on tcgen05 / TMEM for every Swin width (attn_core.cu): window-ordered 16-bit qkv[B*H*W, 3C] (row pitch ldq
 * elements; per row q | k | v, head h in columns 32h..32h+31, as csvit_linear writes it after csvit_layernorm in window mode) ->
 *   ctx = softmax(q k^T * qs + bias + shift_mask) v     per window and head
 * replacing transpose_for_scores, Q K^T, the relative-position-bias gather, the mask add, softmax, P V and the head merge of
 * HF:swin/modeling_swin.py:404-459 (mask: 556-582).  Operand tiles come in by TMA ({64 columns, 49 rows} boxes, 128-byte swizzle),
 * both contractions run as tcgen05.mma with TMEM accumulators, four heads in flight per SM.
 *   bias_log2    [heads*49, 56] fp16, the csvit_swin_attn_fused table: log2(e) * table[rel_pos_index(i, j), h], 0 for j >= 49
 *   token_order  1: ctx rows in token order (window_reverse + roll(+s) folded into the store address, HF:631-636);
 *                0: window order like qkv (the training forward)
 *   q_prescaled  1: q already carries log2(e)/sqrt(32) (folded into the q rows of the Q/K/V weight and bias at packing time);
 *                0: the kernel applies it to the logits */
CSVIT_API int csvit_swin_attn_core(const void* qkv, long long ldq, const void* bias_log2, void* ctx, int dtype, int B, int H,
                                   int W, int C, int heads, int ws, int shift, int token_order, int q_prescaled, void* stream);

/* ---- the fp32 tail of predict_batch (tail.cu) -------------------------------------------------------------------------------
 * axis_angle[i] = matrix_to_axis_angle(rotation_6d_to_matrix(d6[i])) for n rotations (d6 [n,6], axis_angle [n,3]), with the
 * reference's branch structure: Gram-Schmidt rows (b1, b2, b1 x b2), best-conditioned quaternion candidate with real part >= 0,
 * sinc form of the half angle.   ref:cs_vit/utils/geometry.py:111-132, 150-223, 258-298; called at ref:cs_vit/net/ti_poser.py:529-534 */
CSVIT_API int csvit_rot6d_to_axis_angle(const float* d6, float* axis_angle, long long n, void* stream);

/* Poser._pose_fk in one kernel (one sample per CTA): MANO linear-blend skinning + J_regressor_mano + mean bone length +
 * de-normalisation.   ref:cs_vit/net/ti_poser.py:561-607
 *   pose [n,48] axis-angle (global orientation, 15 hand joints), betas [n,10], root_norm [n,3]
 *   v_template [778,3], shapedirs [778,3,10], j_regressor [16,778], lbs_weights [778,16], parents16 (HOST, parent < child, root -1):
 *   the buffers of the MANO layer; posedirs [135, 2334] and pose_mean [45] may be NULL (the stand-in has neither)
 *   j_regressor_out [21,778] = Poser.J_regressor_mano; edges40 (HOST): the 20 (a, b) joint pairs of TARGET_JOINTS_CONNECTION
 *   rodrigues_mode 0: theta = sqrt(|a|^2 + 1e-16) (cs_vit.utils.mano_standin); 1: theta = |a + 1e-8| (smplx batch_rodrigues)
 *   out: joint_cam [n,21,3] and verts_cam [n,778,3] in mm, root-relative + root_transl [n,3] = root_norm * 1e3 * mean bone length */
CSVIT_API int csvit_mano_fk(const float* pose, const float* betas, const float* root_norm, const float* v_template,
                            const float* shapedirs, const float* posedirs, const float* pose_mean, const float* j_regressor,
                            const float* lbs_weights, const float* j_regressor_out, const int* parents16, const int* edges40,
                            int rodrigues_mode, float* joint_cam, float* verts_cam, float* root_transl, int n, void* stream);

/* ---- data-parallel gradient allreduce over NVLink / NVSwitch peer memory (allreduce.cu) --------------------------------------
 * In-place fp32 SUM * scale of one flat bucket that lives at bufs[r] in the symmetric memory of every rank r (HOST arrays of
 * `world` DEVICE pointers; bufs[rank] is this GPU's own copy).  Replaces the bucketed NCCL allreduce that
 * DistributedDataParallel issues for ref:scripts/finetune.py:133-135, 217 (loss.backward()).
 *   flags      per rank a zero-initialised region of CSVIT_ALLREDUCE_FLAG_BYTES in symmetric memory (cross-GPU barriers)
 *   multicast  NVSwitch multicast address of the bucket (multimem.ld_reduce / multimem.st: the switch adds), or NULL for the
 *              two-shot form over plain P2P loads / stores
 *   n          floats, a multiple of 4;  world <= 8;  ctas: grid size, identical on all ranks (0 = default)
 * Every rank must call it with the same n / world / ctas, stream-ordered after the kernels that wrote its bucket; the kernel
 * returns on a rank once every rank's result has landed in that rank's copy. */
#define CSVIT_ALLREDUCE_FLAG_BYTES 4096
CSVIT_API int csvit_allreduce_f32(const void* const* bufs, const void* const* flags, void* multicast, long long n, int rank, int world,
                                  float scale, int ctas, void* stream);

/* ---- SwinV2 (SURVEY.md section 8f row 1; "V2:" = transformers/models/swinv2/modeling_swinv2.py) ---------------------------
 * Scaled-cosine window attention on window-ordered qkv[B*H*W, 3C] (layout as csvit_window_attention):
 *   out = softmax( normalize(Q) normalize(K)^T * logit_scale[h] + bias_tab[h, rel_pos_index(i, j)]
 *                  + mask_repeat * shift_mask ) V, heads merged.                                  V2:421-487
 *   bias_tab    [heads, (2ws-1)^2] fp32 = 16 sigmoid(continuous_position_bias_mlp(relative_coords_table))  V2:460-472, 489-510
 *   logit_scale [heads] fp32 = exp(min(logit_scale, ln 100))                                      V2:455
 *   mask_repeat how often the {0,-100} shift mask is added (HF adds it twice, V2:466-474: pass 2)
 *   out_token_order 1: out rows in TOKEN order (window_reverse + roll(+shift), V2:693-701, folded into the store), 0: window order
 * ws^2 must be a multiple of 16 and <= 256 (window 16: 256 tokens; window 8: 64).  bf16 / fp16: tensor-core kernel with
 * online softmax; fp32: exact kernel (validation mode). */
CSVIT_API int csvit_swinv2_window_attention(const void* qkv, const float* bias_tab, const float* logit_scale, void* out,
                                            int dtype, int B, int H, int W, int C, int heads, int ws, int shift,
                                            int mask_repeat, int out_token_order, void* stream);

/* SwinV2 Q/K/V projection with the cosine normalisation folded into the GEMM epilogue (16-bit operands):
 *   out[M, 3C] = A[M, K] @ W[3C, K]^T + bias, then per row and head h (32 columns):
 *   q_h <- q_h / max(|q_h|, 1e-12) * qscale_log2[h],   k_h <- k_h / max(|k_h|, 1e-12),   v_h unchanged,
 * with qscale_log2[h] = log2(e) * exp(min(logit_scale[h], ln 100)): the product q_h . k_h is then the log2-domain cosine logit of
 * V2:450-455 (both F.normalize and the logit scale), computed on the fp32 accumulator before the one 16-bit rounding. */
CSVIT_API int csvit_swinv2_qkv(const void* A, long long lda, const void* W, long long ldw, int dtype, int M, int C, int K,
                               const float* bias, const float* qscale_log2, void* out, long long ldo, void* stream);

/* SwinV2 cosine window attention for 16 x 16 windows on tcgen05 / TMEM (swinv2_attn_tc.cu), on the output of csvit_swinv2_qkv:
 *   ctx = softmax2( q_h k_h^T + bias_log2[h] + mask_repeat * log2(e) * shift_mask ) v_h     per window and head   (V2:450-487)
 * Operand tiles by TMA ({64 columns, 256 rows} boxes), S = Q K^T [128 x 256] per query tile in TMEM, the 16-bit probabilities
 * written back to TMEM and read from there as the A operand of P V (no shared-memory round trip).
 *   bias_log2   fp32 [heads][31][48]: entry [dy + 15][dx + 15] = log2(e) * 16 sigmoid(cpb_mlp)[(dy + 15) * 31 + dx + 15], dy / dx =
 *               query minus key row / column inside the window (columns 31..47 are padding: conflict-free shared-memory rows)
 *   shift       0 or 8;  token_order as csvit_swinv2_window_attention's out_token_order */
CSVIT_API int csvit_swinv2_attn_tc(const void* qkv, long long ldq, const float* bias_log2, void* ctx, int dtype, int B, int H, int W,
                                   int C, int heads, int shift, int mask_repeat, int token_order, void* stream);

/* Training forward of csvit_swinv2_attn_tc (the same kernel, instantiated to also write the row statistics the backward needs):
 *   ctx   16-bit [B*nW*256, C] in WINDOW order (the out-projection's operand in the differentiable path)
 *   lse2  fp32 [B*nW][heads][256]: log2 of each query row's softmax denominator in the log2 domain, lse2 = max_j z2 + log2 sum_j 2^(z2 - max)
 * Inputs as csvit_swinv2_attn_tc: qkv = q2 | k_hat | v, 16-bit [rows, 3C] (pitch ldq), q2 = F.normalize(q) * log2(e) * logit_scale_h,
 * k_hat = F.normalize(k) (V2:450-455); windows of 16, shift 0 or 8, head_dim 32.  Replaces the forward of V2:450-487 in training. */
CSVIT_API int csvit_swinv2_attn_tc_train(const void* qkv, long long ldq, const float* bias_log2, void* ctx, float* lse2, int dtype, int B,
                                         int H, int W, int C, int heads, int shift, int mask_repeat, void* stream);

/* Backward of csvit_swinv2_attn_tc_train (swinv2_attn_bwd.cu, tcgen05 / TMEM / TMA), log2 domain, per window and head:
 *   P = 2^(z2 - lse2),  D_i = sum_d dO_i,d O_i,d,  dZ2 = ln 2 * P o (dO v^T - D)
 *   dq = dZ2 k_hat,  dk = dZ2^T q2,  dv = P^T dO                  16-bit [rows, C] each (dense, window order; no atomics: reproducible)
 *   dbias_log2[h][dy + 15][dx + 15] = sum over windows and (i, j) at offset (dy, dx) of dZ2[i, j]
 *               fp32 [heads][31][48], zeroed here, accumulated with global reductions (last bits may vary run to run); columns 31..47 stay 0
 * qkv / bias_log2 / shape arguments as given to the forward; ctx = its output O and dctx = dO, dense 16-bit [rows, C].  The gradients
 * of logit_scale and of the CPB-MLP follow from dq and dbias_log2 by the chain rule through q2 = q_hat * log2(e) * scale and
 * bias_log2 = log2(e) * 16 sigmoid(cpb_mlp): this replaces the autograd backward of V2:450-487. */
CSVIT_API int csvit_swinv2_attn_tc_bwd(const void* qkv, long long ldq, const void* ctx, const void* dctx, const float* lse2,
                                       const float* bias_log2, void* dq, void* dk, void* dv, float* dbias_log2, int dtype, int B, int H,
                                       int W, int C, int heads, int shift, int mask_repeat, void* stream);

/* Post-norm residual LayerNorm of SwinV2 (V2:707-712, 387, 282) with the next GEMM's operand copy folded in:
 *   out[r, :] = (resid ? resid[r, :] : 0) + LayerNorm(y[r, :]) * gamma + beta        fp32, rows in token order;
 *   out may alias resid or y (in place); resid / out are dense [rows, C], y has pitch ldy.
 * copy (optional, dtype copy_dtype, pitch ldc) receives the same values at
 *   CSVIT_COPY_IDENTITY  row r                                   (operand of intermediate.dense)
 *   CSVIT_COPY_WINDOW    the (shifted-)window order of (H, W, ws, shift): replaces torch.roll + window_partition  V2:676-684
 *   CSVIT_COPY_MERGE2X2  row (b, y/2, x/2), column block ((y&1) + 2(x&1)) * C: the concat of patch merging       V2:373-384 */
enum { CSVIT_COPY_NONE = 0, CSVIT_COPY_IDENTITY = 1, CSVIT_COPY_WINDOW = 2, CSVIT_COPY_MERGE2X2 = 3 };
CSVIT_API int csvit_layernorm_post(const float* y, long long ldy, const float* resid, const float* gamma, const float* beta,
                                   float eps, float* out, void* copy, int copy_dtype, long long ldc, int copy_mode, int rows,
                                   int C, int H, int W, int ws, int shift, void* stream);

/* Dense multi-head attention for short sequences (S <= 128, head_dim 32), exact fp32 math:
 *   out[s, i, h*32:(h+1)*32] = softmax_j(q[s,i,h] . k[s,j,h] * scale) v[s,j,h]
 * q rows: n_seq*Lq, k/v rows: n_seq*S.  `scale` multiplies the logits (the reference passes sqrt(head_dim),
 * ref:cs_vit/net/transformer_module.py:243,273).  dtype applies to q, k, v and out. */
CSVIT_API int csvit_attention(const void* q, const void* k, const void* v, void* out, int dtype, long long ldq, long long ldk,
                    long long ldv, long long ldo, int n_seq, int Lq, int S, int heads, float scale, void* stream);

/* ---- training step: backward kernels (BASELINE configs[3], the finetune step) ----------------------------
 * torch autograd derives the backward of the reference from its eager ops (HF:591-653 SwinLayer; ref:cs_vit/net/
 * transformer_module.py:250-378; driven by loss.backward() at ref:scripts/finetune.py:224).  The entry points below
 * are what the autograd.Function wrappers of cs_vit/autograd.py bind instead.
 *
 * csvit_gemm_ex: out[M,N] = (accumulate ? out : 0) + sum_k A(m,k) B(n,k), fp32 accumulation on tcgen05.
 *   a_mn = 0: A stored [M,K] (pitch lda >= K);  a_mn = 1: A stored [K,M] (pitch lda >= M).  Same for B / N.
 *   dgrad  dX = dY W      : A = dY [T,out] a_mn=0, B = W [out,in] b_mn=1, M=T, N=in, K=out
 *   wgrad  dW = dY^T X    : A = dY [T,out] a_mn=1, B = X [T,in]   b_mn=1, M=out, N=in, K=T  (split-K, fp32 red.add)
 *   in_dtype BF16/F16 (kind::f16, any layout) or F32 (kind::tf32: K-major operands only; exact FMA in any layout
 *   with impl = CSVIT_GEMM_SIMT_FP32).
 *   split_k 0 = automatic.  accumulate / split-K need an fp32 output. */
CSVIT_API int csvit_gemm_ex(const void* A, long long lda, int a_mn, const void* B, long long ldb, int b_mn, int in_dtype, int M,
                            int N, int K, void* out, long long ldo, int out_dtype, int accumulate, int impl, int split_k,
                            void* stream);

/* dst[c, r] = src[r, c], fp32 (pitches in elements).  csvit_gemm_ex takes MN-major operands in the 16-bit formats
 * only; the fp32 (TF32) head transposes its small backward operands with this instead. */
CSVIT_API int csvit_transpose_f32(const float* src, long long lds, float* dst, long long ldd, int rows, int cols, void* stream);

/* Column reductions over the rows of a[rows, C] (dtype a_dtype, pitch lda), accumulated with atomics into fp32 s1 / s2
 * (caller zeroes them):
 *   CSVIT_CR_SUM      s1[c] += sum_r a          bias gradients (colsum of dY)
 *   CSVIT_CR_CENTERED s1 += sum_r (a - center), s2 += sum_r (a - center)^2     BatchNorm1d batch statistics
 *   CSVIT_CR_DOT      s1 += sum_r a,            s2 += sum_r a * b              BatchNorm1d backward (b fp32, pitch ldb)
 * row_mode CSVIT_LN_WINDOW reads row r from token window_index_map(r) (as csvit_layernorm).  If `copy` is non-NULL the
 * rows are also written out, converted to copy_dtype, in pass order: the fp32 residual gradient becomes a (window-
 * ordered) 16-bit GEMM operand in the same pass.  s1 / s2 may be NULL for a pure cast / gather. */
enum { CSVIT_CR_SUM = 0, CSVIT_CR_CENTERED = 1, CSVIT_CR_DOT = 2 };
CSVIT_API int csvit_col_reduce(const void* a, int a_dtype, long long lda, const float* b, long long ldb, const float* center,
                               int mode, int rows, int C, int row_mode, int H, int W, int ws, int shift, void* copy,
                               int copy_dtype, long long ldc, float* s1, float* s2, void* stream);

/* out[r, :] = (x ? x[r, :] : 0) + s[r / group_rows] * y[r, :] on dense fp32 [rows, C] tensors (C % 4 == 0): stochastic depth of the
 * attention branch in train mode - shortcut + drop_path(attention_output), s[b] = floor(keep + U[0,1)) / keep per sample
 * (HF:swin/modeling_swin.py:353-366, 646); with x = NULL the same scale applied to the incoming gradient in the backward pass. */
CSVIT_API int csvit_row_scale_add(const float* x, const float* y, const float* s, float* out, long long rows, int C, int group_rows,
                                  void* stream);

/* Elementwise, n elements (multiple of 4) of `dtype`:  GELU_FWD out = gelu(a) (exact erf, nn.GELU / HF "gelu");
 * GELU_BWD out = a * gelu'(b) (a = dY, b = pre-activation);  RELU_BWD out = b > 0 ? a : 0 (b = forward output). */
enum { CSVIT_EW_GELU_FWD = 0, CSVIT_EW_GELU_BWD = 1, CSVIT_EW_RELU_BWD = 2 };
CSVIT_API int csvit_eltwise(int op, const void* a, const void* b, void* out, int dtype, long long n, void* stream);

/* out[r,c] = a[c] dy[r,c] + b[c] x[r,c] + c0[c] (+ resid[r,c]), dense fp32 rows: BatchNorm1d backward per channel. */
CSVIT_API int csvit_affine2_rows(const float* dy, const float* x, const float* a, const float* b, const float* c0,
                                 const float* resid, float* out, long long rows, int C, void* stream);

/* Backward of csvit_layernorm (same modes and row maps; x is the fp32 input of the forward, dy the gradient of its
 * output rows in dy_dtype):  dx[map(r)] = (dres ? dres[map(r)] : 0) + dLN;  dgamma / dbeta (fp32, output width) are
 * accumulated with atomics (caller zeroes them).  dx may alias dres. */
CSVIT_API int csvit_layernorm_bwd(const float* x, const void* dy, int dy_dtype, long long ldy, const float* gamma, float eps,
                                  int rows, int C, int mode, int H, int W, int ws, int shift, const float* dres, float* dx,
                                  float* dgamma, float* dbeta, void* stream);

/* Backward of csvit_attention and of csvit_window_attention (pass q = qkv, k = qkv + C, v = qkv + 2C, pitches 3C,
 * n_seq = B*nW, Lq = S = ws*ws, scale = 1/sqrt(32), bias = csvit_expand_rel_bias table, mask_* = the window geometry;
 * mask_shift = 0 disables the shift mask).  Lq, S <= 64 (<= 128 when dbias is NULL: the head attention over 3 + 64 tokens of a
 * 256x256 SwinV2 input), head_dim 32, exact fp32 math, I/O in `dtype`.
 * dbias [heads, Lq, S] fp32 is accumulated (caller zeroes it); bias / dbias may be NULL. */
CSVIT_API int csvit_attention_bwd(const void* q, const void* k, const void* v, const void* dout, void* dq, void* dk, void* dv,
                                  int dtype, long long ldq, long long ldk, long long ldv, long long ldo, long long lddq,
                                  long long lddk, long long lddv, int n_seq, int Lq, int S, int heads, float scale,
                                  const float* bias, float* dbias, int mask_H, int mask_W, int mask_ws, int mask_shift,
                                  void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CSVIT_H_ */
