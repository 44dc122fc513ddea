#pragma once
#include "common.cuh"
#include "gemm.cuh"

namespace csvit {

enum : int { LN_IDENTITY = 0, LN_WINDOW = 1, LN_MERGE2X2 = 2 };

int launch_layernorm(const float* x, const float* gamma, const float* beta, float eps, void* out, int out_dtype,
                     long long ldo, int rows, int C, int mode, const WinGeom& g, cudaStream_t stream);
int launch_affine_rows(const float* x, const float* scale, const float* shift, void* out, int out_dtype, long long rows,
                       int C, cudaStream_t stream);
int launch_patch_im2col(const float* img, void* out, int out_dtype, int B, int S, const float* mean3, const float* std3,
                        cudaStream_t stream);
int launch_window_index_map(int H, int W, int ws, int shift, int* out, cudaStream_t stream);
int launch_shift_mask(int H, int W, int ws, int shift, float* out, cudaStream_t stream);
int launch_rel_index(int ws, int* out, cudaStream_t stream);
int launch_merge_index_map(int H, int W, int* out, cudaStream_t stream);
int launch_expand_rel_bias(const float* table, float* out, int heads, int ws, cudaStream_t stream);

// attn_fused.cu
int launch_swin_attn_fused(const float* x, float eps, const void* wqkv_h, const float* bqkv_h,
                           const void* bias_op, void* ctx, int dtype, int B, int H, int W, int C, int heads, int ws, int shift,
                           cudaStream_t stream);

// attn_core.cu
int launch_swin_attn_core(const void* qkv, long long ldq, const void* bias_log2, void* ctx, int dtype, int B, int H, int W, int C,
                          int heads, int ws, int shift, int token_order, int q_prescaled, cudaStream_t stream);

// crop.cu
int launch_crop_resize(const void* frames, int frames_u8, int N, int H, int W, const float* boxes, float expansion, float* square_out,
                       float* out, int S, cudaStream_t stream);

// tail.cu
int launch_rot6d_to_axis_angle(const float* d6, float* aa, long long n, cudaStream_t stream);
int launch_mano_fk(const float* pose, const float* betas, const float* root_norm, const float* v_template, const float* shapedirs,
                   const float* posedirs, const float* pose_mean, const float* j_regressor, const float* lbs_weights, const float* j_out,
                   const int* parents16, const int* edges40, int rodrigues_mode, float* joint_cam, float* verts_cam, float* root_transl,
                   int n, cudaStream_t stream);

// stream.cu
int launch_stream_update(const float* tok, const float* ts, const int* ids, const bool* reset, int nb, float* tokens, float* stamps,
                         int* hist, int* head, int num_streams, int W, int D, float* window, float* win_stamps, int* key_start,
                         cudaStream_t stream);

// allreduce.cu
int launch_allreduce_f32(void* const* bufs, void* const* flags, void* mc, long long n, int rank, int world, float scale, int ctas,
                         cudaStream_t stream);

// mlp_fused.cu
int launch_mlp_fused(const void* xn, long long ldxn, const void* W1, long long ldw1, const float* b1, const void* W2,
                     long long ldw2, const float* b2, float* x, long long ldx, int dtype, int M, int C, cudaStream_t stream);

// attention_simt.cu
int launch_attention_simt(const void* q, const void* k, const void* v, void* out, int dtype, long long ldq, long long ldk,
                          long long ldv, long long ldo, int n_seq, int Lq, int S, int heads, float scale,
                          const float* bias, int mH, int mW, int mws, int mshift, const int* key_start, cudaStream_t stream);

// gemm_ex.cu
int launch_gemm_ex(const void* A, long long lda, int a_mn, const void* B, long long ldb, int b_mn, int in_dtype, int M, int N,
                   int K, void* out, long long ldo, int out_dtype, int accumulate, int impl, int split_k, cudaStream_t stream);

// backward.cu
int launch_col_reduce(const void* a, int a_dtype, long long lda, const float* b, long long ldb, const float* center, int mode,
                      int rows, int C, int row_mode, const WinGeom& g, void* copy, int copy_dtype, long long ldc, float* s1,
                      float* s2, cudaStream_t stream);
int launch_transpose_f32(const float* src, long long lds, float* dst, long long ldd, int R, int C, cudaStream_t stream);
int launch_row_scale_add(const float* x, const float* y, const float* s, float* out, long long rows, int C, int group_rows,
                         cudaStream_t stream);
int launch_eltwise(int op, const void* a, const void* b, void* out, int dtype, long long n, cudaStream_t stream);
int launch_affine2_rows(const float* dy, const float* x, const float* a, const float* b, const float* c0, const float* resid,
                        float* out, long long rows, int C, cudaStream_t stream);
int launch_layernorm_bwd(const float* x, const void* dy, int dy_dtype, long long ldy, const float* gamma, float eps, int rows, int C,
                         int mode, const WinGeom& g, const float* dres, float* dx, float* dgamma, float* dbeta, cudaStream_t stream);
int launch_attention_bwd(const void* q, const void* k, const void* v, const void* dout, void* dq, void* dk, void* dv, int dtype,
                         long long ldq, long long ldk, long long ldv, long long ldo, long long lddq, long long lddk, long long lddv,
                         int n_seq, int Lq, int S, int heads, float scale, const float* bias, float* dbias, int mH, int mW, int mws,
                         int mshift, cudaStream_t stream);

// swinv2.cu
int launch_swinv2_window_attention(const void* qkv, const float* bias_tab, const float* logit_scale, void* out, int dtype, int B, int H,
                                   int W, int C, int heads, int ws, int shift, int mask_repeat, int tok_order, cudaStream_t stream);
int launch_layernorm_post(const float* y, long long ldy, const float* resid, const float* gamma, const float* beta, float eps,
                          float* xo, void* copy, int copy_dtype, long long ldc, int copy_mode, int rows, int C, const WinGeom& g,
                          float* row_scale, cudaStream_t stream);

// swinv2_attn_tc.cu
int launch_swinv2_attn_tc(const void* qkv, long long ldq, const float* bias_log2, void* ctx, int dtype, int B, int H, int W, int C,
                          int heads, int shift, int mask_repeat, int token_order, cudaStream_t stream);
int launch_swinv2_attn_tc_train(const void* qkv, long long ldq, const float* bias_log2, void* ctx, float* lse2, int dtype, int B, int H,
                                int W, int C, int heads, int shift, int mask_repeat, cudaStream_t stream);
// swinv2_attn_bwd.cu
int launch_swinv2_attn_bwd(const void* qkv, long long ldq, const void* ctx, const void* dctx, const float* lse2, const float* bias_log2,
                           void* dq, void* dk, void* dv, float* dbias_log2, int dtype, int B, int H, int W, int C, int heads, int shift,
                           int mask_repeat, cudaStream_t stream);

// swinv2_attn8.cu (lse2 null: inference)
int launch_swinv2_attn8_tc(const void* qkv, long long ldq, const float* bias_log2, void* ctx, float* lse2, int dtype, int B, int H, int W,
                           int C, int heads, int shift, int mask_repeat, int token_order, cudaStream_t stream);
int launch_swinv2_attn8_bwd(const void* qkv, long long ldq, const void* ctx, const void* dctx, const float* lse2, const float* bias_log2,
                            void* dq, void* dk, void* dv, float* dbias_log2, int dtype, int B, int H, int W, int C, int heads, int shift,
                            int mask_repeat, cudaStream_t stream);

// swinv2_cosnorm_bwd.cu
int launch_swinv2_cosnorm_bwd(const void* qkv, const float* rnorm, const float* qscale_log2, const void* dq2, const void* dk,
                              const void* dv, void* dqkv, float* dqscale, int dtype, int rows, int C, cudaStream_t stream);

// attention_bwd_mma.cu
int launch_window_attention_bwd_mma(const void* qkv, const void* dout, void* dqkv, int dtype, const float* bias, float* dbias, int B,
                                    int H, int W, int C, int heads, int ws, int shift, cudaStream_t stream);

}  // namespace csvit
