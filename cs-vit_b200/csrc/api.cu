// C ABI of libcsvit_sm100.so (declared in include/csvit.h).
#include <cstdarg>
#include <cstdio>
#include <cstdlib>

#include "../../include/csvit.h"
#include "errors.h"
#include "gemm.cuh"
#include "rowops.cuh"

namespace csvit {

static thread_local char g_err[1024] = "";

int set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return 1;
}
const char* last_error() { return g_err; }

bool pdl_enabled() {
  // OFF by default: measured slower on this pool (Swin-B 16.77 k vs 17.25 k img/s, SwinV2-B 10.70 k vs 10.90 k, same box, A/B/A/B)
  static const bool on = [] { const char* e = getenv("CSVIT_PDL"); return e && e[0] == '1'; }();
  return on;
}

}  // namespace csvit

using namespace csvit;

static_assert(int(CSVIT_F32) == int(DT_F32) && int(CSVIT_BF16) == int(DT_BF16) && int(CSVIT_F16) == int(DT_F16), "dtype codes");
static inline bool ok_dtype(int d) { return d == DT_F32 || d == DT_BF16 || d == DT_F16; }
static_assert(int(CSVIT_ACT_GELU) == int(ACT_GELU) && int(CSVIT_ACT_RELU) == int(ACT_RELU), "activation codes");
static_assert(int(CSVIT_LN_WINDOW) == int(LN_WINDOW) && int(CSVIT_LN_MERGE2X2) == int(LN_MERGE2X2), "layernorm modes");
static_assert(int(CSVIT_GEMM_SIMT_FP32) == int(GEMM_SIMT), "gemm impl codes");

static inline cudaStream_t S(void* s) { return static_cast<cudaStream_t>(s); }
static GemmTuning g_tune = {0, 0, -1, -1};

extern "C" {

int csvit_abi_version(void) { return CSVIT_ABI_VERSION; }
const char* csvit_last_error(void) { return last_error(); }

int csvit_window_index_map(int H, int W, int ws, int shift, int32_t* out, void* stream) {
  CSVIT_REQUIRE(ws > 0 && H % ws == 0 && W % ws == 0, "window_index_map: %dx%d not divisible by window %d", H, W, ws);
  CSVIT_REQUIRE(shift >= 0 && shift < ws, "window_index_map: shift %d outside [0,%d)", shift, ws);
  return launch_window_index_map(H, W, ws, shift, out, S(stream));
}
int csvit_shift_mask(int H, int W, int ws, int shift, float* out, void* stream) {
  CSVIT_REQUIRE(ws > 0 && H % ws == 0 && W % ws == 0, "shift_mask: %dx%d not divisible by window %d", H, W, ws);
  CSVIT_REQUIRE(shift >= 0 && shift < ws, "shift_mask: shift %d outside [0,%d)", shift, ws);
  return launch_shift_mask(H, W, ws, shift, out, S(stream));
}
int csvit_rel_pos_index(int ws, int32_t* out, void* stream) {
  CSVIT_REQUIRE(ws > 0, "rel_pos_index: window %d", ws);
  return launch_rel_index(ws, out, S(stream));
}
int csvit_merge_index_map(int H, int W, int32_t* out, void* stream) {
  CSVIT_REQUIRE(H % 2 == 0 && W % 2 == 0, "merge_index_map: %dx%d must be even", H, W);
  return launch_merge_index_map(H, W, out, S(stream));
}
int csvit_host_window_index_map(int H, int W, int ws, int shift, int32_t* out) {
  CSVIT_REQUIRE(ws > 0 && H % ws == 0 && W % ws == 0, "window_index_map: %dx%d not divisible by window %d", H, W, ws);
  CSVIT_REQUIRE(shift >= 0 && shift < ws, "window_index_map: shift %d outside [0,%d)", shift, ws);
  WinGeom g = make_geom(H, W, ws, shift);
  for (int r = 0; r < g.N; ++r) out[r] = win_row_to_token(g, r);
  return 0;
}
int csvit_host_shift_mask(int H, int W, int ws, int shift, float* out) {
  CSVIT_REQUIRE(ws > 0 && H % ws == 0 && W % ws == 0, "shift_mask: %dx%d not divisible by window %d", H, W, ws);
  CSVIT_REQUIRE(shift >= 0 && shift < ws, "shift_mask: shift %d outside [0,%d)", shift, ws);
  WinGeom g = make_geom(H, W, ws, shift);
  const int nW = (H / ws) * (W / ws);
  for (int w = 0; w < nW; ++w)
    for (int i = 0; i < g.L; ++i)
      for (int j = 0; j < g.L; ++j)
        out[(w * g.L + i) * g.L + j] = (shift > 0 && win_region(g, w, i) != win_region(g, w, j)) ? -100.0f : 0.0f;
  return 0;
}
int csvit_host_rel_pos_index(int ws, int32_t* out) {
  CSVIT_REQUIRE(ws > 0, "rel_pos_index: window %d", ws);
  const int L = ws * ws;
  for (int i = 0; i < L; ++i)
    for (int j = 0; j < L; ++j) out[i * L + j] = rel_pos_index(ws, i, j);
  return 0;
}
int csvit_host_merge_index_map(int H, int W, int32_t* out) {
  CSVIT_REQUIRE(H % 2 == 0 && W % 2 == 0, "merge_index_map: %dx%d must be even", H, W);
  for (int t = 0; t < (H / 2) * (W / 2); ++t)
    for (int q = 0; q < 4; ++q) out[t * 4 + q] = merge_src_token(W, t / (W / 2), t % (W / 2), q);
  return 0;
}

int csvit_expand_rel_bias(const float* table, float* out, int heads, int ws, void* stream) {
  CSVIT_REQUIRE(heads > 0 && ws > 0, "expand_rel_bias: heads=%d ws=%d", heads, ws);
  return launch_expand_rel_bias(table, out, heads, ws, S(stream));
}

int csvit_layernorm(const float* x, const float* gamma, const float* beta, float eps, void* out, int out_dtype,
                    long long ldo, int rows, int C, int mode, int H, int W, int ws, int shift, void* stream) {
  CSVIT_REQUIRE(ok_dtype(out_dtype), "layernorm: bad out_dtype %d", out_dtype);
  WinGeom g = make_geom(H > 0 ? H : 1, W > 0 ? W : 1, ws > 0 ? ws : 1, shift);
  if (mode == LN_WINDOW) {
    CSVIT_REQUIRE(ws > 0 && H % ws == 0 && W % ws == 0, "layernorm(window): %dx%d not divisible by window %d", H, W, ws);
    CSVIT_REQUIRE(shift >= 0 && shift < ws, "layernorm(window): shift %d outside [0,%d)", shift, ws);
    CSVIT_REQUIRE(rows % (H * W) == 0, "layernorm(window): rows %d not a multiple of %d tokens", rows, H * W);
  } else if (mode == LN_MERGE2X2) {
    CSVIT_REQUIRE(H % 2 == 0 && W % 2 == 0, "layernorm(merge): %dx%d must be even", H, W);
    CSVIT_REQUIRE(rows % ((H / 2) * (W / 2)) == 0, "layernorm(merge): rows %d not a multiple of %d", rows, (H / 2) * (W / 2));
  } else {
    CSVIT_REQUIRE(mode == LN_IDENTITY, "layernorm: unknown mode %d", mode);
  }
  return launch_layernorm(x, gamma, beta, eps, out, out_dtype, ldo, rows, C, mode, g, S(stream));
}

int csvit_affine_rows(const float* x, const float* scale, const float* shift, void* out, int out_dtype, long long rows,
                      int C, void* stream) {
  CSVIT_REQUIRE(ok_dtype(out_dtype), "affine_rows: bad out_dtype %d", out_dtype);
  return launch_affine_rows(x, scale, shift, out, out_dtype, rows, C, S(stream));
}

int csvit_patch_im2col(const float* img, void* out, int out_dtype, int B, int S_, const float* mean3, const float* std3,
                       void* stream) {
  CSVIT_REQUIRE(ok_dtype(out_dtype), "patch_im2col: bad out_dtype %d", out_dtype);
  return launch_patch_im2col(img, out, out_dtype, B, S_, mean3, std3, S(stream));
}

int csvit_linear(const void* A, long long lda, const void* W, long long ldw, int in_dtype, int M, int N, int K,
                 const float* bias, int act, const float* resid, long long ldr, void* out, long long ldo, int out_dtype,
                 int scatter_H, int scatter_W, int scatter_ws, int scatter_shift, int impl, void* stream) {
  CSVIT_REQUIRE(ok_dtype(in_dtype), "linear: bad in_dtype %d", in_dtype);
  CSVIT_REQUIRE(ok_dtype(out_dtype), "linear: bad out_dtype %d", out_dtype);
  CSVIT_REQUIRE(act >= ACT_NONE && act <= ACT_RELU, "linear: bad activation %d", act);
  CSVIT_REQUIRE(lda >= K && ldw >= K && ldo >= N, "linear: pitches smaller than the logical widths");
  EpiParams ep{};
  ep.bias = bias; ep.resid = resid; ep.out = out; ep.ldo = ldo; ep.ldr = ldr;
  ep.out_dtype = out_dtype; ep.act = act;
  ep.map_mode = ROWMAP_IDENTITY;
  ep.geom = make_geom(1, 1, 1, 0);
  if (scatter_ws > 0) {
    CSVIT_REQUIRE(scatter_H % scatter_ws == 0 && scatter_W % scatter_ws == 0, "linear: scatter grid %dx%d vs window %d",
                  scatter_H, scatter_W, scatter_ws);
    CSVIT_REQUIRE(M % (scatter_H * scatter_W) == 0, "linear: M=%d not a multiple of %d tokens", M, scatter_H * scatter_W);
    ep.map_mode = ROWMAP_WINDOW;
    ep.geom = make_geom(scatter_H, scatter_W, scatter_ws, scatter_shift);
  }
  return launch_gemm(A, lda, W, ldw, in_dtype, M, N, K, ep, impl, g_tune, S(stream));
}

int csvit_mlp_fused(const void* xn, long long ldxn, const void* W1, long long ldw1, const float* b1, const void* W2,
                    long long ldw2, const float* b2, float* x, long long ldx, int dtype, int M, int C, void* stream) {
  CSVIT_REQUIRE(ldxn >= C && ldw1 >= C && ldw2 >= 4 * C && ldx >= C, "mlp_fused: pitches smaller than the logical widths");
  return launch_mlp_fused(xn, ldxn, W1, ldw1, b1, W2, ldw2, b2, x, ldx, dtype, M, C, S(stream));
}

int csvit_last_gemm_kernel(void) { return last_gemm_kernel(); }

int csvit_set_gemm_tuning(int cluster, int tma_store, int max_ctas, int pair) {
  g_tune.pair = pair;
  CSVIT_REQUIRE(cluster == 0 || cluster == 1 || cluster == 2 || cluster == 4, "gemm tuning: cluster %d not in {0,1,2,4}", cluster);
  g_tune.cluster = cluster; g_tune.tma_store = tma_store; g_tune.max_ctas = max_ctas;
  return 0;
}

int csvit_swin_attn_fused(const float* x, float eps, const void* wqkv_h, const float* bqkv_h,
                          const void* bias_op, void* ctx, int dtype, int B, int H, int W, int C, int heads, int ws, int shift,
                          void* stream) {
  CSVIT_REQUIRE(x && wqkv_h && bqkv_h && bias_op && ctx, "swin_attn_fused: null operand");
  return launch_swin_attn_fused(x, eps, wqkv_h, bqkv_h, bias_op, ctx, dtype, B, H, W, C, heads, ws, shift, S(stream));
}

int csvit_swin_attn_core(const void* qkv, long long ldq, const void* bias_log2, void* ctx, int dtype, int B, int H, int W, int C,
                         int heads, int ws, int shift, int token_order, int q_prescaled, void* stream) {
  CSVIT_REQUIRE(qkv && bias_log2 && ctx, "swin_attn_core: null operand");
  return launch_swin_attn_core(qkv, ldq, bias_log2, ctx, dtype, B, H, W, C, heads, ws, shift, token_order, q_prescaled, S(stream));
}

int csvit_window_attention(const void* qkv, const float* bias, void* out, int dtype, int B, int H, int W, int C, int heads, int ws,
                           int shift, void* stream) {
  CSVIT_REQUIRE(dtype == DT_F32, "window_attention: the exact fp32 kernel only (16-bit operands: csvit_swin_attn_core), dtype %d", dtype);
  CSVIT_REQUIRE(bias != nullptr, "window_attention: needs the csvit_expand_rel_bias table");
  CSVIT_REQUIRE(C == heads * 32, "window_attention: head_dim must be 32 (C=%d heads=%d)", C, heads);
  CSVIT_REQUIRE(H % ws == 0 && W % ws == 0, "window_attention: %dx%d not divisible by window %d", H, W, ws);
  const int L = ws * ws, nW = (H / ws) * (W / ws);
  const float* q = static_cast<const float*>(qkv);
  return launch_attention_simt(q, q + C, q + 2 * C, out, DT_F32, 3ll * C, 3ll * C, 3ll * C, C, B * nW, L, L, heads,
                               0.17677669529663687f, bias, H, W, ws, shift, S(stream));
}

int csvit_crop_resize(const void* frames, int frames_u8, int N, int H, int W, const float* boxes, float expansion_ratio,
                      float* square_boxes_out, float* out, int size, void* stream) {
  CSVIT_REQUIRE(frames && boxes && out, "crop_resize: null operand");
  return launch_crop_resize(frames, frames_u8, N, H, W, boxes, expansion_ratio, square_boxes_out, out, size, S(stream));
}

int csvit_rot6d_to_axis_angle(const float* d6, float* axis_angle, long long n, void* stream) {
  CSVIT_REQUIRE(d6 && axis_angle, "rot6d_to_axis_angle: null operand");
  return launch_rot6d_to_axis_angle(d6, axis_angle, n, S(stream));
}

int csvit_mano_fk(const float* pose, const float* betas, const float* root_norm, const float* v_template, const float* shapedirs,
                  const float* posedirs, const float* pose_mean, const float* j_regressor, const float* lbs_weights,
                  const float* j_regressor_out, const int* parents16, const int* edges40, int rodrigues_mode, float* joint_cam,
                  float* verts_cam, float* root_transl, int n, void* stream) {
  CSVIT_REQUIRE(pose && betas && root_norm && v_template && shapedirs && j_regressor && lbs_weights && j_regressor_out && parents16 &&
                    edges40 && joint_cam && verts_cam && root_transl, "mano_fk: null operand");
  CSVIT_REQUIRE(rodrigues_mode == 0 || rodrigues_mode == 1, "mano_fk: rodrigues_mode %d", rodrigues_mode);
  return launch_mano_fk(pose, betas, root_norm, v_template, shapedirs, posedirs, pose_mean, j_regressor, lbs_weights, j_regressor_out,
                        parents16, edges40, rodrigues_mode, joint_cam, verts_cam, root_transl, n, S(stream));
}

int csvit_allreduce_f32(const void* const* bufs, const void* const* flags, void* multicast, long long n, int rank, int world, float scale,
                        int ctas, void* stream) {
  CSVIT_REQUIRE(bufs && flags, "allreduce_f32: null pointer tables");
  return launch_allreduce_f32(const_cast<void* const*>(bufs), const_cast<void* const*>(flags), multicast, n, rank, world, scale, ctas,
                              S(stream));
}

int csvit_attention(const void* q, const void* k, const void* v, void* out, int dtype, long long ldq, long long ldk,
                    long long ldv, long long ldo, int n_seq, int Lq, int S_, int heads, float scale, void* stream) {
  CSVIT_REQUIRE(ok_dtype(dtype), "attention: bad dtype %d", dtype);
  return launch_attention_simt(q, k, v, out, dtype, ldq, ldk, ldv, ldo, n_seq, Lq, S_, heads, scale, nullptr, 0, 0, 0, 0,
                               S(stream));
}

// ---- SwinV2 ------------------------------------------------------------------------------------------------
int csvit_swinv2_window_attention(const void* qkv, const float* bias_tab, const float* logit_scale, void* out, int dtype, int B, int H,
                                  int W, int C, int heads, int ws, int shift, int mask_repeat, int out_token_order, void* stream) {
  CSVIT_REQUIRE(ok_dtype(dtype), "swinv2_window_attention: bad dtype %d", dtype);
  CSVIT_REQUIRE(bias_tab != nullptr && logit_scale != nullptr, "swinv2_window_attention: bias table and logit scale are required");
  CSVIT_REQUIRE(mask_repeat >= 0 && mask_repeat <= 2, "swinv2_window_attention: mask_repeat %d outside [0,2]", mask_repeat);
  return launch_swinv2_window_attention(qkv, bias_tab, logit_scale, out, dtype, B, H, W, C, heads, ws, shift, mask_repeat,
                                        out_token_order ? 1 : 0, S(stream));
}

static int swinv2_qkv(const void* A, long long lda, const void* W, long long ldw, int dtype, int M, int C, int K, const float* bias,
                      const float* qscale_log2, void* out, long long ldo, float* rnorm, void* stream) {
  CSVIT_REQUIRE(dtype == DT_BF16 || dtype == DT_F16, "swinv2_qkv: 16-bit operands only (the fp32 mode normalises inside its attention kernel)");
  CSVIT_REQUIRE(A && W && out && qscale_log2, "swinv2_qkv: null operand");
  CSVIT_REQUIRE(C > 0 && C % 32 == 0 && lda >= K && ldw >= K && ldo >= 3ll * C, "swinv2_qkv: C=%d must be a multiple of 32, pitches >= widths", C);
  CSVIT_REQUIRE(ldo % 8 == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0 && (!bias || (reinterpret_cast<uintptr_t>(bias) & 15) == 0),
                "swinv2_qkv: output rows and bias must be 16-byte aligned");
  EpiParams ep{};
  ep.bias = bias; ep.out = out; ep.ldo = ldo; ep.out_dtype = dtype; ep.act = ACT_NONE;
  ep.map_mode = ROWMAP_IDENTITY;
  ep.geom = make_geom(1, 1, 1, 0);
  ep.cos_scale = qscale_log2; ep.cos_C = C;
  ep.rnorm = rnorm;
  return launch_gemm(A, lda, W, ldw, dtype, M, 3 * C, K, ep, GEMM_TC, g_tune, S(stream));
}

int csvit_swinv2_qkv(const void* A, long long lda, const void* W, long long ldw, int dtype, int M, int C, int K, const float* bias,
                     const float* qscale_log2, void* out, long long ldo, void* stream) {
  return swinv2_qkv(A, lda, W, ldw, dtype, M, C, K, bias, qscale_log2, out, ldo, nullptr, stream);
}

int csvit_swinv2_qkv_train(const void* A, long long lda, const void* W, long long ldw, int dtype, int M, int C, int K, const float* bias,
                           const float* qscale_log2, void* out, long long ldo, float* rnorm, void* stream) {
  CSVIT_REQUIRE(rnorm, "swinv2_qkv_train: null rnorm");
  return swinv2_qkv(A, lda, W, ldw, dtype, M, C, K, bias, qscale_log2, out, ldo, rnorm, stream);
}

int csvit_swinv2_cosnorm_bwd(const void* qkv, const float* rnorm, const float* qscale_log2, const void* dq2, const void* dk, const void* dv,
                             void* dqkv, float* dqscale, int dtype, int rows, int C, void* stream) {
  CSVIT_REQUIRE(dtype == DT_BF16 || dtype == DT_F16, "swinv2_cosnorm_bwd: 16-bit operands only");
  CSVIT_REQUIRE(qkv && rnorm && qscale_log2 && dq2 && dk && dv && dqkv && dqscale, "swinv2_cosnorm_bwd: null operand");
  CSVIT_REQUIRE(C > 0 && C % 32 == 0 && C <= 2048, "swinv2_cosnorm_bwd: C=%d must be a multiple of 32 and <= 2048", C);
  for (const void* p : {qkv, dq2, dk, dv, static_cast<const void*>(dqkv)})
    CSVIT_REQUIRE((reinterpret_cast<uintptr_t>(p) & 15) == 0, "swinv2_cosnorm_bwd: 16-bit operands must be 16-byte aligned");
  return launch_swinv2_cosnorm_bwd(qkv, rnorm, qscale_log2, dq2, dk, dv, dqkv, dqscale, dtype, rows, C, S(stream));
}

int csvit_swinv2_attn_tc(const void* qkv, long long ldq, const float* bias_log2, void* ctx, int dtype, int B, int H, int W, int C,
                         int heads, int shift, int mask_repeat, int token_order, void* stream) {
  CSVIT_REQUIRE(qkv && bias_log2 && ctx, "swinv2_attn_tc: null operand");
  CSVIT_REQUIRE(mask_repeat >= 0 && mask_repeat <= 2, "swinv2_attn_tc: mask_repeat %d outside [0,2]", mask_repeat);
  return launch_swinv2_attn_tc(qkv, ldq, bias_log2, ctx, dtype, B, H, W, C, heads, shift, mask_repeat, token_order, S(stream));
}

int csvit_swinv2_attn_tc_train(const void* qkv, long long ldq, const float* bias_log2, void* ctx, float* lse2, int dtype, int B, int H,
                               int W, int C, int heads, int shift, int mask_repeat, void* stream) {
  CSVIT_REQUIRE(qkv && bias_log2 && ctx && lse2, "swinv2_attn_tc_train: null operand");
  CSVIT_REQUIRE(mask_repeat >= 0 && mask_repeat <= 2, "swinv2_attn_tc_train: mask_repeat %d outside [0,2]", mask_repeat);
  return launch_swinv2_attn_tc_train(qkv, ldq, bias_log2, ctx, lse2, dtype, B, H, W, C, heads, shift, mask_repeat, S(stream));
}

int csvit_swinv2_attn_tc_bwd(const void* qkv, long long ldq, const void* ctx, const void* dctx, const float* lse2, const float* bias_log2,
                             void* dq, void* dk, void* dv, float* dbias_log2, int dtype, int B, int H, int W, int C, int heads, int shift,
                             int mask_repeat, void* stream) {
  CSVIT_REQUIRE(qkv && ctx && dctx && lse2 && bias_log2 && dq && dk && dv && dbias_log2, "swinv2_attn_tc_bwd: null operand");
  return launch_swinv2_attn_bwd(qkv, ldq, ctx, dctx, lse2, bias_log2, dq, dk, dv, dbias_log2, dtype, B, H, W, C, heads, shift, mask_repeat,
                                S(stream));
}

int csvit_swinv2_attn8_tc(const void* qkv, long long ldq, const float* bias_log2, void* ctx, int dtype, int B, int H, int W, int C,
                          int heads, int shift, int mask_repeat, int token_order, void* stream) {
  CSVIT_REQUIRE(qkv && bias_log2 && ctx, "swinv2_attn8_tc: null operand");
  return launch_swinv2_attn8_tc(qkv, ldq, bias_log2, ctx, nullptr, dtype, B, H, W, C, heads, shift, mask_repeat, token_order, S(stream));
}

int csvit_swinv2_attn8_tc_train(const void* qkv, long long ldq, const float* bias_log2, void* ctx, float* lse2, int dtype, int B, int H,
                                int W, int C, int heads, int shift, int mask_repeat, void* stream) {
  CSVIT_REQUIRE(qkv && bias_log2 && ctx && lse2, "swinv2_attn8_tc_train: null operand");
  return launch_swinv2_attn8_tc(qkv, ldq, bias_log2, ctx, lse2, dtype, B, H, W, C, heads, shift, mask_repeat, 0, S(stream));
}

int csvit_swinv2_attn8_tc_bwd(const void* qkv, long long ldq, const void* ctx, const void* dctx, const float* lse2, const float* bias_log2,
                              void* dq, void* dk, void* dv, float* dbias_log2, int dtype, int B, int H, int W, int C, int heads, int shift,
                              int mask_repeat, void* stream) {
  CSVIT_REQUIRE(qkv && ctx && dctx && lse2 && bias_log2 && dq && dk && dv && dbias_log2, "swinv2_attn8_tc_bwd: null operand");
  return launch_swinv2_attn8_bwd(qkv, ldq, ctx, dctx, lse2, bias_log2, dq, dk, dv, dbias_log2, dtype, B, H, W, C, heads, shift,
                                 mask_repeat, S(stream));
}

int csvit_layernorm_post(const float* y, long long ldy, const float* resid, const float* gamma, const float* beta, float eps, float* out,
                         void* copy, int copy_dtype, long long ldc, int copy_mode, int rows, int C, int H, int W, int ws, int shift,
                         void* stream) {
  CSVIT_REQUIRE(ok_dtype(copy_dtype), "layernorm_post: bad copy dtype %d", copy_dtype);
  CSVIT_REQUIRE(ldy >= C, "layernorm_post: pitch smaller than the row width");
  WinGeom g = make_geom(H > 0 ? H : 1, W > 0 ? W : 1, ws > 0 ? ws : 1, shift);
  if (copy_mode == CSVIT_COPY_WINDOW) {
    CSVIT_REQUIRE(ws > 0 && H % ws == 0 && W % ws == 0, "layernorm_post(window): %dx%d not divisible by window %d", H, W, ws);
    CSVIT_REQUIRE(shift >= 0 && shift < ws, "layernorm_post(window): shift %d outside [0,%d)", shift, ws);
    CSVIT_REQUIRE(rows % (H * W) == 0, "layernorm_post(window): rows %d not a multiple of %d tokens", rows, H * W);
    CSVIT_REQUIRE(ldc >= C, "layernorm_post(window): copy pitch smaller than the row width");
  } else if (copy_mode == CSVIT_COPY_MERGE2X2) {
    CSVIT_REQUIRE(H > 0 && W > 0 && H % 2 == 0 && W % 2 == 0, "layernorm_post(merge): %dx%d must be even", H, W);
    CSVIT_REQUIRE(rows % (H * W) == 0, "layernorm_post(merge): rows %d not a multiple of %d tokens", rows, H * W);
    CSVIT_REQUIRE(ldc >= 4 * C, "layernorm_post(merge): copy pitch smaller than 4C");
  }
  return launch_layernorm_post(y, ldy, resid, gamma, beta, eps, out, copy, copy_dtype, ldc, copy_mode, rows, C, g, S(stream));
}

// ---- training step (backward) ----------------------------------------------------------------------------
int csvit_gemm_ex(const void* A, long long lda, int a_mn, const void* B, long long ldb, int b_mn, int in_dtype, int M, int N, int K,
                  void* out, long long ldo, int out_dtype, int accumulate, int impl, int split_k, void* stream) {
  CSVIT_REQUIRE(ok_dtype(in_dtype) && ok_dtype(out_dtype), "gemm_ex: bad dtype (%d, %d)", in_dtype, out_dtype);
  CSVIT_REQUIRE(lda >= (a_mn ? M : K) && ldb >= (b_mn ? N : K) && ldo >= N, "gemm_ex: pitches smaller than the logical widths");
  return launch_gemm_ex(A, lda, a_mn ? 1 : 0, B, ldb, b_mn ? 1 : 0, in_dtype, M, N, K, out, ldo, out_dtype, accumulate ? 1 : 0, impl,
                        split_k, S(stream));
}

int csvit_col_reduce(const void* a, int a_dtype, long long lda, const float* b, long long ldb, const float* center, int mode,
                     int rows, int C, int row_mode, int H, int W, int ws, int shift, void* copy, int copy_dtype, long long ldc,
                     float* s1, float* s2, void* stream) {
  CSVIT_REQUIRE(ok_dtype(a_dtype) && ok_dtype(copy_dtype), "col_reduce: bad dtype (%d, %d)", a_dtype, copy_dtype);
  WinGeom g = make_geom(H > 0 ? H : 1, W > 0 ? W : 1, ws > 0 ? ws : 1, shift);
  if (row_mode == LN_WINDOW) {
    CSVIT_REQUIRE(ws > 0 && H % ws == 0 && W % ws == 0, "col_reduce(window): %dx%d not divisible by window %d", H, W, ws);
    CSVIT_REQUIRE(shift >= 0 && shift < ws, "col_reduce(window): shift %d outside [0,%d)", shift, ws);
    CSVIT_REQUIRE(rows % (H * W) == 0, "col_reduce(window): rows %d not a multiple of %d tokens", rows, H * W);
  }
  return launch_col_reduce(a, a_dtype, lda, b, ldb, center, mode, rows, C, row_mode, g, copy, copy_dtype, ldc, s1, s2, S(stream));
}

int csvit_transpose_f32(const float* src, long long lds, float* dst, long long ldd, int rows, int cols, void* stream) {
  CSVIT_REQUIRE(lds >= cols && ldd >= rows, "transpose: pitches smaller than the logical widths");
  return launch_transpose_f32(src, lds, dst, ldd, rows, cols, S(stream));
}

int csvit_row_scale_add(const float* x, const float* y, const float* s, float* out, long long rows, int C, int group_rows, void* stream) {
  CSVIT_REQUIRE(y && s && out, "row_scale_add: null operand");
  return launch_row_scale_add(x, y, s, out, rows, C, group_rows, S(stream));
}

int csvit_eltwise(int op, const void* a, const void* b, void* out, int dtype, long long n, void* stream) {
  CSVIT_REQUIRE(ok_dtype(dtype), "eltwise: bad dtype %d", dtype);
  return launch_eltwise(op, a, b, out, dtype, n, S(stream));
}

int csvit_affine2_rows(const float* dy, const float* x, const float* a, const float* b, const float* c0, const float* resid,
                       float* out, long long rows, int C, void* stream) {
  return launch_affine2_rows(dy, x, a, b, c0, resid, out, rows, C, S(stream));
}

int csvit_layernorm_bwd(const float* x, const void* dy, int dy_dtype, long long ldy, const float* gamma, float eps, int rows, int C,
                        int mode, int H, int W, int ws, int shift, const float* dres, float* dx, float* dgamma, float* dbeta,
                        void* stream) {
  CSVIT_REQUIRE(ok_dtype(dy_dtype), "layernorm_bwd: bad dy dtype %d", dy_dtype);
  WinGeom g = make_geom(H > 0 ? H : 1, W > 0 ? W : 1, ws > 0 ? ws : 1, shift);
  if (mode == LN_WINDOW) {
    CSVIT_REQUIRE(ws > 0 && H % ws == 0 && W % ws == 0, "layernorm_bwd(window): %dx%d not divisible by window %d", H, W, ws);
    CSVIT_REQUIRE(shift >= 0 && shift < ws, "layernorm_bwd(window): shift %d outside [0,%d)", shift, ws);
    CSVIT_REQUIRE(rows % (H * W) == 0, "layernorm_bwd(window): rows %d not a multiple of %d tokens", rows, H * W);
  } else if (mode == LN_MERGE2X2) {
    CSVIT_REQUIRE(H % 2 == 0 && W % 2 == 0, "layernorm_bwd(merge): %dx%d must be even", H, W);
    CSVIT_REQUIRE(rows % ((H / 2) * (W / 2)) == 0, "layernorm_bwd(merge): rows %d not a multiple of %d", rows, (H / 2) * (W / 2));
  } else {
    CSVIT_REQUIRE(mode == LN_IDENTITY, "layernorm_bwd: unknown mode %d", mode);
  }
  return launch_layernorm_bwd(x, dy, dy_dtype, ldy, gamma, eps, rows, C, mode, g, dres, dx, dgamma, dbeta, S(stream));
}

int csvit_attention_bwd(const void* q, const void* k, const void* v, const void* dout, void* dq, void* dk, void* dv, int dtype,
                        long long ldq, long long ldk, long long ldv, long long ldo, long long lddq, long long lddk, long long lddv,
                        int n_seq, int Lq, int S_, int heads, float scale, const float* bias, float* dbias, int mask_H, int mask_W,
                        int mask_ws, int mask_shift, void* stream) {
  CSVIT_REQUIRE(ok_dtype(dtype), "attention_bwd: bad dtype %d", dtype);
  CSVIT_REQUIRE((bias == nullptr) == (dbias == nullptr) || dbias == nullptr, "attention_bwd: dbias given without bias");
  // Swin windows on packed 16-bit qkv / dqkv tensors: tensor-core kernel (attention_bwd_mma.cu); everything else (fp32, the
  // head's dense MHA, unpacked operands) takes the exact SIMT kernel.
  static int force_simt = -1;
  if (force_simt < 0) { const char* e = getenv("CSVIT_ATTN_BWD_SIMT"); force_simt = (e && e[0] == '1') ? 1 : 0; }
  const long long C = 32ll * heads, es = 2;
  const char *qb = static_cast<const char*>(q), *kb = static_cast<const char*>(k), *vb = static_cast<const char*>(v);
  const char *dqb = static_cast<const char*>(dq), *dkb = static_cast<const char*>(dk), *dvb = static_cast<const char*>(dv);
  if (!force_simt && (dtype == DT_BF16 || dtype == DT_F16) && bias && dbias && Lq == 49 && S_ == 49 && mask_ws == 7 && mask_H > 0 &&
      mask_W > 0 && kb == qb + C * es && vb == qb + 2 * C * es && dkb == dqb + C * es && dvb == dqb + 2 * C * es && ldq == 3 * C &&
      ldk == 3 * C && ldv == 3 * C && lddq == 3 * C && lddk == 3 * C && lddv == 3 * C && ldo == C) {
    const int nW = (mask_H / 7) * (mask_W / 7);
    if (nW > 0 && n_seq % nW == 0 && mask_H % 7 == 0 && mask_W % 7 == 0)
      return launch_window_attention_bwd_mma(q, dout, dq, dtype, bias, dbias, n_seq / nW, mask_H, mask_W, int(C), heads, 7, mask_shift,
                                             S(stream));
  }
  return launch_attention_bwd(q, k, v, dout, dq, dk, dv, dtype, ldq, ldk, ldv, ldo, lddq, lddk, lddv, n_seq, Lq, S_, heads, scale,
                              bias, dbias, mask_H, mask_W, mask_ws, mask_shift, S(stream));
}

}  // extern "C"
