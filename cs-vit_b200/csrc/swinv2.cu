// SwinV2 additions (SURVEY.md §8f row 1: every shipped CS-ViT configuration uses a swinv2 w16 @256 backbone).
//
// What differs from Swin v1 on the hot path (HF:swinv2/modeling_swinv2.py = "V2:"):
//   * scaled-cosine attention: S = normalize(Q) normalize(K)^T * exp(min(logit_scale, ln 100)) + 16 sigmoid(CPB-MLP)[idx]
//     + shift mask added TWICE (V2:455-474); windows of 16x16 = 256 tokens (8x8 = 64 at the last stage of a 256^2 input)
//   * res-post-norm: x = x + LN(attn(x)), x = x + LN(mlp(x))  (V2:707-712): the LayerNorm sits on the branch OUTPUT, the
//     Linear layers read the raw residual stream
//   * patch merging: 2x2 concat -> Linear(4C, 2C) -> LN(2C)   (V2:365-388)
//
//   swinv2_attn_kernel<T>      16-bit tensor-core (mma.sync m16n8k16) cosine window attention, flash-style online softmax over
//                              64-key chunks, one (window, head) per CTA pass, 4 warps = 4 query tiles in flight
//   swinv2_attn_f32_kernel     exact fp32 form of the same (validation mode, 1e-4 bar)
//   ln_post_kernel             xo = (resid) + LN(y) per token, and in the same pass the 16-bit (or fp32) copy of xo that the next
//                              GEMM reads: token order (fc1), the NEXT block's shifted-window order (Q/K/V), or the 2x2-merged
//                              [N/4, 4C] layout (patch merging) - so window partition, roll and concat never run as copies
#include <cuda_fp8.h>

#include "errors.h"
#include "mma_sync.cuh"
#include "rowops.cuh"

namespace csvit {

using namespace mma;

enum : int { COPY_NONE = 0, COPY_IDENTITY = 1, COPY_WINDOW = 2, COPY_MERGE2X2 = 3 };

// ----------------------------------------------------------------------------------------------------
// cosine window attention, 16-bit operands
// ----------------------------------------------------------------------------------------------------
constexpr int V2_THREADS = 128;
constexpr int V2_MAXL = 256;

template <typename T> __device__ __forceinline__ float2 unpack2(uint32_t u);
template <> __device__ __forceinline__ float2 unpack2<__nv_bfloat16>(uint32_t u) {
  return make_float2(__uint_as_float(u << 16), __uint_as_float(u & 0xffff0000u));
}
template <> __device__ __forceinline__ float2 unpack2<__half>(uint32_t u) {
  return __half22float2(*reinterpret_cast<__half2*>(&u));
}

__host__ __device__ inline int v2_smem_bytes(int ws) {
  const int L = ws * ws, tw = 2 * ws - 1;
  const int tb = (tw * tw + 3) & ~3;
  return tb * 4 + 2 * L * 4 + L + 2 * L + 3 * L * ROW_BYTES;   // bias, 1/|q|, 1/|k|, region ids, token ids, Q / K / V
}

__device__ __forceinline__ float ex2_ftz(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
template <typename T> struct Ones16;
template <> struct Ones16<__nv_bfloat16> { static constexpr uint32_t v = 0x3F803F80u; };
template <> struct Ones16<__half> { static constexpr uint32_t v = 0x3C003C00u; };

constexpr float V2_LOG2E = 1.4426950408889634f;
#ifndef V2_TILES16
#define V2_TILES16 2   // query tiles per warp pass for 256-token windows (1 = one tile, 4 CTAs/SM; 2 = two tiles, 3 CTAs/SM)
#endif

// qkv: window-ordered tokens [B*N, 3C] (Q | K | V column blocks, head h at columns 32h), out [B*N, C] window-ordered.
// bias_tab [heads, (2ws-1)^2] = 16 sigmoid(cpb_mlp(coords)) (V2:460-472), logit_scale [heads] = exp(min(ls, ln 100)).
// gridDim.x is a multiple of `heads`: a CTA serves one head (its bias table stays in shared memory) and walks windows.
//
// The kernel is bound by instruction issue on the softmax side (head_dim 32: 2 MMAs per 64 logits), so the per-logit work is
// pared down to  FMUL, FFMA(+bias), max, FADD, MUFU.EX2, half a pack:
//   * logits live in the log2 domain: log2(e) is folded into the per-row scale, the bias table and the mask value
//   * the bias address is (per-thread row base) - (compile-time column term): one LDS with an immediate offset, no index math
//   * row sums come out of the tensor core: P V is extended by a ones column (one extra MMA per 16 keys), which also makes the
//     normaliser the sum of the ROUNDED probabilities that multiply V
template <typename T, int WS, int TILES>
__global__ void __launch_bounds__(V2_THREADS, TILES == 2 ? 3 : 4)
swinv2_attn_kernel(const T* __restrict__ qkv, const float* __restrict__ bias_tab, const float* __restrict__ logit_scale,
                   T* __restrict__ out, int num_windows, int C, int heads, WinGeom g, int nW, float mask_value, int tok_order) {
  static_assert(WS == 8 || WS == 16, "windows of 8x8 and 16x16 tokens");
  constexpr int L = WS * WS, TW = 2 * WS - 1, TB = TW * TW, TBP = (TB + 3) & ~3;
  extern __shared__ __align__(16) uint8_t v2_smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  float* bias_s = reinterpret_cast<float*>(v2_smem);
  float* rq_s = bias_s + TBP;
  float* rk_s = rq_s + L;
  int8_t* region_s = reinterpret_cast<int8_t*>(rk_s + L);
  int16_t* tok_s = reinterpret_cast<int16_t*>(region_s + L);    // tok_order: token id (within the image) of each window slot
  uint8_t* Qs = reinterpret_cast<uint8_t*>(tok_s + L);
  uint8_t* Ks = Qs + L * ROW_BYTES;
  uint8_t* Vs = Ks + L * ROW_BYTES;

  const int h = blockIdx.x % heads;
  for (int i = tid; i < TB; i += V2_THREADS) bias_s[i] = __ldg(bias_tab + h * TB + i) * V2_LOG2E;
  const float scale = __ldg(logit_scale + h) * V2_LOG2E;
  const float mask_l2 = mask_value * V2_LOG2E;

  const int ld_qkv = 3 * C;
  const int nWy = g.H / WS;
  const int wstride = gridDim.x / heads;
  const int q2 = (lane & 3) * 2;
  for (int wg = blockIdx.x / heads; wg < num_windows; wg += wstride) {   // global window = b*nW + w
    __syncthreads();   // the previous window's tiles are consumed (first pass: the bias table above is written)
    const int w = wg % nW;
    const long long row0 = static_cast<long long>(wg) * L;
    const T* src = qkv + row0 * ld_qkv + h * 32;
#pragma unroll 4
    for (int idx = tid; idx < 3 * L * 4; idx += V2_THREADS) {
      const int which = idx / (L * 4), rem = idx - which * (L * 4);
      const int r = rem >> 2, ch = rem & 3;
      cp_async16(Qs + which * (L * ROW_BYTES) + row_off(r, ch), src + static_cast<long long>(r) * ld_qkv + which * C + ch * 8);
    }
    const int wy = w / g.nWx, wx = w - wy * g.nWx;
    const bool masked = g.shift > 0 && (wy == nWy - 1 || wx == g.nWx - 1);   // CTA-uniform
    if (masked)
      for (int i = tid; i < L; i += V2_THREADS) region_s[i] = static_cast<int8_t>(win_region(g, w, i));
    long long obase = row0;          // window-ordered output: row0 + slot;  token-ordered: image base + token id of the slot
    if (tok_order) {                 // window_reverse + roll(+shift) folded into the store: the out-proj GEMM sees plain rows
      for (int i = tid; i < L; i += V2_THREADS) tok_s[i] = static_cast<int16_t>(win_row_to_token(g, w * L + i));
      obase = static_cast<long long>(wg / nW) * g.N;
    }
    cp_async_wait_all();
    __syncthreads();
    // log2(e) * logit_scale / max(|q_i|, 1e-12) and 1 / max(|k_j|, 1e-12)   (F.normalize, V2:452-455)
    for (int i = tid; i < 2 * L; i += V2_THREADS) {
      const int which = i >= L ? 1 : 0, r = i - which * L;
      const uint4* rowp = reinterpret_cast<const uint4*>(Qs + which * (L * ROW_BYTES) + r * ROW_BYTES);
      float ss = 0.f;
#pragma unroll
      for (int ch = 0; ch < 4; ++ch) {
        const uint4 u = rowp[ch];
        const float2 a = unpack2<T>(u.x), b = unpack2<T>(u.y), c = unpack2<T>(u.z), d = unpack2<T>(u.w);
        ss += (a.x * a.x + a.y * a.y) + (b.x * b.x + b.y * b.y) + (c.x * c.x + c.y * c.y) + (d.x * d.x + d.y * d.y);
      }
      const float inv = 1.0f / fmaxf(sqrtf(ss), 1e-12f);
      if (which) rk_s[r] = inv; else rq_s[r] = inv * scale;
    }
    __syncthreads();

    // A warp walks TILES 16-row query tiles at once: the K / V fragments it pulls from shared memory feed TILES MMAs each and the
    // TILES softmax chains are independent, which is what hides the MMA -> softmax -> MMA latency at 12-16 warps per SM.
#pragma unroll 1
    for (int mg = warp; mg < L / (16 * TILES); mg += V2_THREADS / 32) {
      uint32_t qa[TILES][2][4];
      float rq0[TILES], rq1[TILES], mrun0[TILES], mrun1[TILES];
      const float* bp0[TILES];
      const float* bp1[TILES];
      int reg0[TILES], reg1[TILES];
      float o[TILES][5][4];   // o[t][4] = running row sums (ones column)
#pragma unroll
      for (int t = 0; t < TILES; ++t) {
        const int m0 = (mg * TILES + t) * 16;
#pragma unroll
        for (int ks = 0; ks < 2; ++ks)
          ldsm_x4(qa[t][ks], Qs + row_off(m0 + (lane & 7) + ((lane >> 3) & 1) * 8, ks * 2 + (lane >> 4)));
        const int r0 = m0 + (lane >> 2), r1 = r0 + 8;
        rq0[t] = rq_s[r0]; rq1[t] = rq_s[r1];
        // rel_pos_index(i, j) = (iy - jy + WS-1) TW + (ix - jx + WS-1): per-thread row base minus a compile-time column term
        bp0[t] = bias_s + ((r0 / WS) * TW + (r0 % WS) + (WS - 1) * (TW + 1) - q2);
        bp1[t] = bias_s + ((r1 / WS) * TW + (r1 % WS) + (WS - 1) * (TW + 1) - q2);
        reg0[t] = reg1[t] = 0;
        if (masked) { reg0[t] = region_s[r0]; reg1[t] = region_s[r1]; }
        mrun0[t] = mrun1[t] = -INFINITY;
#pragma unroll
        for (int n = 0; n < 5; ++n) o[t][n][0] = o[t][n][1] = o[t][n][2] = o[t][n][3] = 0.f;
      }

#pragma unroll 1
      for (int c0 = 0; c0 < L; c0 += 64) {
        float s[TILES][8][4];
        // ---- S = Q K^T on the raw 16-bit operands ----
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          uint32_t kb[4];
          ldsm_x4(kb, Ks + row_off(c0 + j * 8 + (lane & 7), lane >> 3));
#pragma unroll
          for (int t = 0; t < TILES; ++t) {
            s[t][j][0] = s[t][j][1] = s[t][j][2] = s[t][j][3] = 0.f;
            mma_16816<T>(s[t][j], qa[t][0], kb[0], kb[1]);
            mma_16816<T>(s[t][j], qa[t][1], kb[2], kb[3]);
          }
        }
        // ---- cosine scaling, continuous position bias (log2 domain, fp32) ----
        const float* rkp = rk_s + c0 + q2;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int ct = (WS == 16 ? (j >> 1) * TW + 8 * (j & 1) : j * TW);     // key (c0 + 8j + q2 + e): jy * TW + jx, less q2 + e
          const float2 rk = *reinterpret_cast<const float2*>(rkp + j * 8);
#pragma unroll
          for (int t = 0; t < TILES; ++t) {
            const float* b0 = bp0[t] - (c0 / WS) * TW;
            const float* b1 = bp1[t] - (c0 / WS) * TW;
            s[t][j][0] = fmaf(s[t][j][0] * rq0[t], rk.x, b0[-ct]);
            s[t][j][1] = fmaf(s[t][j][1] * rq0[t], rk.y, b0[-ct - 1]);
            s[t][j][2] = fmaf(s[t][j][2] * rq1[t], rk.x, b1[-ct]);
            s[t][j][3] = fmaf(s[t][j][3] * rq1[t], rk.y, b1[-ct - 1]);
          }
        }
        if (masked) {   // shift mask, only in the last window row / column of a shifted block
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const uint32_t rc = *reinterpret_cast<const uint16_t*>(region_s + c0 + j * 8 + q2);
            const int rc0 = static_cast<int>(rc & 0xffu), rc1 = static_cast<int>(rc >> 8);
#pragma unroll
            for (int t = 0; t < TILES; ++t) {
              if (rc0 != reg0[t]) s[t][j][0] += mask_l2;
              if (rc1 != reg0[t]) s[t][j][1] += mask_l2;
              if (rc0 != reg1[t]) s[t][j][2] += mask_l2;
              if (rc1 != reg1[t]) s[t][j][3] += mask_l2;
            }
          }
        }
        float mn0[TILES], mn1[TILES];
#pragma unroll
        for (int t = 0; t < TILES; ++t) {
          float mx0 = fmaxf(s[t][0][0], s[t][0][1]), mx1 = fmaxf(s[t][0][2], s[t][0][3]);
#pragma unroll
          for (int j = 1; j < 8; ++j) {
            mx0 = fmaxf(mx0, fmaxf(s[t][j][0], s[t][j][1]));
            mx1 = fmaxf(mx1, fmaxf(s[t][j][2], s[t][j][3]));
          }
          mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
          mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
          // ---- online softmax: rescale the running sums to the new row maximum ----
          mn0[t] = fmaxf(mrun0[t], mx0); mn1[t] = fmaxf(mrun1[t], mx1);
          const float corr0 = ex2_ftz(mrun0[t] - mn0[t]), corr1 = ex2_ftz(mrun1[t] - mn1[t]);
          mrun0[t] = mn0[t]; mrun1[t] = mn1[t];
#pragma unroll
          for (int n = 0; n < 5; ++n) { o[t][n][0] *= corr0; o[t][n][1] *= corr0; o[t][n][2] *= corr1; o[t][n][3] *= corr1; }
        }
        // ---- O += P V, row sums += P 1  (P re-used in registers as the A operand) ----
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          uint32_t pa[TILES][4];
#pragma unroll
          for (int t = 0; t < TILES; ++t) {
            pa[t][0] = Half16<T>::pack(ex2_ftz(s[t][2 * kk][0] - mn0[t]), ex2_ftz(s[t][2 * kk][1] - mn0[t]));
            pa[t][1] = Half16<T>::pack(ex2_ftz(s[t][2 * kk][2] - mn1[t]), ex2_ftz(s[t][2 * kk][3] - mn1[t]));
            pa[t][2] = Half16<T>::pack(ex2_ftz(s[t][2 * kk + 1][0] - mn0[t]), ex2_ftz(s[t][2 * kk + 1][1] - mn0[t]));
            pa[t][3] = Half16<T>::pack(ex2_ftz(s[t][2 * kk + 1][2] - mn1[t]), ex2_ftz(s[t][2 * kk + 1][3] - mn1[t]));
          }
#pragma unroll
          for (int np = 0; np < 2; ++np) {
            uint32_t vb[4];
            ldsm_x4_t(vb, Vs + row_off(c0 + kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8, np * 2 + (lane >> 4)));
#pragma unroll
            for (int t = 0; t < TILES; ++t) {
              mma_16816<T>(o[t][2 * np], pa[t], vb[0], vb[1]);
              mma_16816<T>(o[t][2 * np + 1], pa[t], vb[2], vb[3]);
            }
          }
#pragma unroll
          for (int t = 0; t < TILES; ++t) mma_16816<T>(o[t][4], pa[t], Ones16<T>::v, Ones16<T>::v);
        }
      }
      // ---- store (head merge folded into the column offset) ----
#pragma unroll
      for (int t = 0; t < TILES; ++t) {
        int r0 = (mg * TILES + t) * 16 + (lane >> 2), r1 = r0 + 8;
        if (tok_order) { r0 = tok_s[r0]; r1 = tok_s[r1]; }
        const float inv0 = 1.0f / o[t][4][0], inv1 = 1.0f / o[t][4][2];
#pragma unroll
        for (int n = 0; n < 4; ++n) {
          const int col = h * 32 + n * 8 + q2;
          *reinterpret_cast<uint32_t*>(out + (obase + r0) * C + col) = Half16<T>::pack(o[t][n][0] * inv0, o[t][n][1] * inv0);
          *reinterpret_cast<uint32_t*>(out + (obase + r1) * C + col) = Half16<T>::pack(o[t][n][2] * inv1, o[t][n][3] * inv1);
        }
      }
    }
  }
}

// ----------------------------------------------------------------------------------------------------
// cosine window attention, exact fp32 (validation mode)
// ----------------------------------------------------------------------------------------------------
// One CTA (4 warps) per (window, head); K / V rows padded to 33 floats; warp per query row, lane per key (L / 32 keys per lane).
__global__ void __launch_bounds__(V2_THREADS)
swinv2_attn_f32_kernel(const float* __restrict__ qkv, const float* __restrict__ bias_tab, const float* __restrict__ logit_scale,
                       float* __restrict__ out, int num_items, int C, int heads, WinGeom g, int nW, float mask_value, int tok_order) {
  extern __shared__ __align__(16) uint8_t v2_smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int L = g.L, ws = g.ws, tw = 2 * ws - 1, TB = tw * tw;
  float* Ks = reinterpret_cast<float*>(v2_smem);       // [L][33]
  float* Vs = Ks + L * 33;                              // [L][33]
  float* rk_s = Vs + L * 33;                            // [L]
  float* Ps = rk_s + L;                                 // [4][L]
  float* Qs = Ps + 4 * L;                               // [4][32]
  float* bias_s = Qs + 4 * 32;                          // [TB]
  int* region_s = reinterpret_cast<int*>(bias_s + TB);  // [L]
  const int ld = 3 * C;
  const int row_const = (ws - 1) * tw + (ws - 1);
  int cur_h = -1;
  for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
    const int h = item % heads, wg = item / heads, w = wg % nW;
    const long long row0 = static_cast<long long>(wg) * L;
    __syncthreads();
    if (h != cur_h) {
      for (int i = tid; i < TB; i += V2_THREADS) bias_s[i] = bias_tab[h * TB + i];
      cur_h = h;
    }
    for (int idx = tid; idx < L * 32; idx += V2_THREADS) {
      const int r = idx >> 5, d = idx & 31;
      Ks[r * 33 + d] = qkv[(row0 + r) * ld + C + h * 32 + d];
      Vs[r * 33 + d] = qkv[(row0 + r) * ld + 2 * C + h * 32 + d];
    }
    for (int i = tid; i < L; i += V2_THREADS) region_s[i] = g.shift > 0 ? win_region(g, w, i) : 0;
    __syncthreads();
    for (int j = tid; j < L; j += V2_THREADS) {
      float ss = 0.f;
      for (int d = 0; d < 32; ++d) ss = fmaf(Ks[j * 33 + d], Ks[j * 33 + d], ss);
      rk_s[j] = 1.0f / fmaxf(sqrtf(ss), 1e-12f);
    }
    __syncthreads();
    const float scale = logit_scale[h];
    for (int i = warp; i < L; i += V2_THREADS / 32) {
      const float qv = qkv[(row0 + i) * ld + h * 32 + lane];
      Qs[warp * 32 + lane] = qv;
      const float rq = scale / fmaxf(sqrtf(warp_sum(qv * qv)), 1e-12f);
      __syncwarp();
      const int rt = (i / ws) * tw + (i % ws) + row_const;
      float mx = -INFINITY;
      for (int j = lane; j < L; j += 32) {
        float a = 0.f;
#pragma unroll
        for (int d = 0; d < 32; ++d) a = fmaf(Qs[warp * 32 + d], Ks[j * 33 + d], a);
        a = a * rq * rk_s[j] + bias_s[rt - ((j / ws) * tw + (j % ws))];
        if (g.shift > 0 && region_s[j] != region_s[i]) a += mask_value;
        Ps[warp * L + j] = a;
        mx = fmaxf(mx, a);
      }
      mx = warp_max(mx);
      float sum = 0.f;
      for (int j = lane; j < L; j += 32) {
        const float e = expf(Ps[warp * L + j] - mx);
        Ps[warp * L + j] = e;
        sum += e;
      }
      const float inv = 1.0f / warp_sum(sum);
      __syncwarp();
      float acc = 0.f;
      for (int j = 0; j < L; ++j) acc = fmaf(Ps[warp * L + j], Vs[j * 33 + lane], acc);
      const long long orow = tok_order ? static_cast<long long>(wg / nW) * g.N + win_row_to_token(g, w * L + i) : row0 + i;
      out[orow * C + h * 32 + lane] = acc * inv;
      __syncwarp();
    }
  }
}

template <typename T, int WS, int TILES>
static int launch_v2_t(const void* qkv, const float* bias_tab, const float* logit_scale, void* out, int num_windows, int C, int heads,
                       const WinGeom& g, int nW, float mask_value, int tok_order, cudaStream_t stream) {
  auto kern = swinv2_attn_kernel<T, WS, TILES>;
  const int smem = v2_smem_bytes(WS);
  static DeviceOnce once;
  if (once.first()) {
    CSVIT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  }
  int per_head = num_windows;
  const int resident = TILES == 2 ? 3 : 4;
  const int cap = (num_sms() * resident) / heads > 0 ? (num_sms() * resident) / heads : 1;
  if (per_head > cap) per_head = cap;
  kern<<<per_head * heads, V2_THREADS, smem, stream>>>(static_cast<const T*>(qkv), bias_tab, logit_scale, static_cast<T*>(out),
                                                       num_windows, C, heads, g, nW, mask_value, tok_order);
  CSVIT_CUDA(cudaGetLastError());
  return 0;
}

int launch_swinv2_window_attention(const void* qkv, const float* bias_tab, const float* logit_scale, void* out, int dtype, int B, int H,
                                   int W, int C, int heads, int ws, int shift, int mask_repeat, int tok_order, cudaStream_t stream) {
  CSVIT_REQUIRE(C == heads * 32, "swinv2_window_attention: head_dim must be 32 (C=%d heads=%d)", C, heads);
  CSVIT_REQUIRE(ws > 0 && H % ws == 0 && W % ws == 0, "swinv2_window_attention: %dx%d not divisible by window %d", H, W, ws);
  CSVIT_REQUIRE(ws * ws <= V2_MAXL, "swinv2_window_attention: window %d not built (at most %d tokens per window)", ws, V2_MAXL);
  CSVIT_REQUIRE(dtype == DT_F32 || ws == 16 || ws == 8, "swinv2_window_attention: window %d not built (16-bit kernel: windows 16 and 8)", ws);
  CSVIT_REQUIRE(shift >= 0 && shift < ws, "swinv2_window_attention: shift %d outside [0,%d)", shift, ws);
  CSVIT_REQUIRE(H * W < 32768, "swinv2_window_attention: %dx%d tokens per image exceed the 16-bit token table", H, W);
  const int nW = (H / ws) * (W / ws);
  const long long items = static_cast<long long>(B) * nW * heads;
  if (items <= 0) return 0;
  CSVIT_REQUIRE(items < (1ll << 31), "swinv2_window_attention: too many work items");
  const WinGeom g = make_geom(H, W, ws, shift);
  const float mask_value = -100.0f * static_cast<float>(mask_repeat);
  if (dtype == DT_BF16 && ws == 16) return launch_v2_t<__nv_bfloat16, 16, V2_TILES16>(qkv, bias_tab, logit_scale, out, B * nW, C, heads, g, nW, mask_value, tok_order, stream);
  if (dtype == DT_BF16) return launch_v2_t<__nv_bfloat16, 8, 1>(qkv, bias_tab, logit_scale, out, B * nW, C, heads, g, nW, mask_value, tok_order, stream);
  if (dtype == DT_F16 && ws == 16) return launch_v2_t<__half, 16, V2_TILES16>(qkv, bias_tab, logit_scale, out, B * nW, C, heads, g, nW, mask_value, tok_order, stream);
  if (dtype == DT_F16) return launch_v2_t<__half, 8, 1>(qkv, bias_tab, logit_scale, out, B * nW, C, heads, g, nW, mask_value, tok_order, stream);
  CSVIT_REQUIRE(dtype == DT_F32, "swinv2_window_attention: bad dtype %d", dtype);
  const int L = ws * ws, tw = 2 * ws - 1;
  const int smem = (2 * L * 33 + L + 4 * L + 4 * 32 + tw * tw + L) * 4;
  static DeviceOnce once;
  if (once.first()) {
    const int Lm = V2_MAXL, twm = 31;
    CSVIT_CUDA(cudaFuncSetAttribute(swinv2_attn_f32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (2 * Lm * 33 + Lm + 4 * Lm + 4 * 32 + twm * twm + Lm) * 4));
  }
  const int blocks = static_cast<int>(items < num_sms() * 8 ? items : num_sms() * 8);
  swinv2_attn_f32_kernel<<<blocks, V2_THREADS, smem, stream>>>(static_cast<const float*>(qkv), bias_tab, logit_scale,
                                                               static_cast<float*>(out), static_cast<int>(items), C, heads, g, nW,
                                                               mask_value, tok_order);
  CSVIT_CUDA(cudaGetLastError());
  return 0;
}

// ----------------------------------------------------------------------------------------------------
// post-norm residual LayerNorm with operand copy
// ----------------------------------------------------------------------------------------------------
template <typename T> struct St4;
template <> struct St4<float> {
  __device__ static void st(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
};
template <> struct St4<__half> {
  __device__ static void st(__half* p, float4 v) {
    uint2 u; u.x = pack_f16x2(v.x, v.y); u.y = pack_f16x2(v.z, v.w);
    *reinterpret_cast<uint2*>(p) = u;
  }
};
template <> struct St4<__nv_bfloat16> {
  __device__ static void st(__nv_bfloat16* p, float4 v) {
    uint2 u; u.x = pack_bf16x2(v.x, v.y); u.y = pack_bf16x2(v.z, v.w);
    *reinterpret_cast<uint2*>(p) = u;
  }
};

// One warp per R consecutive tokens (rows of y, token order); rows live in registers between the statistics and the output pass
// (same structure as ln_rows_kernel).  xo[row] = (resid ? resid[row] : 0) + LN(y[row]) * gamma + beta, fp32; xo may alias resid
// or y.  copy (optional) receives the same values as CopyT at
//   COPY_IDENTITY  row `row`
//   COPY_WINDOW    row b*N + win_token_to_row(g, t): the (shifted-)window order of geometry g
//   COPY_MERGE2X2  row b*N/4 + (y/2)*(W/2) + x/2, column block ((y&1) + 2(x&1)) * C: the 2x2 concat of patch merging
// CopyT = __nv_fp8_e4m3 (identity / window copies): the copy is the E4M3 operand of an FP8 GEMM with a per-row scale,
//   row_scale[copy row] = amax / 448 and copy = e4m3_rn_satfinite(x * (448 / amax)), amax = max |x| over the row (0 for an all-zero row,
//   whose copy is zero).  Both divisions are correctly rounded, so the copy is bit-identical to the same expression in torch.
template <int MAXJ, int R, typename CopyT>
__global__ void __launch_bounds__(256)
ln_post_kernel(const float* y, long long ldy, const float* resid, const float* __restrict__ gamma,
               const float* __restrict__ beta, float eps, float* xo, CopyT* __restrict__ copy, long long ldc, int copy_mode,
               int rows, int C, WinGeom g, float* __restrict__ row_scale) {
  constexpr bool F8 = sizeof(CopyT) == 1;
  griddep_launch();
  griddep_wait();
  const int lane = threadIdx.x & 31;
  const int n4 = C >> 2;
  const int warps_total = (gridDim.x * blockDim.x) >> 5;
  for (int row0 = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * R; row0 < rows; row0 += warps_total * R) {
    float4 v[R][MAXJ];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int row = row0 + r;
      if (row < rows) {
#pragma unroll
        for (int j = 0; j < MAXJ; ++j) {
          const int i4 = lane + 32 * j;
          if (i4 < n4) v[r][j] = *reinterpret_cast<const float4*>(y + static_cast<long long>(row) * ldy + (i4 << 2));
        }
      }
    }
    // copy destination (row, column block) of token row0 + r, evaluated once by lane r and broadcast below
    int my_crow = 0, my_ccol = 0;
    if (lane < R && row0 + lane < rows) {
      const int row = row0 + lane;
      my_crow = row;
      if (copy_mode == COPY_WINDOW) {
        const int b = row / g.N, t = row - b * g.N;
        my_crow = b * g.N + win_token_to_row(g, t);
      } else if (copy_mode == COPY_MERGE2X2) {
        const int b = row / g.N, t = row - b * g.N;
        const int ty = t / g.W, tx = t - ty * g.W;
        my_crow = b * (g.N >> 2) + (ty >> 1) * (g.W >> 1) + (tx >> 1);
        my_ccol = ((ty & 1) + 2 * (tx & 1)) * C;
      }
    }
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int row = row0 + r;
      if (row >= rows) break;   // warp-uniform
      float sum = 0.f;
#pragma unroll
      for (int j = 0; j < MAXJ; ++j)
        if (lane + 32 * j < n4) sum += (v[r][j].x + v[r][j].y) + (v[r][j].z + v[r][j].w);
      const float mean = warp_sum(sum) / float(C);
      float sq = 0.f;
#pragma unroll
      for (int j = 0; j < MAXJ; ++j) {
        if (lane + 32 * j < n4) {
          const float a = v[r][j].x - mean, b = v[r][j].y - mean, c = v[r][j].z - mean, d = v[r][j].w - mean;
          sq += (a * a + b * b) + (c * c + d * d);
        }
      }
      const float rstd = rsqrtf(warp_sum(sq) / float(C) + eps);
      const long long crow = __shfl_sync(0xffffffffu, my_crow, r);
      const int ccol = __shfl_sync(0xffffffffu, my_ccol, r);
      float amax = 0.f;
#pragma unroll
      for (int j = 0; j < MAXJ; ++j) {
        const int i4 = lane + 32 * j;
        if (i4 < n4) {
          const int e = i4 << 2;
          const float4 gm = __ldg(reinterpret_cast<const float4*>(gamma + e));
          const float4 bt = __ldg(reinterpret_cast<const float4*>(beta + e));
          float4 o;
          o.x = (v[r][j].x - mean) * rstd * gm.x + bt.x; o.y = (v[r][j].y - mean) * rstd * gm.y + bt.y;
          o.z = (v[r][j].z - mean) * rstd * gm.z + bt.z; o.w = (v[r][j].w - mean) * rstd * gm.w + bt.w;
          if (resid) {
            const float4 x0 = *reinterpret_cast<const float4*>(resid + static_cast<long long>(row) * C + e);
            o.x += x0.x; o.y += x0.y; o.z += x0.z; o.w += x0.w;
          }
          if (xo) *reinterpret_cast<float4*>(xo + static_cast<long long>(row) * C + e) = o;
          if constexpr (F8) {
            v[r][j] = o;
            amax = fmaxf(amax, fmaxf(fmaxf(fabsf(o.x), fabsf(o.y)), fmaxf(fabsf(o.z), fabsf(o.w))));
          } else if (copy_mode != COPY_NONE) {
            St4<CopyT>::st(copy + crow * ldc + ccol + e, o);
          }
        }
      }
      if constexpr (F8) {
        amax = warp_max(amax);
        const float q = amax > 0.f ? __fdiv_rn(448.0f, amax) : 0.f;
        if (lane == 0) row_scale[crow] = __fdiv_rn(amax, 448.0f);
#pragma unroll
        for (int j = 0; j < MAXJ; ++j) {
          const int i4 = lane + 32 * j;
          if (i4 < n4) {
            const uint32_t lo = __nv_cvt_float2_to_fp8x2(make_float2(v[r][j].x * q, v[r][j].y * q), __NV_SATFINITE, __NV_E4M3);
            const uint32_t hi = __nv_cvt_float2_to_fp8x2(make_float2(v[r][j].z * q, v[r][j].w * q), __NV_SATFINITE, __NV_E4M3);
            *reinterpret_cast<uint32_t*>(copy + crow * ldc + (i4 << 2)) = lo | (hi << 16);
          }
        }
      }
    }
  }
}

template <int MAXJ, int R, typename CopyT>
static void launch_lnp_cfg(const float* y, long long ldy, const float* resid, const float* gamma, const float* beta, float eps,
                           float* xo, void* copy, long long ldc, int copy_mode, int rows, int C, const WinGeom& g,
                           float* row_scale, cudaStream_t stream) {
  const int warps = (rows + R - 1) / R;
  const int blocks = (warps + 7) / 8;
  (void)launch_pdl(ln_post_kernel<MAXJ, R, CopyT>, dim3(blocks), dim3(256), 0, stream, y, ldy, resid, gamma, beta, eps, xo,
                   static_cast<CopyT*>(copy), ldc, copy_mode, rows, C, g, row_scale);
}

template <typename CopyT>
static int launch_lnp_t(const float* y, long long ldy, const float* resid, const float* gamma, const float* beta, float eps,
                        float* xo, void* copy, long long ldc, int copy_mode, int rows, int C, const WinGeom& g, float* row_scale,
                        cudaStream_t stream) {
  if (C <= 128) launch_lnp_cfg<1, 8, CopyT>(y, ldy, resid, gamma, beta, eps, xo, copy, ldc, copy_mode, rows, C, g, row_scale, stream);
  else if (C <= 256) launch_lnp_cfg<2, 4, CopyT>(y, ldy, resid, gamma, beta, eps, xo, copy, ldc, copy_mode, rows, C, g, row_scale, stream);
  else if (C <= 512) launch_lnp_cfg<4, 2, CopyT>(y, ldy, resid, gamma, beta, eps, xo, copy, ldc, copy_mode, rows, C, g, row_scale, stream);
  else if (C <= 1024) launch_lnp_cfg<8, 2, CopyT>(y, ldy, resid, gamma, beta, eps, xo, copy, ldc, copy_mode, rows, C, g, row_scale, stream);
  else if (C <= 2048) launch_lnp_cfg<16, 1, CopyT>(y, ldy, resid, gamma, beta, eps, xo, copy, ldc, copy_mode, rows, C, g, row_scale, stream);
  else return set_error("layernorm_post: row width %d exceeds 2048", C);
  CSVIT_CUDA(cudaGetLastError());
  return 0;
}

int launch_layernorm_post(const float* y, long long ldy, const float* resid, const float* gamma, const float* beta, float eps,
                          float* xo, void* copy, int copy_dtype, long long ldc, int copy_mode, int rows, int C, const WinGeom& g,
                          float* row_scale, cudaStream_t stream) {
  CSVIT_REQUIRE(C % 4 == 0 && ldy % 4 == 0, "layernorm_post: C=%d and ldy=%lld must be multiples of 4", C, ldy);
  CSVIT_REQUIRE(copy_mode >= COPY_NONE && copy_mode <= COPY_MERGE2X2, "layernorm_post: unknown copy mode %d", copy_mode);
  CSVIT_REQUIRE(copy_mode == COPY_NONE || (copy != nullptr && ldc % 4 == 0), "layernorm_post: copy buffer missing or pitch %lld not a multiple of 4", ldc);
  CSVIT_REQUIRE(xo != nullptr || copy_mode != COPY_NONE, "layernorm_post: no output requested");
  if (copy_dtype == DT_E4M3) {
    CSVIT_REQUIRE(copy_mode == COPY_IDENTITY || copy_mode == COPY_WINDOW, "layernorm_post: E4M3 copies are identity or window ordered");
    CSVIT_REQUIRE(row_scale != nullptr && (reinterpret_cast<uintptr_t>(copy) & 3) == 0, "layernorm_post: E4M3 copy needs row_scale, 4-byte alignment");
  }
  if (rows <= 0) return 0;
  if (copy_dtype == DT_E4M3)
    return launch_lnp_t<__nv_fp8_e4m3>(y, ldy, resid, gamma, beta, eps, xo, copy, ldc, copy_mode, rows, C, g, row_scale, stream);
  if (copy_mode == COPY_NONE || copy_dtype == DT_BF16)
    return launch_lnp_t<__nv_bfloat16>(y, ldy, resid, gamma, beta, eps, xo, copy, ldc, copy_mode, rows, C, g, nullptr, stream);
  if (copy_dtype == DT_F16) return launch_lnp_t<__half>(y, ldy, resid, gamma, beta, eps, xo, copy, ldc, copy_mode, rows, C, g, nullptr, stream);
  return launch_lnp_t<float>(y, ldy, resid, gamma, beta, eps, xo, copy, ldc, copy_mode, rows, C, g, nullptr, stream);
}

}  // namespace csvit
