// GEMM engine interface shared by the tcgen05 kernel, the SIMT fp32 kernel and the C ABI.
//   D[M,N] = epilogue( A[M,K] * W[N,K]^T )        (both operands K-major, i.e. nn.Linear layout)
#pragma once
#include "common.cuh"

namespace csvit {

enum : int { ACT_NONE = 0, ACT_GELU = 1, ACT_RELU = 2 };
enum : int { ROWMAP_IDENTITY = 0, ROWMAP_WINDOW = 1 };
enum : int { DT_F32 = 0, DT_BF16 = 1, DT_F16 = 2 };
__host__ __device__ inline int dtype_size(int dt) { return dt == DT_F32 ? 4 : 2; }

// What happens to one accumulator row-chunk after the MMA:
//   v = acc (+ bias[col]) -> act -> (+ resid[orow, col]) -> out[orow, col]  (fp32, bf16 or fp16)
// orow = row for ROWMAP_IDENTITY; for ROWMAP_WINDOW the GEMM rows are window-ordered tokens and orow is the
// original token row (window_reverse + roll(+shift) folded into the store address, SURVEY.md §8a).
struct EpiParams {
  const float* bias;
  const float* resid;
  void* out;
  long long ldo, ldr;
  int out_dtype;
  int act;
  int M, N;
  int vec_ok;     // 1: rows are 16-byte aligned for 32-column chunks (ldo/ldr/N multiples of 8)
  int tma_store;  // 1: 16-bit output, identity rows, no residual -> staged through smem and written by TMA
  int coalesced;  // 1: fp32 output (+residual, +scatter) -> transposed through smem, 4 full lines per warp access
  int tma_f32;    // 1: fp32 output on identity rows (+residual): residual chunks arrive by TMA, results leave by TMA
  long long* trace;   // trace builds (-DCSVIT_PAIR_TRACE_BUILD, CSVIT_PAIR_TRACE=<file>): clock64 stamps of pair 0 of gemm_pair_kernel
  int red_add;    // 1 (set by the launcher when out aliases resid; resid is then nullptr): tma_f32 chunks leave by TMA reduce-add,
                  // the coalesced path's float4 stores become red.global.add.v4.f32
  int map_mode;
  WinGeom geom;
  // SwinV2 Q/K/V projection (cos_C = C > 0, N = 3C): every head's 32 columns of q and k are L2-normalised per row before the 16-bit
  // store (F.normalize of V2:452-455) and q is multiplied by cos_scale[head] (logit scale, log2 domain); v passes unchanged.
  const float* cos_scale;
  int cos_C;
  // Training form of the above (csvit_swinv2_qkv_train): rnorm[row, j] = 1 / max(|x|, 1e-12) of q head j (j < C / 32) and k head
  // j - C / 32, fp32 [M, 2C / 32] dense, identity rows only.  nullptr: not stored.
  float* rnorm;
};

// The cosine normalisation above on 32 consecutive columns of one row (= one head: col0 is a multiple of 32).
__device__ __forceinline__ void epi_cosnorm32(const EpiParams& ep, long long row, int col0, float (&v)[32]) {
  if (col0 >= 2 * ep.cos_C) return;
  float ss0 = 0.f, ss1 = 0.f;
#pragma unroll
  for (int j = 0; j < 32; j += 2) { ss0 = fmaf(v[j], v[j], ss0); ss1 = fmaf(v[j + 1], v[j + 1], ss1); }
  float inv = 1.0f / fmaxf(sqrtf(ss0 + ss1), 1e-12f);
  if (ep.rnorm && row < ep.M) ep.rnorm[row * (ep.cos_C >> 4) + (col0 >> 5)] = inv;
  if (col0 < ep.cos_C) inv *= __ldg(ep.cos_scale + (col0 >> 5));
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] *= inv;
}

__device__ __forceinline__ long long epi_out_row(const EpiParams& ep, int row) {
  if (ep.map_mode == ROWMAP_WINDOW) {
    int b = row / ep.geom.N, r = row - b * ep.geom.N;
    return static_cast<long long>(b) * ep.geom.N + win_row_to_token(ep.geom, r);
  }
  return row;
}

// Branch-free erf GELU for the tensor-core epilogues: erfc(|x|/sqrt2) = 2^q(|x|) with q a degree-6 polynomial
// fitted to log2(erfc) on |x| <= 4*sqrt2 (beyond that erfc < 1.6e-8).  6 FFMA + 1 MUFU.EX2 + 5 other FP ops, no
// division, no branch.  Max |error| vs 0.5x(1+erf(x/sqrt2)) evaluated in fp32: 4.2e-7 absolute, 1.9e-4 relative in
// the far negative tail - two to three orders below the 16-bit rounding of the value that is stored.  (The
// epilogues of fc1 at stages 0/1 are bound by exactly this arithmetic, profiles/r1_gemm_pipeline_analysis.md.)
// The fp32 validation mode keeps erff() (gelu_erf).
__device__ __forceinline__ float gelu_fast(float x) {
  const float ax = fminf(fabsf(x), 5.6568542f);
  float q = fmaf(ax, 3.382089429e-05f, -7.692634491e-04f);
  q = fmaf(q, ax, 8.055410705e-03f);
  q = fmaf(q, ax, -5.332621707e-02f);
  q = fmaf(q, ax, -4.588742488e-01f);
  q = fmaf(q, ax, -1.151155207e+00f);
  q = fmaf(q, ax, 1.205011077e-06f);
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(q));
  const float hx = 0.5f * x;
  return fmaf(fabsf(hx), 1.0f - e, hx);   // 0.5x(1 + sign(x) erf(|x|/sqrt2)) = hx + |hx| (1 - erfc)
}

// Two GELUs per instruction for 16-bit outputs: the same degree-6 erfc fit evaluated in packed fp16 (HFMA2, one
// MUFU.EX2 for the pair).  The fc1 / fused-MLP epilogues are bound by this arithmetic (stages 0-1: every element of
// the 4C-wide hidden tensor passes through it), and the result is rounded to 16 bit anyway: the packed evaluation
// adds < 2e-4 absolute error, below the bf16 / at the level of the fp16 output rounding.
__device__ __forceinline__ __half2 gelu_h2(__half2 x) {
  const __half2 ax = __hmin2(__habs2(x), __float2half2_rn(5.65625f));
  __half2 q = __hfma2(ax, __float2half2_rn(3.382089429e-05f), __float2half2_rn(-7.692634491e-04f));
  q = __hfma2(q, ax, __float2half2_rn(8.055410705e-03f));
  q = __hfma2(q, ax, __float2half2_rn(-5.332621707e-02f));
  q = __hfma2(q, ax, __float2half2_rn(-4.588742488e-01f));
  q = __hfma2(q, ax, __float2half2_rn(-1.151155207e+00f));
  q = __hfma2(q, ax, __float2half2_rn(-1.0f));            // q - 1: the exponential below is 0.5 erfc(|x| / sqrt2) = Phi(-|x|)
  __half2 e;
  asm("ex2.approx.f16x2 %0, %1;" : "=r"(*reinterpret_cast<uint32_t*>(&e)) : "r"(*reinterpret_cast<const uint32_t*>(&q)));
  // x Phi(x) = relu(x) - |x| Phi(-|x|): two instructions (max, fma) instead of the four of hx + |hx| (1 - erfc)
  return __hfma2(__hneg2(__habs2(x)), e, __hmax2(x, __float2half2_rn(0.0f)));
}
// (a, b) fp32 pre-activations -> GELU -> one packed 16-bit pair in the output format.
__device__ __forceinline__ uint32_t gelu_pack16(bool bf, float a, float b) {
  const __half2 g = gelu_h2(__floats2half2_rn(a, b));
  if (!bf) return *reinterpret_cast<const uint32_t*>(&g);
  const float2 f = __half22float2(g);
  return pack_bf16x2(f.x, f.y);
}

// acc (+ bias) -> GELU -> 16 packed pairs, for 32 consecutive full columns (16-byte aligned bias).
__device__ __forceinline__ void epi_bias_gelu_pack32(const float* bias, bool bf, int col0, const uint32_t (&r)[32], uint32_t* pk) {
  float v[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
  if (bias) {
    const float4* b4 = reinterpret_cast<const float4*>(bias + col0);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float4 b = __ldg(b4 + j);
      v[4 * j + 0] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
    }
  }
#pragma unroll
  for (int j = 0; j < 16; ++j) pk[j] = gelu_pack16(bf, v[2 * j], v[2 * j + 1]);
}

__device__ __forceinline__ float epi_act(int act, float v) {
  if (act == ACT_GELU) return gelu_erf(v);
  if (act == ACT_RELU) return fmaxf(v, 0.0f);
  return v;
}

// Scalar form (SIMT kernel and ragged edges).
__device__ __forceinline__ void epi_store_scalar(const EpiParams& ep, long long orow, int col, float acc) {
  float v = acc;
  if (ep.bias) v += __ldg(ep.bias + col);
  v = epi_act(ep.act, v);
  if (ep.resid) v += ep.resid[orow * ep.ldr + col];
  if (ep.out_dtype == DT_BF16)
    reinterpret_cast<__nv_bfloat16*>(ep.out)[orow * ep.ldo + col] = __float2bfloat16_rn(v);
  else if (ep.out_dtype == DT_F16)
    reinterpret_cast<__half*>(ep.out)[orow * ep.ldo + col] = __float2half_rn(v);
  else
    reinterpret_cast<float*>(ep.out)[orow * ep.ldo + col] = v;
}

// bias + activation on 32 consecutive full columns of GEMM row `row` held in registers (16-byte aligned bias).
__device__ __forceinline__ void epi_bias_act32(const EpiParams& ep, long long row, int col0, float (&v)[32]) {
  if (ep.bias) {
    const float4* b4 = reinterpret_cast<const float4*>(ep.bias + col0);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float4 b = __ldg(b4 + j);
      v[4 * j + 0] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
    }
  }
  if (ep.cos_C > 0) epi_cosnorm32(ep, row, col0, v);
  if (ep.act == ACT_GELU) {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = gelu_fast(v[j]);
  } else if (ep.act == ACT_RELU) {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.0f);
  }
}

__device__ __forceinline__ uint32_t pack16(bool bf, float lo, float hi) { return bf ? pack_bf16x2(lo, hi) : pack_f16x2(lo, hi); }

// 32 consecutive columns of one row held in registers (the tcgen05 epilogue shape), direct global store.
__device__ __forceinline__ void epi_store_chunk32(const EpiParams& ep, long long orow, int col0, const uint32_t (&r)[32]) {
  if (ep.vec_ok && col0 + 32 <= ep.N) {
    float v[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
    epi_bias_act32(ep, orow, col0, v);
    if (ep.resid) {
      const float4* r4 = reinterpret_cast<const float4*>(ep.resid + orow * ep.ldr + col0);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float4 b = r4[j];
        v[4 * j + 0] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
      }
    }
    if (ep.out_dtype != DT_F32) {
      uint4* o = reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(ep.out) + orow * ep.ldo + col0);
      const bool bf = ep.out_dtype == DT_BF16;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        o[j] = make_uint4(pack16(bf, v[8 * j + 0], v[8 * j + 1]), pack16(bf, v[8 * j + 2], v[8 * j + 3]),
                          pack16(bf, v[8 * j + 4], v[8 * j + 5]), pack16(bf, v[8 * j + 6], v[8 * j + 7]));
    } else {
      float4* o = reinterpret_cast<float4*>(reinterpret_cast<float*>(ep.out) + orow * ep.ldo + col0);
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = make_float4(v[4 * j + 0], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    }
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (col0 + j < ep.N) epi_store_scalar(ep, orow, col0 + j, __uint_as_float(r[j]));
  }
}


// ----------------------------------------------------------------------------------------------------
// Tile epilogue shared by the tcgen05 GEMM kernels: one warp drains its 32 TMEM lanes x (BN/2) columns.
// ----------------------------------------------------------------------------------------------------
constexpr int kBM = 128;
constexpr int kGemmThreads = 320;
constexpr int kEpiWarps = 8;
constexpr uint32_t kStageBufBytes = 32 * 128;  // per epilogue warp: 32 rows x 128 B of swizzled staging

// Pull the residual lines a warp will read for tile (m_blk, n_blk) into L2 one tile ahead of their use: the
// residual epilogue was latency-bound on those reads (ncu: long-scoreboard stalls, DRAM 38 %).
template <int BN>
__device__ __forceinline__ void prefetch_resid_tile(const EpiParams& ep, int m_blk, int n_blk, int quad, int half, int lane) {
  if (!ep.resid || !(ep.coalesced || ep.tma_f32)) return;
  const int row = m_blk * kBM + quad * 32 + lane;
  const int col0 = n_blk * BN + half * (BN / 2);
  if (row >= ep.M || col0 >= ep.N) return;
  const char* p = reinterpret_cast<const char*>(ep.resid + epi_out_row(ep, row) * ep.ldr + col0);
  const int bytes = (ep.N - col0 < BN / 2 ? ep.N - col0 : BN / 2) * 4;
  for (int o = 0; o < bytes; o += 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + o));
}

// tma_f32 epilogue, first half: once the previous tile's stores have drained the warp's two staging buffers, request the first
// two 32 x 32 residual chunks of tile (m_blk, n_blk).  epilogue_tile() does this itself unless told that the caller already did
// (the fused MLP issues it at tile start, several microseconds before the accumulator is ready).
template <int BN>
__device__ __forceinline__ void tma_f32_prefetch(const EpiParams& ep, const CUtensorMap* tmR, uint8_t* stg, uint64_t* rbar, int m_blk,
                                                 int n_blk, int quad, int half, int lane) {
  constexpr int NCH = BN / 64;
  const int row0 = m_blk * kBM + quad * 32;
  const int colbase = n_blk * BN + half * (BN / 2);
  if (lane == 0) {
    tma_store_wait_read0();                  // the previous tile's stores have drained both buffers
    if (ep.resid != nullptr && row0 < ep.M) {
#pragma unroll
      for (int c = 0; c < 2 && c < NCH; ++c) {
        if (colbase + 32 * c < ep.N) {
          mbar_arrive_expect_tx(&rbar[c], kStageBufBytes);
          tma_load_2d(stg + c * kStageBufBytes, tmR, &rbar[c], colbase + 32 * c, row0);
        }
      }
    }
  }
  __syncwarp();
}

template <int BN>
__device__ __forceinline__ void epilogue_tile(const EpiParams& ep, const CUtensorMap* tmC, uint8_t* stg, uint32_t tmem_tile,
                                              uint64_t* tfull_bar, uint32_t aph, int m_blk, int n_blk, int quad, int half,
                                              int lane, int nbuf = 1, uint32_t* stg_sel = nullptr, const CUtensorMap* tmR = nullptr,
                                              uint64_t* rbar = nullptr, uint32_t* rph = nullptr, bool prefetched = false) {
  const bool bf = ep.out_dtype == DT_BF16;
  const int row_in_tile = quad * 32 + lane;
        const int row = m_blk * kBM + row_in_tile;
        const bool row_ok = row < ep.M;
        // Residual epilogue: row addresses do not depend on the MMA result, so the first chunk's residual
        // lines are requested BEFORE waiting for the accumulator (and chunk c+1's while chunk c is processed).
        long long orow8[8];
        bool ok8[8];
        float4 res[8];
        const int q = lane & 7;
        auto load_resid = [&](int gcol) {
  #pragma unroll
          for (int j = 0; j < 8; ++j) {
            res[j] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (ep.resid && ok8[j] && gcol < ep.N)
              res[j] = *reinterpret_cast<const float4*>(ep.resid + orow8[j] * ep.ldr + gcol + 4 * q);
          }
        };
        if (ep.tma_f32) {
          // fp32 output on identity rows (out-proj on token-ordered context, fc2, patch embedding, merging): the warp's
          // 32 x 32 fp32 chunks of the residual stream are fetched by TMA into its two 128B-swizzled staging buffers (the first
          // two before the accumulator is even awaited, chunk c+2 as soon as chunk c's store has drained its buffer), each
          // lane adds its accumulator row in place, and the chunk leaves by TMA store.  No LDG / STG, no transposition: the
          // register-staged form of this epilogue ran at 3.4-3.6 TB/s (profiles/r1_gemm_pipeline_analysis.md).
          constexpr int NCH = BN / 64;
          const int row0 = m_blk * kBM + quad * 32;
          const int colbase = n_blk * BN + half * (BN / 2);
          const bool has_res = ep.resid != nullptr;
          const bool rows_ok = row0 < ep.M;          // warp-uniform
          if (!prefetched) tma_f32_prefetch<BN>(ep, tmR, stg, rbar, m_blk, n_blk, quad, half, lane);
          mbar_wait(tfull_bar, aph);
          tc_fence_after();
          const uint32_t t_addr = tmem_tile + (uint32_t(quad * 32) << 16);
  #pragma unroll 1
          for (int ci = 0; ci < NCH; ++ci) {
            const int gcol = colbase + 32 * ci;
            if (gcol >= ep.N) break;  // warp-uniform
            const int b = ci & 1;
            uint8_t* buf = stg + b * kStageBufBytes;
            uint32_t r[32];
            tmem_ld_32x32(t_addr + uint32_t(half * (BN / 2) + 32 * ci), r);
            tmem_ld_wait();
            float v[32];
  #pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
            epi_bias_act32(ep, row, gcol, v);
            if (has_res && rows_ok) {
              mbar_wait(&rbar[b], (*rph >> b) & 1u);
              *rph ^= (1u << b);
            } else if (ci >= 2) {
              if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");   // chunk ci-2's store has drained buf
              __syncwarp();
            }
  #pragma unroll
            for (int k = 0; k < 8; ++k) {
              float4* p = reinterpret_cast<float4*>(buf + lane * 128 + ((k ^ (lane & 7)) << 4));
              float4 t = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
              if (has_res && rows_ok) {
                const float4 x0 = *p;
                t.x += x0.x; t.y += x0.y; t.z += x0.z; t.w += x0.w;
              }
              *p = t;
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0 && rows_ok) {
              if (ep.red_add) tma_reduce_add_2d(tmC, buf, gcol, row0);
              else tma_store_2d(tmC, buf, gcol, row0);
              tma_store_commit();
              if (has_res && ci + 2 < NCH && gcol + 64 < ep.N) {
                tma_store_wait_read0();              // that store has read buf: it can take chunk ci+2's residual
                mbar_arrive_expect_tx(&rbar[b], kStageBufBytes);
                tma_load_2d(buf, tmR, &rbar[b], gcol + 64, row0);
              }
            }
          }
          return;
        }
        if (ep.coalesced) {
  #pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int rr = m_blk * kBM + quad * 32 + 4 * j + (lane >> 3);
            ok8[j] = rr < ep.M;
            orow8[j] = ok8[j] ? epi_out_row(ep, rr) : 0;
          }
          load_resid(n_blk * BN + half * (BN / 2));
        }
        mbar_wait(tfull_bar, aph);
        tc_fence_after();
        const uint32_t t_addr = tmem_tile + (uint32_t(quad * 32) << 16);
        if (ep.tma_store) {
  #pragma unroll 1
          for (int c = 0; c < BN / 2; c += 64) {
            const int col_local = half * (BN / 2) + c;
            const int gcol = n_blk * BN + col_local;
            if (gcol >= ep.N) break;  // warp-uniform
            uint32_t pk[32];          // 64 columns packed to 16 bit
            uint32_t r2[2][32];       // both 32-column TMEM loads are issued before the single wait: their latency overlaps
            tmem_ld_32x32(t_addr + uint32_t(col_local), r2[0]);
            tmem_ld_32x32(t_addr + uint32_t(col_local + 32), r2[1]);
            tmem_ld_wait();
  #pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              if (ep.act == ACT_GELU) {
                epi_bias_gelu_pack32(ep.bias, bf, gcol + 32 * hh, r2[hh], pk + 16 * hh);
              } else {
                float v[32];
    #pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r2[hh][j]);
                epi_bias_act32(ep, row, gcol + 32 * hh, v);
    #pragma unroll
                for (int j = 0; j < 16; ++j) pk[16 * hh + j] = pack16(bf, v[2 * j], v[2 * j + 1]);
              }
            }
            // With two staging buffers per warp only the store issued TWO chunks ago must have drained its buffer,
            // so the TMA engine's read of the previous chunk overlaps this chunk's math and smem writes.
            uint8_t* sbuf = stg;
            if (nbuf == 2) {
              sbuf = stg + (*stg_sel & 1u) * kStageBufBytes;
              *stg_sel ^= 1u;
              if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
            } else if (lane == 0) {
              tma_store_wait_read0();
            }
            __syncwarp();
  #pragma unroll
            for (int q = 0; q < 8; ++q)  // row `lane`, 16-byte chunk q -> swizzled position q ^ (lane & 7)
              *reinterpret_cast<uint4*>(sbuf + lane * 128 + ((q ^ (lane & 7)) << 4)) =
                  make_uint4(pk[4 * q], pk[4 * q + 1], pk[4 * q + 2], pk[4 * q + 3]);
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0 && m_blk * kBM + quad * 32 < ep.M) {
              tma_store_2d(tmC, sbuf, gcol, m_blk * kBM + quad * 32);
              tma_store_commit();
            }
          }
        } else if (ep.coalesced) {
          // fp32 output (+ residual, + row scatter).  Accumulators arrive row-per-thread; a 32x32 fp32 chunk is
          // transposed through the swizzled staging buffer so that every global access of the warp covers 4 full
          // 128-byte lines (8 lanes x 16 B per row) instead of 32 partial ones.
          float* outp = reinterpret_cast<float*>(ep.out);
  #pragma unroll 1
          for (int c = 0; c < BN / 2; c += 32) {
            const int col_local = half * (BN / 2) + c;
            const int gcol = n_blk * BN + col_local;
            if (gcol >= ep.N) break;  // warp-uniform
            uint32_t r[32];
            tmem_ld_32x32(t_addr + uint32_t(col_local), r);
            tmem_ld_wait();
            float v[32];
  #pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
            epi_bias_act32(ep, row, gcol, v);
  #pragma unroll
            for (int k = 0; k < 8; ++k)
              *reinterpret_cast<float4*>(stg + lane * 128 + ((k ^ (lane & 7)) << 4)) =
                  make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
            __syncwarp();
            float4 val[8];
  #pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int i = 4 * j + (lane >> 3);
              const float4 t = *reinterpret_cast<const float4*>(stg + i * 128 + ((q ^ (i & 7)) << 4));
              val[j] = make_float4(t.x + res[j].x, t.y + res[j].y, t.z + res[j].z, t.w + res[j].w);
            }
            if (c + 32 < BN / 2) load_resid(gcol + 32);   // next chunk's residual in flight during the stores
            if (ep.red_add) {      // in-place residual: x += val as a vector reduction in L2 (res[] is zero, nothing was loaded)
  #pragma unroll
              for (int j = 0; j < 8; ++j)
                if (ok8[j]) red_add_f32x4(outp + orow8[j] * ep.ldo + gcol + 4 * q, val[j]);
            } else {
  #pragma unroll
              for (int j = 0; j < 8; ++j)
                if (ok8[j]) *reinterpret_cast<float4*>(outp + orow8[j] * ep.ldo + gcol + 4 * q) = val[j];
            }
            __syncwarp();
          }
        } else {
          const long long orow = row_ok ? epi_out_row(ep, row) : 0;
  #pragma unroll 1
          for (int c = 0; c < BN / 2; c += 32) {
            const int col_local = half * (BN / 2) + c;
            const int gcol = n_blk * BN + col_local;
            if (gcol >= ep.N) break;  // warp-uniform
            uint32_t r[32];
            tmem_ld_32x32(t_addr + uint32_t(col_local), r);
            tmem_ld_wait();
            if (row_ok) epi_store_chunk32(ep, orow, gcol, r);
          }
        }
}

// The 16-bit TMA-store epilogue for SIXTEEN epilogue warps (gemm_pair_kernel<FMT, 16>, GELU outputs at K <= 512): warp (quad, part)
// drains its 32 TMEM lanes x 64 columns (part = 0..3 of a 256-column tile) - one staging buffer, one TMA store per warp and tile.
// Why: a clock64 trace of the 8-warp epilogue (profiles/r2_gemm_pair_trace_before.txt) shows 6600 cycles of GELU epilogue per tile
// against ~4100 cycles of MMAs at K = 512, the issuer waiting ~4000 cycles for the accumulator buffer on EVERY tile; half the columns
// per warp halve that chain (fc1 at Swin-B stage 2: 107 -> 100 us).  Both 32-column loads are in flight before the single wait; the first
// half's 64 bytes per row are in shared memory before the second half's arithmetic starts (96 registers per thread at 576 threads).
// The plain-store epilogue (4500 cycles on 8 warps) does NOT gain from this: once it is short the tile period stays at ~5500 cycles because
// the mainloop alone saturates the SM's shared-memory bandwidth at the tensor floor and the staging traffic comes on top
// (profiles/r2_gemm_epilogue_diagnostics.txt), so plain stores keep the 8-warp kernel.
template <int BN>
__device__ __forceinline__ void epilogue_tile16(const EpiParams& ep, const CUtensorMap* tmC, uint8_t* sbuf, uint32_t tmem_tile,
                                                uint64_t* tfull_bar, uint32_t aph, int m_blk, int n_blk, int quad, int part, int lane) {
  static_assert(BN == 256, "four 64-column parts");
  const bool bf = ep.out_dtype == DT_BF16;
  const int col_local = part * 64;
  const int gcol = n_blk * BN + col_local;
  mbar_wait(tfull_bar, aph);
  tc_fence_after();
  if (gcol >= ep.N) return;  // warp-uniform
  const uint32_t t_addr = tmem_tile + (uint32_t(quad * 32) << 16) + uint32_t(col_local);
  uint32_t r0[32], r1[32];
  tmem_ld_32x32(t_addr, r0);
  tmem_ld_32x32(t_addr + 32u, r1);
  if (lane == 0) tma_store_wait_read0();      // the previous tile's store has read the staging buffer (issued a whole tile ago)
  __syncwarp();
  tmem_ld_wait();
  auto step32 = [&](const uint32_t (&r)[32], int gc, int hh) {
    uint32_t pk[16];
    if (ep.act == ACT_GELU) {
      epi_bias_gelu_pack32(ep.bias, bf, gc, r, pk);
    } else {
      float v[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
      epi_bias_act32(ep, m_blk * kBM + quad * 32 + lane, gc, v);
#pragma unroll
      for (int j = 0; j < 16; ++j) pk[j] = pack16(bf, v[2 * j], v[2 * j + 1]);
    }
#pragma unroll
    for (int q = 0; q < 4; ++q)  // row `lane`, 16-byte chunk 4 hh + q -> swizzled position
      *reinterpret_cast<uint4*>(sbuf + lane * 128 + (((4 * hh + q) ^ (lane & 7)) << 4)) =
          make_uint4(pk[4 * q], pk[4 * q + 1], pk[4 * q + 2], pk[4 * q + 3]);
  };
  step32(r0, gcol, 0);
  step32(r1, gcol + 32, 1);
  fence_proxy_async_smem();
  __syncwarp();
  if (lane == 0 && m_blk * kBM + quad * 32 < ep.M) {
    tma_store_2d(tmC, sbuf, gcol, m_blk * kBM + quad * 32);
    tma_store_commit();
  }
}

// Host launchers (gemm.cu).  in_dtype: DT_BF16 / DT_F16 -> tcgen05 kind::f16 (W in the same format);
// DT_F32 -> tcgen05 kind::tf32 when impl == GEMM_TC, exact fp32 FMA when impl == GEMM_SIMT.
enum : int { GEMM_TC = 0, GEMM_SIMT = 1 };
int last_gemm_kernel();      // 0 none, 1 gemm_pair_kernel, 2 gemm_tc_kernel, 3 gemm_simt_f32_kernel

struct GemmTuning {
  int max_ctas;   // 0 = one per SM
  int cluster;    // 0 = auto, else 1 / 2 / 4 CTAs sharing the weight tile by TMA multicast
  int tma_store;  // -1 = auto, 0 = direct stores, 1 = smem-staged TMA stores where legal
  int pair;       // -1 = auto, 0 = never, 1 = CTA-pair (cta_group::2) kernel where legal
};
int make_tmap(CUtensorMap* tm, const void* ptr, long long ld, long long rows, long long cols, int dtype, int box_rows,
              bool as_tf32);
int make_tmap_sw64(CUtensorMap* tm, const void* ptr, long long ld, long long rows, long long cols, int dtype, int box_rows);
int num_sms();
int red_add_mode();          // CSVIT_RED_ADD: 0 off, 1 (default) every in-place residual epilogue, 2 TMA path only
int launch_gemm_pair(const void* A, long long lda, const void* W, long long ldw, int in_dtype, int M, int N, int K,
                     const EpiParams& ep, const GemmTuning& tune, cudaStream_t stream);
int launch_gemm(const void* A, long long lda, const void* W, long long ldw, int in_dtype, int M, int N, int K,
                const EpiParams& ep, int impl, const GemmTuning& tune, cudaStream_t stream);

}  // namespace csvit
