// SwinV2 scaled-cosine window attention for 8 x 8 windows (64 tokens) on tcgen05 / TMEM: the forward (inference and training) and the
// backward of the last stage of every window-16 configuration and of every stage of the window-8 checkpoints.  Same contract and log2
// domain as the 16 x 16 pair (swinv2_attn_tc.cu / swinv2_attn_bwd.cu), per window and head h:
//     z2  = q2 k_hat^T + bias_log2[h][dy + 7][dx + 7] + mask_repeat * log2(e) * shift_mask        (V2:421-487)
//     ctx = softmax2(z2) v,   lse2 = log2 sum_j 2^z2
//     dZ2 = ln 2 * P o (dO v^T - D),  dq2 = dZ2 k_hat,  dk_hat = dZ2^T q2,  dv = P^T dO,  dbias_log2 = sum of dZ2 by offset
//
// Tile = two consecutive windows (128 rows), work unit = (head, window pair), head-major over a persistent grid of two CTAs per SM (256
// TMEM columns each: the second CTA's MMAs and TMA overlap the first one's softmax).  Q2 / K / V (/ dO) are {32 columns, 128 rows} TMA
// boxes with a 64-byte swizzle; rows past the last window read as zeros, so an odd window count needs no special tile.
//   S = Q2 K^T [128 x 128] in TMEM (and dP = dO V^T next to it in the backward).  Query row r belongs to window e = r / 64 and only its
//   own window's 64 logits are ever read: thread = (row, 32-key half), 8 warps, so no exponential or FMA is spent on the cross-window
//   quadrants.  The 16-bit P (and dZ2) are written once as [128 rows x 128 keys] 128-byte-swizzled tiles; the cross-window quadrants of
//   those tiles are zeroed at kernel start and never written, so they contribute exactly zero to P V, to the row sums and to dQ / dK / dV.
//   Forward: O = P V and the row sums of the rounded probabilities (P times a tile of ones) on tcgen05.
//   Backward: dQ = dZ2 K (dZ2 tile K-major), dK = dZ2^T Q2 (the same bytes MN-major), dV = P^T dO, accumulated in TMEM over S's columns
//   (S / dP are consumed by then): no atomics, bit-reproducible.  The bias-table gradient is reduced per head in shared memory
//   (red.shared, conflict-free with the 24-float table pitch) and flushed with red.global.add when the CTA's head changes.
#include <type_traits>

#include "attn_common.cuh"
#include "errors.h"
#include "gemm.cuh"
#include "rowops.cuh"

namespace csvit {

constexpr int W8_THREADS = 256;
constexpr int W8_L = 64;                                // tokens per window
constexpr uint32_t W8_BOX = 128 * 64;                   // one {32 col, 128 row} 16-bit box, 64-byte rows
constexpr uint32_t W8_PTILE = 32768;                    // [128 rows x 128 keys] 16 bit: two 16 KB 128-byte-swizzled atoms
// Bias table row pitch (15 used): for one key, the 32 lanes of a warp are 32 consecutive query rows of one window - 4 window rows x 8
// columns - and 4 rows x 24 floats land on banks 0, 24, 16, 8: the 32 lanes hit 32 distinct banks (loads and red.shared alike).
constexpr int W8_BROW = 24;
constexpr int W8_TAB = 15 * W8_BROW;
constexpr uint32_t W8_TAB_BYTES = 1536;
constexpr float W8_LN2 = 0.69314718055994531f;

// forward: two stages of Q2 | K | V, the P tile, 2 KB of ones, the bias table, the row-max exchange, barriers
constexpr uint32_t W8F_STAGE = 3 * W8_BOX;
constexpr uint32_t W8F_P_OFF = 2 * W8F_STAGE;
constexpr uint32_t W8F_ONES_OFF = W8F_P_OFF + W8_PTILE;
constexpr uint32_t W8F_BIAS_OFF = W8F_ONES_OFF + 2048;
constexpr uint32_t W8F_XCH_OFF = W8F_BIAS_OFF + W8_TAB_BYTES;
constexpr uint32_t W8F_BAR_OFF = W8F_XCH_OFF + 1024;
constexpr size_t W8F_SMEM = 1024 + size_t(W8F_BAR_OFF) + 64;
// backward: one stage of Q2 | K | V | dO, the P and dZ2 tiles, the bias and dbias tables, barriers
constexpr uint32_t W8B_STAGE = 4 * W8_BOX;
constexpr uint32_t W8B_P_OFF = W8B_STAGE;
constexpr uint32_t W8B_Z_OFF = W8B_P_OFF + W8_PTILE;
constexpr uint32_t W8B_BIAS_OFF = W8B_Z_OFF + W8_PTILE;
constexpr uint32_t W8B_DB_OFF = W8B_BIAS_OFF + W8_TAB_BYTES;
constexpr uint32_t W8B_BAR_OFF = W8B_DB_OFF + W8_TAB_BYTES;
constexpr size_t W8B_SMEM = 1024 + size_t(W8B_BAR_OFF) + 64;

struct W8Params {
  const float* bias;     // fp32 [heads][15][24]: log2(e) * 16 sigmoid(cpb)[(dy + 7) * 15 + dx + 7] at [dy + 7][dx + 7]
  void* ctx;             // forward: 16-bit [rows, C] output
  float* lse2;           // training forward: fp32 [num_windows][heads][64]; backward: its input
  const void* octx;      // backward: O and dO, 16-bit [rows, C] window order
  const void* dctx;
  void* dq;              // backward: 16-bit [rows, C] each
  void* dk;
  void* dv;
  float* dbias;          // backward: fp32 [heads][15][24], zeroed by the launcher
  int num_windows, nW, C, heads, token_order;
  float mask_add;        // log2(e) * (-100) * mask_repeat
  WinGeom g;
};

// Shift-mask addends of a thread's 32 keys (window rows 4 hf .. 4 hf + 3, all columns): HF's regions split the last window row / column
// of a shifted layer at 4, so a key's class is (its row < 4 = hf == 0) x (its column < 4); lo / hi = keys with column < 4 / >= 4.
__device__ __forceinline__ bool w8_mask(const W8Params& p, int wg, int yi, int xi, int hf, float& madd_lo, float& madd_hi) {
  const int w = wg % p.nW, wy = w / p.g.nWx, wx = w - wy * p.g.nWx;
  const bool lastrow = p.g.shift > 0 && wy == p.g.H / p.g.ws - 1, lastcol = p.g.shift > 0 && wx == p.g.nWx - 1;
  const bool ydiff = lastrow && ((yi < 4) != (hf == 0));
  madd_lo = (ydiff || (lastcol && xi >= 4)) ? p.mask_add : 0.0f;
  madd_hi = (ydiff || (lastcol && xi < 4)) ? p.mask_add : 0.0f;
  return lastrow || lastcol;
}

// Table offset of key k (0..31) of the thread's half relative to the thread's entry for key (4 hf, 0).
__host__ __device__ constexpr int w8_koff(int k) { return (k >> 3) * W8_BROW + (k & 7); }

// + bias [+ mask] over the thread's 32 logits and their maximum.
template <bool MASKED>
__device__ __forceinline__ void w8_logits(uint32_t (&v)[32], const float* bt, float madd_lo, float madd_hi, float& mx) {
  float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
  for (int k = 0; k < 32; k += 2) {
    float2 f = __fadd2_rn(make_float2(__uint_as_float(v[k]), __uint_as_float(v[k + 1])),
                          make_float2(bt[-w8_koff(k)], bt[-w8_koff(k) - 1]));
    if (MASKED) f = __fadd2_rn(f, (k & 7) < 4 ? make_float2(madd_lo, madd_lo) : make_float2(madd_hi, madd_hi));
    v[k] = __float_as_uint(f.x); v[k + 1] = __float_as_uint(f.y);
  }
#pragma unroll
  for (int k = 0; k < 32; k += 4) {
    mx0 = fa_max3(mx0, __uint_as_float(v[k]), __uint_as_float(v[k + 1]));
    mx1 = fa_max3(mx1, __uint_as_float(v[k + 2]), __uint_as_float(v[k + 3]));
  }
  mx = fmaxf(mx0, mx1);
}

// The thread's 16 packed 16-bit values -> its four 16-byte chunks of row r of a 128-byte-swizzled [128 x 64] atom (keys 32 hf ..).
__device__ __forceinline__ void w8_store_row(uint32_t row_addr, int hf, int r, const uint32_t (&pk)[16]) {
#pragma unroll
  for (int q = 0; q < 4; ++q)
    sts128(row_addr + (uint32_t((4 * hf + q) ^ (r & 7)) << 4), pk[4 * q], pk[4 * q + 1], pk[4 * q + 2], pk[4 * q + 3]);
}

__device__ __forceinline__ void w8_store16(bool bf, void* dst, const uint32_t (&v)[16], float scale) {
  uint4* o = reinterpret_cast<uint4*>(dst);
#pragma unroll
  for (int q = 0; q < 2; ++q)
    o[q] = make_uint4(pack16(bf, __uint_as_float(v[8 * q]) * scale, __uint_as_float(v[8 * q + 1]) * scale),
                      pack16(bf, __uint_as_float(v[8 * q + 2]) * scale, __uint_as_float(v[8 * q + 3]) * scale),
                      pack16(bf, __uint_as_float(v[8 * q + 4]) * scale, __uint_as_float(v[8 * q + 5]) * scale),
                      pack16(bf, __uint_as_float(v[8 * q + 6]) * scale, __uint_as_float(v[8 * q + 7]) * scale));
}

// Forward.  FMT: 0 = fp16, 1 = bf16.  LSE = 1 (training) also writes lse2 = row max + log2(row sum of the rounded probabilities), so
// that the backward recomputes P = 2^(z2 - lse2) exactly as this kernel normalised it; LSE = 0 is the inference kernel.
// Per unit n: S(n) was issued with P V(n - 1); softmax -> P tile; P V(n), row sums and S(n + 1) are issued together and one commit
// covers them; the epilogue reads O(n) while S(n + 1) is already in TMEM.
template <int FMT, int LSE>
__global__ void __launch_bounds__(W8_THREADS, 2)
swinv2_w8_attn_kernel(const __grid_constant__ CUtensorMap tmQKV, W8Params p) {
  using T16 = typename std::conditional<FMT == 1, __nv_bfloat16, __half>::type;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + W8F_BAR_OFF);      // [2] operand stages
  uint64_t* mma_bar = full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(full + 3);
  float* btab = reinterpret_cast<float*>(smem + W8F_BIAS_OFF);
  float* xmax = reinterpret_cast<float*>(smem + W8F_XCH_OFF);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int quad = warp & 3, hf = warp >> 2;
  const int r = quad * 32 + lane, e = r >> 6, i = r & 63, yi = i >> 3, xi = i & 7;
  const int C = p.C, HEADS = p.heads, NWIN = p.num_windows, PAIRS = (NWIN + 1) >> 1;
  const long long units = static_cast<long long>(PAIRS) * HEADS;
  const int u_begin = int(units * blockIdx.x / gridDim.x), u_end = int(units * (blockIdx.x + 1) / gridDim.x);
  const int total = u_end - u_begin;

  for (int k = threadIdx.x; k < int(W8_PTILE / 16); k += W8_THREADS)       // the cross-window quadrants stay zero
    reinterpret_cast<uint4*>(smem + W8F_P_OFF)[k] = make_uint4(0u, 0u, 0u, 0u);
  for (int k = threadIdx.x; k < 512; k += W8_THREADS)
    reinterpret_cast<uint32_t*>(smem + W8F_ONES_OFF)[k] = FMT == 1 ? 0x3F803F80u : 0x3C003C00u;
  if (threadIdx.x == 0) {
    prefetch_tmap(&tmQKV);
    mbar_init(&full[0], 1); mbar_init(&full[1], 1); mbar_init(mma_bar, 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, 256);
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tl = tmem_base + (uint32_t(quad * 32) << 16);

  auto load_unit = [&](int n) {       // thread 0: the three boxes of unit u_begin + n into stage n & 1
    const int u = u_begin + n, h = u / PAIRS, wp = u - h * PAIRS, st = n & 1;
    uint8_t* sb = smem + size_t(st) * W8F_STAGE;
    mbar_arrive_expect_tx(&full[st], W8F_STAGE);
#pragma unroll
    for (int m = 0; m < 3; ++m) tma_load_2d(sb + m * W8_BOX, &tmQKV, &full[st], m * C + h * 32, wp * 128);
  };
  constexpr uint32_t idesc_s = make_idesc(uint32_t(FMT), 128, 128);
  constexpr uint32_t idesc_o = make_idesc(uint32_t(FMT), 128, 32) | (1u << 16);       // V MN-major
  constexpr uint32_t idesc_1 = make_idesc(uint32_t(FMT), 128, 16) | (1u << 16);
  const uint32_t pt = base + W8F_P_OFF;
  const uint64_t onesd = fa_mnmajor_desc(base + W8F_ONES_OFF);
  auto issue_s = [&](uint32_t sb) {   // S = Q2 K^T, TMEM columns 0-127 (K = 32: two k-steps of 32 bytes in the 64-byte rows)
    const uint64_t qd = vb_sw64_desc(sb), kd = vb_sw64_desc(sb + W8_BOX);
#pragma unroll
    for (int k = 0; k < 2; ++k) umma_ss<false>(tmem_base, qd + uint64_t(2 * k), kd + uint64_t(2 * k), idesc_s, k ? 1u : 0u);
  };
  auto issue_pv = [&](uint32_t sb) {  // O = P V (columns 128-159) and the row sums P 1 (160-175): 8 k-steps of 16 keys
#pragma unroll
    for (int ks = 0; ks < 8; ++ks) {
      const uint64_t ad = make_sw128_kmajor_desc(pt + uint32_t(ks >> 2) * 16384u) + uint64_t(2 * (ks & 3));
      umma_ss<false>(tmem_base + 128u, ad, vb_sw64_desc(sb + 2 * W8_BOX + uint32_t(ks) * 1024u), idesc_o, ks ? 1u : 0u);
    }
#pragma unroll
    for (int ks = 0; ks < 8; ++ks) {
      const uint64_t ad = make_sw128_kmajor_desc(pt + uint32_t(ks >> 2) * 16384u) + uint64_t(2 * (ks & 3));
      umma_ss<false>(tmem_base + 160u, ad, onesd, idesc_1, ks ? 1u : 0u);
    }
  };

  if (threadIdx.x == 0 && total > 0) load_unit(0);
  const bool bf = FMT == 1;
  const uint32_t ts = tl + uint32_t(64 * e + 32 * hf);                 // this thread's 32 logits: its own window's keys only
  const uint32_t p_row = pt + uint32_t(e) * 16384u + uint32_t(r) * 128u;
  const int boff = (yi + 7 - 4 * hf) * W8_BROW + xi + 7;               // table entry of key (4 hf, 0)
  T16* ctx = static_cast<T16*>(p.ctx);
  uint32_t mph = 0;
  int cur_h = -1;
  for (int n = 0; n < total; ++n) {
    const int u = u_begin + n, h = u / PAIRS, wp = u - h * PAIRS, wg = 2 * wp + e;
    if (threadIdx.x == 0 && n + 1 < total) load_unit(n + 1);          // its stage's last reader, P V(n - 1), has completed
    if (h != cur_h) {
      __syncthreads();
      for (int k = threadIdx.x; k < W8_TAB; k += W8_THREADS) btab[k] = p.bias[size_t(h) * W8_TAB + k];
      __syncthreads();
      cur_h = h;
    }
    if (n == 0) {
      if (warp == 0) {
        mbar_wait(&full[0], 0);
        tc_fence_after();
        if (fa_elect_one()) {
          issue_s(base);
          umma_commit(mma_bar);
        }
        __syncwarp();
      }
      mbar_wait(mma_bar, mph);
      mph ^= 1u;
    }
    tc_fence_after();
    float madd_lo, madd_hi, mx;
    const bool masked = w8_mask(p, wg, yi, xi, hf, madd_lo, madd_hi);
    uint32_t v[32];
    tmem_ld_32x32(ts, v);
    tmem_ld_wait();
    if (masked) w8_logits<true>(v, btab + boff, madd_lo, madd_hi, mx);
    else w8_logits<false>(v, btab + boff, 0.f, 0.f, mx);
    xmax[hf * 128 + r] = mx;
    __syncthreads();
    mx = fmaxf(mx, xmax[(hf ^ 1) * 128 + r]);
    uint32_t pk[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const float2 d = __fadd2_rn(make_float2(__uint_as_float(v[2 * k]), __uint_as_float(v[2 * k + 1])), make_float2(-mx, -mx));
      pk[k] = FMT == 1 ? pack_bf16x2(fa_exp2(d.x), fa_exp2(d.y)) : pack_f16x2(fa_exp2(d.x), fa_exp2(d.y));
    }
    w8_store_row(p_row, hf, r, pk);
    fence_proxy_async_smem();          // the P tile is read by the tensor core (async proxy)
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
      if (n + 1 < total) mbar_wait(&full[(n + 1) & 1], (uint32_t(n + 1) >> 1) & 1u);
      tc_fence_after();
      if (fa_elect_one()) {
        issue_pv(base + uint32_t(n & 1) * W8F_STAGE);
        if (n + 1 < total) issue_s(base + uint32_t((n + 1) & 1) * W8F_STAGE);
        umma_commit(mma_bar);
      }
      __syncwarp();
    }
    // ---- epilogue: this half's 16 of the head's 32 output columns
    mbar_wait(mma_bar, mph);
    mph ^= 1u;
    tc_fence_after();
    uint32_t o[16], rs;
    tmem_ld_32x16(tl + 128u + 16u * uint32_t(hf), o);
    tmem_ld_32x1(tl + 160u, rs);
    tmem_ld_wait();
    tc_fence_before();
    if (wg < NWIN) {
      const int b = wg / p.nW, w = wg - b * p.nW;
      const long long row = p.token_order ? static_cast<long long>(b) * p.g.N + win_row_to_token(p.g, w * W8_L + i)
                                          : static_cast<long long>(wg) * W8_L + i;
      w8_store16(bf, ctx + row * C + h * 32 + 16 * hf, o, 1.0f / __uint_as_float(rs));
      if (LSE && hf == 0) p.lse2[(static_cast<long long>(wg) * HEADS + h) * W8_L + i] = mx + __log2f(__uint_as_float(rs));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 256);
}

// Backward.  Per unit: S and dP (TMEM 0-127 / 128-255) -> P, dZ2 tiles and the dbias table -> dQ, dK, dV (TMEM 0-31 / 32-63 / 64-95)
// -> 16-bit rows.  The unit's phases run in sequence; the other CTA on the SM fills the gaps.
template <int FMT>
__global__ void __launch_bounds__(W8_THREADS, 2)
swinv2_w8_bwd_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ CUtensorMap tmDO, W8Params p) {
  using T16 = typename std::conditional<FMT == 1, __nv_bfloat16, __half>::type;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + W8B_BAR_OFF);
  uint64_t* mma_bar = full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(full + 2);
  float* btab = reinterpret_cast<float*>(smem + W8B_BIAS_OFF);
  float* dbt = reinterpret_cast<float*>(smem + W8B_DB_OFF);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int quad = warp & 3, hf = warp >> 2;
  const int r = quad * 32 + lane, e = r >> 6, i = r & 63, yi = i >> 3, xi = i & 7;
  const int C = p.C, HEADS = p.heads, NWIN = p.num_windows, PAIRS = (NWIN + 1) >> 1;
  const long long units = static_cast<long long>(PAIRS) * HEADS;
  const int u_begin = int(units * blockIdx.x / gridDim.x), u_end = int(units * (blockIdx.x + 1) / gridDim.x);
  const int total = u_end - u_begin;

  for (int k = threadIdx.x; k < int(2 * W8_PTILE / 16); k += W8_THREADS)   // P and dZ2: the cross-window quadrants stay zero
    reinterpret_cast<uint4*>(smem + W8B_P_OFF)[k] = make_uint4(0u, 0u, 0u, 0u);
  for (int k = threadIdx.x; k < W8_TAB; k += W8_THREADS) dbt[k] = 0.0f;
  if (threadIdx.x == 0) {
    prefetch_tmap(&tmQKV);
    prefetch_tmap(&tmDO);
    mbar_init(full, 1); mbar_init(mma_bar, 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, 256);
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tl = tmem_base + (uint32_t(quad * 32) << 16);

  auto load_unit = [&](int n) {
    const int u = u_begin + n, h = u / PAIRS, wp = u - h * PAIRS;
    mbar_arrive_expect_tx(full, W8B_STAGE);
#pragma unroll
    for (int m = 0; m < 3; ++m) tma_load_2d(smem + m * W8_BOX, &tmQKV, full, m * C + h * 32, wp * 128);
    tma_load_2d(smem + 3 * W8_BOX, &tmDO, full, h * 32, wp * 128);
  };
  constexpr uint32_t idesc_s = make_idesc(uint32_t(FMT), 128, 128);
  constexpr uint32_t idesc_dq = make_idesc(uint32_t(FMT), 128, 32) | (1u << 16);                 // B (K) MN-major
  constexpr uint32_t idesc_dkv = make_idesc(uint32_t(FMT), 128, 32) | (1u << 15) | (1u << 16);   // A (P / dZ2 transposed), B MN-major
  const uint32_t pt = base + W8B_P_OFF, zt = base + W8B_Z_OFF;
  auto issue_s = [&]() {              // S = Q2 K^T, dP = dO V^T
    const uint64_t qd = vb_sw64_desc(base), kd = vb_sw64_desc(base + W8_BOX);
    const uint64_t vd = vb_sw64_desc(base + 2 * W8_BOX), od = vb_sw64_desc(base + 3 * W8_BOX);
#pragma unroll
    for (int k = 0; k < 2; ++k) umma_ss<false>(tmem_base, qd + uint64_t(2 * k), kd + uint64_t(2 * k), idesc_s, k ? 1u : 0u);
#pragma unroll
    for (int k = 0; k < 2; ++k) umma_ss<false>(tmem_base + 128u, od + uint64_t(2 * k), vd + uint64_t(2 * k), idesc_s, k ? 1u : 0u);
  };
  auto issue_grad = [&]() {           // dQ = dZ2 K, dK = dZ2^T Q2, dV = P^T dO: 8 k-steps of 16 keys / query rows each
#pragma unroll
    for (int ks = 0; ks < 8; ++ks) {
      const uint64_t ad = make_sw128_kmajor_desc(zt + uint32_t(ks >> 2) * 16384u) + uint64_t(2 * (ks & 3));
      umma_ss<false>(tmem_base, ad, vb_sw64_desc(base + W8_BOX + uint32_t(ks) * 1024u), idesc_dq, ks ? 1u : 0u);
    }
#pragma unroll
    for (int ks = 0; ks < 8; ++ks)
      umma_ss<false>(tmem_base + 32u, vb_mn128_desc(zt + uint32_t(ks) * 2048u), vb_sw64_desc(base + uint32_t(ks) * 1024u), idesc_dkv,
                     ks ? 1u : 0u);
#pragma unroll
    for (int ks = 0; ks < 8; ++ks)
      umma_ss<false>(tmem_base + 64u, vb_mn128_desc(pt + uint32_t(ks) * 2048u), vb_sw64_desc(base + 3 * W8_BOX + uint32_t(ks) * 1024u),
                     idesc_dkv, ks ? 1u : 0u);
  };

  if (threadIdx.x == 0 && total > 0) load_unit(0);
  const T16* O = static_cast<const T16*>(p.octx);
  const T16* dO = static_cast<const T16*>(p.dctx);
  const bool bf = FMT == 1;
  const uint32_t ts = tl + uint32_t(64 * e + 32 * hf);
  const uint32_t p_row = pt + uint32_t(e) * 16384u + uint32_t(r) * 128u, z_row = p_row + W8_PTILE;
  const int boff = (yi + 7 - 4 * hf) * W8_BROW + xi + 7;
  const uint32_t dbt_addr = smem_u32(dbt) + 4u * uint32_t(boff);
  uint32_t mph = 0;
  int cur_h = -1;
  for (int n = 0; n < total; ++n) {
    const int u = u_begin + n, h = u / PAIRS, wp = u - h * PAIRS, wg = 2 * wp + e;
    const bool valid = wg < NWIN;      // the second window of an odd count's last tile: zero operands, nothing read or written
    if (h != cur_h) {
      __syncthreads();
      if (cur_h >= 0)
        for (int k = threadIdx.x; k < W8_TAB; k += W8_THREADS) {
          const float g = dbt[k];
          if (g != 0.0f) atomicAdd(p.dbias + size_t(cur_h) * W8_TAB + k, g);
          dbt[k] = 0.0f;
        }
      for (int k = threadIdx.x; k < W8_TAB; k += W8_THREADS) btab[k] = p.bias[size_t(h) * W8_TAB + k];
      __syncthreads();
      cur_h = h;
    }
    if (warp == 0) {
      mbar_wait(full, uint32_t(n) & 1u);
      tc_fence_after();
      if (fa_elect_one()) {
        issue_s();
        umma_commit(mma_bar);
      }
      __syncwarp();
    }
    // the row's lse2 (+inf for a missing window: P = 0) and D = dO . O while S and dP are computed
    const long long row = static_cast<long long>(wg) * W8_L + i;
    float lse = INFINITY, D = 0.f;
    if (valid) {
      lse = p.lse2[(static_cast<long long>(wg) * HEADS + h) * W8_L + i];
      const uint4* po = reinterpret_cast<const uint4*>(O + row * C + h * 32);
      const uint4* pd = reinterpret_cast<const uint4*>(dO + row * C + h * 32);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const uint4 a = po[q], b = pd[q];
        D = vb_dot2<FMT>(a.x, b.x, D); D = vb_dot2<FMT>(a.y, b.y, D);
        D = vb_dot2<FMT>(a.z, b.z, D); D = vb_dot2<FMT>(a.w, b.w, D);
      }
    }
    float madd_lo, madd_hi;
    const bool masked = w8_mask(p, wg, yi, xi, hf, madd_lo, madd_hi);
    mbar_wait(mma_bar, mph);
    mph ^= 1u;
    tc_fence_after();
    uint32_t s[32], dp[32];
    tmem_ld_32x32(ts, s);
    tmem_ld_32x32(ts + 128u, dp);
    tmem_ld_wait();
    uint32_t pp[16], zz[16];
    const float* bt = btab + boff;
#pragma unroll
    for (int k = 0; k < 32; k += 2) {
      float pe[2], g[2];
#pragma unroll
      for (int m = 0; m < 2; ++m) {
        float z = __uint_as_float(s[k + m]) + bt[-w8_koff(k + m)];
        if (masked) z += (k & 7) < 4 ? madd_lo : madd_hi;
        pe[m] = fa_exp2(z - lse);
        g[m] = W8_LN2 * pe[m] * (__uint_as_float(dp[k + m]) - D);
        red_shared_f32(dbt_addr - 4u * uint32_t(w8_koff(k + m)), g[m]);
      }
      pp[k >> 1] = FMT == 1 ? pack_bf16x2(pe[0], pe[1]) : pack_f16x2(pe[0], pe[1]);
      zz[k >> 1] = FMT == 1 ? pack_bf16x2(g[0], g[1]) : pack_f16x2(g[0], g[1]);
    }
    w8_store_row(p_row, hf, r, pp);
    w8_store_row(z_row, hf, r, zz);
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
      tc_fence_after();
      if (fa_elect_one()) {
        issue_grad();
        umma_commit(mma_bar);
      }
      __syncwarp();
    }
    mbar_wait(mma_bar, mph);
    mph ^= 1u;
    tc_fence_after();
    if (threadIdx.x == 0 && n + 1 < total) load_unit(n + 1);          // every reader of the stage has completed
    // epilogue: dQ (lanes = query rows), dK / dV (lanes = key rows); this thread's 16 of the head's 32 columns
#pragma unroll
    for (int m = 0; m < 3; ++m) {
      uint32_t v[16];
      tmem_ld_32x16(tl + 32u * uint32_t(m) + 16u * uint32_t(hf), v);
      tmem_ld_wait();
      if (valid) w8_store16(bf, static_cast<T16*>(m == 0 ? p.dq : (m == 1 ? p.dk : p.dv)) + row * C + h * 32 + 16 * hf, v, 1.0f);
    }
    tc_fence_before();
    __syncthreads();                     // the accumulators are read before the next unit's S overwrites them
  }
  __syncthreads();
  if (cur_h >= 0)
    for (int k = threadIdx.x; k < W8_TAB; k += W8_THREADS) {
      const float g = dbt[k];
      if (g != 0.0f) atomicAdd(p.dbias + size_t(cur_h) * W8_TAB + k, g);
    }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 256);
}

static int w8_geometry(const char* name, int dtype, int H, int W, int C, int heads, int shift, int mask_repeat) {
  CSVIT_REQUIRE(dtype == DT_BF16 || dtype == DT_F16, "%s: 16-bit operand formats only", name);
  CSVIT_REQUIRE(C == heads * 32 && heads >= 1, "%s: head_dim 32 only (C=%d heads=%d)", name, C, heads);
  CSVIT_REQUIRE(H > 0 && W > 0 && H % 8 == 0 && W % 8 == 0 && (shift == 0 || shift == 4), "%s: windows of 8, shift 0 or 4 (%dx%d shift %d)",
                name, H, W, shift);
  CSVIT_REQUIRE(mask_repeat >= 0 && mask_repeat <= 2, "%s: mask_repeat %d outside [0,2]", name, mask_repeat);
  return 0;
}

static W8Params w8_params(const float* bias_log2, int B, int H, int W, int C, int heads, int shift, int mask_repeat) {
  W8Params p{};
  p.bias = bias_log2;
  p.nW = (H / 8) * (W / 8);
  p.num_windows = B * p.nW;
  p.C = C; p.heads = heads;
  p.mask_add = -100.0f * 1.4426950408889634f * static_cast<float>(mask_repeat);
  p.g = make_geom(H, W, 8, shift);
  return p;
}

static int w8_ctas(const W8Params& p) {
  const long long units = static_cast<long long>((p.num_windows + 1) / 2) * p.heads;
  return units < 2ll * num_sms() ? int(units) : 2 * num_sms();
}

template <int FMT, int LSE>
static int launch_w8(const CUtensorMap& tm, const W8Params& p, cudaStream_t stream) {
  auto kern = swinv2_w8_attn_kernel<FMT, LSE>;
  CSVIT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(W8F_SMEM)));
  kern<<<w8_ctas(p), W8_THREADS, W8F_SMEM, stream>>>(tm, p);
  CSVIT_CUDA(cudaGetLastError());
  return 0;
}

// qkv: 16-bit [B*nW*64, 3C] rows in window order (pitch ldq), q2 | k_hat | v as csvit_swinv2_qkv writes them.  lse2 null = inference.
int launch_swinv2_attn8_tc(const void* qkv, long long ldq, const float* bias_log2, void* ctx, float* lse2, int dtype, int B, int H, int W,
                           int C, int heads, int shift, int mask_repeat, int token_order, cudaStream_t stream) {
  const char* name = lse2 ? "swinv2_attn8_tc_train" : "swinv2_attn8_tc";
  if (int e = w8_geometry(name, dtype, H, W, C, heads, shift, mask_repeat)) return e;
  CSVIT_REQUIRE(B >= 0, "%s: negative batch", name);
  const uintptr_t al = reinterpret_cast<uintptr_t>(qkv) | reinterpret_cast<uintptr_t>(ctx) | reinterpret_cast<uintptr_t>(bias_log2) |
                       reinterpret_cast<uintptr_t>(lse2);
  CSVIT_REQUIRE((al & 15) == 0 && ldq >= 3ll * C && (ldq & 7) == 0, "%s: operands must be 16-byte aligned, pitch >= 3C", name);
  CSVIT_REQUIRE(!(lse2 && token_order), "%s: the training forward writes window order", name);
  const long long windows = static_cast<long long>(B) * (H / 8) * (W / 8);
  if (windows <= 0) return 0;
  CSVIT_REQUIRE(windows * W8_L < (1ll << 31) && windows * heads < (1ll << 31), "%s: too many rows", name);
  W8Params p = w8_params(bias_log2, B, H, W, C, heads, shift, mask_repeat);
  p.ctx = ctx; p.lse2 = lse2; p.token_order = token_order ? 1 : 0;
  CUtensorMap tm;
  if (int e = make_tmap_sw64(&tm, qkv, ldq, windows * W8_L, 3ll * C, dtype, 128)) return e;
  const bool bf = dtype == DT_BF16;
  if (lse2) return bf ? launch_w8<1, 1>(tm, p, stream) : launch_w8<0, 1>(tm, p, stream);
  return bf ? launch_w8<1, 0>(tm, p, stream) : launch_w8<0, 0>(tm, p, stream);
}

template <int FMT>
static int launch_w8_bwd(const CUtensorMap& tmQKV, const CUtensorMap& tmDO, const W8Params& p, cudaStream_t stream) {
  auto kern = swinv2_w8_bwd_kernel<FMT>;
  CSVIT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(W8B_SMEM)));
  kern<<<w8_ctas(p), W8_THREADS, W8B_SMEM, stream>>>(tmQKV, tmDO, p);
  CSVIT_CUDA(cudaGetLastError());
  return 0;
}

// ctx (O) / dctx (dO): dense 16-bit [rows, C], window order.  Writes dq / dk / dv (dense 16-bit [rows, C]) and dbias_log2 (fp32
// [heads][15][24], columns 15..23 stay 0).
int launch_swinv2_attn8_bwd(const void* qkv, long long ldq, const void* ctx, const void* dctx, const float* lse2, const float* bias_log2,
                            void* dq, void* dk, void* dv, float* dbias_log2, int dtype, int B, int H, int W, int C, int heads, int shift,
                            int mask_repeat, cudaStream_t stream) {
  const char* name = "swinv2_attn8_tc_bwd";
  if (int e = w8_geometry(name, dtype, H, W, C, heads, shift, mask_repeat)) return e;
  CSVIT_REQUIRE(B >= 0, "%s: negative batch", name);
  const uintptr_t al = reinterpret_cast<uintptr_t>(qkv) | reinterpret_cast<uintptr_t>(ctx) | reinterpret_cast<uintptr_t>(dctx) |
                       reinterpret_cast<uintptr_t>(lse2) | reinterpret_cast<uintptr_t>(bias_log2) | reinterpret_cast<uintptr_t>(dq) |
                       reinterpret_cast<uintptr_t>(dk) | reinterpret_cast<uintptr_t>(dv) | reinterpret_cast<uintptr_t>(dbias_log2);
  CSVIT_REQUIRE((al & 15) == 0 && ldq >= 3ll * C && (ldq & 7) == 0, "%s: operands must be 16-byte aligned, pitch >= 3C", name);
  CSVIT_CUDA(cudaMemsetAsync(dbias_log2, 0, size_t(heads) * W8_TAB * sizeof(float), stream));
  const long long windows = static_cast<long long>(B) * (H / 8) * (W / 8);
  if (windows <= 0) return 0;
  CSVIT_REQUIRE(windows * W8_L < (1ll << 31) && windows * heads < (1ll << 31), "%s: too many rows", name);
  W8Params p = w8_params(bias_log2, B, H, W, C, heads, shift, mask_repeat);
  p.lse2 = const_cast<float*>(lse2); p.octx = ctx; p.dctx = dctx;
  p.dq = dq; p.dk = dk; p.dv = dv; p.dbias = dbias_log2;
  CUtensorMap tmQKV, tmDO;
  if (int e = make_tmap_sw64(&tmQKV, qkv, ldq, windows * W8_L, 3ll * C, dtype, 128)) return e;
  if (int e = make_tmap_sw64(&tmDO, dctx, C, windows * W8_L, C, dtype, 128)) return e;
  return dtype == DT_BF16 ? launch_w8_bwd<1>(tmQKV, tmDO, p, stream) : launch_w8_bwd<0>(tmQKV, tmDO, p, stream);
}

}  // namespace csvit
