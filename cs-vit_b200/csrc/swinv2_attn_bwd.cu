// Backward of the SwinV2 cosine window attention for 16 x 16 windows (256 tokens) on tcgen05 / TMEM: the differentiable counterpart of
// swinv2_attn_tc.cu for the finetune step.  Log2 domain, per window and head h (q2 = q_hat * logit_scale_h * log2 e, k_hat, v 16 bit):
//     z2  = q2 k_hat^T + bias_log2[h][dy + 15][dx + 15] + mask_repeat * log2(e) * shift_mask        (V2:421-487)
//     P   = 2^(z2 - lse2)       (lse2 from the training forward, swinv2_attn_tc_kernel<FMT, 1>)
//     D_i = sum_d dO_i,d O_i,d
//     dZ2 = ln 2 * P o (dO v^T - D)            dq2 = dZ2 k_hat     dk_hat = dZ2^T q2     dv = P^T dO
//     dbias_log2[h][dy + 15][dx + 15] = sum over windows and (i, j) at offset (dy, dx) of dZ2[i, j]
//
// Work unit = (head, window), head-major over the grid (persistent, one CTA per SM): a CTA's contiguous range stays on one or two heads.
// The unit's Q2 / K / V / dO are four {32 columns, 256 rows} TMA boxes with a 64-byte swizzle (one head per box, 16 KB each; odd head
// counts need no phantom head), double-buffered across units.  Per query tile t (128 rows) and key block kb (128 keys):
//   S  = Q2_t K_kb^T, dP = dO_t V_kb^T                  [128 x 128] each, TMEM columns 0-127 / 128-255
//   8 warps, thread = (query row, key half): + bias (one LDS from the 48-pitch table) + closed-form shift mask, P = 2^(z2 - lse2),
//       dZ2 = ln2 P (dP - D); dZ2 into the shared-memory dbias table (red.shared: for one key the 32 lanes of a warp - 32 consecutive
//       query rows - hit 32 distinct (dy, dx) bins, lanes 16-31 one table row = 48 floats = 16 banks after lanes 0-15: conflict-free);
//       P and dZ2 written ONCE each as 16-bit [128 query rows x 128 keys] 128-byte-swizzled tiles
//   dQ_t  += dZ2 K_kb           A = the dZ2 tile read K-major           TMEM 256 + 32 t
//   dK_kb += dZ2^T Q2_t         A = the same bytes read MN-major        TMEM 320 + 32 kb
//   dV_kb += P^T dO_t           A = the P tile read MN-major            TMEM 384 + 32 kb
// then dQ, dK, dV leave TMEM as 16 bit into the head's 32 columns of the window-ordered [rows, C] outputs.  dq / dk / dv involve no
// atomics (bit-reproducible); the dbias table is flushed with red.global.add when the CTA's head changes (a few thousand global
// reductions per launch; the last bits of dbias depend on their order).
// The MMA issuer is warp 0, converged, one elected lane.  The phases of a unit run in sequence (the MMAs of a step overlap nothing but
// the TMA of the next unit): this kernel is bound by the per-logit instructions of the softmax-gradient warps.
#include <cstdio>
#include <type_traits>

#include "attn_common.cuh"
#include "errors.h"
#include "gemm.cuh"

namespace csvit {

constexpr int VB_THREADS = 256;
constexpr int VB_L = 256;
constexpr uint32_t VB_BOX = 256 * 64;                  // one {32 col, 256 row} 16-bit box, 64-byte rows
constexpr uint32_t VB_STAGE = 4 * VB_BOX;              // Q2, K, V, dO of one unit
constexpr uint32_t VB_PZ_OFF = 2 * VB_STAGE;           // P tile then dZ2 tile: [128 rows x 128 keys] 16 bit = two 16 KB 128-byte atoms each
constexpr uint32_t VB_PZ_TILE = 32768;
constexpr int VB_BROW = 48;
constexpr int VB_TAB = 31 * VB_BROW;                   // floats of one head's bias / dbias table
constexpr uint32_t VB_BIAS_OFF = VB_PZ_OFF + 2 * VB_PZ_TILE;
constexpr uint32_t VB_DB_OFF = VB_BIAS_OFF + 6144;
constexpr uint32_t VB_BAR_OFF = VB_DB_OFF + 6144;
constexpr size_t VB_SMEM = 1024 + size_t(VB_BAR_OFF) + 64;
constexpr float VB_LN2 = 0.69314718055994531f;

struct VbParams {
  const float* bias;     // fp32 [heads][31][48] (csvit_swinv2_attn_tc's layout)
  const void* ctx;       // O: 16-bit [rows, C] window order (the training forward's output)
  const void* dctx;      // dO: 16-bit [rows, C]
  const float* lse2;     // fp32 [num_windows][heads][256]
  void* dq;              // 16-bit [rows, C] each
  void* dk;
  void* dv;
  float* dbias;          // fp32 [heads][31][48], zeroed by the launcher, accumulated with red.global.add
  int num_windows, nW, C, heads;
  float mask_add;        // log2(e) * (-100) * mask_repeat
  WinGeom g;
};

// K-major operand with a 64-byte swizzle: rows of 64 B (32 16-bit elements), 8-row atoms of 512 B (SBO), layout type 4 = SWIZZLE_64B.
// The same descriptor reads a box MN-major ([K rows x 32 MN elements], one MN chunk: LBO unused).
__device__ __forceinline__ uint64_t vb_sw64_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(512 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(4) << 61;
  return d;
}
// MN-major 128-byte-swizzled operand spanning two 64-element MN chunks 16 KB apart (LBO); rows = k, 8-row atoms of 1024 B (SBO).
__device__ __forceinline__ uint64_t vb_mn128_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(16384 >> 4) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
__device__ __forceinline__ void red_shared_f32(uint32_t addr, float v) {
  asm volatile("red.shared.add.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

template <int FMT>
__device__ __forceinline__ float vb_dot2(uint32_t a, uint32_t b, float acc) {
  float2 fa, fb;
  if (FMT == 1) {
    fa = __bfloat1622float2(__halves2bfloat162(__ushort_as_bfloat16(uint16_t(a)), __ushort_as_bfloat16(uint16_t(a >> 16))));
    fb = __bfloat1622float2(__halves2bfloat162(__ushort_as_bfloat16(uint16_t(b)), __ushort_as_bfloat16(uint16_t(b >> 16))));
  } else {
    fa = __half22float2(__halves2half2(__ushort_as_half(uint16_t(a)), __ushort_as_half(uint16_t(a >> 16))));
    fb = __half22float2(__halves2half2(__ushort_as_half(uint16_t(b)), __ushort_as_half(uint16_t(b >> 16))));
  }
  return fmaf(fa.x, fb.x, fmaf(fa.y, fb.y, acc));
}

// One 32-key chunk of a thread's row: keys 32 c4 .. 32 c4 + 31 of the key block.  Writes P / dZ2 (16 bit) to the swizzled tiles and
// dZ2 into the dbias table.
template <int FMT, bool MASKED>
__device__ __forceinline__ void vb_chunk(const uint32_t (&s)[32], const uint32_t (&dp)[32], const float* bt, uint32_t dbt_addr, int c4,
                                         float madd_lo, float madd_hi, float lse, float D, uint32_t p_row, uint32_t z_row, int r) {
  uint32_t pp[16], zz[16];
#pragma unroll
  for (int k = 0; k < 32; k += 2) {
    float e[2], g[2];
#pragma unroll
    for (int m = 0; m < 2; ++m) {
      const int c = 32 * c4 + k + m;                      // key (8 kb + (c >> 4), c & 15) of the block
      const int off = (c >> 4) * VB_BROW + (c & 15);
      float z = __uint_as_float(s[k + m]) + bt[-off];
      if (MASKED) z += ((c & 15) < 8) ? madd_lo : madd_hi;
      e[m] = fa_exp2(z - lse);
      g[m] = VB_LN2 * e[m] * (__uint_as_float(dp[k + m]) - D);
      red_shared_f32(dbt_addr - 4u * uint32_t(off), g[m]);
    }
    pp[k >> 1] = FMT == 1 ? pack_bf16x2(e[0], e[1]) : pack_f16x2(e[0], e[1]);
    zz[k >> 1] = FMT == 1 ? pack_bf16x2(g[0], g[1]) : pack_f16x2(g[0], g[1]);
  }
  // 128-byte swizzle, K-major [rows x 64 keys] atoms: key c at atom c >> 6, 16-byte chunk ((c & 63) >> 3) ^ (row & 7)
  const uint32_t atom = uint32_t(c4 >> 1) * 16384u;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const uint32_t ch = uint32_t((4 * (c4 & 1) + q) ^ (r & 7)) << 4;
    sts128(p_row + atom + ch, pp[4 * q], pp[4 * q + 1], pp[4 * q + 2], pp[4 * q + 3]);
    sts128(z_row + atom + ch, zz[4 * q], zz[4 * q + 1], zz[4 * q + 2], zz[4 * q + 3]);
  }
}

// Flush the CTA's dbias table of head h into global memory and clear it (all threads; caller synchronises around it).
__device__ __forceinline__ void vb_flush(float* dbt, float* gdb) {
  for (int k = threadIdx.x; k < VB_TAB; k += VB_THREADS) {
    const float v = dbt[k];
    if (v != 0.0f) atomicAdd(gdb + k, v);
    dbt[k] = 0.0f;
  }
}

template <int FMT>
__global__ void __launch_bounds__(VB_THREADS, 1)
swinv2_attn_bwd_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ CUtensorMap tmDO, VbParams p) {
  using T16 = typename std::conditional<FMT == 1, __nv_bfloat16, __half>::type;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + VB_BAR_OFF);
  uint64_t* full = bars;               // [2] operand stages
  uint64_t* mma_bar = bars + 2;        // every MMA batch commits here
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3);
  float* btab = reinterpret_cast<float*>(smem + VB_BIAS_OFF);
  float* dbt = reinterpret_cast<float*>(smem + VB_DB_OFF);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int quad = warp & 3, hf = warp >> 2;
  const int r = quad * 32 + lane;                       // row of the 128-row tile = TMEM lane
  const int C = p.C, HEADS = p.heads, NWIN = p.num_windows;
  const long long units = static_cast<long long>(NWIN) * HEADS;
  const int u_begin = int(units * blockIdx.x / gridDim.x), u_end = int(units * (blockIdx.x + 1) / gridDim.x);
  const int total = u_end - u_begin;

  for (int k = threadIdx.x; k < VB_TAB; k += VB_THREADS) dbt[k] = 0.0f;
  if (threadIdx.x == 0) {
    prefetch_tmap(&tmQKV);
    prefetch_tmap(&tmDO);
    mbar_init(&full[0], 1); mbar_init(&full[1], 1); mbar_init(mma_bar, 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tlane = tmem_base + (uint32_t(quad * 32) << 16);

  auto load_unit = [&](int n) {       // thread 0: the four boxes of unit u_begin + n into stage n & 1
    const int u = u_begin + n, h = u / NWIN, w = u - h * NWIN, st = n & 1;
    uint8_t* sb = smem + size_t(st) * VB_STAGE;
    mbar_arrive_expect_tx(&full[st], VB_STAGE);
#pragma unroll
    for (int m = 0; m < 3; ++m) tma_load_2d(sb + m * VB_BOX, &tmQKV, &full[st], m * C + h * 32, w * VB_L);
    tma_load_2d(sb + 3 * VB_BOX, &tmDO, &full[st], h * 32, w * VB_L);
  };
  constexpr uint32_t idesc_s = make_idesc(uint32_t(FMT), 128, 128);
  constexpr uint32_t idesc_dq = make_idesc(uint32_t(FMT), 128, 32) | (1u << 16);                 // B (K_kb) MN-major
  constexpr uint32_t idesc_dkv = make_idesc(uint32_t(FMT), 128, 32) | (1u << 15) | (1u << 16);   // A (P / dZ2 transposed), B MN-major
  const uint32_t pz = base + VB_PZ_OFF;
  // S = Q2_t K_kb^T and dP = dO_t V_kb^T (K = 32: two k-steps of 32 bytes in the 64-byte rows)
  auto issue_s = [&](uint32_t sb, int t, int kb) {
    const uint64_t qd = vb_sw64_desc(sb + uint32_t(t) * 8192u), kd = vb_sw64_desc(sb + VB_BOX + uint32_t(kb) * 8192u);
    const uint64_t od = vb_sw64_desc(sb + 3 * VB_BOX + uint32_t(t) * 8192u), vd = vb_sw64_desc(sb + 2 * VB_BOX + uint32_t(kb) * 8192u);
#pragma unroll
    for (int k = 0; k < 2; ++k) umma_ss<false>(tmem_base, qd + uint64_t(2 * k), kd + uint64_t(2 * k), idesc_s, k ? 1u : 0u);
#pragma unroll
    for (int k = 0; k < 2; ++k) umma_ss<false>(tmem_base + 128u, od + uint64_t(2 * k), vd + uint64_t(2 * k), idesc_s, k ? 1u : 0u);
  };
  // dQ_t += dZ2 K_kb, dK_kb += dZ2^T Q2_t, dV_kb += P^T dO_t: 8 k-steps of 16 (keys / query rows) each
  auto issue_grad = [&](uint32_t sb, int t, int kb) {
#pragma unroll
    for (int ks = 0; ks < 8; ++ks) {
      const uint64_t ad = make_sw128_kmajor_desc(pz + VB_PZ_TILE + uint32_t(ks >> 2) * 16384u) + uint64_t(2 * (ks & 3));
      const uint64_t bd = vb_sw64_desc(sb + VB_BOX + uint32_t(kb) * 8192u + uint32_t(ks) * 1024u);
      umma_ss<false>(tmem_base + 256u + 32u * uint32_t(t), ad, bd, idesc_dq, (kb | ks) ? 1u : 0u);
    }
#pragma unroll
    for (int ks = 0; ks < 8; ++ks) {
      const uint64_t ad = vb_mn128_desc(pz + VB_PZ_TILE + uint32_t(ks) * 2048u);
      const uint64_t bd = vb_sw64_desc(sb + uint32_t(t) * 8192u + uint32_t(ks) * 1024u);
      umma_ss<false>(tmem_base + 320u + 32u * uint32_t(kb), ad, bd, idesc_dkv, (t | ks) ? 1u : 0u);
    }
#pragma unroll
    for (int ks = 0; ks < 8; ++ks) {
      const uint64_t ad = vb_mn128_desc(pz + uint32_t(ks) * 2048u);
      const uint64_t bd = vb_sw64_desc(sb + 3 * VB_BOX + uint32_t(t) * 8192u + uint32_t(ks) * 1024u);
      umma_ss<false>(tmem_base + 384u + 32u * uint32_t(kb), ad, bd, idesc_dkv, (t | ks) ? 1u : 0u);
    }
  };

  if (threadIdx.x == 0 && total > 0) load_unit(0);
  const T16* O = static_cast<const T16*>(p.ctx);
  const T16* dO = static_cast<const T16*>(p.dctx);
  const int nWy = p.g.H / p.g.ws;
  const bool bf = FMT == 1;
  const uint32_t p_row = pz + uint32_t(r) * 128u, z_row = pz + VB_PZ_TILE + uint32_t(r) * 128u;
  const uint32_t dbt_u32 = smem_u32(dbt);
  uint32_t mph = 0;
  int cur_h = -1;
  for (int n = 0; n < total; ++n) {
    const int u = u_begin + n, h = u / NWIN, w = u - h * NWIN, st = n & 1;
    const uint32_t sb = base + uint32_t(st) * VB_STAGE;
    if (threadIdx.x == 0 && n + 1 < total) load_unit(n + 1);     // the other stage's last reader (unit n - 1's MMAs) has completed
    if (h != cur_h) {
      __syncthreads();
      if (cur_h >= 0) vb_flush(dbt, p.dbias + size_t(cur_h) * VB_TAB);
      for (int k = threadIdx.x; k < VB_TAB; k += VB_THREADS) btab[k] = p.bias[size_t(h) * VB_TAB + k];
      __syncthreads();
      cur_h = h;
    }
    // the row's lse2 and D = dO . O for both query tiles
    float lse[2], Dv[2];
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      const int i = 128 * t + r;
      const long long row = static_cast<long long>(w) * VB_L + i;
      lse[t] = p.lse2[(static_cast<long long>(w) * HEADS + h) * VB_L + i];
      const uint4* po = reinterpret_cast<const uint4*>(O + row * C + h * 32);
      const uint4* pd = reinterpret_cast<const uint4*>(dO + row * C + h * 32);
      float acc = 0.f;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const uint4 a = po[q], b = pd[q];
        acc = vb_dot2<FMT>(a.x, b.x, acc); acc = vb_dot2<FMT>(a.y, b.y, acc);
        acc = vb_dot2<FMT>(a.z, b.z, acc); acc = vb_dot2<FMT>(a.w, b.w, acc);
      }
      Dv[t] = acc;
    }
    // shift-mask geometry of the window (only the last window row / column of a shifted layer has masked pairs)
    const int wl = w % p.nW, wy = wl / p.g.nWx, wx = wl - wy * p.g.nWx;
    const bool lastrow = p.g.shift > 0 && wy == nWy - 1, lastcol = p.g.shift > 0 && wx == p.g.nWx - 1;
    const int xi = r & 15;

    if (warp == 0) {
      mbar_wait(&full[st], (uint32_t(n) >> 1) & 1u);
      tc_fence_after();
      if (fa_elect_one()) {
        issue_s(sb, 0, 0);
        umma_commit(mma_bar);
      }
      __syncwarp();
    }
    for (int it = 0; it < 4; ++it) {
      const int t = it >> 1, kb = it & 1;
      const int yi = 8 * t + (r >> 4);
      const bool ydiff = lastrow && (t != kb);            // query row y < 8 iff t == 0, key row y < 8 iff kb == 0
      const float madd_lo = (ydiff || (lastcol && xi >= 8)) ? p.mask_add : 0.0f;
      const float madd_hi = (ydiff || (lastcol && xi < 8)) ? p.mask_add : 0.0f;
      const bool masked = lastrow || lastcol;
      const int boff = (yi + 15 - 8 * kb) * VB_BROW + xi + 15;      // table entry of key (8 kb, 0)
      const float* bt = btab + boff;
      const uint32_t dbt_addr = dbt_u32 + 4u * uint32_t(boff);
      mbar_wait(mma_bar, mph);
      mph ^= 1u;
      tc_fence_after();
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        const int c4 = 2 * hf + cc;
        uint32_t s[32], dp[32];
        tmem_ld_32x32(tlane + uint32_t(32 * c4), s);
        tmem_ld_32x32(tlane + 128u + uint32_t(32 * c4), dp);
        tmem_ld_wait();
        if (masked) vb_chunk<FMT, true>(s, dp, bt, dbt_addr, c4, madd_lo, madd_hi, lse[t], Dv[t], p_row, z_row, r);
        else vb_chunk<FMT, false>(s, dp, bt, dbt_addr, c4, 0.f, 0.f, lse[t], Dv[t], p_row, z_row, r);
      }
      fence_proxy_async_smem();          // the P / dZ2 tiles are read by the tensor core (async proxy)
      tc_fence_before();
      __syncthreads();
      if (warp == 0) {
        tc_fence_after();
        if (fa_elect_one()) {
          issue_grad(sb, t, kb);
          if (it < 3) issue_s(sb, (it + 1) >> 1, (it + 1) & 1);
          umma_commit(mma_bar);
        }
        __syncwarp();
      }
    }
    // epilogue: dQ_t (lanes = query rows), dK_kb / dV_kb (lanes = key rows); this thread's 16 of the head's 32 columns
    mbar_wait(mma_bar, mph);
    mph ^= 1u;
    tc_fence_after();
#pragma unroll
    for (int m = 0; m < 6; ++m) {
      const int blk = m & 1;                               // t for dQ, kb for dK / dV
      T16* dst = static_cast<T16*>(m < 2 ? p.dq : (m < 4 ? p.dk : p.dv));
      uint32_t v[16];
      tmem_ld_32x16(tlane + 256u + 32u * uint32_t(m) + 16u * uint32_t(hf), v);
      tmem_ld_wait();
      const long long row = static_cast<long long>(w) * VB_L + 128 * blk + r;
      uint4* o = reinterpret_cast<uint4*>(dst + row * C + h * 32 + 16 * hf);
#pragma unroll
      for (int q = 0; q < 2; ++q)
        o[q] = make_uint4(pack16(bf, __uint_as_float(v[8 * q]), __uint_as_float(v[8 * q + 1])),
                          pack16(bf, __uint_as_float(v[8 * q + 2]), __uint_as_float(v[8 * q + 3])),
                          pack16(bf, __uint_as_float(v[8 * q + 4]), __uint_as_float(v[8 * q + 5])),
                          pack16(bf, __uint_as_float(v[8 * q + 6]), __uint_as_float(v[8 * q + 7])));
    }
    tc_fence_before();
    __syncthreads();                     // the accumulators are read before the next unit's MMAs overwrite them
  }
  __syncthreads();
  if (cur_h >= 0) vb_flush(dbt, p.dbias + size_t(cur_h) * VB_TAB);
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 512);
}

template <int FMT>
static int launch_vb(const CUtensorMap& tmQKV, const CUtensorMap& tmDO, const VbParams& p, cudaStream_t stream) {
  auto kern = swinv2_attn_bwd_kernel<FMT>;
  CSVIT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(VB_SMEM)));
  const long long units = static_cast<long long>(p.num_windows) * p.heads;
  const int ctas = units < num_sms() ? int(units) : num_sms();
  kern<<<ctas, VB_THREADS, VB_SMEM, stream>>>(tmQKV, tmDO, p);
  CSVIT_CUDA(cudaGetLastError());
  return 0;
}

// qkv: the training forward's 16-bit [rows, 3C] operand (pitch ldq): q2 | k_hat | v, window order.  ctx (O) / dctx (dO): dense 16-bit
// [rows, C].  Writes dq / dk / dv (dense 16-bit [rows, C]) and dbias_log2 (fp32 [heads][31][48], columns 31..47 stay 0).
int launch_swinv2_attn_bwd(const void* qkv, long long ldq, const void* ctx, const void* dctx, const float* lse2, const float* bias_log2,
                           void* dq, void* dk, void* dv, float* dbias_log2, int dtype, int B, int H, int W, int C, int heads, int shift,
                           int mask_repeat, cudaStream_t stream) {
  constexpr int ws = 16;
  CSVIT_REQUIRE(dtype == DT_BF16 || dtype == DT_F16, "swinv2_attn_tc_bwd: 16-bit operand formats only");
  CSVIT_REQUIRE(C == heads * 32 && heads >= 1, "swinv2_attn_tc_bwd: head_dim 32 only (C=%d heads=%d)", C, heads);
  CSVIT_REQUIRE(H % ws == 0 && W % ws == 0 && (shift == 0 || shift == 8),
                "swinv2_attn_tc_bwd: windows of 16, shift 0 or 8 (%dx%d shift %d)", H, W, shift);
  CSVIT_REQUIRE(mask_repeat >= 0 && mask_repeat <= 2, "swinv2_attn_tc_bwd: mask_repeat %d outside [0,2]", mask_repeat);
  const uintptr_t al = reinterpret_cast<uintptr_t>(qkv) | reinterpret_cast<uintptr_t>(ctx) | reinterpret_cast<uintptr_t>(dctx) |
                       reinterpret_cast<uintptr_t>(lse2) | reinterpret_cast<uintptr_t>(bias_log2) | reinterpret_cast<uintptr_t>(dq) |
                       reinterpret_cast<uintptr_t>(dk) | reinterpret_cast<uintptr_t>(dv) | reinterpret_cast<uintptr_t>(dbias_log2);
  CSVIT_REQUIRE((al & 15) == 0 && ldq >= 3ll * C && (ldq & 7) == 0, "swinv2_attn_tc_bwd: operands must be 16-byte aligned, pitch >= 3C");
  const int nW = (H / ws) * (W / ws);
  const long long windows = static_cast<long long>(B) * nW;
  CSVIT_CUDA(cudaMemsetAsync(dbias_log2, 0, size_t(heads) * VB_TAB * sizeof(float), stream));
  if (windows <= 0) return 0;
  CSVIT_REQUIRE(windows * VB_L < (1ll << 31) && windows * heads < (1ll << 31), "swinv2_attn_tc_bwd: too many rows");
  VbParams p{};
  p.bias = bias_log2; p.ctx = ctx; p.dctx = dctx; p.lse2 = lse2;
  p.dq = dq; p.dk = dk; p.dv = dv; p.dbias = dbias_log2;
  p.num_windows = static_cast<int>(windows); p.nW = nW; p.C = C; p.heads = heads;
  p.mask_add = -100.0f * 1.4426950408889634f * static_cast<float>(mask_repeat);
  p.g = make_geom(H, W, ws, shift);
  CUtensorMap tmQKV, tmDO;
  if (int e = make_tmap_sw64(&tmQKV, qkv, ldq, windows * VB_L, 3ll * C, dtype, VB_L)) return e;
  if (int e = make_tmap_sw64(&tmDO, dctx, C, windows * VB_L, C, dtype, VB_L)) return e;
  return dtype == DT_BF16 ? launch_vb<1>(tmQKV, tmDO, p, stream) : launch_vb<0>(tmQKV, tmDO, p, stream);
}

}  // namespace csvit
