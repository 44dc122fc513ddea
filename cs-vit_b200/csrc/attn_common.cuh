// Helpers shared by the tcgen05 window-attention kernels (attn_fused.cu: LN + QKV + attention for C <= 256; attn_core.cu: the
// attention core on Q/K/V loaded by TMA for every width).
#pragma once
#include "common.cuh"

namespace csvit {

constexpr int FA_L = 49;                            // tokens per 7 x 7 window
constexpr uint32_t FA_BIAS_BYTES = 49 * 56 * 2;     // one head's bias rows [49][56] fp16 (log2 domain, query-slot-major)
constexpr uint32_t FA_BIAS_STAGE = 5632;
constexpr float FA_MASK_LOG2 = -100.0f * 1.4426950408889634f;

__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ uint64_t fa_mnmajor_desc(uint32_t smem_addr) {
  // MN-major operand of one 128-byte MN chunk (64 elements): rows = k, 8-row swizzle atoms of 1024 B (layout of gemm_ex.cu)
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(8192 >> 4) << 16;    // LBO: next MN chunk (unused, N = 64 is one chunk)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;    // SBO: next group of 8 k-rows
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
__device__ __forceinline__ float fa_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ void tmem_ld_32x1(uint32_t taddr, uint32_t& r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r) : "r"(taddr) : "memory");
}
// a += lo(h2), b += hi(h2): fp16 addends, fp32 sums (one FHADD each)
__device__ __forceinline__ void fa_add_h2(float& a, float& b, uint32_t h2) {
  asm("{\n\t.reg .f16 lo, hi;\n\tmov.b32 {lo, hi}, %2;\n\tadd.rn.f32.f16 %0, lo, %0;\n\tadd.rn.f32.f16 %1, hi, %1;\n\t}" : "+f"(a), "+f"(b) : "r"(h2));
}
__device__ __forceinline__ void fa_bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ float fa_max3(float a, float b, float c) {
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}


// Shift mask of query slot j in window w of the image (HF get_attn_mask, HF:swin/modeling_swin.py:556-582) as a bit mask over the
// 49 key slots: bit c set = key slot c lies in another region (the logit gets -100).  Only windows on the last window row /
// column of a shifted layer have masked pairs.
__device__ __forceinline__ unsigned long long fa_row_mask(const WinGeom& g, int w, int j) {
  if (g.shift <= 0) return 0ull;
  const int nWy = g.H / g.ws;
  const int wy = w / g.nWx, wx = w - wy * g.nWx;
  const int iy = j / 7, ix = j - iy * 7, th = g.ws - g.shift;
  unsigned long long dm = 0;
  if (wy == nWy - 1) {      // key slots whose row side (iy < th) differs from mine
    const unsigned long long rows_lo = (1ull << (7 * th)) - 1ull;
    dm |= (iy < th) ? ~rows_lo : rows_lo;
  }
  if (wx == g.nWx - 1) {      // key slots whose column side (ix < th) differs from mine: th low bits of every 7-bit row group
    const unsigned long long cols_lo = ((1ull << th) - 1ull) * 0x40810204081ull;      // sum of 2^(7 i), i = 0..6
    dm |= (ix < th) ? ~cols_lo : cols_lo;
  }
  return dm & ((1ull << FA_L) - 1ull);
}

// Adds the shift mask of fa_row_mask (as two 32-bit halves) to a row's 49 log2-domain logits.  For the Swin geometry (window 7,
// shift 3) the key slots fall into four fixed classes - (iy < 4 or not) x (ix < 4 or not) - so the row needs four addends read off
// four representative bits and 49 plain additions with compile-time class selection; other shifts take the bit-by-bit form.
__device__ __forceinline__ void fa_add_mask(float (&sv)[50], uint32_t dm_lo, uint32_t dm_hi, bool th4) {
  if ((dm_lo | dm_hi) == 0u) return;
  if (th4) {
    const float m[2][2] = {{(dm_lo & 1u) ? FA_MASK_LOG2 : 0.0f, (dm_lo & (1u << 4)) ? FA_MASK_LOG2 : 0.0f},
                           {(dm_lo & (1u << 28)) ? FA_MASK_LOG2 : 0.0f, (dm_hi & 1u) ? FA_MASK_LOG2 : 0.0f}};
#pragma unroll
    for (int c = 0; c < FA_L; ++c) sv[c] += m[(c / 7) >= 4][(c % 7) >= 4];
  } else {
#pragma unroll
    for (int c = 0; c < FA_L; ++c) {
      const uint32_t bit = c < 32 ? (dm_lo >> c) & 1u : (dm_hi >> (c - 32)) & 1u;
      sv[c] += bit ? FA_MASK_LOG2 : 0.0f;
    }
  }
}

// ---- operands of the SwinV2 tcgen05 backward kernels (swinv2_attn_bwd.cu, swinv2_attn8.cu)
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

}  // namespace csvit
