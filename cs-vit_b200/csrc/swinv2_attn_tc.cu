// SwinV2 scaled-cosine window attention for 16 x 16 windows (256 tokens) on tcgen05 / TMEM:
//     ctx = concat_h softmax( normalize(q_h) normalize(k_h)^T * logit_scale_h + 16 sigmoid(CPB-MLP)[rel_index] + 2 * shift_mask ) v_h
// i.e. the two F.normalize, both bmm, the logit scale, the continuous-position-bias gather, the (twice added) shift mask, the softmax,
// the head merge and - in token order - window_reverse + roll(+s) of HF:swinv2/modeling_swinv2.py:421-487, 693-701.
// It replaces the round-1 mma.sync kernel (swinv2.cu) for the 256-token windows of stages 0-2; the 8 x 8 windows of the last stage
// stay there.
//
// Input: the window-ordered 16-bit [rows, 3C] output of csvit_swinv2_qkv, whose epilogue already normalised every head's q and k
// rows and multiplied q by log2(e) * logit_scale_h - so the raw tensor-core product IS the log2-domain cosine logit.
//
// Work unit = (window, head pair).  One pipeline stage holds the pair's three {64 columns, 256 rows} TMA boxes (128-byte swizzle =
// the K-major / MN-major operand tiles tcgen05 reads, head e of the pair = the k-slice at +64 e bytes) and the two heads' bias tables.
//   S(e, t)  [128 x 256] = Q_e[rows 128 t ..] K_e^T   2 MMAs (K = 32) into TMEM slot t (256 columns): a query row's 256 logits
//   X1       thread (row, key half): + bias (one LDS per logit, conflict-free: the table is padded to 48-float rows) [+ mask], row
//            max, logits written back to TMEM in place; the two halves of a row meet in shared memory for the max
//   X2       exp2(logit - max) -> 16-bit P written to TMEM over the consumed logits (tcgen05.st, two keys per column)
//   PV       O'[128 x 32] = P[128 x 256] V_e[256 x 32] with P read FROM TMEM as the A operand (16 MMAs, K = 16); V' is MN-major and the B
//            descriptor starts 64 e bytes into the pair's 128-byte rows, so only the head's own value columns are multiplied;
//            16 more MMAs of P against a 2 KB tile of ones put the row sums of the ROUNDED probabilities next to O' (N = 16)
//   E        O' / rowsum -> 16 bit -> ctx row (token order: window_reverse + un-shift folded into the address)
// P never touches shared memory: the softmax thread that owns a row writes it where the tensor core reads it.
// TMEM slot (256 columns): S in 0-255; P of key half hf in 128 hf .. 128 hf + 63 (over logits already consumed); O' in 64-95 and the row
// sums in 96-111 (both written only after every logit of the tile has been read).
// Roles: warp 0 TMA producer (2-stage ring), warp 1 MMA issuer (whole warp converged, one elected lane issues), warps 4-19 = two
// softmax sets (one per TMEM slot / query tile of the head) of two warpgroups (key halves).  X2 is MUFU-heavy and the sets share the
// SM's MUFU pipes: they take turns on X2 (named-barrier ping-pong), so that one set's exponentials hide the other's X1, E and MMA round
// trips - left alone, both sets run X2 together and then idle together (clock64 trace, profiles/r2_swinv2_attn_tc_trace.txt).
// The kernel is bound by the instructions of X1 / X2 (about 4.5 issue slots per logit), not by bytes, MMAs or MUFU throughput.
#include <cstdio>
#include <cstdlib>
#include <type_traits>
#include <vector>

#include "attn_common.cuh"
#include "errors.h"
#include "gemm.cuh"
#include "rowops.cuh"

namespace csvit {

constexpr int VT_THREADS = 640;
constexpr int VT_L = 256;                               // tokens per window
constexpr uint32_t VT_TILE = 256 * 128;                 // 256 rows x 64 16-bit columns
constexpr int VT_BROW = 48;                             // bias table row pitch (31 used): lanes 16-31 land 16 banks after lanes 0-15
constexpr uint32_t VT_BIAS_BYTES = 31 * VT_BROW * 4;
constexpr uint32_t VT_STAGE_USED = 3 * VT_TILE + 2 * VT_BIAS_BYTES;
constexpr uint32_t VT_STAGE = (VT_STAGE_USED + 1023u) & ~1023u;
constexpr uint32_t VT_XCH_OFF = 2 * VT_STAGE;           // float xmax[2 sets][2 halves][128], xsum[2][2][128]
constexpr uint32_t VT_ONES_OFF = VT_XCH_OFF + 4096;      // 2 KB of 1.0 (16 bit): the B operand of the row-sum MMA, any layout
constexpr uint32_t VT_BAR_OFF = VT_ONES_OFF + 2048;
constexpr size_t VT_SMEM = 1024 + size_t(VT_BAR_OFF) + 256;

struct VtParams {
  const float* bias;     // fp32 [heads][31][48]: log2(e) * 16 sigmoid(cpb)[(dy + 15) * 31 + dx + 15] at [dy + 15][dx + 15]
  void* ctx;             // 16-bit [B*N, C]
  int num_windows;       // B * nW
  int nW;
  int C, heads;
  int token_order;
  float mask_add;        // log2(e) * (-100) * mask_repeat
  WinGeom g;
  long long* trace;      // debugging (CSVIT_V2_TRACE): clock64 at the phase boundaries of CTA 0's first tiles, else null
  float* lse2;           // LSE = 1 (training forward): fp32 [num_windows][heads][256], log2 of each query row's softmax denominator
};
constexpr int VT_TRACE_TILES = 24;
#define VT_STAMP(k) do { if (tr) tr[k] = clock64(); } while (0)

__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]),
        "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]),
        "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// D[tmem] (+)= A[tmem: 128 lanes x 8 columns = 16 packed 16-bit k-elements per row] * B[smem]
__device__ __forceinline__ void umma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}
__device__ __forceinline__ void named_bar_arrive(int id, int threads) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(threads) : "memory");
}
__device__ __forceinline__ uint32_t ex2_h2(uint32_t x) {
  uint32_t y;
  asm("ex2.approx.f16x2 %0, %1;" : "=r"(y) : "r"(x));
  return y;
}

// X1 on one 32-column chunk (keys 32 c4 .. 32 c4 + 31 of the thread's half): + bias [+ mask], running max, write back.
template <bool MASKED>
__device__ __forceinline__ void vt_pass1_chunk(uint32_t taddr, uint32_t (&v)[32], const float* bt, int c4, float madd_lo, float madd_hi,
                                               float& mx0, float& mx1) {
#pragma unroll
  for (int k = 0; k < 32; k += 2) {                              // two logits per packed f32x2 add
    const int c = 32 * c4 + k;                                   // key (8 hf + (c >> 4), c & 15)
    float2 f = __fadd2_rn(make_float2(__uint_as_float(v[k]), __uint_as_float(v[k + 1])),
                          make_float2(bt[-((c >> 4) * VT_BROW + (c & 15))], bt[-((c >> 4) * VT_BROW + (c & 15) + 1)]));
    if (MASKED) f = __fadd2_rn(f, ((c & 15) < 8) ? make_float2(madd_lo, madd_lo) : make_float2(madd_hi, madd_hi));
    v[k] = __float_as_uint(f.x); v[k + 1] = __float_as_uint(f.y);
  }
#pragma unroll
  for (int k = 0; k < 32; k += 4) {
    mx0 = fa_max3(mx0, __uint_as_float(v[k]), __uint_as_float(v[k + 1]));
    mx1 = fa_max3(mx1, __uint_as_float(v[k + 2]), __uint_as_float(v[k + 3]));
  }
  tmem_st_32x32(taddr, v);
}

// X1 over the thread's four chunks; chunk c + 1 is requested from TMEM before chunk c is processed.
template <bool MASKED>
__device__ __forceinline__ void vt_pass1(uint32_t ts, const float* bt, float madd_lo, float madd_hi, float& mx0, float& mx1) {
  uint32_t a[32], b[32];
  tmem_ld_32x32(ts, a);
  tmem_ld_wait();
  tmem_ld_32x32(ts + 32u, b);
  vt_pass1_chunk<MASKED>(ts, a, bt, 0, madd_lo, madd_hi, mx0, mx1);
  tmem_ld_wait();
  tmem_ld_32x32(ts + 64u, a);
  vt_pass1_chunk<MASKED>(ts + 32u, b, bt, 1, madd_lo, madd_hi, mx0, mx1);
  tmem_ld_wait();
  tmem_ld_32x32(ts + 96u, b);
  vt_pass1_chunk<MASKED>(ts + 64u, a, bt, 2, madd_lo, madd_hi, mx0, mx1);
  tmem_ld_wait();
  vt_pass1_chunk<MASKED>(ts + 96u, b, bt, 3, madd_lo, madd_hi, mx0, mx1);
}

// X2 on one chunk: exp2(logit - max) -> 16 packed pairs; SUM: also accumulate the row sum in registers.
template <int FMT, bool SUM>
__device__ __forceinline__ void vt_pass2_chunk(const uint32_t (&v)[32], uint32_t (&pk)[16], float mx, float& sum0, float& sum1) {
  // fp32 MUFU.EX2 for both formats: ex2.approx.f16x2 is two MUFU.EX2.F16 plus a PRMT, one instruction more per pair
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    const float2 d = __fadd2_rn(make_float2(__uint_as_float(v[2 * k]), __uint_as_float(v[2 * k + 1])), make_float2(-mx, -mx));
    const float e0 = fa_exp2(d.x), e1 = fa_exp2(d.y);
    if (SUM) { sum0 += e0; sum1 += e1; }
    pk[k] = FMT == 1 ? pack_bf16x2(e0, e1) : pack_f16x2(e0, e1);
  }
}

// FMT: 0 = fp16, 1 = bf16.  LSE = 1 is the training forward: it also writes lse2 = row max + log2(row sum of the rounded
// probabilities), so that the backward (swinv2_attn_bwd.cu) recomputes P = 2^(z2 - lse2) exactly as this kernel normalised it; LSE = 0
// is the inference kernel, whose code the flag does not touch.  (Exponentials on the FMA pipes for one or two of the four X2 chunks -
// a degree-4 polynomial, FA4's MUFU relief - measured SLOWER, 28.3 -> 29.8 / 30.6 ns: the kernel is bound by issued instructions,
// not by MUFU.)
// (P V runs on the head's own 32 value columns - the B descriptor starts 64 e bytes into the pair's 128-byte rows - and the row sums
// come from the tensor core: P times a tile of ones.  Both were measured against the alternatives: 38 -> 32 ns per (window, head).)
template <int FMT, int LSE>
__global__ void __launch_bounds__(VT_THREADS, 1)
swinv2_attn_tc_kernel(const __grid_constant__ CUtensorMap tmQ, VtParams p) {
  using T16 = typename std::conditional<FMT == 1, __nv_bfloat16, __half>::type;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + VT_BAR_OFF);
  uint64_t* st_full = bars;            // [2] stages
  uint64_t* st_empty = st_full + 2;
  uint64_t* s_full = st_empty + 2;     // [2] by TMEM slot, like everything below
  uint64_t* p_full = s_full + 2;
  uint64_t* o_full = p_full + 2;
  uint64_t* o_empty = o_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int C = p.C, HEADS = p.heads;
  const int PAIRS = (HEADS + 1) >> 1;       // an odd head count (SwinV2-T: 3) leaves a phantom head that is computed and dropped
  const long long units = static_cast<long long>(p.num_windows) * PAIRS;
  const int u_begin = int(units * blockIdx.x / gridDim.x), u_end = int(units * (blockIdx.x + 1) / gridDim.x);
  const int total_units = u_end - u_begin;

  constexpr bool N32 = true, ONES = true;
  for (uint32_t k = threadIdx.x; k < 512; k += VT_THREADS)
    reinterpret_cast<uint32_t*>(smem + VT_ONES_OFF)[k] = FMT == 1 ? 0x3F803F80u : 0x3C003C00u;
  if (threadIdx.x == 0) {
    prefetch_tmap(&tmQ);
    for (int s = 0; s < 2; ++s) {
      mbar_init(&st_full[s], 1); mbar_init(&st_empty[s], 1);
      mbar_init(&s_full[s], 1); mbar_init(&p_full[s], 8);
      mbar_init(&o_full[s], 1); mbar_init(&o_empty[s], 8);
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  griddep_launch();      // PDL: the next kernel's prologue may overlap this kernel's tail ...
  griddep_wait();        // ... and this kernel touches global memory only after its predecessors have completed

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    if (warp == 0 && lane == 0) {
      // ---------------- TMA producer: one (window, head pair) per stage: q / k / v boxes + the two bias tables
      for (int gp = 0; gp < total_units; ++gp) {
        const int st = gp & 1;
        const int wg = (u_begin + gp) / PAIRS, hp = (u_begin + gp) - wg * PAIRS;
        mbar_wait(&st_empty[st], ((uint32_t(gp) >> 1) & 1u) ^ 1u);
        mbar_arrive_expect_tx(&st_full[st], VT_STAGE_USED);
        uint8_t* sb = smem + size_t(st) * VT_STAGE;
#pragma unroll
        for (int m = 0; m < 3; ++m) tma_load_2d(sb + m * VT_TILE, &tmQ, &st_full[st], m * C + hp * 64, wg * VT_L);
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int h = min(2 * hp + e, HEADS - 1);
          fa_bulk_load(sb + 3 * VT_TILE + e * VT_BIAS_BYTES, reinterpret_cast<const char*>(p.bias) + size_t(h) * VT_BIAS_BYTES,
                       VT_BIAS_BYTES, &st_full[st]);
        }
      }
    } else if (warp == 1) {
      // ---------------- MMA issuer: query tile gq = 4 unit + 2 e + t uses TMEM slot t; S(gq), then PV(gq - 1).  The whole warp walks
      // the loop converged and one elected lane issues: in divergent code every tcgen05.mma costs a six-instruction loop with a branch.
      constexpr uint32_t idesc_s = make_idesc(uint32_t(FMT), 128, 256);
      constexpr uint32_t idesc_o = make_idesc(uint32_t(FMT), 128, N32 ? 32 : 64) | (1u << 16);       // V' is MN-major
      constexpr uint32_t idesc_1 = make_idesc(uint32_t(FMT), 128, 16) | (1u << 16);
      const uint64_t onesd = fa_mnmajor_desc(base + VT_ONES_OFF);
      const int QT = 4 * total_units;
      for (int gq = 0; gq <= QT; ++gq) {
        if (gq < QT) {
          const int gp = gq >> 2, e = (gq >> 1) & 1, t = gq & 1;
          const uint32_t n = uint32_t(gq) >> 1;                      // this slot's n-th tile
          if ((gq & 3) == 0) mbar_wait(&st_full[gp & 1], (uint32_t(gp) >> 1) & 1u);
          mbar_wait(&o_empty[t], (n & 1u) ^ 1u);                     // E of the slot's previous tile has drained O'
          tc_fence_after();
          if (fa_elect_one()) {
            const uint32_t sb = base + uint32_t(gp & 1) * VT_STAGE;
            const uint64_t qd = make_sw128_kmajor_desc(sb + uint32_t(t) * 16384u) + uint64_t(4 * e);
            const uint64_t kd = make_sw128_kmajor_desc(sb + VT_TILE) + uint64_t(4 * e);
#pragma unroll
            for (int k = 0; k < 2; ++k)
              umma_ss<false>(tmem_base + uint32_t(t) * 256u, qd + uint64_t(2 * k), kd + uint64_t(2 * k), idesc_s, k ? 1u : 0u);
            umma_commit(&s_full[t]);
          }
          __syncwarp();
        }
        if (gq >= 1) {
          const int q = gq - 1, gp = q >> 2, t = q & 1, e = (q >> 1) & 1;
          const uint32_t n = uint32_t(q) >> 1;
          mbar_wait(&p_full[t], n & 1u);
          tc_fence_after();
          if (fa_elect_one()) {
            const uint32_t sb = base + uint32_t(gp & 1) * VT_STAGE;
            const uint64_t vd = fa_mnmajor_desc(sb + 2 * VT_TILE) + uint64_t(N32 ? 4 * e : 0);    // N32: head e's 32 columns, 64 bytes in
            const uint32_t slot = tmem_base + uint32_t(t) * 256u;
#pragma unroll
            for (int hf = 0; hf < 2; ++hf)
#pragma unroll
              for (int ks = 0; ks < 8; ++ks)     // 16 keys per step: 8 packed TMEM columns of P, 16 key rows (2048 B) of V'
                umma_ts(slot + 64u, slot + uint32_t(128 * hf + 8 * ks), vd + uint64_t(128 * (8 * hf + ks)), idesc_o, (hf | ks) ? 1u : 0u);
            if (ONES) {
#pragma unroll
              for (int hf = 0; hf < 2; ++hf)
#pragma unroll
                for (int ks = 0; ks < 8; ++ks)     // every column of this 16-column result = the row's sum of rounded probabilities
                  umma_ts(slot + 64u + (N32 ? 32u : 64u), slot + uint32_t(128 * hf + 8 * ks), onesd, idesc_1, (hf | ks) ? 1u : 0u);
            }
            umma_commit(&o_full[t]);
            if ((q & 3) == 3) umma_commit(&st_empty[gp & 1]);      // the unit's last P V: its stage may be reloaded
          }
          __syncwarp();
        }
      }
    }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 104;");
    // ---------------- softmax: set = query tile of the head = TMEM slot; hf = key half; thread = (row, half)
    const int sw = warp - 4;
    const int set = sw >> 3, hf = (sw >> 2) & 1, quad = warp & 3;
    const int r = quad * 32 + lane;
    const int i = set * 128 + r;                 // query slot in the window
    const int yi = i >> 4, xi = i & 15;
    const bool bf = FMT == 1;
    const uint32_t tslot = tmem_base + (uint32_t(quad * 32) << 16) + uint32_t(set) * 256u;
    const uint32_t ts = tslot + uint32_t(hf) * 128u;
    float* xmax = reinterpret_cast<float*>(smem + VT_XCH_OFF) + set * 256;
    float* xsum = xmax + 512;
    const int boff = (yi + 15 - 8 * hf) * VT_BROW + xi + 15;      // bias element of this half's first key (8 hf, 0)
    T16* ctx = static_cast<T16*>(p.ctx);
    const int nWy = p.g.H / p.g.ws;
    long long tok_off = 0;
    float madd_lo = 0.f, madd_hi = 0.f;
    bool masked = false;
    int cur_w = -1;
    const int total_tiles = 2 * total_units;
    int wg = u_begin / PAIRS, hp = u_begin - wg * PAIRS;      // (window, head pair) of the current unit, advanced without divisions
    // X2 is MUFU-bound and the two sets share the SM's MUFU pipes: they take turns (set 0 first), so that one set's exponentials
    // overlap the other's X1 / E / MMA round trips instead of both queueing on the same pipe and then idling together.
    if (set == 1) named_bar_arrive(3, 512);
    for (int n = 0; n < total_tiles; ++n) {
      const int gp = n >> 1, e = n & 1;
      const int h = 2 * hp + e;
      const uint32_t ph = uint32_t(n) & 1u;
      const uint8_t* sb = smem + size_t(gp & 1) * VT_STAGE;
      if (wg != cur_w) {      // where the row goes, and its shift-mask addends for the key columns x < 8 / x >= 8
        cur_w = wg;
        const int b = wg / p.nW, w = wg - b * p.nW;
        const long long row = p.token_order ? static_cast<long long>(b) * p.g.N + win_row_to_token(p.g, w * VT_L + i)
                                            : static_cast<long long>(wg) * VT_L + i;
        tok_off = row * C;
        const int wy = w / p.g.nWx, wx = w - wy * p.g.nWx;
        const bool lastrow = p.g.shift > 0 && wy == nWy - 1, lastcol = p.g.shift > 0 && wx == p.g.nWx - 1;
        masked = lastrow || lastcol;
        const bool ydiff = lastrow && ((yi < 8) != (hf == 0));
        madd_lo = (ydiff || (lastcol && xi >= 8)) ? p.mask_add : 0.0f;
        madd_hi = (ydiff || (lastcol && xi < 8)) ? p.mask_add : 0.0f;
      }
      long long* tr = (p.trace && blockIdx.x == 0 && lane == 0 && quad == 0 && n < VT_TRACE_TILES)
                          ? p.trace + ((set * 2 + hf) * VT_TRACE_TILES + n) * 8 : nullptr;
      VT_STAMP(0);
      if (e == 0) mbar_wait(&st_full[gp & 1], (uint32_t(gp) >> 1) & 1u);      // the bias tables (async-proxy writes) are visible
      const float* bt = reinterpret_cast<const float*>(sb + 3 * VT_TILE + e * VT_BIAS_BYTES) + boff;
      // ---- X1: biased logits, row max
      mbar_wait(&s_full[set], ph);
      tc_fence_after();
      VT_STAMP(1);
      float mx0 = -INFINITY, mx1 = -INFINITY;
      if (masked) vt_pass1<true>(ts, bt, madd_lo, madd_hi, mx0, mx1);
      else vt_pass1<false>(ts, bt, 0.f, 0.f, mx0, mx1);
      tmem_st_wait();
      float mx = fmaxf(mx0, mx1);
      xmax[hf * 128 + r] = mx;
      uint32_t va[32], vb[32], pk[16];
      tmem_ld_32x32(ts, va);                       // X2's first chunk travels while the halves exchange their maxima
      VT_STAMP(2);
      named_bar_sync(1 + set, 256);
      VT_STAMP(3);
      mx = fmaxf(mx, xmax[(hf ^ 1) * 128 + r]);
      // ---- X2: unnormalised probabilities, 16 bit, into TMEM over the consumed logits (two keys per column)
      float sum0 = 0.f, sum1 = 0.f;
      named_bar_sync(3 + set, 512);                // my turn on the MUFU pipes
      tmem_ld_wait();
      tmem_ld_32x32(ts + 32u, vb);
      vt_pass2_chunk<FMT, !ONES>(va, pk, mx, sum0, sum1);
      tmem_st_32x16(ts, pk);
      tmem_ld_wait();
      tmem_ld_32x32(ts + 64u, va);
      vt_pass2_chunk<FMT, !ONES>(vb, pk, mx, sum0, sum1);
      tmem_st_32x16(ts + 16u, pk);
      tmem_ld_wait();
      tmem_ld_32x32(ts + 96u, vb);
      vt_pass2_chunk<FMT, !ONES>(va, pk, mx, sum0, sum1);
      tmem_st_32x16(ts + 32u, pk);
      tmem_ld_wait();
      vt_pass2_chunk<FMT, !ONES>(vb, pk, mx, sum0, sum1);
      tmem_st_32x16(ts + 48u, pk);
      named_bar_arrive(4 - set, 512);              // the other set's turn (handing over a chunk earlier is slower: 36 vs 29 ns)
      tmem_st_wait();
      if (!ONES) xsum[hf * 128 + r] = sum0 + sum1;
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_full[set]);
      VT_STAMP(4);
      // ---- E: this half's 16 of the head's 32 output columns
      mbar_wait(&o_full[set], ph);
      tc_fence_after();
      uint32_t o[16], rs1 = 0;
      tmem_ld_32x16(tslot + 64u + uint32_t((N32 ? 0 : 32 * e) + 16 * hf), o);
      if (ONES) tmem_ld_32x1(tslot + 64u + (N32 ? 32u : 64u), rs1);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&o_empty[set]);
      VT_STAMP(5);
      if (h < HEADS && wg < p.num_windows) {
        const float inv = 1.0f / (ONES ? __uint_as_float(rs1) : xsum[r] + xsum[128 + r]);
        uint4* dst = reinterpret_cast<uint4*>(ctx + tok_off + h * 32 + 16 * hf);
#pragma unroll
        for (int q = 0; q < 2; ++q)
          dst[q] = make_uint4(pack16(bf, __uint_as_float(o[8 * q]) * inv, __uint_as_float(o[8 * q + 1]) * inv),
                              pack16(bf, __uint_as_float(o[8 * q + 2]) * inv, __uint_as_float(o[8 * q + 3]) * inv),
                              pack16(bf, __uint_as_float(o[8 * q + 4]) * inv, __uint_as_float(o[8 * q + 5]) * inv),
                              pack16(bf, __uint_as_float(o[8 * q + 6]) * inv, __uint_as_float(o[8 * q + 7]) * inv));
        if (LSE && hf == 0) p.lse2[(static_cast<long long>(wg) * HEADS + h) * VT_L + i] = mx + __log2f(__uint_as_float(rs1));
      }
      if (e == 1 && ++hp == PAIRS) { hp = 0; ++wg; }
    }
  }

  if (warp >= 4 && ((warp - 4) >> 3) == 0) named_bar_sync(3, 512);      // absorbs set 1's last hand-over
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

template <int FMT, int LSE>
static int launch_vt(const CUtensorMap& tmQ, const VtParams& p, cudaStream_t stream) {
  auto kern = swinv2_attn_tc_kernel<FMT, LSE>;
  CSVIT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(VT_SMEM)));
  const long long units = static_cast<long long>(p.num_windows) * ((p.heads + 1) / 2);
  const int ctas = units < num_sms() ? int(units) : num_sms();
  CSVIT_CUDA(launch_pdl(kern, dim3(ctas), dim3(VT_THREADS), VT_SMEM, stream, tmQ, p));
  return 0;
}

// qkv: 16-bit [B*nW*256, 3C] rows in window order (row pitch ldq elements), q and k cosine-normalised per head, q carrying
// log2(e) * logit_scale (csvit_swinv2_qkv).  bias_log2: fp32 [heads][31][48].
// lse2 (training forward): fp32 [B*nW][heads][256], written with window-ordered ctx; null = inference.
static int launch_vt_any(const void* qkv, long long ldq, const float* bias_log2, void* ctx, float* lse2, int dtype, int B, int H, int W,
                         int C, int heads, int shift, int mask_repeat, int token_order, cudaStream_t stream) {
  constexpr int ws = 16;
  CSVIT_REQUIRE(dtype == DT_BF16 || dtype == DT_F16, "swinv2_attn_tc: 16-bit operand formats only");
  CSVIT_REQUIRE(C == heads * 32 && heads >= 1, "swinv2_attn_tc: head_dim 32 only (C=%d heads=%d)", C, heads);
  CSVIT_REQUIRE(H % ws == 0 && W % ws == 0 && (shift == 0 || shift == 8), "swinv2_attn_tc: windows of 16, shift 0 or 8 (%dx%d shift %d)",
                H, W, shift);
  CSVIT_REQUIRE((reinterpret_cast<uintptr_t>(ctx) & 15) == 0 && (reinterpret_cast<uintptr_t>(bias_log2) & 15) == 0 && ldq >= 3ll * C,
                "swinv2_attn_tc: operands must be 16-byte aligned, pitch >= 3C");
  const int nW = (H / ws) * (W / ws);
  const long long windows = static_cast<long long>(B) * nW;
  if (windows <= 0) return 0;
  CSVIT_REQUIRE(windows * VT_L < (1ll << 31), "swinv2_attn_tc: too many rows");
  VtParams p{};
  p.trace = nullptr;
  p.lse2 = lse2;
  p.bias = bias_log2; p.ctx = ctx;
  p.num_windows = static_cast<int>(windows); p.nW = nW; p.C = C; p.heads = heads;
  p.token_order = token_order ? 1 : 0;
  p.mask_add = -100.0f * 1.4426950408889634f * static_cast<float>(mask_repeat);
  p.g = make_geom(H, W, ws, shift);
  CUtensorMap tmQ;
  if (int e = make_tmap(&tmQ, qkv, ldq, windows * VT_L, 3ll * C, dtype, VT_L, false)) return e;
  // CSVIT_V2_VAR (ablation): bit 0 = P V on the head's own 32 value columns, bit 1 = row sums from the tensor core
  const bool bf = dtype == DT_BF16;
  if (lse2) {
    CSVIT_REQUIRE((reinterpret_cast<uintptr_t>(lse2) & 15) == 0 && !token_order, "swinv2_attn_tc_train: lse2 16-byte aligned, window order");
    return bf ? launch_vt<1, 1>(tmQ, p, stream) : launch_vt<0, 1>(tmQ, p, stream);
  }
  static const char* trace_path = getenv("CSVIT_V2_TRACE");
  if (trace_path) {      // debugging: one traced launch, timestamps written as text
    const size_t nb = size_t(4) * VT_TRACE_TILES * 8 * sizeof(long long);
    CSVIT_CUDA(cudaMalloc(&p.trace, nb));
    CSVIT_CUDA(cudaMemsetAsync(p.trace, 0, nb, stream));
    int e = bf ? launch_vt<1, 0>(tmQ, p, stream) : launch_vt<0, 0>(tmQ, p, stream);
    if (e) { cudaFree(p.trace); return e; }
    CSVIT_CUDA(cudaStreamSynchronize(stream));
    std::vector<long long> h(nb / sizeof(long long));
    CSVIT_CUDA(cudaMemcpy(h.data(), p.trace, nb, cudaMemcpyDeviceToHost));
    cudaFree(p.trace);
    if (FILE* f = fopen(trace_path, "w")) {
      long long t0 = 0;
      for (long long v : h) if (v && (!t0 || v < t0)) t0 = v;
      fprintf(f, "# clock64 relative to the first stamp; rows: set hf tile | loop top, S ready, X1 done, max exchanged, P published, O read\n");
      for (int w = 0; w < 4; ++w)
        for (int n = 0; n < VT_TRACE_TILES; ++n) {
          fprintf(f, "%d %d %2d |", w >> 1, w & 1, n);
          for (int k = 0; k < 6; ++k) fprintf(f, " %8lld", h[(w * VT_TRACE_TILES + n) * 8 + k] ? h[(w * VT_TRACE_TILES + n) * 8 + k] - t0 : -1);
          fprintf(f, "\n");
        }
      fclose(f);
    }
    return 0;
  }
  return bf ? launch_vt<1, 0>(tmQ, p, stream) : launch_vt<0, 0>(tmQ, p, stream);
}

int launch_swinv2_attn_tc(const void* qkv, long long ldq, const float* bias_log2, void* ctx, int dtype, int B, int H, int W, int C,
                          int heads, int shift, int mask_repeat, int token_order, cudaStream_t stream) {
  return launch_vt_any(qkv, ldq, bias_log2, ctx, nullptr, dtype, B, H, W, C, heads, shift, mask_repeat, token_order, stream);
}

int launch_swinv2_attn_tc_train(const void* qkv, long long ldq, const float* bias_log2, void* ctx, float* lse2, int dtype, int B, int H,
                                int W, int C, int heads, int shift, int mask_repeat, cudaStream_t stream) {
  CSVIT_REQUIRE(lse2, "swinv2_attn_tc_train: null lse2");
  return launch_vt_any(qkv, ldq, bias_log2, ctx, lse2, dtype, B, H, W, C, heads, shift, mask_repeat, 0, stream);
}

}  // namespace csvit
