// Shared device helpers for the CS-ViT sm_100a kernels: PTX wrappers (mbarrier, TMA, tcgen05/TMEM),
// the closed-form Swin index maps, and small numeric utilities.
//
// Index maps restate SURVEY.md §8(a) "closed-form integer maps" (verified there against
// HF:swin/modeling_swin.py:141-160 window_partition/window_reverse, :615-616/:635-636 torch.roll and
// :556-582 get_attn_mask); they are the single source of truth for every kernel in this library and for
// the csvit_*_map test entry points, so the bit-exact tests exercise exactly what the hot path uses.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace csvit {

// ----------------------------------------------------------------------------------------------------
// Swin index maps
// ----------------------------------------------------------------------------------------------------
struct WinGeom {
  int H, W;    // token grid of one image
  int ws;      // window side (7)
  int shift;   // cyclic shift (0 or ws/2)
  int nWx;     // windows per row
  int L;       // tokens per window (ws*ws)
  int N;       // tokens per image (H*W)
};

__host__ __device__ inline WinGeom make_geom(int H, int W, int ws, int shift) {
  WinGeom g;
  g.H = H; g.W = W; g.ws = ws; g.shift = shift;
  g.nWx = W / ws; g.L = ws * ws; g.N = H * W;
  return g;
}

// Row r of the window-ordered token stream (r = w*L + i within one image) -> flat token id y*W + x of the
// un-shifted, un-partitioned image.  The same address serves the gather (LN -> roll(-s) -> partition) and
// the scatter (reverse -> roll(+s)), so the residual add is in place.
__host__ __device__ inline int win_row_to_token(const WinGeom& g, int r) {
  int w = r / g.L, i = r - w * g.L;
  int wy = w / g.nWx, wx = w - wy * g.nWx;
  int iy = i / g.ws, ix = i - iy * g.ws;
  int y = wy * g.ws + iy + g.shift; if (y >= g.H) y -= g.H;
  int x = wx * g.ws + ix + g.shift; if (x >= g.W) x -= g.W;
  return y * g.W + x;
}

// Inverse of win_row_to_token: flat token id -> row of the window-ordered stream.
__host__ __device__ inline int win_token_to_row(const WinGeom& g, int t) {
  int y = t / g.W, x = t - y * g.W;
  int ys = y - g.shift; if (ys < 0) ys += g.H;
  int xs = x - g.shift; if (xs < 0) xs += g.W;
  int wy = ys / g.ws, wx = xs / g.ws;
  return (wy * g.nWx + wx) * g.L + (ys - wy * g.ws) * g.ws + (xs - wx * g.ws);
}

// Shift-mask region id of slot i in window w, on SHIFTED coordinates (HF get_attn_mask slices).
__host__ __device__ inline int win_region(const WinGeom& g, int w, int i) {
  int wy = w / g.nWx, wx = w - wy * g.nWx;
  int iy = i / g.ws, ix = i - iy * g.ws;
  int p = wy * g.ws + iy, q = wx * g.ws + ix;
  int rp = p < g.H - g.ws ? 0 : (p < g.H - g.shift ? 1 : 2);
  int rq = q < g.W - g.ws ? 0 : (q < g.W - g.shift ? 1 : 2);
  return 3 * rp + rq;
}

// relative_position_index[i][j] for a ws x ws window (HF create_relative_position_index).
__host__ __device__ inline int rel_pos_index(int ws, int i, int j) {
  int iy = i / ws, ix = i - iy * ws, jy = j / ws, jx = j - jy * ws;
  return (iy - jy + ws - 1) * (2 * ws - 1) + (ix - jx + ws - 1);
}

// Patch merging: output token (Y,X), quadrant q in concat order (0,0),(1,0),(0,1),(1,1)
// (HF:swin/modeling_swin.py:338-345) -> source token of the H x W grid.
__host__ __device__ inline int merge_src_token(int W, int Y, int X, int q) {
  int dy = q & 1, dx = q >> 1;
  return (2 * Y + dy) * W + (2 * X + dx);
}

// ----------------------------------------------------------------------------------------------------
// Numerics
// ----------------------------------------------------------------------------------------------------
__device__ __forceinline__ float gelu_erf(float x) {
  // exact-erf GELU, as nn.GELU() / HF "gelu" (HF:swin/modeling_swin.py:510-519)
  return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f));
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
  __half2 v = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
// 16-bit operand formats of the tensor-core path: bf16 (8-bit mantissa) and fp16 (11-bit mantissa, same MMA rate).
template <typename T> struct Half16;
template <> struct Half16<__nv_bfloat16> {
  static __device__ __forceinline__ uint32_t pack(float lo, float hi) { return pack_bf16x2(lo, hi); }
  static __device__ __forceinline__ __nv_bfloat16 from(float v) { return __float2bfloat16_rn(v); }
  static __device__ __forceinline__ float to(__nv_bfloat16 v) { return __bfloat162float(v); }
};
template <> struct Half16<__half> {
  static __device__ __forceinline__ uint32_t pack(float lo, float hi) { return pack_f16x2(lo, hi); }
  static __device__ __forceinline__ __half from(float v) { return __float2half_rn(v); }
  static __device__ __forceinline__ float to(__half v) { return __half2float(v); }
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ----------------------------------------------------------------------------------------------------
// PTX: shared-memory addresses, mbarrier, TMA, tcgen05
// ----------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// Non-blocking probe (try_wait may suspend the thread for a hardware time slice; event loops that poll several barriers use this).
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must surface as a CUDA error (trap), never as a hung GPU.  try_wait suspends the thread for a
// hardware time slice per attempt, so the attempt counter bounds the wait to seconds; no timer reads or printf at the ~30 wait
// sites of the warp-specialised kernels (instruction-cache footprint).
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 26)) __trap();
  }
}

__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* t) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(t)) : "memory");
}
// 2-D tiled TMA load global -> shared, completion on an mbarrier (bytes of the full box, OOB zero-filled).
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar, int x, int y) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(x), "r"(y)
      : "memory");
}

// Same, delivered to the same shared-memory offset of every CTA in `cta_mask` (each CTA's own mbarrier at
// that offset receives the complete_tx): one L2 read feeds the whole cluster.
__device__ __forceinline__ void tma_load_2d_mc(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar, int x, int y, uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(x), "r"(y), "h"(cta_mask)
      : "memory");
}
// 2-D tiled TMA store shared -> global (bulk async group; OOB rows/cols are clipped).
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* tmap, const void* smem_src, int x, int y) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(smem_src)), "r"(x), "r"(y) : "memory");
}
// The same as a reduction: global[box] += shared[box] (element type of the tensor map, here fp32), performed in L2 - the result tile of an
// in-place residual GEMM (x += A W^T + b) leaves this way, so the residual stream is never loaded into the SM.
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* tmap, const void* smem_src, int x, int y) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(smem_src)), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ void red_add_f32x4(float* p, float4 v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// Programmatic dependent launch (errors.h::launch_pdl): let the next kernel of the stream be scheduled / wait until every kernel
// before this one has completed and its writes are visible.  No-ops for kernels launched without the attribute.
#ifdef CSVIT_PDL_NO_TRIGGER      // experiment: no early trigger - the dependent kernel is released as this kernel's CTAs exit
__device__ __forceinline__ void griddep_launch() {}
#else
__device__ __forceinline__ void griddep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#endif
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// One lane of a CONVERGED warp.  The MMA issuers walk their loops with the whole warp and issue under this predicate: ptxas then emits
// back-to-back UTCHMMA, whereas under `lane == 0` (divergent code) every tcgen05.mma becomes a six-instruction loop with a branch.
__device__ __forceinline__ bool fa_elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// D[tmem] (+)= A[smem] * B[smem]; kind::f16 covers bf16/fp16 inputs, kind::tf32 covers fp32-as-tf32.
template <bool kTF32>
__device__ __forceinline__ void umma_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  if constexpr (kTF32) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}
// The same with 8-bit operands (kind::f8f6f4, here E4M3 x E4M3 per make_idesc(kE4M3, ...)): one MMA consumes K = 32 elements,
// the same 32 bytes of each 128-byte swizzled row as one kind::f16 MMA, so the descriptors advance exactly as for 16-bit operands.
__device__ __forceinline__ void umma_ss_f8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier once every tcgen05.mma previously issued by this thread has completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// Same arrive, delivered to the mbarrier at this shared-memory offset in every CTA of `cta_mask`.
__device__ __forceinline__ void umma_commit_mc(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"(cta_mask) : "memory");
}

// ---- CTA-pair (cta_group::2) forms: two CTAs of a cluster act as one 256-row MMA ------------------------
// Address of the same shared-memory variable in CTA `rank` of the cluster (shared::cluster window).
__device__ __forceinline__ uint32_t mapa_u32(uint32_t smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_expect_tx_cluster(uint32_t cluster_bar_addr, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cluster.b64 _, [%0], %1;" ::"r"(cluster_bar_addr), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_bar_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar_addr) : "memory");
}
// TMA load into THIS CTA's shared memory whose completion bytes are credited to an mbarrier that may live in
// the peer CTA (cluster address), as the leader CTA's MMA thread waits for both halves on one barrier.
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* tmap, uint32_t cluster_bar_addr, int x, int y) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(cluster_bar_addr), "r"(x), "r"(y)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs] (+)= A[128 rows in each CTA's smem] * B[N/2 rows in each CTA's smem]; leader CTA issues.
__device__ __forceinline__ void umma_ss_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_ss_pair_f8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"(cta_mask) : "memory");
}

// TMEM -> registers: this warp's 32 lanes x 32 consecutive fp32 columns (thread t <- lane base+t).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, 128-byte-swizzled shared-memory operand descriptor (sm_100 "version 1").
// Rows are 128 B (64 bf16 / 32 tf32), 8-row swizzle atoms of 1024 B stacked along M/N: SBO = 1024 B,
// LBO unused for swizzled K-major (encoded 1), layout type 2 = SWIZZLE_128B.
__device__ __forceinline__ uint64_t make_sw128_kmajor_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);  // start address, bits [0,14)
  d |= static_cast<uint64_t>(1) << 16;                        // leading byte offset (ignored)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;                // stride byte offset, bits [32,46)
  d |= static_cast<uint64_t>(1) << 46;                        // descriptor version (Blackwell)
  d |= static_cast<uint64_t>(2) << 61;                        // SWIZZLE_128B
  return d;
}

// Instruction descriptor for kind::f16 / kind::tf32 / kind::f8f6f4, fp32 accumulate, both operands K-major.  The a/b format fields are
// interpreted by the instruction's kind (PTX ISA, tcgen05 instruction descriptor): under kind::f16 0 = F16, 1 = BF16; under kind::tf32
// 2 = TF32; under kind::f8f6f4 0 = E4M3, 1 = E5M2, 3 = E2M3, 4 = E3M2, 5 = E2M1.
constexpr uint32_t kE4M3 = 0;
__host__ __device__ constexpr uint32_t make_idesc(uint32_t fmt, int M, int N) {
  return (1u << 4)                 // c_format = F32
         | (fmt << 7)              // a_format
         | (fmt << 10)             // b_format
         | (0u << 15) | (0u << 16) // a_major, b_major = K
         | (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}

}  // namespace csvit
