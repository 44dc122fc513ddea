// CTA-pair GEMM: two CTAs of a cluster (one TPC) execute `tcgen05.mma.cta_group::2` on a 256 x 256 output tile.
//
// Why: the single-CTA kernel (gemm.cu) is bounded by bytes entering each SM's shared memory - a 128x256 tile
// needs 16 KB of A and 32 KB of W per 512 MMA cycles (96 B/clk), and multicasting W does not lower that
// (profiles/r1_gemm_sweep_cluster_tmastore.txt).  With a pair, each CTA holds its own 128 rows of A and only
// HALF of the 256-row weight tile; the MMA reads the two halves from both SMs.  Ingest per CTA drops to
// 16 + 16 KB per 512 cycles (64 B/clk) and the smem ring deepens from 4 to 5 stages.
//
// Protocol (rank 0 = leader):
//   full[s]   lives in the leader, count 2: each CTA's producer arms it (remote arrive.expect_tx) with its own
//             32 KB and issues its TMA loads with `.cta_group::2`, crediting the leader's barrier.
//   MMA       issued by the leader's elected thread only; `tcgen05.commit.cta_group::2` multicasts the arrival
//             to empty[s] (slot free) and tfull[a] (accumulator ready) of BOTH CTAs.
//   tempty[a] lives in the leader, count 2 * EPW: the epilogue warps of both CTAs arrive on it (remote for rank 1).
//   TMEM      allocated with cta_group::2 by the same warp of both CTAs; each CTA drains its own 128 lanes.
#include <cstdio>
#include <cstdlib>

#include "errors.h"
#include "gemm.cuh"

namespace csvit {

#ifdef CSVIT_PAIR_TRACE_BUILD
#define PAIR_STAMP(tr, k) do { if (tr) (tr)[k] = clock64(); } while (0)
#else
#define PAIR_STAMP(tr, k) do { } while (0)
#endif

constexpr int kPairBN = 256;
constexpr int kPairStages = 5;   // 6th stage traded for a second staging buffer per epilogue warp
constexpr uint32_t kPairABytes = kBM * 128;               // 128 rows x 128 B
constexpr uint32_t kPairBBytes = (kPairBN / 2) * 128;     // this CTA's half of the weight tile
constexpr uint32_t kPairStageBytes = kPairABytes + kPairBBytes;
constexpr uint32_t kPairTiles = kPairStages * kPairStageBytes;
constexpr uint32_t kPairStg = 2 * kEpiWarps * kStageBufBytes;      // 8 warps x 2 buffers, or 16 warps x 1 buffer (EPW = 16) of 4 KB
constexpr size_t kPairSmem = 1024 + size_t(kPairTiles) + kPairStg + 512;

// EPW = epilogue warps per CTA: 8 (every epilogue) or 16 (16-bit TMA-store outputs only - used for GELU at K <= 512: epilogue_tile16, one
// staging buffer per warp, no tail split)
template <int FMT, int EPW>  // FMT: 0 = fp16, 1 = bf16, 3 = E4M3 (kind::f8f6f4, 128 elements per 128-byte row, scaled epilogue)
__device__ __forceinline__ void gemm_pair_body(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmB2, const CUtensorMap& tmC,
                                               const CUtensorMap& tmR, int K, int split_tail, const EpiParams& ep) {
  constexpr bool F8 = FMT == 3;
  constexpr int BN = kPairBN, STAGES = kPairStages, BK = F8 ? 128 : 64;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
  uint8_t* tiles = smem;
  uint8_t* staging = smem + kPairTiles;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kPairTiles + kPairStg);
  uint64_t* full = bars;                     // [STAGES]  (used in the leader)
  uint64_t* empty = bars + STAGES;           // [STAGES]
  uint64_t* tfull = bars + 2 * STAGES;       // [2]
  uint64_t* tempty = bars + 2 * STAGES + 2;  // [2]       (used in the leader)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);
  uint64_t* rbar = bars + 2 * STAGES + 6;    // [kEpiWarps][2] residual-chunk arrivals (tma_f32 epilogue)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair_id = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;
  const int num_mp = (ep.M + 2 * kBM - 1) / (2 * kBM);
  const int num_n = (ep.N + BN - 1) / BN;
  const int num_ptiles = num_mp * num_n;
  const int num_kb = (K + BK - 1) / BK;
  // Tail split: after the full rounds (every pair the same number of 256 x 256 tiles) the `rem` left-over tiles would occupy rem of the
  // num_pairs pairs for a whole tile time.  When 2 rem <= num_pairs they run as 2 rem tiles of 256 x 128 instead (MMA N = 128, the
  // B box of tmB2 = 64 rows per CTA), one per pair: the last round costs half a tile time (Swin-B stage 2, N = 512: 5.3 -> 5.5 instead of 6 rounds).
  const int full_tiles = (num_ptiles / num_pairs) * num_pairs;
  const int rem = num_ptiles - full_tiles;
  const bool split = split_tail != 0 && rem > 0 && 2 * rem <= num_pairs;
  const int main_end = split ? full_tiles : num_ptiles;
  const bool has_half = split && pair_id < 2 * rem;
  const int half_pt = full_tiles + (pair_id >> 1), half_nh = pair_id & 1;      // this pair's half tile: tile half_pt, columns 128 half_nh ..

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    if (ep.tma_store || ep.tma_f32) prefetch_tmap(&tmC);
    if (ep.tma_f32 && ep.resid) prefetch_tmap(&tmR);
    for (int i = 0; i < 2 * kEpiWarps; ++i) mbar_init(&rbar[i], 1);
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 2); mbar_init(&empty[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], 2 * EPW); }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc_pair(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  griddep_launch();      // PDL: the next kernel's prologue may overlap this kernel's tail ...
  griddep_wait();        // ... and this kernel touches global memory only after its predecessors have completed

  if (warp == 0) {
    // ---------------- TMA producer (both CTAs) ----------------
    if (lane == 0) {
      int s = 0; uint32_t ph = 0;
      for (int pt = pair_id; pt < main_end; pt += num_pairs) {
        const int mp = pt / num_n, n_blk = pt - mp * num_n;
        const int m_blk = mp * 2 + int(rank);
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty[s], ph ^ 1u);
          const uint32_t lfull = mapa_u32(smem_u32(&full[s]), 0);
          mbar_arrive_expect_tx_cluster(lfull, kPairStageBytes);
          uint8_t* sa = tiles + size_t(s) * kPairStageBytes;
          tma_load_2d_pair(sa, &tmA, lfull, kb * BK, m_blk * kBM);
          tma_load_2d_pair(sa + kPairABytes, &tmB, lfull, kb * BK, n_blk * BN + int(rank) * (BN / 2));
          if (++s == STAGES) { s = 0; ph ^= 1u; }
        }
      }
      if (has_half) {
        const int mp = half_pt / num_n, n_blk = half_pt - mp * num_n;
        const int m_blk = mp * 2 + int(rank);
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty[s], ph ^ 1u);
          const uint32_t lfull = mapa_u32(smem_u32(&full[s]), 0);
          mbar_arrive_expect_tx_cluster(lfull, kPairABytes + kPairBBytes / 2);
          uint8_t* sa = tiles + size_t(s) * kPairStageBytes;
          tma_load_2d_pair(sa, &tmA, lfull, kb * BK, m_blk * kBM);
          tma_load_2d_pair(sa + kPairABytes, &tmB2, lfull, kb * BK, n_blk * BN + half_nh * (BN / 2) + int(rank) * (BN / 4));
          if (++s == STAGES) { s = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ---------------- MMA issuer (leader CTA only) ----------------
    if (rank == 0) {      // converged warp, one elected lane issues (see fa_elect_one)
      constexpr uint32_t idesc = make_idesc(F8 ? kE4M3 : uint32_t(FMT), 2 * kBM, BN);
      int s = 0; uint32_t ph = 0;
      int as = 0; uint32_t aph = 0;
      constexpr uint32_t idesc_half = make_idesc(F8 ? kE4M3 : uint32_t(FMT), 2 * kBM, BN / 2);
      const int rounds = (main_end - pair_id + num_pairs - 1) / num_pairs + (has_half ? 1 : 0);
      for (int it = 0; it < rounds; ++it) {
        const uint32_t idesc_t = (has_half && it == rounds - 1) ? idesc_half : idesc;
#ifdef CSVIT_PAIR_TRACE_BUILD
        long long* tr = (ep.trace && pair_id == 0 && lane == 0 && it < 32) ? ep.trace + it * 8 : nullptr;
#endif
        PAIR_STAMP(tr, 3);
        mbar_wait(&tempty[as], aph ^ 1u);
        tc_fence_after();
        PAIR_STAMP(tr, 4);
        const uint32_t d_tmem = tmem_base + uint32_t(as * BN);
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full[s], ph);
          tc_fence_after();
          if (fa_elect_one()) {
            const uint32_t sa = base + uint32_t(s) * kPairStageBytes;
            const uint64_t adesc = make_sw128_kmajor_desc(sa);
            const uint64_t bdesc = make_sw128_kmajor_desc(sa + kPairABytes);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              if constexpr (F8) umma_ss_pair_f8(d_tmem, adesc + uint64_t(2 * k), bdesc + uint64_t(2 * k), idesc_t, (kb | k) ? 1u : 0u);
              else umma_ss_pair(d_tmem, adesc + uint64_t(2 * k), bdesc + uint64_t(2 * k), idesc_t, (kb | k) ? 1u : 0u);
            }
            umma_commit_pair(&empty[s], 3);
            if (kb == num_kb - 1) umma_commit_pair(&tfull[as], 3);
          }
          __syncwarp();
          if (++s == STAGES) { s = 0; ph ^= 1u; }
        }
        PAIR_STAMP(tr, 5);
        if (++as == 2) { as = 0; aph ^= 1u; }
      }
    }
  } else {
    // ---------------- epilogue (both CTAs, own 128 TMEM lanes) ----------------
    const int e = warp - 2;
    const int quad = warp & 3;
    const int half = e >> 2;
    if constexpr (EPW == 16) {
      uint8_t* stg16 = staging + e * kStageBufBytes;
      int as = 0; uint32_t aph = 0;
      for (int pt = pair_id; pt < num_ptiles; pt += num_pairs) {
        const int mp = pt / num_n, n_blk = pt - mp * num_n;
        const int m_blk = mp * 2 + int(rank);
        epilogue_tile16<BN, F8>(ep, &tmC, stg16, tmem_base + uint32_t(as * BN), &tfull[as], aph, m_blk, n_blk, quad, half, lane);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(mapa_u32(smem_u32(&tempty[as]), 0));
        if (++as == 2) { as = 0; aph ^= 1u; }
      }
      if (lane == 0) tma_store_wait_all();
    } else {
    uint8_t* stg = staging + e * 2 * kStageBufBytes;
    uint32_t stg_sel = 0, rph = 0;
    int as = 0; uint32_t aph = 0;
    for (int pt = pair_id; pt < main_end; pt += num_pairs) {
      const int mp = pt / num_n, n_blk = pt - mp * num_n;
      const int m_blk = mp * 2 + int(rank);
      {
        const int npt = pt + num_pairs;
        if (pt == pair_id) prefetch_resid_tile<BN>(ep, m_blk, n_blk, quad, half, lane);
        if (npt < main_end) prefetch_resid_tile<BN>(ep, (npt / num_n) * 2 + int(rank), npt % num_n, quad, half, lane);
      }
#ifdef CSVIT_PAIR_TRACE_BUILD
      const int tidx = (pt - pair_id) / num_pairs;
      long long* tr = (ep.trace && pair_id == 0 && rank == 0 && e == 0 && lane == 0 && tidx < 32) ? ep.trace + tidx * 8 : nullptr;
      if (tr) { tr[0] = clock64(); mbar_wait(&tfull[as], aph); tr[1] = clock64(); }
#endif
      epilogue_tile<BN, F8>(ep, &tmC, stg, tmem_base + uint32_t(as * BN), &tfull[as], aph, m_blk, n_blk, quad, half, lane, 2, &stg_sel,
                            &tmR, rbar + 2 * e, &rph);
      tc_fence_before();
      __syncwarp();
      PAIR_STAMP(tr, 2);
      if (lane == 0) mbar_arrive_cluster(mapa_u32(smem_u32(&tempty[as]), 0));
      if (++as == 2) { as = 0; aph ^= 1u; }
    }
    if (has_half) {      // the 256 x 128 tail tile: the BN = 128 epilogue on column block 2 n_blk + half_nh (64 columns per warp)
      const int mp = half_pt / num_n, n_blk = half_pt - mp * num_n;
      const int m_blk = mp * 2 + int(rank);
      epilogue_tile<BN / 2, F8>(ep, &tmC, stg, tmem_base + uint32_t(as * BN), &tfull[as], aph, m_blk, 2 * n_blk + half_nh, quad, half, lane, 2,
                            &stg_sel, &tmR, rbar + 2 * e, &rph);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(mapa_u32(smem_u32(&tempty[as]), 0));
    }
    if ((ep.tma_store || ep.tma_f32) && lane == 0) tma_store_wait_all();
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 1) tmem_dealloc_pair(tmem_base, 512);
}

template <int FMT, int EPW>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__((2 + EPW) * 32, 1)
gemm_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmB2,
                 const __grid_constant__ CUtensorMap tmC, const __grid_constant__ CUtensorMap tmR, int K, int split_tail, EpiParams ep) {
  gemm_pair_body<FMT, EPW>(tmA, tmB, tmB2, tmC, tmR, K, split_tail, ep);
}
// The E4M3 instantiation under its own name (its SASS is told apart from the 16-bit kernels' by name).
template <int EPW>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__((2 + EPW) * 32, 1)
gemm_pair_fp8_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmB2,
                     const __grid_constant__ CUtensorMap tmC, const __grid_constant__ CUtensorMap tmR, int K, int split_tail, EpiParams ep) {
  gemm_pair_body<3, EPW>(tmA, tmB, tmB2, tmC, tmR, K, split_tail, ep);
}

template <int FMT, int EPW>
static int launch_pair(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmB2, const CUtensorMap& tmC, const CUtensorMap& tmR,
                       int K, int split_tail, const EpiParams& ep, int max_ctas, cudaStream_t stream) {
  static DeviceOnce once;
  auto kern = [] {
    if constexpr (FMT == 3) return gemm_pair_fp8_kernel<EPW>;
    else return gemm_pair_kernel<FMT, EPW>;
  }();
  if (once.first()) {
    CSVIT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kPairSmem)));
  }
  const int num_mp = (ep.M + 2 * kBM - 1) / (2 * kBM), num_n = (ep.N + kPairBN - 1) / kPairBN;
  int pairs = (max_ctas > 0 ? max_ctas : num_sms()) / 2;
  if (pairs > num_mp * num_n) pairs = num_mp * num_n;
  if (pairs < 1) pairs = 1;
  CSVIT_CUDA(launch_pdl(kern, dim3(pairs * 2), dim3((2 + EPW) * 32), kPairSmem, stream, tmA, tmB, tmB2, tmC, tmR, K, split_tail, ep));
  return 0;
}

int launch_gemm_pair(const void* A, long long lda, const void* W, long long ldw, int in_dtype, int M, int N, int K,
                     const EpiParams& ep_in, const GemmTuning& tune, cudaStream_t stream) {
  EpiParams ep = ep_in;
#ifdef CSVIT_PAIR_TRACE_BUILD
  static const char* trace_path = getenv("CSVIT_PAIR_TRACE");
  if (trace_path) { CSVIT_CUDA(cudaMalloc(&ep.trace, 32 * 8 * sizeof(long long))); CSVIT_CUDA(cudaMemsetAsync(ep.trace, 0, 32 * 8 * sizeof(long long), stream)); }
#endif
  CUtensorMap tmA, tmB, tmB2, tmC, tmR;
  if (int e = make_tmap(&tmA, A, lda, M, K, in_dtype, kBM, true)) return e;
  if (int e = make_tmap(&tmB, W, ldw, N, K, in_dtype, kPairBN / 2, true)) return e;
  if (int e = make_tmap(&tmB2, W, ldw, N, K, in_dtype, kPairBN / 4, true)) return e;      // the tail's 256 x 128 tiles: 64 weight rows per CTA
  static const int split_tail = [] { const char* e = getenv("CSVIT_PAIR_TAIL"); return (e && e[0] == '0') ? 0 : 1; }();
  if (ep.tma_store || ep.tma_f32) {
    if (int e = make_tmap(&tmC, ep.out, ep.ldo, M, N, ep.out_dtype, 32, false)) return e;
  } else {
    tmC = tmA;
  }
  tmR = tmC;
  if (ep.tma_f32 && ep.resid)
    if (int e = make_tmap(&tmR, ep.resid, ep.ldr, M, N, DT_F32, 32, false)) return e;
  // CSVIT_PAIR_EPW=8: the 8-warp epilogue for the GELU outputs too; =16: sixteen warps for every 16-bit store (ablations)
  static const int epw = [] { const char* e = getenv("CSVIT_PAIR_EPW"); return e ? atoi(e) : 0; }();
  const bool epw16 = ep.tma_store && epw != 8 && (epw == 16 || (ep.act == ACT_GELU && K <= 512));
  int rc;
  if (in_dtype == DT_E4M3)
    rc = epw16 ? launch_pair<3, 16>(tmA, tmB, tmB2, tmC, tmR, K, 0, ep, tune.max_ctas, stream)
               : launch_pair<3, 8>(tmA, tmB, tmB2, tmC, tmR, K, split_tail, ep, tune.max_ctas, stream);
  else if (epw16)
    rc = in_dtype == DT_BF16 ? launch_pair<1, 16>(tmA, tmB, tmB2, tmC, tmR, K, 0, ep, tune.max_ctas, stream)
                             : launch_pair<0, 16>(tmA, tmB, tmB2, tmC, tmR, K, 0, ep, tune.max_ctas, stream);
  else
    rc = in_dtype == DT_BF16 ? launch_pair<1, 8>(tmA, tmB, tmB2, tmC, tmR, K, split_tail, ep, tune.max_ctas, stream)
                             : launch_pair<0, 8>(tmA, tmB, tmB2, tmC, tmR, K, split_tail, ep, tune.max_ctas, stream);
#ifdef CSVIT_PAIR_TRACE_BUILD
  if (trace_path && rc == 0) {      // one traced launch written as text (cycles relative to the issuer's first stamp)
    CSVIT_CUDA(cudaStreamSynchronize(stream));
    long long h[32 * 8];
    CSVIT_CUDA(cudaMemcpy(h, ep.trace, sizeof(h), cudaMemcpyDeviceToHost));
    cudaFree(ep.trace);
    if (FILE* f = fopen(trace_path, "a")) {
      fprintf(f, "# gemm_pair M=%d N=%d K=%d act=%d: pair 0; per tile: issuer [wait tempty | issue all k-blocks], epilogue warp 0 [wait tfull | work]\n", M, N, K, ep.act);
      const long long t0 = h[3];
      for (int t = 0; t < 32; ++t) {
        const long long* r = h + t * 8;
        if (!r[5]) continue;
        fprintf(f, "tile %2d  issuer start %7lld wait %5lld issue %5lld | epilogue ready %7lld wait %5lld work %5lld done %7lld", t, r[3] - t0, r[4] - r[3], r[5] - r[4],
                r[0] - t0, r[1] - r[0], r[2] - r[1], r[2] - t0);
        if (r[7]) fprintf(f, "  (16 warps: staging wait %lld, TMEM load wait %lld, arithmetic + store %lld)", r[6] - r[1], r[7] - r[6], r[2] - r[7]);
        fprintf(f, "\n");
      }
      fclose(f);
    }
  }
#endif
  return rc;
}

}  // namespace csvit
