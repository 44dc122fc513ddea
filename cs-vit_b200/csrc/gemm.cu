// GEMM engine: persistent warp-specialised TMA + tcgen05/TMEM kernel (bf16 / fp16 / tf32 operands, fp32
// accumulate) and an exact-fp32 SIMT kernel used by the fp32 validation mode.
//
// Every Linear on the CS-ViT hot path goes through here: Swin Q/K/V, attention out-proj, MLP fc1/fc2, patch
// merging reduction, patch embedding (K1, K4, K10, K12, K13 of SURVEY.md §2.3) and the head's projections
// (K15-K18).  The reference runs each as an `addmm` (HF:swin/modeling_swin.py:404-406,479,514,527,347;
// ref:cs_vit/net/transformer_module.py:262-264,282,290-294).
#include <cudaTypedefs.h>

#include "errors.h"
#include <cstdlib>
#include "gemm.cuh"

namespace csvit {

// ----------------------------------------------------------------------------------------------------
// tcgen05 kernel
//   warp 0      : TMA producer (one elected lane)
//   warp 1      : MMA issuer   (one elected lane) - owns the TMEM allocation
//   warps 2..9  : epilogue, 2 warps per TMEM lane quadrant, each taking half of the tile's columns
// Pipelines: smem ring full/empty (TMA <-> MMA) and a 2-deep TMEM accumulator ring (MMA <-> epilogue), so
// the epilogue of tile i overlaps the MMAs of tile i+1.
//
// Cluster mode (CS = 2 or 4): the CS CTAs of a cluster work on CS consecutive 128-row blocks of the SAME
// column block, so they need the same weight tile.  Each CTA fetches 1/CS of it and TMA-multicasts the slice
// to all of them; L2 -> SM traffic per MMA drops from 48 KB to 16 + 32/CS KB per 128x256x64 step.  Measured
// without it (profiles/r1_gemm_baseline.md): the kernel ran at the L2 output cap (~10 TB/s), tensor pipe 42 %.
//
// Store path: 16-bit outputs with identity rows are converted in registers, staged in 128-byte-swizzled smem
// (bank-conflict free) and written by TMA (cp.async.bulk.tensor store) - full 128-byte lines instead of
// per-thread 16-byte fragments.  Residual / scatter epilogues keep direct stores: there each thread owns a
// whole 128-byte line of the fp32 residual stream.
// ----------------------------------------------------------------------------------------------------

template <int BN>
struct TcCfg {
  static constexpr int STAGES = BN == 256 ? 3 : 5;   // one stage traded for a second staging buffer per epilogue warp
  static constexpr uint32_t A_BYTES = kBM * 128;
  static constexpr uint32_t B_BYTES = BN * 128;
  static constexpr uint32_t STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr uint32_t TMEM_COLS = 2 * BN <= 256 ? 256 : 512;  // two accumulator buffers, power of 2
  static constexpr uint32_t TILES_BYTES = STAGES * STAGE_BYTES;
  static constexpr uint32_t STG_BYTES = 2 * kEpiWarps * kStageBufBytes;
  static constexpr size_t SMEM = 1024 + size_t(TILES_BYTES) + STG_BYTES + 256;
};

template <int BN, int FMT, int CS>  // FMT: 0 = fp16, 1 = bf16, 2 = tf32 operands (UMMA format codes)
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmC, const __grid_constant__ CUtensorMap tmR, int K, EpiParams ep) {
  using Cfg = TcCfg<BN>;
  constexpr bool TF32 = FMT == 2;
  constexpr int STAGES = Cfg::STAGES;
  constexpr int BK = TF32 ? 32 : 64;  // elements per 128-byte swizzled row
  constexpr uint16_t kMask = uint16_t((1u << CS) - 1u);
  constexpr int B_SLICE_ROWS = BN / CS;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
  uint8_t* tiles = smem;
  uint8_t* staging = smem + Cfg::TILES_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::TILES_BYTES + Cfg::STG_BYTES);
  uint64_t* full = bars;                     // [STAGES]
  uint64_t* empty = bars + STAGES;           // [STAGES]
  uint64_t* tfull = bars + 2 * STAGES;       // [2]
  uint64_t* tempty = bars + 2 * STAGES + 2;  // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);
  uint64_t* rbar = bars + 16;                // [kEpiWarps][2] residual-chunk arrivals (tma_f32 epilogue)

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int rank = CS > 1 ? int(cluster_ctarank()) : 0;
  const int cluster_id = blockIdx.x / CS;
  const int num_clusters = gridDim.x / CS;

  const int num_m = (ep.M + kBM - 1) / kBM;
  const int num_n = (ep.N + BN - 1) / BN;
  const int num_ctiles = ((num_m + CS - 1) / CS) * num_n;  // cluster tiles: CS row blocks x 1 column block
  const int num_kb = (K + BK - 1) / BK;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    if (ep.tma_store || ep.tma_f32) prefetch_tmap(&tmC);
    if (ep.tma_f32 && ep.resid) prefetch_tmap(&tmR);
    for (int i = 0; i < 2 * kEpiWarps; ++i) mbar_init(&rbar[i], 1);
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], CS); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], kEpiWarps); }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  if constexpr (CS > 1) cluster_sync_all();  // peers' barriers are initialised before any remote arrive / multicast
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  griddep_launch();      // PDL: the next kernel's prologue may overlap this kernel's tail ...
  griddep_wait();        // ... and this kernel touches global memory only after its predecessors have completed

  if (warp == 0) {
    // ---------------- TMA producer ----------------
    if (lane == 0) {
      int s = 0; uint32_t ph = 0;
      for (int ct = cluster_id; ct < num_ctiles; ct += num_clusters) {
        const int mg = ct / num_n, n_blk = ct - mg * num_n;
        const int m_blk = mg * CS + rank;  // may be >= num_m in the last group: TMA zero-fills, epilogue skips
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty[s], ph ^ 1u);   // every CTA of the cluster has consumed this slot
          mbar_arrive_expect_tx(&full[s], Cfg::STAGE_BYTES);
          uint8_t* sa = tiles + size_t(s) * Cfg::STAGE_BYTES;
          tma_load_2d(sa, &tmA, &full[s], kb * BK, m_blk * kBM);
          if constexpr (CS == 1) {
            tma_load_2d(sa + Cfg::A_BYTES, &tmB, &full[s], kb * BK, n_blk * BN);
          } else {
            tma_load_2d_mc(sa + Cfg::A_BYTES + rank * B_SLICE_ROWS * 128, &tmB, &full[s], kb * BK,
                           n_blk * BN + rank * B_SLICE_ROWS, kMask);
          }
          if (++s == STAGES) { s = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ---------------- MMA issuer (converged warp, one elected lane issues: see fa_elect_one) ----------------
    {
      constexpr uint32_t idesc = make_idesc(uint32_t(FMT), kBM, BN);
      int s = 0; uint32_t ph = 0;
      int as = 0; uint32_t aph = 0;
      for (int ct = cluster_id; ct < num_ctiles; ct += num_clusters) {
        mbar_wait(&tempty[as], aph ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + uint32_t(as * BN);
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full[s], ph);
          tc_fence_after();
          if (fa_elect_one()) {
            const uint32_t sa = base + uint32_t(s) * Cfg::STAGE_BYTES;
            const uint64_t adesc = make_sw128_kmajor_desc(sa);
            const uint64_t bdesc = make_sw128_kmajor_desc(sa + Cfg::A_BYTES);
#pragma unroll
            for (int k = 0; k < 4; ++k)  // 4 x 32-byte K slices per 128-byte row; +32 B = +2 in the >>4 field
              umma_ss<TF32>(d_tmem, adesc + uint64_t(2 * k), bdesc + uint64_t(2 * k), idesc, (kb | k) ? 1u : 0u);
            if constexpr (CS == 1) umma_commit(&empty[s]);
            else umma_commit_mc(&empty[s], kMask);   // release the slot in every CTA that multicasts into it
            if (kb == num_kb - 1) umma_commit(&tfull[as]);
          }
          __syncwarp();
          if (++s == STAGES) { s = 0; ph ^= 1u; }
        }
        if (++as == 2) { as = 0; aph ^= 1u; }
      }
    }
  } else {
    // ---------------- epilogue ----------------
    const int e = warp - 2;
    const int quad = warp & 3;            // TMEM lane quadrant this warp may read
    const int half = e >> 2;              // which half of the tile's columns
    uint8_t* stg = staging + e * 2 * kStageBufBytes;
    uint32_t stg_sel = 0, rph = 0;
    int as = 0; uint32_t aph = 0;
    for (int ct = cluster_id; ct < num_ctiles; ct += num_clusters) {
      const int mg = ct / num_n, n_blk = ct - mg * num_n;
      const int m_blk = mg * CS + rank;
      {
        const int nct = ct + num_clusters;
        if (ct == cluster_id) prefetch_resid_tile<BN>(ep, m_blk, n_blk, quad, half, lane);
        if (nct < num_ctiles) prefetch_resid_tile<BN>(ep, (nct / num_n) * CS + rank, nct % num_n, quad, half, lane);
      }
      epilogue_tile<BN>(ep, &tmC, stg, tmem_base + uint32_t(as * BN), &tfull[as], aph, m_blk, n_blk, quad, half, lane, 2, &stg_sel,
                        &tmR, rbar + 2 * e, &rph);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[as]);
      if (++as == 2) { as = 0; aph ^= 1u; }
    }
    if ((ep.tma_store || ep.tma_f32) && lane == 0) tma_store_wait_all();
  }

  tc_fence_before();
  __syncthreads();
  if constexpr (CS > 1) cluster_sync_all();  // no CTA exits while a peer may still multicast into it / signal it
  if (warp == 1) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
}

// ----------------------------------------------------------------------------------------------------
// Exact fp32 SIMT kernel (validation mode; also the on-device cross-check for the tensor-core path)
// ----------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
gemm_simt_f32_kernel(const float* __restrict__ A, long long lda, const float* __restrict__ W, long long ldw, int K, EpiParams ep) {
  __shared__ float As[16][64 + 4];
  __shared__ float Ws[16][64 + 4];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += 16) {
    for (int i = threadIdx.x; i < 64 * 16; i += 256) {
      int r = i >> 4, k = i & 15;
      int gm = m0 + r, gn = n0 + r, gk = k0 + k;
      As[k][r] = (gm < ep.M && gk < K) ? A[gm * lda + gk] : 0.0f;
      Ws[k][r] = (gn < ep.N && gk < K) ? W[gn * ldw + gk] : 0.0f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = As[k][ty * 4 + i]; b[i] = Ws[k][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int row = m0 + ty * 4 + i;
    if (row >= ep.M) continue;
    long long orow = epi_out_row(ep, row);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int col = n0 + tx * 4 + j;
      if (col < ep.N) epi_store_scalar(ep, orow, col, acc[i][j]);
    }
  }
}

// ----------------------------------------------------------------------------------------------------
// Host side
// ----------------------------------------------------------------------------------------------------
static PFN_cuTensorMapEncodeTiled_v12000 get_tmap_encoder() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  }
  return fn;
}

// rows x cols row-major tensor, box = box_rows x 128 bytes, 128-byte swizzle, OOB zero fill / clipping.
int make_tmap(CUtensorMap* tm, const void* ptr, long long ld, long long rows, long long cols, int dtype, int box_rows,
                     bool as_tf32) {
  auto enc = get_tmap_encoder();
  if (!enc) return set_error("cuTensorMapEncodeTiled entry point not available (driver too old?)");
  const size_t es = dtype_size(dtype);
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) || ((ld * es) & 15))
    return set_error("GEMM operand must be 16-byte aligned with a 16-byte-multiple row pitch (ptr=%p ld=%lld)", ptr, ld);
  cuuint64_t gdim[2] = {cuuint64_t(cols), cuuint64_t(rows)};
  cuuint64_t gstr[1] = {cuuint64_t(ld * es)};
  cuuint32_t box[2] = {cuuint32_t(128 / es), cuuint32_t(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapDataType tdt = dtype == DT_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                                  : (dtype == DT_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16
                                                     : (as_tf32 ? CU_TENSOR_MAP_DATA_TYPE_TFLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32));
  CUresult r = enc(tm, tdt, 2, const_cast<void*>(ptr), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%lld cols=%lld ld=%lld)", int(r), rows, cols, ld);
  return 0;
}

// 16-bit operand boxes of box_cols x box_rows with a 64-byte swizzle (box_cols = 32: one 32-column attention head per 64-byte row).
int make_tmap_sw64(CUtensorMap* tm, const void* ptr, long long ld, long long rows, long long cols, int dtype, int box_rows) {
  auto enc = get_tmap_encoder();
  if (!enc) return set_error("cuTensorMapEncodeTiled entry point not available (driver too old?)");
  if (dtype != DT_BF16 && dtype != DT_F16) return set_error("make_tmap_sw64: 16-bit operands only");
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) || ((ld * 2) & 15))
    return set_error("operand must be 16-byte aligned with a 16-byte-multiple row pitch (ptr=%p ld=%lld)", ptr, ld);
  cuuint64_t gdim[2] = {cuuint64_t(cols), cuuint64_t(rows)};
  cuuint64_t gstr[1] = {cuuint64_t(ld * 2)};
  cuuint32_t box[2] = {32u, cuuint32_t(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapDataType tdt = dtype == DT_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  CUresult r = enc(tm, tdt, 2, const_cast<void*>(ptr), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%lld cols=%lld ld=%lld)", int(r), rows, cols, ld);
  return 0;
}

// CSVIT_RED_ADD=0 keeps the load-add-store form of the in-place residual epilogue, 2 = reduce-add on the TMA path only (ablations)
int red_add_mode() {
  static const int m = [] { const char* e = getenv("CSVIT_RED_ADD"); return (e && e[0] >= '0' && e[0] <= '2') ? e[0] - '0' : 1; }();
  return m;
}
// CSVIT_TMA_F32=0 falls back to the register-staged fp32 epilogue (ablation)
static const bool g_tma_f32 = [] { const char* e = getenv("CSVIT_TMA_F32"); return !(e && e[0] == '0'); }();
static int g_num_sms = 0;
int num_sms() {
  if (!g_num_sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
    if (g_num_sms <= 0) g_num_sms = 148;
  }
  return g_num_sms;
}

template <int BN, int FMT, int CS>
static int launch_tc(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC, const CUtensorMap& tmR, int K,
                     const EpiParams& ep, int max_ctas, cudaStream_t stream) {
  using Cfg = TcCfg<BN>;
  static DeviceOnce once;
  auto kern = gemm_tc_kernel<BN, FMT, CS>;
  if (once.first()) {
    CSVIT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(Cfg::SMEM)));
  }
  const int num_m = (ep.M + kBM - 1) / kBM, num_n = (ep.N + BN - 1) / BN;
  const int ctiles = ((num_m + CS - 1) / CS) * num_n;
  int ctas = max_ctas > 0 ? max_ctas : num_sms();
  int clusters = ctas / CS;
  if (clusters > ctiles) clusters = ctiles;
  if (clusters < 1) clusters = 1;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(unsigned(clusters * CS));
  cfg.blockDim = dim3(kGemmThreads);
  cfg.dynamicSmemBytes = Cfg::SMEM;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CS;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;      // PDL, see errors.h::launch_pdl
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 2 : 1;
  CSVIT_CUDA(cudaLaunchKernelEx(&cfg, kern, tmA, tmB, tmC, tmR, K, ep));
  return 0;
}

template <int BN, int FMT>
static int launch_tc_cs(int cs, const CUtensorMap& a, const CUtensorMap& b, const CUtensorMap& c, const CUtensorMap& r, int K,
                        const EpiParams& ep, int max_ctas, cudaStream_t st) {
  if (cs == 4) return launch_tc<BN, FMT, 4>(a, b, c, r, K, ep, max_ctas, st);
  if (cs == 2) return launch_tc<BN, FMT, 2>(a, b, c, r, K, ep, max_ctas, st);
  return launch_tc<BN, FMT, 1>(a, b, c, r, K, ep, max_ctas, st);
}

static thread_local int g_last_gemm_kernel = 0;      // which kernel the last launch_gemm() of this thread chose (bench.py labels its roofline by it)
int last_gemm_kernel() { return g_last_gemm_kernel; }

int launch_gemm(const void* A, long long lda, const void* W, long long ldw, int in_dtype, int M, int N, int K,
                const EpiParams& ep_in, int impl, const GemmTuning& tune, cudaStream_t stream) {
  g_last_gemm_kernel = 0;
  if (M <= 0 || N <= 0 || K <= 0) return 0;
  EpiParams ep = ep_in;
  ep.M = M; ep.N = N;
  const size_t oes = dtype_size(ep.out_dtype);
  ep.vec_ok = (N % 8 == 0) && ((ep.ldo * oes) % 16 == 0) && ((reinterpret_cast<uintptr_t>(ep.out) & 15) == 0) &&
              (!ep.resid || ((ep.ldr % 4 == 0) && (reinterpret_cast<uintptr_t>(ep.resid) & 15) == 0)) &&
              (!ep.bias || (reinterpret_cast<uintptr_t>(ep.bias) & 15) == 0);
  ep.tma_store = 0;
  if (impl == GEMM_SIMT) {
    if (in_dtype != DT_F32) return set_error("SIMT GEMM takes fp32 operands only");
    dim3 grid((N + 63) / 64, (M + 63) / 64);
    gemm_simt_f32_kernel<<<grid, 256, 0, stream>>>(static_cast<const float*>(A), lda, static_cast<const float*>(W), ldw, K, ep);
    CSVIT_CUDA(cudaGetLastError());
    g_last_gemm_kernel = 3;
    return 0;
  }
  // Tile width: 256 halves the per-MMA shared-memory operand traffic; narrower tiles only where N is small
  // or 256 would leave most SMs idle.
  int BN = 256;
  if (N <= 128 || (N % 256 != 0 && N % 128 == 0)) BN = 128;
  const int num_m = (M + kBM - 1) / kBM;
  if (BN == 256 && num_m * ((N + 255) / 256) < num_sms()) BN = 128;
  // Cluster size: share the weight tile across row blocks when there are enough of them to keep every SM busy.
  int cs = tune.cluster;
  if (cs == 0) cs = 1;  // measured (profiles/r1_gemm_sweep.md): multicast does not help - the limit is per-SM ingest, not L2 output
  if (cs != 1 && cs != 2 && cs != 4) return set_error("gemm: cluster size %d not in {1,2,4}", cs);
  // TMA store: 16-bit output, plain rows, no residual, whole 64-column chunks.
  const bool can_tma_store = ep.out_dtype != DT_F32 && !ep.resid && ep.map_mode == ROWMAP_IDENTITY && (N % 64 == 0) &&
                             ep.vec_ok;
  ep.tma_store = (tune.tma_store != 0 && can_tma_store) ? 1 : 0;
  // fp32 output on identity rows: residual in / result out by TMA (32 x 32 fp32 boxes).  Scattered rows keep the register path.
  // Measured (tools/bench_gemm.py, out-proj shapes): 406 -> 475 TFLOP/s at N = 512, 749 -> 905 at N = 1024, but 157 -> 139 at
  // N = 128, where the register path already streams at the HBM rate and a tile has only two chunks per warp: N >= 256 only.
  ep.tma_f32 = (tune.tma_store != 0 && ep.out_dtype == DT_F32 && ep.map_mode == ROWMAP_IDENTITY && ep.vec_ok && (N % 32 == 0) && N >= 256 &&
                ((ep.ldo * 4) % 16 == 0) && (!ep.resid || (ep.ldr * 4) % 16 == 0) && g_tma_f32) ? 1 : 0;
  // In-place residual (x += A W^T + b: out-proj on token-ordered context, fc2): the tile leaves by TMA reduce-add (fp32 add in L2), the
  // residual stream never enters the SM - no residual TMA loads, no load -> add -> store chain on the two staging buffers per warp.
  ep.coalesced = (!ep.tma_store && !ep.tma_f32 && tune.tma_store != 0 && ep.out_dtype == DT_F32 && ep.vec_ok && (N % 32 == 0)) ? 1 : 0;
  // (the coalesced register path - scattered rows, N < 256 - does the same with red.global.add.v4.f32 instead of load + add + store)
  ep.red_add = 0;
  if ((ep.tma_f32 ? red_add_mode() != 0 : (ep.coalesced && red_add_mode() == 1)) && ep.resid && static_cast<const void*>(ep.resid) == ep.out &&
      ep.ldr == ep.ldo) {
    ep.red_add = 1;
    ep.resid = nullptr;
  }
  // CTA pairs (cta_group::2): 256x256 tiles with the weight tile split across the two SMs - a third less
  // shared-memory ingest per MMA than the single-CTA kernel, which is what bounds the large-K GEMMs.
  const bool pair_ok = in_dtype != DT_F32 && N % 256 == 0 && num_m * (N / 256) >= 2 * num_sms();
  if (pair_ok && tune.pair != 0) {
    g_last_gemm_kernel = 1;
    return launch_gemm_pair(A, lda, W, ldw, in_dtype, M, N, K, ep, tune, stream);
  }
  g_last_gemm_kernel = 2;
  CUtensorMap tmA, tmB, tmC, tmR;
  if (int e = make_tmap(&tmA, A, lda, M, K, in_dtype, kBM, true)) return e;
  if (int e = make_tmap(&tmB, W, ldw, N, K, in_dtype, BN / cs, true)) return e;
  if (ep.tma_store || ep.tma_f32) {
    if (int e = make_tmap(&tmC, ep.out, ep.ldo, M, N, ep.out_dtype, 32, false)) return e;
  } else {
    tmC = tmA;
  }
  tmR = tmC;
  if (ep.tma_f32 && ep.resid)
    if (int e = make_tmap(&tmR, ep.resid, ep.ldr, M, N, DT_F32, 32, false)) return e;
  const int mc = tune.max_ctas;
  if (BN == 256) {
    if (in_dtype == DT_F32) return launch_tc_cs<256, 2>(cs, tmA, tmB, tmC, tmR, K, ep, mc, stream);
    if (in_dtype == DT_BF16) return launch_tc_cs<256, 1>(cs, tmA, tmB, tmC, tmR, K, ep, mc, stream);
    return launch_tc_cs<256, 0>(cs, tmA, tmB, tmC, tmR, K, ep, mc, stream);
  }
  if (in_dtype == DT_F32) return launch_tc_cs<128, 2>(cs, tmA, tmB, tmC, tmR, K, ep, mc, stream);
  if (in_dtype == DT_BF16) return launch_tc_cs<128, 1>(cs, tmA, tmB, tmC, tmR, K, ep, mc, stream);
  return launch_tc_cs<128, 0>(cs, tmA, tmB, tmC, tmR, K, ep, mc, stream);
}

}  // namespace csvit
