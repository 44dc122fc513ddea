// Backward of the SwinV2 cosine normalisation that csvit_swinv2_qkv_train folds into the Q/K/V GEMM epilogue (V2:450-455):
//   q2 = q / |q| * qs[h],  k_hat = k / |k|,  v unchanged    ->    dqkv [rows, 3C] = dq | dk | dv,  dqs[h] += sum_rows q_hat . dq2
// with q_hat = q2 / qs[h] and 1 / |q|, 1 / |k| taken from the forward's rnorm.  HBM-bound: per row it reads the 2C 16-bit values of
// q2 | k_hat, the 3C of the incoming gradients and 2C / 32 floats of rnorm, and writes 3C 16-bit values - one pass, fp32 arithmetic.
#include "errors.h"
#include "gemm.cuh"
#include "rowops.cuh"

namespace csvit {

template <typename T>
__device__ __forceinline__ void load8(const T* p, float (&f)[8]) {
  const uint4 u = __ldg(reinterpret_cast<const uint4*>(p));
  const T* h = reinterpret_cast<const T*>(&u);
#pragma unroll
  for (int j = 0; j < 8; ++j) f[j] = Half16<T>::to(h[j]);
}

template <typename T>
__device__ __forceinline__ void store8(T* p, const float (&f)[8]) {
  *reinterpret_cast<uint4*>(p) = make_uint4(Half16<T>::pack(f[0], f[1]), Half16<T>::pack(f[2], f[3]), Half16<T>::pack(f[4], f[5]),
                                            Half16<T>::pack(f[6], f[7]));
}

// A CTA is R rows x (C / 8) threads; thread x of a row owns columns [8x, 8x + 8) of q, k and v, so four consecutive lanes hold one
// 32-wide head and its dot products are two shuffles.  The thread's head never changes, so its share of dqs stays in a register over
// the grid-stride loop and meets the CTA's other rows once in shared memory: one red.global.add per head and CTA.
template <typename T>
__global__ void __launch_bounds__(256)
swinv2_cosnorm_bwd_kernel(const T* __restrict__ qkv, const float* __restrict__ rnorm, const float* __restrict__ qs,
                          const T* __restrict__ dq2, const T* __restrict__ dk, const T* __restrict__ dv, T* __restrict__ dqkv,
                          float* __restrict__ dqs, int rows, int C, int R) {
  extern __shared__ float s_dqs[];
  const int cpr = C >> 3, heads = C >> 5;
  const int x = threadIdx.x % cpr, ry = threadIdx.x / cpr, h = x >> 2;
  const unsigned lanes = __activemask();      // the last warp is partial when R * C / 8 is not a multiple of 32 (C = 96)
  for (int i = threadIdx.x; i < heads; i += blockDim.x) s_dqs[i] = 0.f;
  __syncthreads();
  const float s = __ldg(qs + h), inv_s = 1.0f / s;
  float acc = 0.f;
  const int nblk = (rows + R - 1) / R;
  for (int rb = blockIdx.x; rb < nblk; rb += gridDim.x) {      // uniform trip count across the CTA: the shuffles see every lane
    const long long r = static_cast<long long>(rb) * R + ry;
    const bool ok = r < rows;
    float q[8], k[8], gq[8], gk[8];
    uint4 v = make_uint4(0, 0, 0, 0);
    float rq = 0.f, rk = 0.f;
    if (ok) {
      const T* src = qkv + r * 3 * C + 8 * x;
      const long long g = r * C + 8 * x;
      load8(src, q);
      load8(src + C, k);
      load8(dq2 + g, gq);
      load8(dk + g, gk);
      v = __ldg(reinterpret_cast<const uint4*>(dv + g));
      rq = __ldg(rnorm + r * 2 * heads + h);
      rk = __ldg(rnorm + r * 2 * heads + heads + h);
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) q[j] = k[j] = gq[j] = gk[j] = 0.f;
    }
    float dotq = 0.f, dotk = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      q[j] *= inv_s;
      dotq = fmaf(q[j], gq[j], dotq);
      dotk = fmaf(k[j], gk[j], dotk);
    }
    dotq += __shfl_xor_sync(lanes, dotq, 1);
    dotk += __shfl_xor_sync(lanes, dotk, 1);
    dotq += __shfl_xor_sync(lanes, dotq, 2);
    dotk += __shfl_xor_sync(lanes, dotk, 2);
    acc += dotq;
    if (ok) {
      const float sq = rq * s;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        gq[j] = sq * fmaf(-q[j], dotq, gq[j]);
        gk[j] = rk * fmaf(-k[j], dotk, gk[j]);
      }
      T* dst = dqkv + r * 3 * C + 8 * x;
      store8(dst, gq);
      store8(dst + C, gk);
      *reinterpret_cast<uint4*>(dst + 2 * C) = v;
    }
  }
  if ((x & 3) == 0) atomicAdd(&s_dqs[h], acc);
  __syncthreads();
  for (int i = threadIdx.x; i < heads; i += blockDim.x) atomicAdd(dqs + i, s_dqs[i]);
}

int launch_swinv2_cosnorm_bwd(const void* qkv, const float* rnorm, const float* qscale_log2, const void* dq2, const void* dk,
                              const void* dv, void* dqkv, float* dqscale, int dtype, int rows, int C, cudaStream_t stream) {
  if (rows <= 0) return 0;
  const int cpr = C / 8;
  const int R = cpr >= 256 ? 1 : 256 / cpr;
  const int threads = R * cpr;
  const int nblk = (rows + R - 1) / R;
  const int resident = num_sms() * (1024 / threads);      // 61-64 registers a thread: four CTAs of 256 threads per SM
  const int grid = nblk < resident ? nblk : resident;
  const size_t smem = sizeof(float) * (C / 32);
  if (dtype == DT_BF16) {
    swinv2_cosnorm_bwd_kernel<__nv_bfloat16><<<grid, threads, smem, stream>>>(
        static_cast<const __nv_bfloat16*>(qkv), rnorm, qscale_log2, static_cast<const __nv_bfloat16*>(dq2),
        static_cast<const __nv_bfloat16*>(dk), static_cast<const __nv_bfloat16*>(dv), static_cast<__nv_bfloat16*>(dqkv), dqscale, rows,
        C, R);
  } else {
    swinv2_cosnorm_bwd_kernel<__half><<<grid, threads, smem, stream>>>(
        static_cast<const __half*>(qkv), rnorm, qscale_log2, static_cast<const __half*>(dq2), static_cast<const __half*>(dk),
        static_cast<const __half*>(dv), static_cast<__half*>(dqkv), dqscale, rows, C, R);
  }
  CSVIT_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace csvit
