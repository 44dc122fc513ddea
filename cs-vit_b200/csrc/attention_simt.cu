// Exact-fp32 dense attention for short sequences (<= 128 keys, head_dim 32): the CS-ViT head's MHA
// (ref:cs_vit/net/transformer_module.py:250-282), whose logits are MULTIPLIED by sqrt(head_dim) (line 273,
// quirk Q1: near-argmax softmax, kept in fp32 on purpose), and the fp32 validation mode of the Swin window
// attention (bias table + closed-form shift mask).
#include "errors.h"
#include "rowops.cuh"

namespace csvit {

// ----------------------------------------------------------------------------------------------------
// (2) exact fp32 dense attention for short sequences
// ----------------------------------------------------------------------------------------------------
template <typename T> __device__ __forceinline__ float to_f(T v);
template <> __device__ __forceinline__ float to_f<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <> __device__ __forceinline__ float to_f<__half>(__half v) { return __half2float(v); }
template <typename T> __device__ __forceinline__ T from_f(float v);
template <> __device__ __forceinline__ float from_f<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ __half from_f<__half>(float v) { return __float2half_rn(v); }

constexpr int SA_MAXS = 128;   // 3 query tokens + 64 patches of a 256^2 SwinV2 backbone = 67 keys in the "encoder" head
constexpr int SA_KPL = SA_MAXS / 32;   // keys per lane
constexpr int SA_HD = 32;

// One CTA (4 warps) per (sequence, head); warp per query row, lane per key (up to SA_KPL keys per lane).
template <typename T>
__global__ void __launch_bounds__(128)
attention_simt_kernel(const T* __restrict__ q, const T* __restrict__ k, const T* __restrict__ v, T* __restrict__ out,
                      long long ldq, long long ldk, long long ldv, long long ldo, int num_items, int Lq, int S, int heads,
                      float scale, const float* __restrict__ bias, WinGeom g, int nW, const int* __restrict__ key_start) {
  __shared__ float Ks[SA_MAXS][SA_HD + 1];
  __shared__ float Vs[SA_MAXS][SA_HD + 1];
  __shared__ float Qs[4][SA_HD];
  __shared__ float Ps[4][SA_MAXS];
  __shared__ int region_s[SA_MAXS];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int item = blockIdx.x; item < num_items; item += gridDim.x) {
    const int h = item % heads, seq = item / heads;
    // Ragged keys: this sequence sees rows [seq*S + k0, seq*S + S) only.  Valid key j goes to shared row j, so everything
    // below runs exactly as a plain call with Sv = S - k0 keys would (same lanes, same shuffles, same P.V order).
    const int k0 = key_start ? min(max(__ldg(key_start + seq), 0), S - 1) : 0;
    const int Sv = S - k0;
    const long long krow0 = static_cast<long long>(seq) * S + k0;
    __syncthreads();
    for (int idx = tid; idx < Sv * SA_HD; idx += 128) {
      int r = idx >> 5, d = idx & 31;
      Ks[r][d] = to_f<T>(k[(krow0 + r) * ldk + h * SA_HD + d]);
      Vs[r][d] = to_f<T>(v[(krow0 + r) * ldv + h * SA_HD + d]);
    }
    if (tid < SA_MAXS) region_s[tid] = (g.shift > 0 && tid < S) ? win_region(g, seq % nW, tid) : 0;
    __syncthreads();
    for (int i = warp; i < Lq; i += 4) {
      Qs[warp][lane] = to_f<T>(q[(static_cast<long long>(seq) * Lq + i) * ldq + h * SA_HD + lane]);
      __syncwarp();
      float sc[SA_KPL];
#pragma unroll
      for (int t = 0; t < SA_KPL; ++t) {
        const int j = lane + 32 * t;
        float a = -INFINITY;
        if (j < Sv) {
          a = 0.f;
#pragma unroll
          for (int d = 0; d < SA_HD; ++d) a = fmaf(Qs[warp][d], Ks[j][d], a);
          a *= scale;
          if (bias) a += __ldg(bias + (static_cast<long long>(h) * Lq + i) * S + j);
          if (g.shift > 0 && region_s[j] != region_s[i]) a += -100.0f;
        }
        sc[t] = a;
      }
      float mx = sc[0];
#pragma unroll
      for (int t = 1; t < SA_KPL; ++t) mx = fmaxf(mx, sc[t]);
      mx = warp_max(mx);
      float esum = 0.f;
#pragma unroll
      for (int t = 0; t < SA_KPL; ++t) {
        sc[t] = lane + 32 * t < Sv ? expf(sc[t] - mx) : 0.f;
        esum += sc[t];
      }
      const float inv = 1.0f / warp_sum(esum);
#pragma unroll
      for (int t = 0; t < SA_KPL; ++t) Ps[warp][lane + 32 * t] = sc[t] * inv;
      __syncwarp();
      float acc = 0.f;
      for (int j = 0; j < Sv; ++j) acc = fmaf(Ps[warp][j], Vs[j][lane], acc);
      out[(static_cast<long long>(seq) * Lq + i) * ldo + h * SA_HD + lane] = from_f<T>(acc);
      __syncwarp();
    }
  }
}

int launch_attention_simt(const void* q, const void* k, const void* v, void* out, int dtype, long long ldq, long long ldk,
                          long long ldv, long long ldo, int n_seq, int Lq, int S, int heads, float scale,
                          const float* bias, int mH, int mW, int mws, int mshift, const int* key_start, cudaStream_t stream) {
  CSVIT_REQUIRE(S >= 1 && S <= SA_MAXS, "attention_simt: key length %d outside [1,%d]", S, SA_MAXS);
  CSVIT_REQUIRE(!key_start || (!bias && mshift <= 0), "attention_simt: per-sequence key ranges take no bias and no window mask");
  CSVIT_REQUIRE(Lq >= 1, "attention_simt: empty query");
  const long long items = static_cast<long long>(n_seq) * heads;
  if (items <= 0) return 0;
  CSVIT_REQUIRE(items < (1ll << 31), "attention_simt: too many work items");
  WinGeom g = make_geom(mH > 0 ? mH : 1, mW > 0 ? mW : 1, mws > 0 ? mws : 1, mshift);
  int nW = mshift > 0 ? (mH / mws) * (mW / mws) : 1;
  if (mshift > 0) CSVIT_REQUIRE(S == mws * mws && Lq == S, "attention_simt: window mask needs Lq == S == ws^2");
  int blocks = static_cast<int>(items < 148 * 16 ? items : 148 * 16);
  if (dtype == DT_F16)
    attention_simt_kernel<__half><<<blocks, 128, 0, stream>>>(
        static_cast<const __half*>(q), static_cast<const __half*>(k), static_cast<const __half*>(v),
        static_cast<__half*>(out), ldq, ldk, ldv, ldo, static_cast<int>(items), Lq, S, heads, scale, bias, g, nW, key_start);
  else if (dtype == DT_BF16)
    attention_simt_kernel<__nv_bfloat16><<<blocks, 128, 0, stream>>>(
        static_cast<const __nv_bfloat16*>(q), static_cast<const __nv_bfloat16*>(k), static_cast<const __nv_bfloat16*>(v),
        static_cast<__nv_bfloat16*>(out), ldq, ldk, ldv, ldo, static_cast<int>(items), Lq, S, heads, scale, bias, g, nW, key_start);
  else
    attention_simt_kernel<float><<<blocks, 128, 0, stream>>>(
        static_cast<const float*>(q), static_cast<const float*>(k), static_cast<const float*>(v), static_cast<float*>(out),
        ldq, ldk, ldv, ldo, static_cast<int>(items), Lq, S, heads, scale, bias, g, nW, key_start);
  CSVIT_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace csvit
