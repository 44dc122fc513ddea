// Per-step state update of the streaming sessions (cs_vit/stream.py): one launch moves the new frames of the nb rows of a step
// into their streams' history and gathers the operands of the temporal part for those rows.
//
// State, for num_streams streams and a window of W frames:
//   tokens [num_streams, W, 3, D] fp32 and (realtime model) stamps [num_streams, W] fp32: a ring per stream, head[s] is the slot of
//   stream s's newest frame; hist[s] int32 is the number of frames since its last reset, at most W.  Only the streams named in
//   ids are read or written, so a stream that is not in a step keeps its state exactly.
// Operands, row r = stream ids[r]:
//   window [3, nb, W, D]: the three per-encoder token sequences, right-aligned (newest frame in slot W-1), zeros outside the history;
//   win_stamps [nb, W]: the stream's timestamps, the newest one outside the history;  key_start [nb] = W - hist.
//   A padding row (ids[r] = -1) gets zeros and key_start = W - 1 and touches no state.
// The operands equal the right-aligned shift of the previous sessions' _push (cat + where over the window) bit for bit: every value
// is a copy.
#include "errors.h"
#include "rowops.cuh"

namespace csvit {

constexpr int SU_THREADS = 512;

__global__ void __launch_bounds__(SU_THREADS)
stream_update_kernel(const float4* __restrict__ tok, const float* __restrict__ ts, const int* __restrict__ ids,
                     const bool* __restrict__ reset, int nb, float4* __restrict__ tokens, float* __restrict__ stamps,
                     int* __restrict__ hist, int* __restrict__ head, int num_streams, int W, int D4,
                     float4* __restrict__ window, float* __restrict__ win_stamps, int* __restrict__ key_start) {
  const int r = blockIdx.x;
  const int s = ids[r];
  const bool pad = s < 0 || s >= num_streams;
  int h = 0, p = 0;                    // history length after this frame, ring slot of this frame
  if (!pad) {
    h = min((reset != nullptr && reset[r]) ? 1 : hist[s] + 1, W);
    p = head[s] + 1 == W ? 0 : head[s] + 1;
  }
  __syncthreads();                     // every thread has read hist[s] / head[s] before thread 0 overwrites them
  if (threadIdx.x == 0) {
    key_start[r] = pad ? W - 1 : W - h;
    if (!pad) { hist[s] = h; head[s] = p; }
  }
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  const long long ring = static_cast<long long>(pad ? 0 : s) * W;
  const int per_q = W * D4;
  for (int i = threadIdx.x; i < 3 * per_q; i += SU_THREADS) {
    const int q = i / per_q, rem = i - q * per_q, j = rem / D4, d = rem - j * D4;
    const int age = W - 1 - j;         // frames between slot j and the newest frame
    float4 v = zero;
    if (!pad && age < h) {
      if (age == 0) {
        v = tok[(static_cast<long long>(r) * 3 + q) * D4 + d];
        tokens[((ring + p) * 3 + q) * D4 + d] = v;
      } else {
        const int slot = p >= age ? p - age : p - age + W;    // != p: ages 1..W-1 only
        v = tokens[((ring + slot) * 3 + q) * D4 + d];
      }
    }
    window[((static_cast<long long>(q) * nb + r) * W + j) * D4 + d] = v;
  }
  if (win_stamps != nullptr) {
    const float newest = pad ? 0.f : ts[r];
    for (int j = threadIdx.x; j < W; j += SU_THREADS) {
      const int age = W - 1 - j;
      float v = newest;
      if (!pad && age == 0) {
        stamps[ring + p] = newest;
      } else if (!pad && age < h) {
        v = stamps[ring + (p >= age ? p - age : p - age + W)];
      }
      win_stamps[static_cast<long long>(r) * W + j] = v;
    }
  }
}

int launch_stream_update(const float* tok, const float* ts, const int* ids, const bool* reset, int nb, float* tokens, float* stamps,
                         int* hist, int* head, int num_streams, int W, int D, float* window, float* win_stamps, int* key_start,
                         cudaStream_t stream) {
  if (nb <= 0) return 0;
  stream_update_kernel<<<nb, SU_THREADS, 0, stream>>>(reinterpret_cast<const float4*>(tok), ts, ids, reset, nb,
                                                      reinterpret_cast<float4*>(tokens), stamps, hist, head, num_streams, W, D / 4,
                                                      reinterpret_cast<float4*>(window), win_stamps, key_start);
  CSVIT_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace csvit
