// Shared device/host helpers for the mLSTM kernels (sm_100a).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/mlstm_b200.h"

namespace mlstm {

// Host-side launch bookkeeping, defined in mlstm_api.cu.
void set_error(const char* fmt, ...);
void count_launch(int n = 1);
void clear_error();
int bind_device(const void* dev_ptr);   // make the device owning dev_ptr current on this thread

// Per-family launchers (each returns an mlstm_status).
int simt_fwd(const mlstm_params& p, cudaStream_t st);
int simt_bwd(const mlstm_params& p, cudaStream_t st, int part = -1);  // part -1: both kernels
size_t simt_bwd_workspace(const mlstm_params& p);
bool simt_supported(const mlstm_params& p);

int tc_fwd(const mlstm_params& p, cudaStream_t st);
int tc_bwd(const mlstm_params& p, cudaStream_t st, int part = -1);
size_t tc_bwd_workspace(const mlstm_params& p);
size_t tc_state_bytes(const mlstm_params& p);
bool tc_use_two_phase(const mlstm_params& p);
bool tc_use_fused_bwd(const mlstm_params& p);
bool tc_supported(const mlstm_params& p);

__host__ __device__ inline float resolve_scale(const mlstm_params& p) {
  return p.qk_scale > 0.f ? p.qk_scale : rsqrtf((float)p.DHQK);
}

#ifdef __CUDACC__
template <typename T> __device__ __forceinline__ float to_f32(T x);
template <> __device__ __forceinline__ float to_f32<float>(float x) { return x; }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 x) { return __bfloat162float(x); }
template <typename T> __device__ __forceinline__ T from_f32(float x);
template <> __device__ __forceinline__ float from_f32<float>(float x) { return x; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float x) { return __float2bfloat16_rn(x); }

// log(sigmoid(x)) without overflow: min(x,0) - log1p(exp(-|x|))
__device__ __forceinline__ float log_sigmoid(float x) {
  return fminf(x, 0.f) - log1pf(__expf(-fabsf(x)));
}

// Input-gate pre-activation as it enters the log-space recurrence, and its derivative
// (gate_mode 1: sigmoid input gate, log-gate = logsigmoid(i); d/di = sigmoid(-i)).
__device__ __forceinline__ float igate_log(const mlstm_params& p, float i_raw) {
  return p.gate_mode ? log_sigmoid(i_raw) : i_raw;
}
__device__ __forceinline__ float igate_dlog(const mlstm_params& p, float i_raw) {
  return p.gate_mode ? 1.f / (1.f + __expf(i_raw)) : 1.f;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// Fixed-order (deterministic) sum of n_part partials spaced `stride` floats apart, by a group of 8 adjacent lanes: lane l adds
// partials l, l+8, ... , then the eight lane sums are added in lane order.  Every lane of the warp must call it (clamp the
// element index instead of returning early); the total comes back in all eight lanes.
__device__ __forceinline__ float ordered_sum8(const float* base, int n_part, size_t stride) {
  const int l8 = threadIdx.x & 7;
  float acc = 0.f;
  for (int r = l8; r < n_part; r += 8) acc += base[(size_t)r * stride];
  float tot = 0.f;
#pragma unroll
  for (int l = 0; l < 8; ++l) tot += __shfl_sync(0xffffffffu, acc, l, 8);
  return tot;
}
// inclusive scans across the 32 lanes of a warp
__device__ __forceinline__ float warp_scan_add(float v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    float t = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += t;
  }
  return v;
}
__device__ __forceinline__ float warp_scan_max(float v, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    float t = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v = fmaxf(v, t);
  }
  return v;
}
#endif  // __CUDACC__

}  // namespace mlstm
