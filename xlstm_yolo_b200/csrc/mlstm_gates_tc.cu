// Gate projection forward on the tensor cores (bf16 activations, 2*NH <= 16 gate outputs, D % 64 == 0).
//
// Reference (vision_lstm2.py:895-897): i, f = Linear(cat[q, k, v]) — per token 2*NH dot products of length 3*D.  The SIMT kernel
// (mlstm_gates.cu) spends 16 FMAs per input element on it and is issue-bound (83 us at T = 51 200, D = 512 for 157 MB of input);
// as a GEMM it is M = tokens, N = 2*NH, K = 3*D — far too skinny to fill a tensor core, but the tensor core takes the FMAs off the
// SM's issue slots and leaves a pure streaming kernel:
//   * a persistent CTA per SM walks 128-token tiles; the 3*D columns of [q | k | v] stream through a seven-stage TMA ring in
//     64-column slices (16 KB each), straight from the three tensors (no concatenation); one lane loads, another issues MMAs;
//   * the fp32 weights are split once per CTA into three bf16 parts (hi + mid + lo = the fp32 value to 2^-24) stacked as the N
//     rows of one K-major B operand (rows [0, NOP) = hi, [NOP, 2 NOP) = mid, [2 NOP, 3 NOP) = lo, NOP = 8 or 16): one
//     N = 32 / 48 MMA per k-step accumulates all three, the epilogue adds them — fp32 weights at fp32 accuracy, as the SIMT kernel;
//   * two TMEM accumulators alternate between tiles, so the epilogue of one tile (128 threads: one token row each, bias, two
//     float4 stores) runs under the MMAs of the next.
#include "tc_common.cuh"

namespace mlstm {
namespace {

using namespace tc;

constexpr int GT_NT = 192;        // four epilogue warps (one TMEM lane quadrant each), the MMA warp and the load warp
constexpr int GT_ST = 7;          // ring stages of one [128 tokens][64 columns] slice

struct GateMaps { CUtensorMap q, k, v; };

struct SmemGT {
  alignas(1024) uint8_t ring[GT_ST][TILE];
  uint64_t full[GT_ST], empty[GT_ST], acc_full[2], acc_empty[2];
  uint32_t tmem_base;
  float bias[16];
  // followed by the B operand: [3*D / 64 slices][32 or 48 rows][64 columns] bf16, 128-byte swizzled (dynamic size)
};

template <int NOP>   // padded gate outputs: 8 or 16
__global__ void __launch_bounds__(GT_NT, 1) gates_fwd_tc_kernel(const __grid_constant__ GateMaps maps, const mlstm_gate_proj_params p,
                                                                const int n_tiles) {
  constexpr int NR = (NOP == 8) ? 32 : 48;       // rows of the B operand (hi | mid | lo, padded to a multiple of 16)
  constexpr int WSL = NR * 128;                  // bytes of one weight slice tile
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  SmemGT& sm = *reinterpret_cast<SmemGT*>(smem_raw);
  uint8_t* wB = smem_raw + ((sizeof(SmemGT) + 1023) & ~(size_t)1023);
  if ((smem_u32(smem_raw) & 1023u) != 0) __trap();

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool issuer = tid == 128, loader = tid == 160;
  const int D = p.D, C3 = 3 * D, NO = 2 * p.NH;
  const int n_sl = C3 / 64, sl_per_src = D / 64;

  if (loader) {
    tma_prefetch_desc(&maps.q); tma_prefetch_desc(&maps.k); tma_prefetch_desc(&maps.v);
    for (int i = 0; i < GT_ST; ++i) { mbar_init(&sm.full[i], 1); mbar_init(&sm.empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&sm.acc_full[i], 1); mbar_init(&sm.acc_empty[i], 128); }
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(&sm.tmem_base, 128);
  const int my_tiles = ((int)blockIdx.x < n_tiles) ? (n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const int total = my_tiles * n_sl;
  int next_load = 0;
  auto load_slice = [&](int g) {
    const int slot = g % GT_ST, n = g / n_sl, s = g - n * n_sl;
    if (g >= GT_ST) mbar_wait(&sm.empty[slot], ((g / GT_ST) - 1) & 1);
    const int t0 = ((int)blockIdx.x + n * (int)gridDim.x) * 128;
    const int src = s / sl_per_src, col = (s - src * sl_per_src) * 64;
    mbar_arrive_expect_tx(&sm.full[slot], TILE);
    tma_load_2d(sm.ring[slot], src == 0 ? &maps.q : (src == 1 ? &maps.k : &maps.v), &sm.full[slot], col, t0);
  };
  if (loader)     // it initialised the barriers itself, so the ring fills while the weights are split
    for (; next_load < GT_ST && next_load < total; ++next_load) load_slice(next_load);
  // weights: bf16 hi / mid / lo split, gate output o in rows o, NOP + o and 2 NOP + o; rows of unused outputs and the padding are
  // zero.  Thread = column, the NOP loads of a column (and of the unrolled neighbours) are in flight together.
#pragma unroll 2
  for (int c = tid; c < C3; c += GT_NT) {
    float w[NOP];
#pragma unroll
    for (int o = 0; o < NOP; ++o)
      w[o] = o < NO ? __ldg((o < p.NH ? p.w_i + (size_t)o * C3 : p.w_f + (size_t)(o - p.NH) * C3) + c) : 0.f;
    uint8_t* base = wB + (size_t)(c >> 6) * WSL;
#pragma unroll
    for (int o = 0; o < NOP; ++o) {
      const __nv_bfloat16 hi = __float2bfloat16_rn(w[o]);
      const float r1 = w[o] - __bfloat162float(hi);
      const __nv_bfloat16 mid = __float2bfloat16_rn(r1);
      const __nv_bfloat16 lo = __float2bfloat16_rn(r1 - __bfloat162float(mid));
      *reinterpret_cast<__nv_bfloat16*>(base + swz128(o, c & 63)) = hi;
      *reinterpret_cast<__nv_bfloat16*>(base + swz128(NOP + o, c & 63)) = mid;
      *reinterpret_cast<__nv_bfloat16*>(base + swz128(2 * NOP + o, c & 63)) = lo;
      if (NR > 3 * NOP) *reinterpret_cast<__nv_bfloat16*>(base + swz128(3 * NOP + o, c & 63)) = __float2bfloat16_rn(0.f);
    }
  }
  if (tid < 16) {
    float b = 0.f;
    if (tid < NO) {
      const float* bp = tid < p.NH ? p.b_i : p.b_f;
      b = bp ? bp[tid < p.NH ? tid : tid - p.NH] : 0.f;
    }
    sm.bias[tid] = b;
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tm = sm.tmem_base;

  if (issuer) {
    // ---- MMA lane: the flat slice sequence g = tile * n_sl + slice of this CTA's tiles -------------------------------------
    constexpr uint32_t idM = make_idesc_bf16(128, NR, 0, 0);
    for (int n = 0; n < my_tiles; ++n) {
      const int buf = n & 1;
      if (n >= 2) mbar_wait(&sm.acc_empty[buf], ((n >> 1) - 1) & 1);   // the epilogue of tile n - 2 has read this accumulator
      tc_fence_after();
      for (int s = 0; s < n_sl; ++s) {
        const int g = n * n_sl + s, slot = g % GT_ST;
        mbar_wait(&sm.full[slot], (g / GT_ST) & 1);
        tc_fence_after();
        const uint64_t dA = make_sdesc(smem_u32(sm.ring[slot]), 16, 1024);
        const uint64_t dB = make_sdesc(smem_u32(wB + (size_t)s * WSL), 16, 1024);
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) umma_bf16_ss(tm + buf * 64, dA + kstep(ks), dB + kstep(ks), idM, (s > 0 || ks > 0) ? 1u : 0u);
        umma_commit(&sm.empty[slot]);
      }
      umma_commit(&sm.acc_full[buf]);
    }
  } else if (loader) {
    // ---- load lane: refills a slot as soon as the MMAs that read it have retired --------------------------------------------
    for (; next_load < total; ++next_load) load_slice(next_load);
  } else if (tid < 128) {
    // ---- epilogue warps: thread = token row of the tile ------------------------------------------------------------------------
    const uint32_t lane_sel = (uint32_t)(warp * 32) << 16;
    for (int n = 0; n < my_tiles; ++n) {
      const int buf = n & 1;
      mbar_wait(&sm.acc_full[buf], (n >> 1) & 1);
      tc_fence_after();
      float a[48];
      tmem_ld32(tm + buf * 64 + lane_sel, reinterpret_cast<float(&)[32]>(a));
      if (NR > 32) tmem_ld16(tm + buf * 64 + 32 + lane_sel, reinterpret_cast<float(&)[16]>(a[32]));
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(&sm.acc_empty[buf]);
      const int t = ((int)blockIdx.x + n * (int)gridDim.x) * 128 + warp * 32 + lane;
      if (t < p.T) {
        float* oi = p.i + (size_t)t * p.NH;
        float* of = p.f + (size_t)t * p.NH;
#pragma unroll
        for (int o = 0; o < NOP; ++o) {
          if (o < NO) {
            const float val = (a[o] + a[NOP + o]) + a[2 * NOP + o] + sm.bias[o];
            if (o < p.NH) oi[o] = val; else of[o - p.NH] = val;
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tm, 128);
}

}  // namespace

bool gates_tc_ok(const mlstm_gate_proj_params& p) {
  if (p.dtype != MLSTM_BF16 || p.D % 64 != 0 || 2 * p.NH > 16 || p.ld % 8 != 0) return false;
  // TMA needs 16-byte aligned base addresses; views that start mid-row at an odd offset stay on the SIMT kernel
  if (((reinterpret_cast<uintptr_t>(p.q) | reinterpret_cast<uintptr_t>(p.k) | reinterpret_cast<uintptr_t>(p.v)) & 15u) != 0) return false;
  const size_t wbytes = (size_t)(3 * p.D / 64) * (2 * p.NH > 8 ? 48 : 32) * 128;
  return ((sizeof(SmemGT) + 1023) & ~(size_t)1023) + wbytes <= 220 * 1024;
}

int gates_fwd_tc(const mlstm_gate_proj_params& p, cudaStream_t st) {
  GateMaps maps;
  int r = 0;
  r |= make_mat_tmap(&maps.q, p.q, p.D, p.T, p.ld);
  r |= make_mat_tmap(&maps.k, p.k, p.D, p.T, p.ld);
  r |= make_mat_tmap(&maps.v, p.v, p.D, p.T, p.ld);
  if (r) {
    set_error("cuTensorMapEncodeTiled failed (%d): q, k, v must be 16-byte aligned", r);
    return r == -1 ? MLSTM_ERR_NO_DEVICE : MLSTM_ERR_INVALID_ARG;
  }
  const int NOP = 2 * p.NH > 8 ? 16 : 8;
  const size_t smem = ((sizeof(SmemGT) + 1023) & ~(size_t)1023) + (size_t)(3 * p.D / 64) * (NOP == 8 ? 32 : 48) * 128;
  const int n_tiles = (p.T + 127) / 128;
  const int sms = sm_count_of(p.q);
  const int grid = n_tiles < sms ? n_tiles : sms;
  cudaError_t e;
  if (NOP == 8) {
    e = set_max_smem_once(reinterpret_cast<const void*>(gates_fwd_tc_kernel<8>), smem);
    if (e == cudaSuccess) gates_fwd_tc_kernel<8><<<grid, GT_NT, smem, st>>>(maps, p, n_tiles);
  } else {
    e = set_max_smem_once(reinterpret_cast<const void*>(gates_fwd_tc_kernel<16>), smem);
    if (e == cudaSuccess) gates_fwd_tc_kernel<16><<<grid, GT_NT, smem, st>>>(maps, p, n_tiles);
  }
  if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(gates_fwd_tc, %zu B): %s", smem, cudaGetErrorString(e)); return MLSTM_ERR_CUDA; }
  count_launch();
  e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("gates_fwd_tc launch failed: %s", cudaGetErrorString(e)); return MLSTM_ERR_CUDA; }
  return MLSTM_OK;
}

}  // namespace mlstm
