// Gate projection forward on the tensor cores (bf16 activations, 2*NH <= 32 gate outputs, D % 64 == 0).
//
// Reference (vision_lstm2.py:895-897): i, f = Linear(cat[q, k, v]) — per token 2*NH dot products of length 3*D.  The SIMT kernel
// (mlstm_gates.cu) spends 16 FMAs per input element on it and is issue-bound (83 us at T = 51 200, D = 512 for 157 MB of input);
// as a GEMM it is M = tokens, N = 2*NH, K = 3*D — far too skinny to fill a tensor core, but the tensor core takes the FMAs off the
// SM's issue slots and leaves a pure streaming kernel:
//   * the fp32 weights are split into three bf16 parts (hi + mid + lo = the fp32 value to 2^-24) stacked as the N rows of one
//     K-major B operand (rows [0, NOP) = hi, [NOP, 2 NOP) = mid, [2 NOP, 3 NOP) = lo, NOP = 8, 16 or 32, padded to NR = 32,
//     48 or 96 rows): one N = NR MMA per k-step accumulates all three, the epilogue adds them — fp32 weights at fp32
//     accuracy, as the SIMT kernel;
//   * a persistent CTA per SM walks 128-token tiles; the 3*D columns of [q | k | v] stream through a seven-stage TMA ring in
//     64-column slices (16 KB each), straight from the three tensors (no concatenation); one lane loads, another issues MMAs;
//   * where the whole split B operand fits in shared memory next to the ring (RES: D <= 512 at 8 outputs, <= 320 at 16), each
//     CTA splits the weights into it once, while the ring fills, and the call is one launch with no workspace.  Otherwise a
//     small first kernel splits them into the caller's workspace, and every ring slot carries the [NR][64] weight slice of
//     its columns next to the activations (L2-resident after the first tile), so shared memory does not grow with D;
//   * a tile's K is accumulated in segments of GT_SEG slices (K = 256): the tensor core's fp32 accumulation truncates, and
//     its error grows with the number of k-steps summed into one accumulator (up to 6e-6 relative at K = 3 * 2048 in one
//     piece); the epilogue adds the segments' partial sums in fp32 registers.  Two TMEM accumulators alternate between
//     segments, so the epilogue of one (128 threads: one token row each; bias and the NH + NH fp32 stores after the last)
//     runs under the MMAs of the next.
#include "tc_common.cuh"

namespace mlstm {
namespace {

using namespace tc;

constexpr int GT_NT = 192;        // four epilogue warps (one TMEM lane quadrant each), the MMA warp and the load warp
constexpr int GT_ST = 7;          // ring stages of one [128 tokens][64 columns] slice (and, streamed, its [NR][64] weight slice)
constexpr size_t GT_SMEM_MAX = 220 * 1024;
constexpr int GT_SEG = 4;         // 64-column slices accumulated in TMEM before the epilogue takes the partial sum

struct GateMaps { CUtensorMap q, k, v, w; };

__host__ __device__ constexpr int gt_nop(int NO) { return NO <= 8 ? 8 : (NO <= 16 ? 16 : 32); }   // padded gate outputs
__host__ __device__ constexpr int gt_rows(int NOP) { return NOP == 8 ? 32 : (NOP == 16 ? 48 : 96); }   // hi | mid | lo, x16

struct SmemGT {
  alignas(1024) uint8_t ring[GT_ST][TILE];
  uint64_t full[GT_ST], empty[GT_ST], acc_full[2], acc_empty[2];
  uint32_t tmem_base;
  float bias[32];
  // followed (1024-aligned) by the B operand, [slices][NR rows][64 columns] bf16, 128-byte swizzled; NR * 128 is a multiple
  // of 1024, so every slice stays swizzle-aligned.  Resident: all 3*D / 64 slices; streamed: one per ring stage.
};
constexpr size_t GT_HEAD = (sizeof(SmemGT) + 1023) & ~(size_t)1023;

// shared memory of a launch: the ring and barriers, then the B operand slices
inline size_t gt_smem(int D, int NR, bool resident) { return GT_HEAD + (size_t)(resident ? 3 * D / 64 : GT_ST) * NR * 128; }

// B operand in the workspace: (3*D / 64) slices of [NR rows][64 columns] bf16, row-major, read by TMA with the 128-byte
// swizzle.  Element (slice s, row r, column cc) is part r / NOP of gate output r % NOP at input column 64 s + cc; zero for
// unused outputs and the padding rows.
__global__ void gates_split_kernel(const mlstm_gate_proj_params p, __nv_bfloat16* __restrict__ wB, const int NOP, const int NR) {
  const int C3 = 3 * p.D, NO = 2 * p.NH;
  const long long n = (long long)C3 * NR;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < n; idx += (long long)gridDim.x * blockDim.x) {
    const int s = (int)(idx / (NR * 64)), rc = (int)(idx - (long long)s * NR * 64), r = rc >> 6, c = s * 64 + (rc & 63);
    const int part = r / NOP, o = r - part * NOP;
    float v = 0.f;
    if (part < 3 && o < NO) {
      const float w = __ldg((o < p.NH ? p.w_i + (size_t)o * C3 : p.w_f + (size_t)(o - p.NH) * C3) + c);
      const float r1 = w - __bfloat162float(__float2bfloat16_rn(w));
      const float r2 = r1 - __bfloat162float(__float2bfloat16_rn(r1));
      v = part == 0 ? w : (part == 1 ? r1 : r2);
    }
    wB[idx] = __float2bfloat16_rn(v);
  }
}

template <int NOP, bool RES>   // RES: the whole B operand resident in shared memory, split by the CTA; else streamed
__global__ void __launch_bounds__(GT_NT, 1) gates_fwd_tc_kernel(const __grid_constant__ GateMaps maps, const mlstm_gate_proj_params p,
                                                                const int n_tiles) {
  constexpr int NR = gt_rows(NOP);               // rows of the B operand
  constexpr int WSL = NR * 128;                  // bytes of one weight slice tile
  constexpr int ACC = NR <= 64 ? 64 : 128;       // TMEM columns between the two accumulators
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  SmemGT& sm = *reinterpret_cast<SmemGT*>(smem_raw);
  uint8_t* wB = smem_raw + GT_HEAD;
  if ((smem_u32(smem_raw) & 1023u) != 0) __trap();

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool issuer = tid == 128, loader = tid == 160;
  const int D = p.D, NO = 2 * p.NH;
  const int n_sl = 3 * D / 64, sl_per_src = D / 64, n_seg = (n_sl + GT_SEG - 1) / GT_SEG;

  if (loader) {
    tma_prefetch_desc(&maps.q); tma_prefetch_desc(&maps.k); tma_prefetch_desc(&maps.v);
    if (!RES) tma_prefetch_desc(&maps.w);
    for (int i = 0; i < GT_ST; ++i) { mbar_init(&sm.full[i], 1); mbar_init(&sm.empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&sm.acc_full[i], 1); mbar_init(&sm.acc_empty[i], 128); }
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(&sm.tmem_base, 2 * ACC);
  const int my_tiles = ((int)blockIdx.x < n_tiles) ? (n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const int total = my_tiles * n_sl;
  int next_load = 0;
  auto load_slice = [&](int g) {   // activations (and, streamed, the weight slice) of flat slice g into ring slot g % GT_ST
    const int slot = g % GT_ST, n = g / n_sl, s = g - n * n_sl;
    if (g >= GT_ST) mbar_wait(&sm.empty[slot], ((g / GT_ST) - 1) & 1);
    const int t0 = ((int)blockIdx.x + n * (int)gridDim.x) * 128;
    const int src = s / sl_per_src, col = (s - src * sl_per_src) * 64;
    mbar_arrive_expect_tx(&sm.full[slot], TILE + (RES ? 0 : WSL));
    tma_load_2d(sm.ring[slot], src == 0 ? &maps.q : (src == 1 ? &maps.k : &maps.v), &sm.full[slot], col, t0);
    if (!RES) tma_load_2d(wB + (size_t)slot * WSL, &maps.w, &sm.full[slot], 0, s * NR);
  };
  if (RES) {
    if (loader)   // it initialised the barriers itself, so the ring fills while the weights are split
      for (; next_load < GT_ST && next_load < total; ++next_load) load_slice(next_load);
    // resident B operand: gate output o in rows o, NOP + o and 2 NOP + o of every slice; rows of unused outputs and the padding
    // are zero.  Thread = column, the NOP loads of a column (and of the unrolled neighbour) are in flight together.
    const int C3 = 3 * D;
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
    fence_proxy_async_smem();
  }
  if (tid < 32) {
    float b = 0.f;
    if (tid < NO) {
      const float* bp = tid < p.NH ? p.b_i : p.b_f;
      b = bp ? bp[tid < p.NH ? tid : tid - p.NH] : 0.f;
    }
    sm.bias[tid] = b;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tm = sm.tmem_base;

  if (issuer) {
    // ---- MMA lane: the flat slice sequence g = tile * n_sl + slice of this CTA's tiles -------------------------------------
    constexpr uint32_t idM = make_idesc_bf16(128, NR, 0, 0);
    for (int u = 0; u < my_tiles * n_seg; ++u) {   // unit u = segment u % n_seg of tile u / n_seg
      const int buf = u & 1, n = u / n_seg, s0 = (u - n * n_seg) * GT_SEG, s1 = min(s0 + GT_SEG, n_sl);
      if (u >= 2) mbar_wait(&sm.acc_empty[buf], ((u >> 1) - 1) & 1);   // the epilogue has read unit u - 2 from this accumulator
      tc_fence_after();
      for (int s = s0; s < s1; ++s) {
        const int g = n * n_sl + s, slot = g % GT_ST;
        mbar_wait(&sm.full[slot], (g / GT_ST) & 1);
        tc_fence_after();
        const uint64_t dA = make_sdesc(smem_u32(sm.ring[slot]), 16, 1024);
        const uint64_t dB = make_sdesc(smem_u32(wB + (size_t)(RES ? s : slot) * WSL), 16, 1024);
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) umma_bf16_ss(tm + buf * ACC, dA + kstep(ks), dB + kstep(ks), idM, (s > s0 || ks > 0) ? 1u : 0u);
        umma_commit(&sm.empty[slot]);
      }
      umma_commit(&sm.acc_full[buf]);
    }
  } else if (loader) {
    // ---- load lane: refills a slot as soon as the MMAs that read it have retired ---------------------------------------------
    for (; next_load < total; ++next_load) load_slice(next_load);
  } else if (tid < 128) {
    // ---- epilogue warps: thread = token row of the tile ------------------------------------------------------------------------
    const uint32_t lane_sel = (uint32_t)(warp * 32) << 16;
    float sum[NOP];
    for (int u = 0; u < my_tiles * n_seg; ++u) {
      const int buf = u & 1, n = u / n_seg, seg = u - n * n_seg;
      mbar_wait(&sm.acc_full[buf], (u >> 1) & 1);
      tc_fence_after();
      float a[NR];
#pragma unroll
      for (int c = 0; c + 32 <= NR; c += 32) tmem_ld32(tm + buf * ACC + c + lane_sel, reinterpret_cast<float(&)[32]>(a[c]));
      if constexpr (NR % 32 != 0) tmem_ld16(tm + buf * ACC + (NR & ~31) + lane_sel, reinterpret_cast<float(&)[16]>(a[NR & ~31]));
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(&sm.acc_empty[buf]);
#pragma unroll
      for (int o = 0; o < NOP; ++o) {
        const float part = (a[o] + a[NOP + o]) + a[2 * NOP + o];
        sum[o] = seg == 0 ? part : sum[o] + part;
      }
      if (seg < n_seg - 1) continue;
      const int t = ((int)blockIdx.x + n * (int)gridDim.x) * 128 + warp * 32 + lane;
      if (t < p.T) {
        float* oi = p.i + (size_t)t * p.NH;
        float* of = p.f + (size_t)t * p.NH;
#pragma unroll
        for (int o = 0; o < NOP; ++o) {
          if (o < NO) {
            const float val = sum[o] + sm.bias[o];
            if (o < p.NH) oi[o] = val; else of[o - p.NH] = val;
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tm, 2 * ACC);
}

template <int NOP, bool RES>
int launch_fwd_tc(const GateMaps& maps, const mlstm_gate_proj_params& p, cudaStream_t st) {
  const size_t smem = gt_smem(p.D, gt_rows(NOP), RES);
  const int n_tiles = (p.T + 127) / 128;
  const int sms = sm_count_of(p.q);
  const int grid = n_tiles < sms ? n_tiles : sms;
  const cudaError_t e = set_max_smem_once(reinterpret_cast<const void*>(gates_fwd_tc_kernel<NOP, RES>), smem);
  if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(gates_fwd_tc, %zu B): %s", smem, cudaGetErrorString(e)); return MLSTM_ERR_CUDA; }
  gates_fwd_tc_kernel<NOP, RES><<<grid, GT_NT, smem, st>>>(maps, p, n_tiles);
  return MLSTM_OK;
}

template <bool RES>
int launch_fwd_tc(const GateMaps& maps, const mlstm_gate_proj_params& p, cudaStream_t st, int NOP) {
  return NOP == 8 ? launch_fwd_tc<8, RES>(maps, p, st) : (NOP == 16 ? launch_fwd_tc<16, RES>(maps, p, st) : launch_fwd_tc<32, RES>(maps, p, st));
}

// the split B operand fits in shared memory next to the ring: one launch, no workspace
bool gates_tc_resident(const mlstm_gate_proj_params& p) { return gt_smem(p.D, gt_rows(gt_nop(2 * p.NH)), true) <= GT_SMEM_MAX; }

}  // namespace

// The shape alone selects the kernel: bf16 q, k, v with 16-byte aligned rows, D % 64 == 0 and 2*NH <= 32 gate outputs run
// here; fp32 activations, unaligned views and wider gate sets stay on the SIMT kernel.
bool gates_tc_ok(const mlstm_gate_proj_params& p) {
  if (p.dtype != MLSTM_BF16 || p.D % 64 != 0 || 2 * p.NH > 32 || p.ld % 8 != 0) return false;
  // TMA needs 16-byte aligned base addresses; views that start mid-row at an odd offset stay on the SIMT kernel
  return ((reinterpret_cast<uintptr_t>(p.q) | reinterpret_cast<uintptr_t>(p.k) | reinterpret_cast<uintptr_t>(p.v)) & 15u) == 0;
}

// workspace of a shape gates_tc_ok takes: the split B operand when it is streamed, 0 when it is resident
size_t gates_tc_workspace_bytes(const mlstm_gate_proj_params& p) {
  return gates_tc_resident(p) ? 0 : (size_t)(3 * p.D / 64) * gt_rows(gt_nop(2 * p.NH)) * 128;
}

int gates_fwd_tc(const mlstm_gate_proj_params& p, cudaStream_t st) {
  const int NOP = gt_nop(2 * p.NH), NR = gt_rows(NOP);
  const bool res = gates_tc_resident(p);
  GateMaps maps;
  memset(&maps, 0, sizeof(maps));
  int r = 0;
  r |= make_mat_tmap(&maps.q, p.q, p.D, p.T, p.ld);
  r |= make_mat_tmap(&maps.k, p.k, p.D, p.T, p.ld);
  r |= make_mat_tmap(&maps.v, p.v, p.D, p.T, p.ld);
  if (!res) r |= make_state_tmap(&maps.w, p.workspace, (size_t)(3 * p.D / 64) * NR, 64, NR);
  if (r) {
    set_error("cuTensorMapEncodeTiled failed (%d): q, k, v and the workspace must be 16-byte aligned", r);
    return r == -1 ? MLSTM_ERR_NO_DEVICE : MLSTM_ERR_INVALID_ARG;
  }
  cudaError_t e;
  if (!res) {
    const long long n = (long long)3 * p.D * NR;
    const int split_grid = (int)((n + 255) / 256 < 4 * 148 ? (n + 255) / 256 : 4 * 148);
    gates_split_kernel<<<split_grid, 256, 0, st>>>(p, reinterpret_cast<__nv_bfloat16*>(p.workspace), NOP, NR);
    count_launch();
    e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("gates_split launch failed: %s", cudaGetErrorString(e)); return MLSTM_ERR_CUDA; }
  }
  const int rc = res ? launch_fwd_tc<true>(maps, p, st, NOP) : launch_fwd_tc<false>(maps, p, st, NOP);
  if (rc) return rc;
  count_launch();
  e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("gates_fwd_tc launch failed: %s", cudaGetErrorString(e)); return MLSTM_ERR_CUDA; }
  return MLSTM_OK;
}

}  // namespace mlstm
