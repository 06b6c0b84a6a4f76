// Gate projection of the mLSTM cell, forward and backward, as two streaming kernels.
//
// Reference (nn/modules/vision_lstm/vision_lstm2.py:895-897):
//     if_gate_input = torch.cat([q, k, v], dim=-1)            # (B, S, 3*dim) copy
//     i = self.igate(if_gate_input) ; f = self.fgate(if_gate_input)   # two nn.Linear(3*dim, NH)
// i.e. two skinny GEMMs (N = NH) over a materialised concatenation.  Here q, k, v are read once in
// place (no cat), both gates come out of one pass, and the backward updates the cell's dq, dk, dv
// IN PLACE (dx += di W_i + df W_f) while accumulating dW / db, so autograd never materialises three
// extra (B,S,dim) gradients.  Pure HBM-bound row work: plain coalesced loads, fp32 FMAs, no tensor
// cores (2*NH outputs per token is far below any MMA tile).
//
// Determinism: the dW / db reduction over tokens goes through per-CTA partials in the workspace and a
// fixed-order second kernel; no atomics (cfg/default.yaml: deterministic: True).
#include "mlstm_common.cuh"

namespace mlstm {
bool gates_tc_ok(const mlstm_gate_proj_params& p);                     // mlstm_gates_tc.cu
size_t gates_tc_workspace_bytes(const mlstm_gate_proj_params& p);
int gates_fwd_tc(const mlstm_gate_proj_params& p, cudaStream_t st);
namespace {

constexpr int OG = 8;            // gate outputs per pass (i_0..i_{NH-1}, f_0..f_{NH-1} in groups of 8)
constexpr int FW_NT = 256;       // forward: 8 warps, each warp a tile of TT tokens
constexpr int TT = 4;
constexpr int BW_NT = 128;       // backward: each thread owns BW_CP adjacent columns of [q | k | v]
constexpr int BW_CP = 4;
constexpr int BW_SLAB = BW_CP * BW_NT;      // 512 columns per CTA column slab
constexpr int BW_TU = 4;         // tokens in flight per thread
constexpr int BW_TILE = 64;      // tokens per staged gate-gradient tile

// weight row / bias of gate output o (o < NH: input gate head o; else forget gate head o-NH)
__device__ __forceinline__ const float* w_row(const mlstm_gate_proj_params& p, int o) {
  return (o < p.NH ? p.w_i + (size_t)o * 3 * p.D : p.w_f + (size_t)(o - p.NH) * 3 * p.D);
}
__device__ __forceinline__ float bias_of(const mlstm_gate_proj_params& p, int o) {
  const float* b = o < p.NH ? p.b_i : p.b_f;
  return b ? b[o < p.NH ? o : o - p.NH] : 0.f;
}

template <typename T> struct Vec8;   // 8 adjacent elements: raw load now, unpack to fp32 later
template <> struct Vec8<__nv_bfloat16> {
  using Raw = uint4;
  static __device__ __forceinline__ Raw load_raw(const __nv_bfloat16* ptr) { return *reinterpret_cast<const uint4*>(ptr); }
  static __device__ __forceinline__ void unpack(const Raw& w, float* x) {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&w);
#pragma unroll
    for (int e = 0; e < 4; ++e) { const float2 f2 = __bfloat1622float2(h[e]); x[2 * e] = f2.x; x[2 * e + 1] = f2.y; }
  }
};
template <> struct Vec8<float> {
  struct Raw { float4 a, b; };
  static __device__ __forceinline__ Raw load_raw(const float* ptr) {
    return Raw{reinterpret_cast<const float4*>(ptr)[0], reinterpret_cast<const float4*>(ptr)[1]};
  }
  static __device__ __forceinline__ void unpack(const Raw& r, float* x) {
    x[0] = r.a.x; x[1] = r.a.y; x[2] = r.a.z; x[3] = r.a.w; x[4] = r.b.x; x[5] = r.b.y; x[6] = r.b.z; x[7] = r.b.w;
  }
};

template <typename T> struct Cols;   // BW_CP = 4 adjacent columns
template <> struct Cols<__nv_bfloat16> {
  static __device__ __forceinline__ void load(const __nv_bfloat16* ptr, float* x, bool valid) {
    uint2 w = make_uint2(0u, 0u);
    if (valid) w = *reinterpret_cast<const uint2*>(ptr);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&w);
    const float2 a = __bfloat1622float2(h[0]), b = __bfloat1622float2(h[1]);
    x[0] = a.x; x[1] = a.y; x[2] = b.x; x[3] = b.y;
  }
  static __device__ __forceinline__ void store(__nv_bfloat16* ptr, const float* x) {
    __nv_bfloat162 h[2] = {__floats2bfloat162_rn(x[0], x[1]), __floats2bfloat162_rn(x[2], x[3])};
    *reinterpret_cast<uint2*>(ptr) = *reinterpret_cast<const uint2*>(h);
  }
};
template <> struct Cols<float> {
  static __device__ __forceinline__ void load(const float* ptr, float* x, bool valid) {
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    if (valid) a = *reinterpret_cast<const float4*>(ptr);
    x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w;
  }
  static __device__ __forceinline__ void store(float* ptr, const float* x) {
    *reinterpret_cast<float4*>(ptr) = make_float4(x[0], x[1], x[2], x[3]);
  }
};

// ---------------------------------------------------------------------------------------------
// Forward: i[t, h], f[t, h] = [q_t | k_t | v_t] . W[h] + b[h]
// Weights of the current output group live in shared memory (fp32, [OG][3D]); a warp owns TT tokens,
// its lanes stride the 3D columns in 8-element (16/32-byte) chunks, then a butterfly reduction.
// ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(FW_NT, 2) gates_fwd_kernel(const mlstm_gate_proj_params p) {
  extern __shared__ float wsm[];   // [OG][3D]
  const int D = p.D, C3 = 3 * D, NO = 2 * p.NH;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int warps = FW_NT / 32;
  for (int g0 = 0; g0 < NO; g0 += OG) {
    __syncthreads();
    for (int e = tid; e < OG * C3; e += FW_NT) {
      const int o = g0 + e / C3;
      wsm[e] = o < NO ? w_row(p, o)[e % C3] : 0.f;
    }
    __syncthreads();
    for (int tile = blockIdx.x * warps + warp; tile * TT < p.T; tile += gridDim.x * warps) {
      const int t0 = tile * TT;
      float acc[TT][OG];
#pragma unroll
      for (int tt = 0; tt < TT; ++tt)
#pragma unroll
        for (int o = 0; o < OG; ++o) acc[tt][o] = 0.f;
      // chunks of 8 columns at c = lane*8 + 256*ci over the concatenated [q | k | v] row; the raw loads
      // of chunk ci+1 are issued before the FMAs of chunk ci (D % 8 == 0: a chunk never straddles sources)
      const int nchunk = (C3 - lane * 8 + 255) / 256;
      typename Vec8<T>::Raw raw[TT], nxt[TT];
      auto fetch = [&](int ci, typename Vec8<T>::Raw* dst) {
        const int c = lane * 8 + 256 * ci;
        const int s = c / D, col = c - s * D;
        const T* base = reinterpret_cast<const T*>(s == 0 ? p.q : (s == 1 ? p.k : p.v)) + col;
#pragma unroll
        for (int tt = 0; tt < TT; ++tt) dst[tt] = Vec8<T>::load_raw(base + (size_t)min(t0 + tt, p.T - 1) * p.ld);
      };
      if (nchunk > 0) fetch(0, raw);
      for (int ci = 0; ci < nchunk; ++ci) {
        if (ci + 1 < nchunk) fetch(ci + 1, nxt);
        const int c = lane * 8 + 256 * ci;
        float x[TT][8];
#pragma unroll
        for (int tt = 0; tt < TT; ++tt) Vec8<T>::unpack(raw[tt], x[tt]);
#pragma unroll
        for (int o = 0; o < OG; ++o) {
          const float4 wa = *reinterpret_cast<const float4*>(&wsm[o * C3 + c]);
          const float4 wb = *reinterpret_cast<const float4*>(&wsm[o * C3 + c + 4]);
          const float w[8] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
#pragma unroll
          for (int tt = 0; tt < TT; ++tt)
#pragma unroll
            for (int e = 0; e < 8; ++e) acc[tt][o] = fmaf(x[tt][e], w[e], acc[tt][o]);
        }
#pragma unroll
        for (int tt = 0; tt < TT; ++tt) raw[tt] = nxt[tt];
      }
#pragma unroll
      for (int tt = 0; tt < TT; ++tt)
#pragma unroll
        for (int o = 0; o < OG; ++o) acc[tt][o] = warp_sum(acc[tt][o]);
      if (lane < TT * OG) {
        const int tt = lane / OG, o = g0 + lane % OG, t = t0 + tt;
        float val = 0.f;
#pragma unroll
        for (int a = 0; a < TT; ++a)
#pragma unroll
          for (int b = 0; b < OG; ++b) val = (a == tt && b == lane % OG) ? acc[a][b] : val;
        if (t < p.T && o < NO) {
          float* out = o < p.NH ? p.i + (size_t)t * p.NH + o : p.f + (size_t)t * p.NH + (o - p.NH);
          *out = val + bias_of(p, o);
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Backward: dx[t, c] += sum_o dg[t, o] W[o, c]   (in place on dq | dk | dv)
//           dW[o, c]  = sum_t dg[t, o] x[t, c] ,  db[o] = sum_t dg[t, o]
// grid = (token ranges, column slabs), one launch per output group; a thread owns BW_CP adjacent
// columns with their weights and dW accumulators in registers and streams over the tokens of its
// range (gate gradients staged through shared memory a tile at a time).
// Partials: ws_w[range][NO][3D], ws_b[range][NO].
// ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(BW_NT) gates_bwd_kernel(const mlstm_gate_proj_params p, float* __restrict__ ws_w,
                                                          float* __restrict__ ws_b, const int g0) {
  __shared__ __align__(16) float dgs[BW_TILE][OG];   // gate gradients of the current token tile
  const int D = p.D, C3 = 3 * D, NO = 2 * p.NH;
  const int tid = threadIdx.x;
  const int per = (p.T + gridDim.x - 1) / gridDim.x;
  const int t_begin = blockIdx.x * per, t_end = min(p.T, t_begin + per);
  // this thread's BW_CP adjacent columns of the concatenated [q | k | v] row
  const int c = blockIdx.y * BW_SLAB + BW_CP * tid;
  const bool ok = c < C3;
  const int cc = ok ? c : 0;
  const int sidx = cc / D, col = cc - sidx * D;   // D % 8 == 0 and BW_CP | 8: never straddles two sources
  const T* xs = reinterpret_cast<const T*>(sidx == 0 ? p.q : (sidx == 1 ? p.k : p.v)) + col;
  T* ds = reinterpret_cast<T*>(sidx == 0 ? p.dq : (sidx == 1 ? p.dk : p.dv)) + col;

  float w[OG][BW_CP], dw[OG][BW_CP], dbs[OG];
#pragma unroll
  for (int o = 0; o < OG; ++o) {
    const bool oo = ok && (g0 + o < NO);
    dbs[o] = 0.f;
#pragma unroll
    for (int e = 0; e < BW_CP; ++e) {
      w[o][e] = oo ? w_row(p, g0 + o)[cc + e] : 0.f;
      dw[o][e] = 0.f;
    }
  }

  for (int tile = t_begin; tile < t_end; tile += BW_TILE) {
    __syncthreads();
    for (int e = tid; e < BW_TILE * OG; e += BW_NT) {
      const int t = tile + e / OG, oo = g0 + e % OG;
      dgs[e / OG][e % OG] = (t < t_end && oo < NO) ? (oo < p.NH ? p.di[(size_t)t * p.NH + oo] : p.df[(size_t)t * p.NH + (oo - p.NH)]) : 0.f;
    }
    __syncthreads();
    const int nt = min(BW_TILE, t_end - tile);
    for (int u0 = 0; u0 < nt; u0 += BW_TU) {
      float x[BW_TU][BW_CP], d[BW_TU][BW_CP];
#pragma unroll
      for (int u = 0; u < BW_TU; ++u) {
        const bool v = ok && (u0 + u < nt);
        const size_t row = (size_t)(tile + (v ? u0 + u : 0)) * p.ld;
        Cols<T>::load(xs + row, x[u], v);
        Cols<T>::load(ds + (size_t)(tile + (v ? u0 + u : 0)) * p.ld_d, d[u], v);
      }
#pragma unroll
      for (int u = 0; u < BW_TU; ++u) {
        const float4 ga = *reinterpret_cast<const float4*>(&dgs[u0 + u][0]);
        const float4 gb = *reinterpret_cast<const float4*>(&dgs[u0 + u][4]);
        const float dg[OG] = {ga.x, ga.y, ga.z, ga.w, gb.x, gb.y, gb.z, gb.w};
#pragma unroll
        for (int o = 0; o < OG; ++o) {
          dbs[o] += dg[o];
#pragma unroll
          for (int e = 0; e < BW_CP; ++e) {
            dw[o][e] = fmaf(dg[o], x[u][e], dw[o][e]);
            d[u][e] = fmaf(dg[o], w[o][e], d[u][e]);
          }
        }
        if (ok && (u0 + u < nt)) Cols<T>::store(ds + (size_t)(tile + u0 + u) * p.ld_d, d[u]);
      }
    }
  }
  if (ok) {
    float* out_w = ws_w + (size_t)blockIdx.x * NO * C3 + c;
#pragma unroll
    for (int o = 0; o < OG; ++o)
      if (g0 + o < NO)
#pragma unroll
        for (int e = 0; e < BW_CP; ++e) out_w[(size_t)(g0 + o) * C3 + e] = dw[o][e];
  }
  if (blockIdx.y == 0 && tid == 0) {
#pragma unroll
    for (int o = 0; o < OG; ++o)
      if (g0 + o < NO) ws_b[(size_t)blockIdx.x * NO + g0 + o] = dbs[o];
  }
}

// fixed-order sum of the per-range partials
__global__ void gates_reduce_kernel(const mlstm_gate_proj_params p, const float* __restrict__ ws_w,
                                    const float* __restrict__ ws_b, const int ranges) {
  const int C3 = 3 * p.D, NO = 2 * p.NH;
  const int e0 = (blockIdx.x * blockDim.x + threadIdx.x) >> 3;   // eight lanes per output element
  const bool lead = (threadIdx.x & 7) == 0;
  {
    const int e = min(e0, NO * C3 - 1);
    const float acc = ordered_sum8(ws_w + e, ranges, (size_t)NO * C3);
    const int o = e / C3, c = e - o * C3;
    float* out = o < p.NH ? p.dw_i + (size_t)o * C3 + c : p.dw_f + (size_t)(o - p.NH) * C3 + c;
    if (lead && e0 < NO * C3) *out = acc;
  }
  if (e0 < ((NO + 31) & ~31)) {   // warp-uniform (NO is rounded up to whole warps of element groups)
    const int e = min(e0, NO - 1);
    const float acc = ordered_sum8(ws_b + e, ranges, (size_t)NO);
    float* out = e < p.NH ? (p.db_i ? p.db_i + e : nullptr) : (p.db_f ? p.db_f + (e - p.NH) : nullptr);
    if (lead && e0 < NO && out) *out = acc;
  }
}

int sm_count() {
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  return sms > 0 ? sms : 148;
}

int bwd_ranges(const mlstm_gate_proj_params& p) {
  const int slabs = (3 * p.D + BW_SLAB - 1) / BW_SLAB;
  int r = (4 * 148) / slabs;                      // <= 4 CTAs per SM over the whole grid, rounded DOWN: one CTA beyond the resident
                                                  // 592 would run as a second wave of its own (198 x 3 = 594 CTAs: 172 us; 197 x 3: one wave)
                                                  // (fixed, not the device's SM count: keeps the
  const int max_r = (p.T + 4 * BW_TU - 1) / (4 * BW_TU);   // workspace size independent of the device)
  if (r > max_r) r = max_r;
  return r < 1 ? 1 : r;
}

int validate(const mlstm_gate_proj_params* p, bool bwd) {
  if (!p) { set_error("params is NULL"); return MLSTM_ERR_INVALID_ARG; }
  if (p->abi_version != MLSTM_B200_ABI_VERSION) {
    set_error("ABI version mismatch: caller %d, library %d", p->abi_version, MLSTM_B200_ABI_VERSION);
    return MLSTM_ERR_INVALID_ARG;
  }
  if (p->T < 0 || p->D < 1 || p->NH < 1) { set_error("bad sizes T=%d D=%d NH=%d", p->T, p->D, p->NH); return MLSTM_ERR_INVALID_ARG; }
  if (p->dtype != MLSTM_F32 && p->dtype != MLSTM_BF16) { set_error("unknown dtype %d", p->dtype); return MLSTM_ERR_UNSUPPORTED; }
  if (p->D % 8 != 0 || p->ld % 8 != 0 || p->ld < p->D) {
    set_error("gate projection needs D and the row stride to be multiples of 8 (D=%d, ld=%lld)", p->D, (long long)p->ld);
    return MLSTM_ERR_UNSUPPORTED;
  }
  if ((size_t)OG * 3 * p->D * sizeof(float) > 200 * 1024) { set_error("D=%d too large for the weight tile", p->D); return MLSTM_ERR_UNSUPPORTED; }
  if (bwd && (p->ld_d % 8 != 0 || p->ld_d < p->D)) {
    set_error("gate projection backward needs the row stride of dq, dk, dv to be a multiple of 8 and >= D (D=%d, ld_d=%lld)", p->D, (long long)p->ld_d);
    return MLSTM_ERR_UNSUPPORTED;
  }
  if (p->T == 0) return MLSTM_OK;
  if (!p->q || !p->k || !p->v || !p->w_i || !p->w_f) { set_error("q, k, v, w_i, w_f must be non-NULL"); return MLSTM_ERR_INVALID_ARG; }
  const uintptr_t al = (uintptr_t)p->q | (uintptr_t)p->k | (uintptr_t)p->v | (bwd ? ((uintptr_t)p->dq | (uintptr_t)p->dk | (uintptr_t)p->dv) : 0);
  if (al % 16) { set_error("q, k, v (dq, dk, dv) must be 16-byte aligned"); return MLSTM_ERR_INVALID_ARG; }
  if (!bwd && (!p->i || !p->f)) { set_error("i, f outputs must be non-NULL"); return MLSTM_ERR_INVALID_ARG; }
  if (bwd) {
    if (!p->di || !p->df || !p->dq || !p->dk || !p->dv || !p->dw_i || !p->dw_f) {
      set_error("backward needs di, df, dq, dk, dv, dw_i, dw_f");
      return MLSTM_ERR_INVALID_ARG;
    }
    const size_t need = mlstm_b200_gates_workspace_bytes(p);
    if (!p->workspace || p->workspace_bytes < need) {
      set_error("workspace too small: need %zu bytes, got %zu", need, p->workspace_bytes);
      return MLSTM_ERR_WORKSPACE;
    }
  }
  return MLSTM_OK;
}

int finish(const char* what) {
  count_launch();
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("%s launch failed: %s", what, cudaGetErrorString(e)); return MLSTM_ERR_CUDA; }
  return MLSTM_OK;
}

}  // namespace
}  // namespace mlstm

using namespace mlstm;

extern "C" {

int mlstm_b200_gates_supported(int D, int64_t ld) {
  return D >= 8 && D % 8 == 0 && ld % 8 == 0 && ld >= D && (size_t)OG * 3 * (size_t)D * sizeof(float) <= 200 * 1024;
}

size_t mlstm_b200_gates_workspace_bytes(const mlstm_gate_proj_params* p) {
  if (!p || p->T <= 0) return 0;
  const size_t NO = 2 * (size_t)p->NH, C3 = 3 * (size_t)p->D;
  return sizeof(float) * (size_t)bwd_ranges(*p) * (NO * C3 + NO);
}

size_t mlstm_b200_gates_fwd_workspace_bytes(const mlstm_gate_proj_params* p) {
  if (!p || p->T <= 0 || p->D < 1 || p->NH < 1 || !mlstm_b200_gates_supported(p->D, p->ld) || !gates_tc_ok(*p)) return 0;
  return gates_tc_workspace_bytes(*p);
}

int mlstm_b200_gates_fwd(const mlstm_gate_proj_params* p, void* cuda_stream) {
  clear_error();
  int rc = validate(p, false);
  if (rc || p->T == 0) return rc;
  if (gates_tc_ok(*p)) {   // bf16, D % 64 == 0, <= 32 gate outputs: the tensor-core kernel (streamed weights need the workspace)
    const size_t need = gates_tc_workspace_bytes(*p);
    if (need && (!p->workspace || p->workspace_bytes < need || (uintptr_t)p->workspace % 16)) {
      set_error("forward workspace too small or misaligned: need %zu bytes (16-byte aligned), got %zu", need, p->workspace_bytes);
      return MLSTM_ERR_WORKSPACE;
    }
  }
  if ((rc = bind_device(p->q))) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(cuda_stream);
  if (gates_tc_ok(*p)) return gates_fwd_tc(*p, st);
  const size_t smem = (size_t)OG * 3 * p->D * sizeof(float);
  const int tiles = (p->T + TT - 1) / TT, warps = FW_NT / 32;
  int grid = (tiles + warps - 1) / warps;
  const int cap = 2 * sm_count();
  if (grid > cap) grid = cap;
  cudaError_t e;
  if (p->dtype == MLSTM_BF16) {
    e = cudaFuncSetAttribute(gates_fwd_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) gates_fwd_kernel<__nv_bfloat16><<<grid, FW_NT, smem, st>>>(*p);
  } else {
    e = cudaFuncSetAttribute(gates_fwd_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) gates_fwd_kernel<float><<<grid, FW_NT, smem, st>>>(*p);
  }
  if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(%zu B): %s", smem, cudaGetErrorString(e)); return MLSTM_ERR_CUDA; }
  return finish("gates_fwd");
}

int mlstm_b200_gates_bwd(const mlstm_gate_proj_params* p, void* cuda_stream) {
  clear_error();
  int rc = validate(p, true);
  if (rc || p->T == 0) return rc;
  if ((rc = bind_device(p->q))) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(cuda_stream);
  const int NO = 2 * p->NH, C3 = 3 * p->D;
  const int ranges = bwd_ranges(*p), slabs = (C3 + BW_SLAB - 1) / BW_SLAB;
  float* ws_w = reinterpret_cast<float*>(p->workspace);
  float* ws_b = ws_w + (size_t)ranges * NO * C3;
  for (int g0 = 0; g0 < NO; g0 += OG) {
    if (p->dtype == MLSTM_BF16) gates_bwd_kernel<__nv_bfloat16><<<dim3(ranges, slabs), BW_NT, 0, st>>>(*p, ws_w, ws_b, g0);
    else gates_bwd_kernel<float><<<dim3(ranges, slabs), BW_NT, 0, st>>>(*p, ws_w, ws_b, g0);
    if ((rc = finish("gates_bwd"))) return rc;
  }
  const int n = NO * C3;
  gates_reduce_kernel<<<(n * 8 + 255) / 256, 256, 0, st>>>(*p, ws_w, ws_b, ranges);
  return finish("gates_reduce");
}

}  // extern "C"
