// Shared pieces of the tcgen05 kernel family (forward and backward):
// thread-role constants, chunk geometry, the per-chunk gate vectors and the one-warp routines
// that build them, the layout of the per-chunk state workspace, and small device helpers.
#pragma once
#include "mlstm_common.cuh"
#include "tc_ptx.cuh"
#include "tc_tmap.cuh"

namespace mlstm {
namespace tc {

using namespace ptx;

constexpr int L = 128;                 // chunk rows (tokens per chunk)
constexpr int CT = 512;                // compute threads: 16 warps = 4 row groups x 4 column blocks
constexpr int GT0 = CT + 32;           // first thread of the gate warp (after the control warp)
constexpr int NT = GT0 + 32;           // 18 warps per CTA
constexpr int TILE = L * 128;          // bytes of one [128 rows][64 bf16] 128B-swizzled tile
constexpr float LOG2E = 1.4426950408889634f;

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void named_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
// log(sigmoid(x)) with fast intrinsics (abs error < 1e-7, enough for the bf16 path)
__device__ __forceinline__ float log_sigmoid_fast(float x) { return fminf(x, 0.f) - __logf(1.f + __expf(-fabsf(x))); }

// descriptor advance per k-step (added to the 64-bit descriptor: start-address field, >>4 units)
__device__ __forceinline__ constexpr uint64_t kstep(int ks, int atom_stride = TILE) {   // K-major operand
  return (uint64_t)((((ks >> 2) * atom_stride) + (ks & 3) * 32) >> 4);
}
__device__ __forceinline__ constexpr uint64_t mnstep(int ks) { return (uint64_t)((ks * 2048) >> 4); }  // MN-major

// ---- chunk geometry -------------------------------------------------------------------------
// Chunks are anchored at token 0 in both scan directions: memory chunk mc covers tokens
// [mc*L, mc*L + nvalid).  In scan order the chunk index is sc; reverse mode walks memory chunks
// from the last to the first and, inside a tile, from the last valid row to row 0.
__host__ __device__ inline int num_chunks(int S) { return (S + L - 1) / L; }
__device__ __forceinline__ int mem_chunk(int sc, int NC, bool rev) { return rev ? (NC - 1 - sc) : sc; }

// ---- per-chunk state workspace (written by the forward, read by the backward) -----------------
// For every (b,h) and scan chunk sc: the ENTRY state of that chunk,
//   Cs : bf16 [DH dk][DH dv]   (row-major; the MN-major / K-major MMA operand tile)
//   ns : fp32 [DH]
//   ms : fp32 scalar
// plus, for the backward, dCs / dns of the same shapes (gradient w.r.t. the state LEAVING chunk sc).
struct StateLayout {
  size_t cs_off, ns_off, ms_off, total;
  __host__ __device__ StateLayout(int B, int NH, int S, int DH) {
    const size_t n = (size_t)B * NH * num_chunks(S);
    cs_off = 0;
    ns_off = cs_off + n * DH * DH * 2;
    ms_off = ns_off + n * DH * 4;
    total = (ms_off + n * 4 + 255) & ~(size_t)255;
  }
};

// ---- gate vectors of one chunk, indexed by tile row --------------------------------------------
struct alignas(16) GateBuf {
  float u2[L];      // u * log2e                     (u_j = i_j - b_j)
  float M2[L];      // M * log2e                     (M_t = max(m_prev, cummax u))
  float w[L];       // exp(m_prev - M_t)             (weight of the inter-chunk term)
  float mrow[L];    // m_t = b_t + M_t
  float kw[L];      // exp(u_j - M_L)                (key weight in the state update)
  float invN[L];    // 1 / (max(|n_t|, e^-m_t) + eps)          (backward only)
  float dnf[L];     // -[|n_t| >= e^-m_t] sign(n_t) / N_t      (backward only: dn_t = dnf_t (dh_t . h_t))
  float sig[L];     // sigmoid(-f_t)                           (backward only)
  float dn[L];      // dn_t                                    (backward only)
  float c2[L];      // M2_t - log2(invN_t)  (+inf for invalid rows)   (backward only)
  float decay;      // exp(m_prev - M_L)
  float m_next;     // b_L + M_L
  float m_prev;
  float pad;
};

// Forward-style gates: one warp, lane l owns scan-local indices 4l..4l+3; m_prev is known.
__device__ __forceinline__ void gates_warp_fwd(GateBuf& G, const mlstm_params& p, int b, int h, int mc, int lane, float m_prev) {
  if (p.gate_mode) m_prev = 0.f;   // sigmoid input gate: every log-weight is <= 0, no stabiliser
  const int tok0 = mc * L;
  const int nvalid = min(L, p.S - tok0);
  float ii[4], bs[4], fraw[4];
  int r[4];
  // all global loads first (independent), then the dependent math: one memory latency, not eight
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const int t = lane * 4 + e;
    const bool valid = t < nvalid;
    r[e] = (p.reverse && valid) ? (nvalid - 1 - t) : t;   // tile row of scan-local index t
    ii[e] = -INFINITY;
    fraw[e] = INFINITY;                                     // logsigmoid(+inf) = 0
    if (valid) {
      const int tok = tok0 + r[e];
      fraw[e] = p.f.ptr[(int64_t)b * p.f.stride_b + (int64_t)h * p.f.stride_h + (int64_t)tok * p.f.stride_s];
      ii[e] = igate_log(p, p.i.ptr[(int64_t)b * p.i.stride_b + (int64_t)h * p.i.stride_h + (int64_t)tok * p.i.stride_s]);
    }
  }
  float run = 0.f;
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    run += (lane * 4 + e < nvalid) ? log_sigmoid_fast(fraw[e]) : 0.f;
    bs[e] = run;
  }
  const float incl = warp_scan_add(run, lane);
  const float excl = incl - run;
  const float g_tot = __shfl_sync(0xffffffffu, incl, 31);
  float u[4], cm[4];
  float lmax = -INFINITY;
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    bs[e] += excl;
    u[e] = ii[e] - bs[e];
    lmax = fmaxf(lmax, u[e]);
    cm[e] = lmax;
  }
  const float imax = warp_scan_max(lmax, lane);
  float emax = __shfl_up_sync(0xffffffffu, imax, 1);
  if (lane == 0) emax = -INFINITY;
  const float ML = p.gate_mode ? -g_tot : fmaxf(m_prev, __shfl_sync(0xffffffffu, imax, 31));
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float M = p.gate_mode ? -bs[e] : fmaxf(m_prev, fmaxf(emax, cm[e]));   // sigmoid gate: m_t = b_t + M_t == 0
    G.u2[r[e]] = u[e] * LOG2E;
    G.M2[r[e]] = M * LOG2E;
    G.w[r[e]] = __expf(m_prev - M);
    G.mrow[r[e]] = bs[e] + M;
    G.kw[r[e]] = __expf(u[e] - ML);
  }
  if (lane == 0) {
    G.decay = __expf(m_prev - ML);
    G.m_next = g_tot + ML;
    G.m_prev = m_prev;
  }
  __syncwarp();
}

// Backward-style gates: everything rebuilt from i, f and the saved rows (n_t, m_t); no carry.
__device__ __forceinline__ void gates_warp_bwd(GateBuf& G, const mlstm_params& p, int b, int h, int bh, int mc, int lane,
                                               const float* ws_dn = nullptr) {
  const int tok0 = mc * L;
  const int nvalid = min(L, p.S - tok0);
  const bool rev = p.reverse != 0;
  float ii[4], bs[4], mr[4], nr[4], fi[4], dnv[4];
  int r[4];
  // all global loads first (independent), then the dependent math
  const int ptok = rev ? (tok0 + nvalid) : (tok0 - 1);
  const float m_prev = p.gate_mode ? 0.f
                       : ((ptok >= 0 && ptok < p.S) ? p.m_row[(int64_t)bh * p.S + ptok] : (p.m_initial ? p.m_initial[bh] : 0.f));
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const int t = lane * 4 + e;
    const bool valid = t < nvalid;
    r[e] = (rev && valid) ? (nvalid - 1 - t) : t;
    ii[e] = -INFINITY; mr[e] = 0.f; nr[e] = 0.f; fi[e] = 0.f; dnv[e] = 0.f;
    if (valid) {
      const int tok = tok0 + r[e];
      fi[e] = p.f.ptr[(int64_t)b * p.f.stride_b + (int64_t)h * p.f.stride_h + (int64_t)tok * p.f.stride_s];
      ii[e] = igate_log(p, p.i.ptr[(int64_t)b * p.i.stride_b + (int64_t)h * p.i.stride_h + (int64_t)tok * p.i.stride_s]);
      mr[e] = p.m_row[(int64_t)bh * p.S + tok];
      nr[e] = p.n_row[(int64_t)bh * p.S + tok];
      if (ws_dn) dnv[e] = ws_dn[(int64_t)bh * p.S + tok];
    }
  }
  float run = 0.f;
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    run += (lane * 4 + e < nvalid) ? log_sigmoid_fast(fi[e]) : 0.f;
    bs[e] = run;
  }
  const float incl = warp_scan_add(run, lane);
  const float excl = incl - run;
  float M[4], u[4];
  float cand = 0.f;
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    bs[e] += excl;
    u[e] = ii[e] - bs[e];
    M[e] = mr[e] - bs[e];
    if (lane * 4 + e == nvalid - 1) cand = M[e];
  }
  const float ML = __shfl_sync(0xffffffffu, cand, (nvalid - 1) >> 2);   // M at the last valid scan index
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const bool valid = lane * 4 + e < nvalid;
    const float Me = valid ? M[e] : ML;
    const float floor_ = __expf(-mr[e]);
    const float N = fmaxf(fabsf(nr[e]), floor_) + p.eps;
    G.u2[r[e]] = u[e] * LOG2E;
    G.M2[r[e]] = Me * LOG2E;
    G.w[r[e]] = __expf(m_prev - Me);
    G.mrow[r[e]] = mr[e];
    G.kw[r[e]] = __expf(u[e] - ML);
    G.invN[r[e]] = valid ? 1.f / N : 0.f;
    G.dnf[r[e]] = (valid && fabsf(nr[e]) >= floor_) ? -copysignf(1.f, nr[e]) / N : 0.f;
    G.sig[r[e]] = 1.f / (1.f + __expf(fi[e]));
    G.dn[r[e]] = dnv[e];
    G.c2[r[e]] = valid ? (Me * LOG2E + log2f(N)) : INFINITY;
  }
  if (lane == 0) {
    G.decay = __expf(m_prev - ML);
    G.m_prev = m_prev;
  }
  __syncwarp();
}

// rows of a [128][DH] swizzled bf16 tile set scaled in place by rowscale[row]; CT compute threads
template <int DH>
__device__ __forceinline__ void scale_rows(uint8_t* tile, const float* rowscale, int tid) {
  constexpr int KT = DH / 64;
#pragma unroll
  for (int it = 0; it < KT * TILE / 16 / CT; ++it) {
    const uint32_t o = (uint32_t)(tid + it * CT) * 16u;
    const float s = rowscale[(o >> 7) & (L - 1)];
    uint4 w = *reinterpret_cast<uint4*>(tile + o);
    __nv_bfloat162* kk = reinterpret_cast<__nv_bfloat162*>(&w);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float2 f2 = __bfloat1622float2(kk[e]);
      kk[e] = __floats2bfloat162_rn(f2.x * s, f2.y * s);
    }
    *reinterpret_cast<uint4*>(tile + o) = w;
  }
}

// 32 bf16 (64 bytes) of a row held as 16 packed words -> global memory
__device__ __forceinline__ void store_row32(__nv_bfloat16* dst, const uint32_t (&pk)[16]) {
#pragma unroll
  for (int x = 0; x < 4; ++x)
    *reinterpret_cast<uint4*>(dst + x * 8) = make_uint4(pk[4 * x], pk[4 * x + 1], pk[4 * x + 2], pk[4 * x + 3]);
}

// 2-D tensor map over a [rows][DH] bf16 matrix stack (the Cs / dCs workspace): dims (DH, rows_total)
// (box = 64 columns x box_rows rows; box_rows = 0 means DH: one whole [DH][64] state tile per load)
inline int make_state_tmap(CUtensorMap* out, const void* ptr, size_t rows_total, int DH, int box_rows = 0) {
  if (box_rows == 0) box_rows = DH;
  TmapKey key;
  memset(&key, 0, sizeof(key));
  key.ptr = ptr; key.s0 = (int64_t)rows_total; key.d0 = DH; key.box_rows = box_rows; key.kind = 2;
  if (tmap_cache_lookup(key, out, false)) return 0;
  PFN_tmapEncodeTiled enc = get_tmap_encoder();
  if (!enc) return -1;
  cuuint64_t dims[2] = {(cuuint64_t)DH, (cuuint64_t)rows_total};
  cuuint64_t strides[1] = {(cuuint64_t)DH * 2};
  cuuint32_t box[2] = {64u, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1u, 1u};
  const int r = (int)enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r == 0) tmap_cache_lookup(key, out, true);
  return r;
}

}  // namespace tc

// 2-D map (columns, rows) of a (T, D) 16-bit matrix with row stride ld; box 64 x 128
inline int make_mat_tmap(CUtensorMap* out, const void* ptr, int D, int T, int64_t ld) {
  TmapKey key;
  memset(&key, 0, sizeof(key));
  key.ptr = ptr; key.s0 = ld; key.d0 = D; key.d1 = T; key.box_rows = 128; key.kind = 8;
  if (tmap_cache_lookup(key, out, false)) return 0;
  PFN_tmapEncodeTiled enc = get_tmap_encoder();
  if (!enc) return -1;
  cuuint64_t dims[2] = {(cuuint64_t)D, (cuuint64_t)T};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {64u, 128u};
  cuuint32_t estr[2] = {1u, 1u};
  const int r = (int)enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r == 0) tmap_cache_lookup(key, out, true);
  return r;
}

}  // namespace mlstm
