// The element-wise / row-reduce tail of a ViL layer fused into one streaming kernel per direction.
//
// Reference (nn/modules/vision_lstm/vision_lstm2.py), four separate HBM round trips over (B,S,inner):
//     h = self.outnorm(h)                        :950   MultiHeadLayerNorm: per-head layer norm over DH,
//                                                       weight applied as (1 + w), optional bias (:1281-1325)
//     h_tilde_state_skip = h + learnable_skip * x_mlstm_conv_act      :498
//     h_state = h_tilde_state_skip * F.silu(z)                        :499
// Here:  y = (LN_head(h) (1 + w) + b + skip * c) * silu(z)  in one pass (read h, c, z; write y), and the
// backward in one pass (read dy, h, c, z; write dh, dc, dz) with the parameter gradients (dw, db, dskip)
// reduced through per-CTA partials in fixed order (deterministic, no atomics).
//
// Layout: rows are tokens; h is the cell's output with heads merged, i.e. the (B,S,NH,DH) storage the
// cell kernels write, seen as (T, D); every operand has its own row stride (z is a column slice of
// proj_up's output).  A warp owns one 256-column segment of a token row (whole heads: DH divides 256),
// a lane 8 adjacent columns (one 16-byte bf16 load); per-head statistics are xor-shuffle reductions over
// the DH/8 lanes of the head.  A CTA is a whole number of rows: (8 / nseg) * nseg warps for nseg = D / 256
// segments (8 warps at D = 256, 512, 1024, 2048; 6 at D = 768 and 1536; 5 at 1280; 7 at 1792), so warp w
// of a CTA always owns segment w % nseg.  HBM-bound row work: no shared-memory staging, no tensor cores.
#include "mlstm_common.cuh"

namespace mlstm {
namespace {

constexpr int GL_NT = 256;                 // at most 8 warps
constexpr int GL_EPL = 8;                  // elements per lane
constexpr int GL_SEG = 32 * GL_EPL;        // columns per warp segment

// warps per CTA: the most whole rows of D / GL_SEG segments that fit in GL_NT threads
__host__ __device__ __forceinline__ int glue_warps(int D) {
  const int nseg = D / GL_SEG;
  return (GL_NT / 32 / nseg) * nseg;
}

template <typename T> struct Ld8;
template <> struct Ld8<__nv_bfloat16> {
  static __device__ __forceinline__ void load(const void* base, size_t idx, float* x) {
    const uint4 w = *reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(base) + idx);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&w);
#pragma unroll
    for (int e = 0; e < 4; ++e) { const float2 f2 = __bfloat1622float2(h[e]); x[2 * e] = f2.x; x[2 * e + 1] = f2.y; }
  }
  static __device__ __forceinline__ void store(void* base, size_t idx, const float* x) {
    __nv_bfloat162 h[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) h[e] = __floats2bfloat162_rn(x[2 * e], x[2 * e + 1]);
    *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(base) + idx) = *reinterpret_cast<const uint4*>(h);
  }
};
template <> struct Ld8<float> {
  static __device__ __forceinline__ void load(const void* base, size_t idx, float* x) {
    const float4* p4 = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(base) + idx);
    const float4 a = p4[0], b = p4[1];
    x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
  }
  static __device__ __forceinline__ void store(void* base, size_t idx, const float* x) {
    float4* p4 = reinterpret_cast<float4*>(reinterpret_cast<float*>(base) + idx);
    p4[0] = make_float4(x[0], x[1], x[2], x[3]);
    p4[1] = make_float4(x[4], x[5], x[6], x[7]);
  }
};

__device__ __forceinline__ void load_param8(const float* ptr, int col, float* x, float fill) {
  if (ptr) {
    const float4 a = *reinterpret_cast<const float4*>(ptr + col), b = *reinterpret_cast<const float4*>(ptr + col + 4);
    x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
  } else {
#pragma unroll
    for (int e = 0; e < 8; ++e) x[e] = fill;
  }
}

// sum over the `lph` lanes of this lane's head (lph a power of two, heads aligned to lph lanes)
__device__ __forceinline__ float head_sum(float v, int lph) {
  for (int o = 1; o < lph; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// per-head statistics of the 8 values this lane holds: normalised values and rstd
__device__ __forceinline__ void head_norm(const float* x, int lph, float inv_dh, float eps, float* xhat, float& rstd) {
  float s = 0.f;
#pragma unroll
  for (int e = 0; e < 8; ++e) s += x[e];
  const float mean = head_sum(s, lph) * inv_dh;
  float ss = 0.f;
#pragma unroll
  for (int e = 0; e < 8; ++e) { xhat[e] = x[e] - mean; ss = fmaf(xhat[e], xhat[e], ss); }
  rstd = rsqrtf(head_sum(ss, lph) * inv_dh + eps);
#pragma unroll
  for (int e = 0; e < 8; ++e) xhat[e] *= rstd;
}

template <typename T>
__global__ void __launch_bounds__(GL_NT) glue_fwd_kernel(const mlstm_glue_params p) {
  const int lane = threadIdx.x & 31, wpc = blockDim.x >> 5;
  const int gw = blockIdx.x * wpc + (threadIdx.x >> 5), nw = gridDim.x * wpc;
  const int nseg = p.D / GL_SEG, DH = p.D / p.NH, lph = DH / GL_EPL;
  const int seg = gw % nseg, col = seg * GL_SEG + lane * GL_EPL;
  const float inv_dh = 1.f / (float)DH;
  float w1[8], bb[8], sk[8];
  load_param8(p.w, col, w1, 0.f);
  load_param8(p.b, col, bb, 0.f);
  load_param8(p.skip, col, sk, 1.f);
#pragma unroll
  for (int e = 0; e < 8; ++e) w1[e] += 1.f;
  const int step = nw / nseg;
  for (int t0 = gw / nseg; t0 < p.T; t0 += 2 * step) {   // two tokens in flight per warp
    float h[2][8], c[2][8], z[2][8];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int t = min(t0 + u * step, p.T - 1);
      Ld8<T>::load(p.h, (size_t)t * p.ld_h + col, h[u]);
      Ld8<T>::load(p.c, (size_t)t * p.ld_c + col, c[u]);
      Ld8<T>::load(p.z, (size_t)t * p.ld_z + col, z[u]);
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int t = t0 + u * step;
      float xhat[8], y[8], rstd;
      head_norm(h[u], lph, inv_dh, p.eps, xhat, rstd);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float pre = fmaf(xhat[e], w1[e], bb[e]) + sk[e] * c[u][e];
        y[e] = pre * z[u][e] / (1.f + __expf(-z[u][e]));
      }
      if (t < p.T) Ld8<T>::store(p.y, (size_t)t * p.ld_y + col, y);
    }
  }
}

// ws: [gridDim.x][3][D] per-CTA partials of (dw, db, dskip)
template <typename T>
__global__ void __launch_bounds__(GL_NT, 2) glue_bwd_kernel(const mlstm_glue_params p, float* __restrict__ ws) {
  __shared__ float red[GL_NT / 32][3][GL_SEG];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpc = blockDim.x >> 5;
  const int gw = blockIdx.x * wpc + warp, nw = gridDim.x * wpc;
  const int nseg = p.D / GL_SEG, DH = p.D / p.NH, lph = DH / GL_EPL;
  const int seg = gw % nseg, col = seg * GL_SEG + lane * GL_EPL;
  const float inv_dh = 1.f / (float)DH;
  float w1[8], bb[8], sk[8], aw[8], ab[8], as[8];
  load_param8(p.w, col, w1, 0.f);
  load_param8(p.b, col, bb, 0.f);
  load_param8(p.skip, col, sk, 1.f);
#pragma unroll
  for (int e = 0; e < 8; ++e) { w1[e] += 1.f; aw[e] = 0.f; ab[e] = 0.f; as[e] = 0.f; }
  const int step = nw / nseg;
  for (int t0 = gw / nseg; t0 < p.T; t0 += 2 * step) {   // two tokens in flight per warp
    float hh[2][8], cc[2][8], zz[2][8], dd[2][8];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int t = min(t0 + u * step, p.T - 1);
      Ld8<T>::load(p.h, (size_t)t * p.ld_h + col, hh[u]);
      Ld8<T>::load(p.c, (size_t)t * p.ld_c + col, cc[u]);
      Ld8<T>::load(p.z, (size_t)t * p.ld_z + col, zz[u]);
      Ld8<T>::load(p.dy, (size_t)t * p.ld_dy + col, dd[u]);
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int t = t0 + u * step;
      const bool live = t < p.T;                 // warp-uniform
      const float* h = hh[u]; const float* c = cc[u]; const float* z = zz[u]; const float* dy = dd[u];
      float xhat[8], rstd;
      head_norm(h, lph, inv_dh, p.eps, xhat, rstd);
      float dz[8], dc[8], dx[8], m1 = 0.f, m2 = 0.f;
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float sg = 1.f / (1.f + __expf(-z[e]));
        const float silu = z[e] * sg;
        const float pre = fmaf(xhat[e], w1[e], bb[e]) + sk[e] * c[e];
        const float g = live ? dy[e] * silu : 0.f;                     // d pre
        dz[e] = dy[e] * pre * sg * (1.f + z[e] * (1.f - sg));
        dc[e] = g * sk[e];
        as[e] = fmaf(g, c[e], as[e]);
        aw[e] = fmaf(g, xhat[e], aw[e]);
        ab[e] += g;
        dx[e] = g * w1[e];                                             // d xhat
        m1 += dx[e];
        m2 = fmaf(dx[e], xhat[e], m2);
      }
      m1 = head_sum(m1, lph) * inv_dh;
      m2 = head_sum(m2, lph) * inv_dh;
      float dh[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) dh[e] = rstd * (dx[e] - m1 - xhat[e] * m2);
      if (live) {
        Ld8<T>::store(p.dh, (size_t)t * p.ld_dh + col, dh);
        Ld8<T>::store(p.dc, (size_t)t * p.ld_dc + col, dc);
        Ld8<T>::store(p.dz, (size_t)t * p.ld_dz + col, dz);
      }
    }
  }
  // CTA-level reduction over the warps that own the same segment, then one partial row per CTA
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    red[warp][0][lane * 8 + e] = aw[e];
    red[warp][1][lane * 8 + e] = ab[e];
    red[warp][2][lane * 8 + e] = as[e];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 3 * p.D; i += blockDim.x) {
    const int k = i / p.D, cd = i - k * p.D, sg = cd / GL_SEG, cc = cd - sg * GL_SEG;
    float acc = 0.f;
    for (int w = sg; w < wpc; w += nseg) acc += red[w][k][cc];   // warp w of a CTA owns segment w % nseg
    ws[((size_t)blockIdx.x * 3 + k) * p.D + cd] = acc;
  }
}

__global__ void glue_reduce_kernel(const mlstm_glue_params p, const float* __restrict__ ws, const int ctas) {
  const int i0 = (blockIdx.x * blockDim.x + threadIdx.x) >> 3;   // eight lanes per output element
  const int i = min(i0, 3 * p.D - 1);
  const int k = i / p.D, cd = i - k * p.D;
  const float acc = ordered_sum8(ws + (size_t)k * p.D + cd, ctas, (size_t)3 * p.D);
  float* out = k == 0 ? p.dw : (k == 1 ? p.db : p.dskip);
  if (out && i0 < 3 * p.D && (threadIdx.x & 7) == 0) out[cd] = acc;
}

int glue_grid(const mlstm_glue_params& p) {
  const int nseg = p.D / GL_SEG;
  const long long units = (long long)p.T * nseg, wpc = glue_warps(p.D);   // (token, segment) work units, one per warp step
  long long g = (units + wpc * 4 - 1) / (wpc * 4);                  // >= 4 units per warp
  if (g > 2 * 148) g = 2 * 148;                                  // fixed cap: workspace size independent of the device
  return g < 1 ? 1 : (int)g;
}

int validate(const mlstm_glue_params* p, bool bwd) {
  if (!p) { set_error("params is NULL"); return MLSTM_ERR_INVALID_ARG; }
  if (p->abi_version != MLSTM_B200_ABI_VERSION) {
    set_error("abi_version %d != %d", p->abi_version, MLSTM_B200_ABI_VERSION);
    return MLSTM_ERR_INVALID_ARG;
  }
  if (p->T < 0 || p->D < 1 || p->NH < 1 || p->D % p->NH) { set_error("bad sizes T=%d D=%d NH=%d", p->T, p->D, p->NH); return MLSTM_ERR_INVALID_ARG; }
  if (p->dtype != MLSTM_F32 && p->dtype != MLSTM_BF16) { set_error("unknown dtype %d", p->dtype); return MLSTM_ERR_UNSUPPORTED; }
  const int DH = p->D / p->NH;
  if (p->D % GL_SEG || p->D > GL_SEG * (GL_NT / 32) || DH % GL_EPL || GL_SEG % DH) {
    set_error("fused layer tail needs D a multiple of 256 (<= 2048) and DH in {8,...,256} dividing 256 (D=%d, DH=%d)", p->D, DH);
    return MLSTM_ERR_UNSUPPORTED;
  }
  if (p->T == 0) return MLSTM_OK;
  const int64_t lds[7] = {p->ld_h, p->ld_c, p->ld_z, bwd ? 8 : p->ld_y, bwd ? p->ld_dy : 8, bwd ? p->ld_dh : 8, bwd ? p->ld_dc : 8};
  for (int i = 0; i < 7; ++i)
    if (lds[i] % 8) { set_error("row strides must be multiples of 8 elements"); return MLSTM_ERR_INVALID_ARG; }
  if (bwd && p->ld_dz % 8) { set_error("row strides must be multiples of 8 elements"); return MLSTM_ERR_INVALID_ARG; }
  uintptr_t al = (uintptr_t)p->h | (uintptr_t)p->c | (uintptr_t)p->z | (uintptr_t)p->w | (uintptr_t)p->b | (uintptr_t)p->skip;
  if (!p->h || !p->c || !p->z) { set_error("h, c, z must be non-NULL"); return MLSTM_ERR_INVALID_ARG; }
  if (!bwd) {
    if (!p->y) { set_error("y must be non-NULL"); return MLSTM_ERR_INVALID_ARG; }
    al |= (uintptr_t)p->y;
  } else {
    if (!p->dy || !p->dh || !p->dc || !p->dz) { set_error("backward needs dy, dh, dc, dz"); return MLSTM_ERR_INVALID_ARG; }
    al |= (uintptr_t)p->dy | (uintptr_t)p->dh | (uintptr_t)p->dc | (uintptr_t)p->dz;
    const size_t need = mlstm_b200_glue_workspace_bytes(p);
    if (!p->workspace || p->workspace_bytes < need) {
      set_error("workspace too small: need %zu bytes, got %zu", need, p->workspace_bytes);
      return MLSTM_ERR_WORKSPACE;
    }
  }
  if (al % 16) { set_error("all pointers must be 16-byte aligned"); return MLSTM_ERR_INVALID_ARG; }
  return MLSTM_OK;
}

int done(const char* what) {
  count_launch();
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("%s launch failed: %s", what, cudaGetErrorString(e)); return MLSTM_ERR_CUDA; }
  return MLSTM_OK;
}

}  // namespace
}  // namespace mlstm

using namespace mlstm;

extern "C" {

int mlstm_b200_glue_supported(int D, int NH) {
  if (D < 1 || NH < 1 || D % NH) return 0;
  const int DH = D / NH;
  return !(D % GL_SEG || D > GL_SEG * (GL_NT / 32) || DH % GL_EPL || GL_SEG % DH);
}

size_t mlstm_b200_glue_workspace_bytes(const mlstm_glue_params* p) {
  if (!p || p->T <= 0 || p->D < GL_SEG || p->D > GL_SEG * (GL_NT / 32)) return 0;
  return sizeof(float) * 3 * (size_t)p->D * glue_grid(*p);
}

int mlstm_b200_glue_fwd(const mlstm_glue_params* p, void* cuda_stream) {
  clear_error();
  int rc = validate(p, false);
  if (rc || p->T == 0) return rc;
  if ((rc = bind_device(p->h))) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(cuda_stream);
  const int grid = glue_grid(*p);
  if (p->dtype == MLSTM_BF16) glue_fwd_kernel<__nv_bfloat16><<<grid, 32 * glue_warps(p->D), 0, st>>>(*p);
  else glue_fwd_kernel<float><<<grid, 32 * glue_warps(p->D), 0, st>>>(*p);
  return done("glue_fwd");
}

int mlstm_b200_glue_bwd(const mlstm_glue_params* p, void* cuda_stream) {
  clear_error();
  int rc = validate(p, true);
  if (rc || p->T == 0) return rc;
  if ((rc = bind_device(p->h))) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(cuda_stream);
  const int grid = glue_grid(*p);
  float* ws = reinterpret_cast<float*>(p->workspace);
  if (p->dtype == MLSTM_BF16) glue_bwd_kernel<__nv_bfloat16><<<grid, 32 * glue_warps(p->D), 0, st>>>(*p, ws);
  else glue_bwd_kernel<float><<<grid, 32 * glue_warps(p->D), 0, st>>>(*p, ws);
  if ((rc = done("glue_bwd"))) return rc;
  glue_reduce_kernel<<<(3 * p->D * 8 + 255) / 256, 256, 0, st>>>(*p, ws, grid);
  return done("glue_reduce");
}

}  // extern "C"
