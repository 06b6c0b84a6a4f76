// extern "C" entry points of libmlstm_b200.so (declared in include/mlstm_b200.h):
// argument validation, kernel-family dispatch, error reporting.  No torch types.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include "mlstm_common.cuh"
#include "tc_tmap.cuh"

namespace mlstm {

static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }
void clear_error() { g_err[0] = 0; }

// ---------------------------------------------------------------------------------------------------------------------
// Head dims the tcgen05 kernels are not written for, on the tensor cores anyway (bf16): DHqk != DHv (the reference's
// mLSTMLayerVision: qk_dim_factor = 0.5, mlstm_large.py:46,186-187) and head dims below / between 64, 128, 256 (the
// reference's default qkv_block_size = 16, vision_lstm2.py:416-417, gives DH = 16).
// Every q / k dependent quantity of the cell is an inner product over DHqk (S = Q K^T, q . C, q . n, the rows of C = K^T V
// and of n = sum k) and every column of v only meets its own column of C, h and dh, so q, k, v, dh padded with zero columns
// to a common DP in {64, 128, 256} give the same h, dq, dk, dv in the leading columns (zeros behind them), the same di, df
// and the same leading block of the carried C, n.  The padded bf16 copies ((B, S, NH, DP), dense) of q, k, v and the padded h
// live behind the chunk states in the caller's `states` buffer (written by the forward, read again by the backward); dh is
// padded and dq, dk, dv are produced padded in the workspace and cropped out; initial / last states are padded / cropped the
// same way; the 1 / sqrt(DHqk) scale is passed explicitly.
// ---------------------------------------------------------------------------------------------------------------------
namespace {

inline size_t al256(size_t x) { return (x + 255) & ~(size_t)255; }

int padded_dim(const mlstm_params& p) {
  const int d = p.DHQK > p.DHV ? p.DHQK : p.DHV;
  return d <= 64 ? 64 : (d <= 128 ? 128 : (d <= 256 ? 256 : 0));
}

struct PadLayout {
  int DP;
  size_t inner, act, cst, nst;             // bytes: padded problem's own states | one padded activation | C | n
  size_t act_c;                            // room per copy in the states buffer and in the workspace (0 where none are made)
  size_t q_off, k_off, v_off, h_off, c0_off, n0_off, cl_off, nl_off, total;
  size_t ws_inner, dh_off, dq_off, dk_off, dv_off, ws_total;
};

mlstm_params padded_params(const mlstm_params& p) {
  mlstm_params pp = p;
  pp.qk_scale = resolve_scale(p);
  pp.DHQK = pp.DHV = padded_dim(p);
  return pp;
}

// Where every access of a kernel variant to q, k, v, h, dh, dq, dk, dv goes through TMA, the padding costs nothing: the tensor
// maps are encoded with the true row length and TMA supplies / clips the rest (tc_tmap.cuh: ExtentOverride).  That holds for
// every DP = 64 and 128 kernel: where they touch rows with plain loads or stores (the two-phase forward's h rows, tc_dn_kernel,
// two row reads of the DH = 128 fused walk) they take the true row length as an argument.  The DH = 256 family runs on copies.
bool zero_copy(const mlstm_params& pp) { return pp.DHV <= 128; }

PadLayout pad_layout(const mlstm_params& p) {
  const mlstm_params pp = padded_params(p);
  PadLayout l;
  l.DP = pp.DHV;
  l.inner = al256(tc_state_bytes(pp));
  l.act = al256((size_t)p.B * p.S * p.NH * l.DP * 2);
  l.cst = al256((size_t)p.B * p.NH * l.DP * l.DP * 4);
  l.nst = al256((size_t)p.B * p.NH * l.DP * 4);
  // copies of q, k, v, h (made by the forward, read again by the backward) and of dh, dq, dk, dv
  l.act_c = zero_copy(pp) ? 0 : l.act;
  l.q_off = l.inner;
  l.k_off = l.q_off + l.act_c;
  l.v_off = l.k_off + l.act_c;
  l.h_off = l.v_off + l.act_c;
  l.c0_off = l.h_off + l.act_c;
  l.n0_off = l.c0_off + l.cst;
  l.cl_off = l.n0_off + l.nst;
  l.nl_off = l.cl_off + l.cst;
  l.total = l.nl_off + l.nst;
  l.ws_inner = al256(tc_bwd_workspace(pp));
  l.dh_off = l.ws_inner;
  l.dq_off = l.dh_off + l.act_c;
  l.dk_off = l.dq_off + l.act_c;
  l.dv_off = l.dk_off + l.act_c;
  l.ws_total = l.dv_off + l.act_c;
  return l;
}

bool pad_path(const mlstm_params& p) {
  if (p.dtype != MLSTM_BF16 || p.DHQK % 8 != 0 || p.DHV % 8 != 0 || p.DHQK < 16 || p.DHV < 16) return false;
  if (padded_dim(p) == 0 || tc_supported(p)) return false;
  return tc_supported(padded_params(p));
}

// rows (b, s, h) of up to three strided bf16 activations <-> rows of their dense padded copies, 16 bytes per thread
struct PadJob { mlstm_act a; __nv_bfloat16* d; int D; };
struct PadJobs { PadJob j[3]; };

__global__ void __launch_bounds__(256) pad_rows_kernel(const PadJobs jobs, const int B, const int S, const int NH, const int DP,
                                                       const int to_padded) {
  const int cpr = DP / 8;                                    // 16-byte chunks per padded row
  const int64_t n = (int64_t)B * S * NH * cpr;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(e % cpr);
    const int64_t row = e / cpr;
    const int h = (int)(row % NH);
    const int64_t bs = row / NH;
    const int s_ = (int)(bs % S), b = (int)(bs / S);
#pragma unroll
    for (int w = 0; w < 3; ++w) {
      const PadJob& jb = jobs.j[w];
      if (!jb.a.ptr) continue;
      const bool live = c * 8 < jb.D;
      __nv_bfloat16* src = reinterpret_cast<__nv_bfloat16*>(jb.a.ptr) + (int64_t)b * jb.a.stride_b + (int64_t)h * jb.a.stride_h +
                           (int64_t)s_ * jb.a.stride_s + c * 8;
      uint4* pad = reinterpret_cast<uint4*>(jb.d + row * DP + c * 8);
      if (to_padded) *pad = live ? *reinterpret_cast<const uint4*>(src) : make_uint4(0, 0, 0, 0);
      else if (live) *reinterpret_cast<uint4*>(src) = *pad;
    }
  }
}

// fp32 states: C (B*NH, DK, DV) <-> (B*NH, DP, DP), n (B*NH, DK) <-> (B*NH, DP)
__global__ void __launch_bounds__(256) pad_states_kernel(float* __restrict__ c_small, float* __restrict__ n_small,
                                                         float* __restrict__ c_pad, float* __restrict__ n_pad, const int BH,
                                                         const int DK, const int DV, const int DP, const int to_padded) {
  const int64_t nc = (int64_t)BH * DP * DP, nn = (int64_t)BH * DP;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nc + nn; e += (int64_t)gridDim.x * blockDim.x) {
    if (e < nc) {
      const int col = (int)(e % DP), r = (int)((e / DP) % DP);
      const int64_t bh = e / ((int64_t)DP * DP);
      const bool live = r < DK && col < DV;
      if (to_padded) c_pad[e] = live ? c_small[(bh * DK + r) * DV + col] : 0.f;
      else if (live) c_small[(bh * DK + r) * DV + col] = c_pad[e];
    } else {
      const int64_t x = e - nc;
      const int r = (int)(x % DP);
      const int64_t bh = x / DP;
      if (to_padded) n_pad[x] = r < DK ? n_small[bh * DK + r] : 0.f;
      else if (r < DK) n_small[bh * DK + r] = n_pad[x];
    }
  }
}

int pad_launched(const char* what) {
  count_launch();
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("%s launch failed: %s", what, cudaGetErrorString(e)); return MLSTM_ERR_CUDA; }
  return MLSTM_OK;
}

mlstm_act dense_act(void* ptr, const mlstm_params& p, int DP) {
  mlstm_act a;
  a.ptr = ptr;
  a.stride_b = (int64_t)p.S * p.NH * DP;
  a.stride_s = (int64_t)p.NH * DP;
  a.stride_h = DP;
  return a;
}

PadJob job(const mlstm_act& a, const mlstm_act& padded, int D) {
  PadJob j;
  j.a = a;
  j.d = reinterpret_cast<__nv_bfloat16*>(padded.ptr);
  j.D = D;
  return j;
}
PadJob no_job() {
  PadJob j;
  j.a.ptr = nullptr; j.a.stride_b = j.a.stride_h = j.a.stride_s = 0;
  j.d = nullptr; j.D = 0;
  return j;
}

int grid_for(int64_t n) { return (int)((n + 255) / 256 < 148 * 8 ? (n + 255) / 256 : 148 * 8); }

int pad_rows(const mlstm_params& p, int DP, PadJob j0, PadJob j1, PadJob j2, int to_padded, cudaStream_t st, const char* what) {
  PadJobs jobs;
  jobs.j[0] = j0; jobs.j[1] = j1; jobs.j[2] = j2;
  pad_rows_kernel<<<grid_for((int64_t)p.B * p.S * p.NH * (DP / 8)), 256, 0, st>>>(jobs, p.B, p.S, p.NH, DP, to_padded);
  return pad_launched(what);
}

// the padded problem of a forward or backward call: pointers into the caller's states / workspace buffers
int make_padded(const mlstm_params& p, int is_bwd, mlstm_params* out, PadLayout* lay) {
  const PadLayout l = pad_layout(p);
  if (!p.states || p.states_bytes < l.total) {
    set_error("head dims (%d, %d) run zero-padded to %d on the tensor cores: the states buffer must hold mlstm_b200_state_bytes() = "
              "%zu bytes (have %zu)", p.DHQK, p.DHV, l.DP, l.total, p.states ? p.states_bytes : (size_t)0);
    return MLSTM_ERR_WORKSPACE;
  }
  if ((reinterpret_cast<uintptr_t>(p.states) & 255u) != 0) { set_error("states buffer must be 256-byte aligned"); return MLSTM_ERR_INVALID_ARG; }
  uint8_t* sb = reinterpret_cast<uint8_t*>(p.states);
  mlstm_params pp = padded_params(p);
  pp.states_bytes = l.inner;
  if (l.inner == 0) pp.states = nullptr;   // forward-only single-pass call: the padded problem keeps its states on chip
  // a side that already has the padded width runs on the caller's own tensors (DHqk < DHv = DP: only q, k are copied);
  // so does everything at DP = 64 and 128
  const bool zc = zero_copy(pp);
  const bool pad_qk = p.DHQK != l.DP && !zc, pad_v = p.DHV != l.DP && !zc;
  if (pad_qk) { pp.q = dense_act(sb + l.q_off, p, l.DP); pp.k = dense_act(sb + l.k_off, p, l.DP); }
  if (pad_v) { pp.v = dense_act(sb + l.v_off, p, l.DP); pp.h = dense_act(sb + l.h_off, p, l.DP); }
  if (p.c_initial) { pp.c_initial = reinterpret_cast<float*>(sb + l.c0_off); pp.n_initial = reinterpret_cast<float*>(sb + l.n0_off); }
  if (p.c_last) { pp.c_last = reinterpret_cast<float*>(sb + l.cl_off); pp.n_last = reinterpret_cast<float*>(sb + l.nl_off); }
  if (is_bwd) {
    uint8_t* ws = reinterpret_cast<uint8_t*>(p.workspace);
    pp.workspace_bytes = l.ws_inner;
    if (pad_qk) { pp.dq = dense_act(ws + l.dq_off, p, l.DP); pp.dk = dense_act(ws + l.dk_off, p, l.DP); }
    if (pad_v) { pp.dh = dense_act(ws + l.dh_off, p, l.DP); pp.dv = dense_act(ws + l.dv_off, p, l.DP); }
  }
  *out = pp;
  *lay = l;
  return MLSTM_OK;
}

int tcpad_fwd(const mlstm_params& p, cudaStream_t st) {
  mlstm_params pp;
  PadLayout l;
  int rc = make_padded(p, 0, &pp, &l);
  if (rc) return rc;
  const bool zc = zero_copy(pp);
  const bool pad_qk = p.DHQK != l.DP && !zc, pad_v = p.DHV != l.DP && !zc;
  ExtentScope ext;
  if (zc) {
    ext.add(p.q.ptr, p.DHQK); ext.add(p.k.ptr, p.DHQK);
    ext.add(p.v.ptr, p.DHV); ext.add(p.h.ptr, p.DHV);
  }
  if ((pad_qk || pad_v) &&
      (rc = pad_rows(p, l.DP, pad_qk ? job(p.q, pp.q, p.DHQK) : no_job(), pad_qk ? job(p.k, pp.k, p.DHQK) : no_job(),
                     pad_v ? job(p.v, pp.v, p.DHV) : no_job(), 1, st, "pad_rows")))
    return rc;
  const int64_t nst = (int64_t)p.B * p.NH * l.DP * (l.DP + 1);
  if (p.c_initial) {
    if (!p.n_initial) { set_error("c_initial without n_initial"); return MLSTM_ERR_INVALID_ARG; }
    pad_states_kernel<<<grid_for(nst), 256, 0, st>>>(const_cast<float*>(p.c_initial), const_cast<float*>(p.n_initial),
                                                     const_cast<float*>(pp.c_initial), const_cast<float*>(pp.n_initial),
                                                     p.B * p.NH, p.DHQK, p.DHV, l.DP, 1);
    if ((rc = pad_launched("pad_states"))) return rc;
  }
  if ((rc = tc_fwd(pp, st))) return rc;
  if (pad_v && (rc = pad_rows(p, l.DP, job(p.h, pp.h, p.DHV), no_job(), no_job(), 0, st, "crop_rows"))) return rc;
  if (p.c_last) {
    pad_states_kernel<<<grid_for(nst), 256, 0, st>>>(p.c_last, p.n_last, pp.c_last, pp.n_last, p.B * p.NH, p.DHQK, p.DHV, l.DP, 0);
    if ((rc = pad_launched("crop_states"))) return rc;
  }
  return MLSTM_OK;
}

int tcpad_bwd(const mlstm_params& p, cudaStream_t st, int part) {
  mlstm_params pp;
  PadLayout l;
  int rc = make_padded(p, 1, &pp, &l);   // q, k, v, h, the initial states: the copies the forward left in the states buffer
  if (rc) return rc;
  const bool zc = zero_copy(pp);
  const bool pad_qk = p.DHQK != l.DP && !zc, pad_v = p.DHV != l.DP && !zc;
  ExtentScope ext;
  if (zc) {
    ext.add(p.q.ptr, p.DHQK); ext.add(p.k.ptr, p.DHQK); ext.add(p.dq.ptr, p.DHQK); ext.add(p.dk.ptr, p.DHQK);
    ext.add(p.v.ptr, p.DHV); ext.add(p.h.ptr, p.DHV); ext.add(p.dh.ptr, p.DHV); ext.add(p.dv.ptr, p.DHV);
    return tc_bwd(pp, st, part);
  }
  if (pad_v && (rc = pad_rows(p, l.DP, job(p.dh, pp.dh, p.DHV), no_job(), no_job(), 1, st, "pad_rows"))) return rc;
  if ((rc = tc_bwd(pp, st, part))) return rc;
  // all of them after either part: which part produces dq depends on the variant (the fused walk writes everything in part 1)
  return pad_rows(p, l.DP, pad_qk ? job(p.dq, pp.dq, p.DHQK) : no_job(), pad_qk ? job(p.dk, pp.dk, p.DHQK) : no_job(),
                  pad_v ? job(p.dv, pp.dv, p.DHV) : no_job(), 0, st, "crop_rows");
}

}  // namespace

namespace {

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// Null check for every family; for the tcgen05 family (bf16, TMA tensor maps over the caller's strided storage) also
// the layout the tensor maps need, so a bad view is reported by name here and not as a cuTensorMapEncodeTiled code later.
int check_act(const char* name, const mlstm_act& a, bool required, bool tma, const mlstm_params& p, int dh) {
  if (!a.ptr) {
    if (required) { set_error("%s: null pointer", name); return MLSTM_ERR_INVALID_ARG; }
    return MLSTM_OK;
  }
  if (!tma) return MLSTM_OK;
  if (!aligned16(a.ptr)) {
    set_error("%s: base pointer %p is not 16-byte aligned (TMA needs it; pass an aligned view or a copy)", name, a.ptr);
    return MLSTM_ERR_INVALID_ARG;
  }
  const int64_t st[3] = {a.stride_b, a.stride_h, a.stride_s};
  const int32_t ext[3] = {p.B, p.NH, p.S};
  const char* which[3] = {"batch", "head", "token"};
  for (int d = 0; d < 3; ++d) {
    if (ext[d] <= 1) continue;   // the stride of a size-1 dimension is never used
    if (st[d] % 8 != 0 || st[d] < dh) {
      set_error("%s: %s stride %lld elements must be a multiple of 8 and >= the head dim %d (bf16 TMA rows are 16-byte units)",
                name, which[d], (long long)st[d], dh);
      return MLSTM_ERR_INVALID_ARG;
    }
  }
  return MLSTM_OK;
}

int validate(const mlstm_params* p, int is_bwd) {
  if (!p) { set_error("params is NULL"); return MLSTM_ERR_INVALID_ARG; }
  if (p->abi_version != MLSTM_B200_ABI_VERSION) {
    set_error("abi_version %d != %d", p->abi_version, MLSTM_B200_ABI_VERSION);
    return MLSTM_ERR_INVALID_ARG;
  }
  if (p->B < 0 || p->NH <= 0 || p->S < 0 || p->DHQK <= 0 || p->DHV <= 0) {
    set_error("bad sizes B=%d NH=%d S=%d DHQK=%d DHV=%d", p->B, p->NH, p->S, p->DHQK, p->DHV);
    return MLSTM_ERR_INVALID_ARG;
  }
  if (p->dtype != MLSTM_F32 && p->dtype != MLSTM_BF16) {
    set_error("unsupported dtype %d", p->dtype);
    return MLSTM_ERR_UNSUPPORTED;
  }
  if (p->gate_mode != MLSTM_IGATE_EXP && p->gate_mode != MLSTM_IGATE_SIGMOID) {
    set_error("unknown gate_mode %d", p->gate_mode);
    return MLSTM_ERR_INVALID_ARG;
  }
  if (p->B == 0 || p->S == 0) return MLSTM_OK;  // empty input: nothing to do
  int rc;
  const bool tma = p->dtype == MLSTM_BF16 && (tc_supported(*p) || pad_path(*p));
  if ((rc = check_act("q", p->q, true, tma, *p, p->DHQK)) || (rc = check_act("k", p->k, true, tma, *p, p->DHQK)) ||
      (rc = check_act("v", p->v, true, tma, *p, p->DHV)) || (rc = check_act("h", p->h, true, tma, *p, p->DHV)))
    return rc;
  if (!p->i.ptr || !p->f.ptr) { set_error("gate pre-activations i/f: null pointer"); return MLSTM_ERR_INVALID_ARG; }
  if ((p->c_last != nullptr) != (p->n_last != nullptr) || (p->c_last != nullptr) != (p->m_last != nullptr)) {
    set_error("c_last/n_last/m_last must be given together");
    return MLSTM_ERR_INVALID_ARG;
  }
  if ((p->n_row != nullptr) != (p->m_row != nullptr)) {
    set_error("n_row/m_row must be given together");
    return MLSTM_ERR_INVALID_ARG;
  }
  if (is_bwd) {
    if ((rc = check_act("dh", p->dh, true, tma, *p, p->DHV)) || (rc = check_act("dq", p->dq, true, tma, *p, p->DHQK)) ||
        (rc = check_act("dk", p->dk, true, tma, *p, p->DHQK)) || (rc = check_act("dv", p->dv, true, tma, *p, p->DHV)))
      return rc;
    if (!p->di.ptr || !p->df.ptr) { set_error("di/df: null pointer"); return MLSTM_ERR_INVALID_ARG; }
    if (!p->n_row || !p->m_row) { set_error("backward needs n_row and m_row from the forward"); return MLSTM_ERR_INVALID_ARG; }
    size_t need = mlstm_b200_workspace_bytes(p, 1);
    if (need && (!p->workspace || p->workspace_bytes < need)) {
      set_error("workspace too small: have %zu, need %zu", p->workspace ? p->workspace_bytes : (size_t)0, need);
      return MLSTM_ERR_WORKSPACE;
    }
    if (need && !aligned16(p->workspace)) { set_error("workspace must be 16-byte aligned"); return MLSTM_ERR_INVALID_ARG; }
  }
  return MLSTM_OK;
}

}  // namespace

// Bind the device that owns the buffers to the calling thread.  PyTorch runs the backward on
// an autograd worker thread that may not have a current CUDA context yet, and the driver-side
// tensor-map encoder needs one.
int bind_device(const void* dev_ptr) {
  cudaPointerAttributes attr;
  cudaError_t e = cudaPointerGetAttributes(&attr, dev_ptr);
  if (e != cudaSuccess || attr.type != cudaMemoryTypeDevice) {
    (void)cudaGetLastError();
    set_error("q does not point to device memory (%s)", e == cudaSuccess ? "host/unregistered pointer" : cudaGetErrorString(e));
    return MLSTM_ERR_INVALID_ARG;
  }
  // Once per thread and device: later calls only check that the device is still current.  (cudaFree is not allowed while a
  // stream of the process is being captured into a CUDA graph; with the binding cached, forward and backward are plain kernel
  // launches and can be captured.)
  thread_local int bound = -1;
  int cur = -1;
  if (bound == attr.device && cudaGetDevice(&cur) == cudaSuccess && cur == attr.device) return MLSTM_OK;
  e = cudaSetDevice(attr.device);
  if (e == cudaSuccess) e = cudaFree(nullptr);   // forces the primary context current on this thread
  if (e == cudaSuccess) bound = attr.device;
  if (e != cudaSuccess) {
    set_error("cudaSetDevice(%d): %s", attr.device, cudaGetErrorString(e));
    return MLSTM_ERR_CUDA;
  }
  return MLSTM_OK;
}

namespace {

enum Family { FAM_NONE = 0, FAM_SIMT = 1, FAM_TC = 2, FAM_TCPAD = 3 };

Family pick(const mlstm_params& p) {
  if (p.dtype == MLSTM_BF16 && tc_supported(p)) return FAM_TC;
  if (pad_path(p)) return FAM_TCPAD;
  if (simt_supported(p)) return FAM_SIMT;
  return FAM_NONE;
}

}  // namespace
}  // namespace mlstm

using namespace mlstm;

extern "C" {

int mlstm_b200_abi_version(void) { return MLSTM_B200_ABI_VERSION; }

size_t mlstm_b200_workspace_bytes(const mlstm_params* p, int is_backward) {
  if (!p || p->B <= 0 || p->S <= 0) return 0;
  if (!is_backward) return 0;
  switch (pick(*p)) {
    case FAM_TC: return tc_bwd_workspace(*p);
    case FAM_TCPAD: return pad_layout(*p).ws_total;
    case FAM_SIMT: return simt_bwd_workspace(*p);
    default: return 0;
  }
}

size_t mlstm_b200_state_bytes(const mlstm_params* p) {
  if (!p || p->B <= 0 || p->S <= 0) return 0;
  const Family fam = pick(*p);
  return fam == FAM_TC ? tc_state_bytes(*p) : (fam == FAM_TCPAD ? pad_layout(*p).total : 0);
}

const char* mlstm_b200_kernel_name(const mlstm_params* p, int /*is_backward*/) {
  if (!p) return nullptr;
  switch (pick(*p)) {
    case FAM_TC: return "tcgen05";
    case FAM_TCPAD: return "tcgen05";
    case FAM_SIMT: return "simt";
    default: return nullptr;
  }
}

const char* mlstm_b200_kernel_variant(const mlstm_params* p, int is_backward) {
  if (!p) return nullptr;
  mlstm_params pp_;
  if (pick(*p) == FAM_TCPAD) { pp_ = padded_params(*p); p = &pp_; }
  switch (pick(*p)) {
    case FAM_TC:
      if (is_backward) return tc_use_fused_bwd(*p) ? "fused_walk" : "chunk_parallel";
      return tc_use_two_phase(*p) ? "two_phase" : "single_pass";
    case FAM_SIMT: return "simt";
    default: return nullptr;
  }
}

int mlstm_b200_fwd(const mlstm_params* p, void* cuda_stream) {
  g_err[0] = 0;
  int rc = validate(p, 0);
  if (rc) return rc;
  if (p->B == 0 || p->S == 0) return MLSTM_OK;
  if ((rc = bind_device(p->q.ptr))) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(cuda_stream);
  switch (pick(*p)) {
    case FAM_TC: return tc_fwd(*p, st);
    case FAM_TCPAD: return tcpad_fwd(*p, st);
    case FAM_SIMT: return simt_fwd(*p, st);
    default:
      set_error("no kernel for dtype=%d DHQK=%d DHV=%d", p->dtype, p->DHQK, p->DHV);
      return MLSTM_ERR_UNSUPPORTED;
  }
}

static int bwd_impl(const mlstm_params* p, int part, void* cuda_stream) {
  g_err[0] = 0;
  int rc = validate(p, 1);
  if (rc) return rc;
  if (part < -1 || part > 1) { set_error("bad backward part %d", part); return MLSTM_ERR_INVALID_ARG; }
  if (p->B == 0 || p->S == 0) return MLSTM_OK;
  if ((rc = bind_device(p->q.ptr))) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(cuda_stream);
  switch (pick(*p)) {
    case FAM_TC: return tc_bwd(*p, st, part);
    case FAM_TCPAD: return tcpad_bwd(*p, st, part);
    case FAM_SIMT: return simt_bwd(*p, st, part);
    default:
      set_error("no kernel for dtype=%d DHQK=%d DHV=%d", p->dtype, p->DHQK, p->DHV);
      return MLSTM_ERR_UNSUPPORTED;
  }
}

int mlstm_b200_bwd(const mlstm_params* p, void* cuda_stream) { return bwd_impl(p, -1, cuda_stream); }

int mlstm_b200_bwd_part(const mlstm_params* p, int part, void* cuda_stream) { return bwd_impl(p, part, cuda_stream); }

uint64_t mlstm_b200_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

const char* mlstm_b200_last_error(void) { return g_err; }

}  // extern "C"
