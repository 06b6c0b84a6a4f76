/*
 * mlstm_b200.h — C ABI of the B200-native mLSTM cell (chunkwise matrix-memory LSTM, fwd + bwd).
 *
 * This is the drop-in boundary for the ONE hot path of DJT777/xlstm-yolo that this repo
 * accelerates.  The reference has no native ABI for this path: it reaches the arithmetic
 * through the Python operator seam
 *
 *     mlstm_kernels.torch.backend_module.mLSTMBackend.forward(q, k, v, i, f,
 *         c_initial=None, n_initial=None, m_initial=None, return_last_states=None, mode=None)
 *
 * called at  nn/modules/vision_lstm/vision_lstm2.py:912-948  (MatrixLSTMCell.forward),
 *            nn/modules/vision_lstm/mlstm_large.py:295-330   (mLSTMLayerVision.forward),
 *            nn/modules/vision_lstm/xlstm/xlstm_large/model.py:425-434,
 * and, on CPU, through the in-tree PyTorch functions
 *            nn/modules/vision_lstm/xlstm/blocks/mlstm/backends.py:149 (chunkwise_simple),
 *            :93 (recurrent_step_stabilized_simple), :9 (parallel_stabilized_simple).
 * Each entry point below names the reference call it replaces.  INTEGRATION.md shows the
 * ctypes stub a maintainer of the reference would add.
 *
 * Conventions
 *   - Plain C: raw device pointers, element strides, sizes.  No torch / C++ types.
 *   - The caller (PyTorch) owns every buffer, including the workspace; the library borrows
 *     pointers for the duration of the launch, allocates nothing persistent on the device
 *     and keeps no mutable global state except a launch counter and a thread-local error
 *     string.  All work is enqueued on the CUDA stream passed in; no host synchronisation;
 *     after one warm-up call on the thread (which binds the device) the calls can be captured
 *     into a CUDA graph.
 *   - Every function returns 0 on success or a negative mlstm_status; no C++ exception
 *     crosses the ABI.  mlstm_b200_last_error() describes the last failure on this thread.
 *   - Re-entrant: forward is called from the main thread, backward from autograd's worker
 *     thread; DDP is one process per GPU.
 *   - Tensors q,k,v,h,dh,dq,dk,dv are logically (B, NH, S, DH) with arbitrary element
 *     strides for B, NH, S and unit stride for DH — so the reference's native
 *     (B, S, NH, DH) storage viewed as (B, NH, S, DH) (vision_lstm2.py:900-902) is consumed
 *     without a .contiguous() copy.  Gates i,f / di,df are fp32 (B, NH, S) with strides.
 */
#ifndef MLSTM_B200_H_
#define MLSTM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MLSTM_B200_ABI_VERSION 5

typedef enum mlstm_status {
  MLSTM_OK = 0,
  MLSTM_ERR_INVALID_ARG = -1,   /* null pointer, bad size, misaligned pointer/stride        */
  MLSTM_ERR_UNSUPPORTED = -2,   /* head dim / dtype combination without a kernel            */
  MLSTM_ERR_WORKSPACE = -3,     /* workspace missing or too small                            */
  MLSTM_ERR_CUDA = -4,          /* a CUDA runtime / driver call failed (see last_error)      */
  MLSTM_ERR_NO_DEVICE = -5      /* no sm_100 device / driver entry points unavailable        */
} mlstm_status;

typedef enum mlstm_igate { MLSTM_IGATE_EXP = 0, MLSTM_IGATE_SIGMOID = 1 } mlstm_igate;

typedef enum mlstm_dtype {
  MLSTM_F32 = 0,   /* fp32 I/O, fp32 SIMT arithmetic ("fp32 mode", tolerance 1e-4)          */
  MLSTM_BF16 = 1   /* bf16 I/O, tcgen05 bf16 MMAs with fp32 accumulation (tolerance 1e-2)   */
} mlstm_dtype;

/* One strided (B, NH, S, DH) activation tensor; innermost stride is 1 element. */
typedef struct mlstm_act {
  void* ptr;
  int64_t stride_b, stride_h, stride_s; /* in elements */
} mlstm_act;

/* One strided fp32 (B, NH, S) per-token scalar tensor (gate pre-activations and their grads). */
typedef struct mlstm_gate {
  float* ptr;
  int64_t stride_b, stride_h, stride_s; /* in elements */
} mlstm_gate;

typedef struct mlstm_params {
  int32_t abi_version;  /* must be MLSTM_B200_ABI_VERSION */
  int32_t B, NH, S;     /* batch, heads, tokens (S = H*W of the feature map) */
  int32_t DHQK, DHV;    /* head dims of q/k and of v/h */
  int32_t dtype;        /* mlstm_dtype of q,k,v,h,dh,dq,dk,dv */
  int32_t reverse;      /* 0: scan from token 0 (ROWWISE_FROM_TOP_LEFT);
                           1: scan from token S-1 (ROWWISE_FROM_BOT_RIGHT) — replaces the
                              flip pair at vision_lstm2.py:479-480,505-506 */
  int32_t chunk_size;   /* the reference's config knob (vision_lstm2.py:823); results do not
                           depend on it, the kernels pick their own tile */
  float eps;            /* normaliser epsilon (5e-5 in MatrixLSTMCell, vision_lstm2.py:827) */
  float qk_scale;       /* 0 -> DHQK^-1/2 (backends.py:168) */

  /* forward inputs */
  mlstm_act q, k, v;
  mlstm_gate i, f;                      /* gate pre-activations, fp32 */
  const float* c_initial;               /* optional (B,NH,DHQK,DHV) contiguous fp32, or NULL */
  const float* n_initial;               /* optional (B,NH,DHQK)     contiguous fp32, or NULL */
  const float* m_initial;               /* optional (B,NH)          contiguous fp32, or NULL */
  /* forward outputs */
  mlstm_act h;
  float* n_row;                         /* (B,NH,S) contiguous fp32: signed normaliser sum   */
  float* m_row;                         /* (B,NH,S) contiguous fp32: stabiliser m_t          */
                                        /* both may be NULL when no backward will follow     */
  float* c_last; float* n_last; float* m_last; /* optional last states, shapes as *_initial */

  /* backward inputs (in addition to q,k,v,i,f,h,n_row,m_row and *_initial above) */
  mlstm_act dh;
  /* backward outputs */
  mlstm_act dq, dk, dv;
  mlstm_gate di, df;

  void* workspace;                      /* device scratch, >= mlstm_b200_workspace_bytes()  */
  size_t workspace_bytes;

  /* Per-chunk entry states (bf16 C, fp32 n, m for every 128-token chunk), written by the
   * forward's state kernel and read by its chunk-parallel kernel and by the backward.  Size
   * mlstm_b200_state_bytes(); keep it with q,k,v,i,f,h,n_row,m_row until the backward has run.
   * 0 bytes (NULL allowed) for the SIMT kernel family.  For bf16 head dims other than
   * DHQK = DHV in {64, 128, 256} the buffer also holds the zero-padded copies of q, k, v, h and of the
   * initial / last states the tensor-core kernels run on (the backward reads them back from here);
   * 256-byte aligned in that case. */
  void* states;
  size_t states_bytes;

  /* Input gate: MLSTM_IGATE_EXP (0) = exponential input gate with max-stabiliser m, the arithmetic of
   * chunkwise_simple (backends.py:149-263) and of upstream's "chunkwise--native_autograd";
   * MLSTM_IGATE_SIGMOID (1) = sigmoid input gate ("...xl_chunk_siging", the kernel string HEAD asks for
   * on CUDA, vision_lstm2.py:835,866): log-gate logsigmoid(i), no stabiliser (m == 0, m_initial ignored,
   * m_row / m_last written as 0), normaliser max(|n|, 1) + eps. */
  int32_t gate_mode;
  int32_t reserved_;
} mlstm_params;

/* ---------------------------------------------------------------------------------------------
 * Gate projection of the cell (reference: vision_lstm2.py:895-897 -- cat[q,k,v] followed by the two
 * nn.Linear(3*dim, NH) `igate` / `fgate`).  Forward reads q, k, v in place (no concatenation) and
 * writes both gate pre-activations; backward adds the gates' contribution to the cell's dq, dk, dv
 * IN PLACE and produces the weight / bias gradients (deterministic two-stage reduction).
 * Rows are tokens: q, k, v (and dq, dk, dv) are (T, D) with row stride `ld` elements, D % 8 == 0,
 * 16-byte aligned; weights fp32 (NH, 3*D) row-major exactly as nn.Linear stores them (columns
 * [q | k | v]); i, f, di, df fp32 (T, NH) row-major, i.e. (B,S,NH) storage that the cell kernels
 * read as (B,NH,S) strided views. */
typedef struct mlstm_gate_proj_params {
  int32_t abi_version;                  /* MLSTM_B200_ABI_VERSION */
  int32_t T;                            /* tokens (B * S) */
  int32_t D;                            /* cell dim = NH * DH */
  int32_t NH;
  int32_t dtype;                        /* mlstm_dtype of q,k,v,dq,dk,dv */
  int64_t ld;                           /* row stride of q,k,v (elements) */
  const void *q, *k, *v;
  const float *w_i, *w_f;               /* (NH, 3*D) */
  const float *b_i, *b_f;               /* (NH) or NULL */
  float *i, *f;                         /* forward outputs (T, NH) */
  const float *di, *df;                 /* backward inputs (T, NH) */
  void *dq, *dk, *dv;                   /* backward in/out (T, D): dx += di W_i[:, x] + df W_f[:, x] */
  int64_t ld_d;                         /* row stride of dq,dk,dv (elements; ABI 4: independent of `ld`, the
                                           cell's gradients are dense even when q,k,v are column slices) */
  float *dw_i, *dw_f;                   /* backward outputs (NH, 3*D), overwritten */
  float *db_i, *db_f;                   /* backward outputs (NH), overwritten; NULL allowed */
  void* workspace;                      /* >= mlstm_b200_gates_workspace_bytes() (backward only) */
  size_t workspace_bytes;
} mlstm_gate_proj_params;

/* 1 when the gate kernels take a (T, D) operand with row stride ld: D % 8 == 0, ld % 8 == 0, ld >= D and
 * the 8 x 3D fp32 weight tile fits in shared memory (D <= 2133). */
int mlstm_b200_gates_supported(int D, int64_t ld);
size_t mlstm_b200_gates_workspace_bytes(const mlstm_gate_proj_params* p);
int mlstm_b200_gates_fwd(const mlstm_gate_proj_params* p, void* cuda_stream);
int mlstm_b200_gates_bwd(const mlstm_gate_proj_params* p, void* cuda_stream);

/* ---------------------------------------------------------------------------------------------
 * Fused tail of a ViL layer (reference: vision_lstm2.py:950 out-norm -- MultiHeadLayerNorm :1309-1325,
 * weight applied as 1 + w -- then :498 `+ learnable_skip * conv_act` and :499 `* silu(z)`):
 *     y = (LN_head(h) * (1 + w) + b + skip * c) * silu(z)
 * in one pass, and its backward (dh, dc, dz and the parameter gradients) in one pass.  Rows are
 * tokens; h is the cell output with heads merged, (T, D) over the (B,S,NH,DH) storage the cell
 * kernels write; every operand has its own row stride in elements (z is a column slice of proj_up's
 * output).  D % 256 == 0, D <= 2048, DH = D / NH divides 256; all pointers 16-byte aligned. */
typedef struct mlstm_glue_params {
  int32_t abi_version;                  /* MLSTM_B200_ABI_VERSION */
  int32_t T, D, NH;
  int32_t dtype;                        /* mlstm_dtype of h, c, z, y and their gradients */
  float eps;                            /* out-norm epsilon (1e-3 at vision_lstm2.py:812) */
  const void* h;  int64_t ld_h;
  const void* c;  int64_t ld_c;         /* conv_act */
  const void* z;  int64_t ld_z;
  const float* w;                       /* out-norm weight (D), applied as 1 + w; NULL = 0 */
  const float* b;                       /* out-norm bias (D) or NULL */
  const float* skip;                    /* learnable_skip (D); NULL = 1 */
  void* y;        int64_t ld_y;         /* forward output */
  const void* dy; int64_t ld_dy;        /* backward input */
  void* dh;       int64_t ld_dh;        /* backward outputs */
  void* dc;       int64_t ld_dc;
  void* dz;       int64_t ld_dz;
  float *dw, *db, *dskip;               /* (D) fp32, overwritten; each may be NULL */
  void* workspace;                      /* >= mlstm_b200_glue_workspace_bytes() (backward only) */
  size_t workspace_bytes;
} mlstm_glue_params;

/* 1 when the fused tail handles (D, NH): D % 256 == 0 with D / 256 in {1, 2, 4, 8}, DH = D / NH a multiple of 8
 * dividing 256. */
int mlstm_b200_glue_supported(int D, int NH);
size_t mlstm_b200_glue_workspace_bytes(const mlstm_glue_params* p);
int mlstm_b200_glue_fwd(const mlstm_glue_params* p, void* cuda_stream);
int mlstm_b200_glue_bwd(const mlstm_glue_params* p, void* cuda_stream);

/* ---------------------------------------------------------------------------------------------
 * Producer of the cell's operands (ABI 5; SURVEY.md 8 row f2).  Reference, four separate HBM round trips
 * over (B,S,inner) in ViLLayer.forward (vision_lstm2.py:482-491):
 *     x_conv = SequenceConv2d(x_mlstm)        vision_lstm_util.py:96-129  depthwise 3x3 over the H x W token grid, zero padded
 *     c      = silu(x_conv)
 *     q, k   = LinearHeadwiseExpand(c)        vision_lstm2.py:987-1022    block-diagonal: one (d, d) matrix per head + bias
 *     v      = LinearHeadwiseExpand(x_mlstm)
 * Here one kernel: a 128-token x d-channel tile of x (with its halo rows) is staged in shared memory once,
 * the conv + SiLU runs on it, and the three projections are tcgen05 MMAs on the staged tiles; c, q, k, v
 * leave through TMA stores.  Rows are tokens of a row-major (GH x GW) grid per batch element; x is (B*S, D)
 * with row stride ld_x elements (a column slice of proj_up's output), outputs dense (ld = D).
 * `rotate` = 1 convolves with the kernel rotated by 180 degrees (the ROWWISE_FROM_BOT_RIGHT layer on the
 * un-flipped sequence).  x_dtype 0: bf16, 1: fp16 (the trainer's autocast dtype; wv then has to be fp16
 * too: the v projection runs as an fp16 x fp16 MMA); outputs are always bf16, what the cell kernels read. */
typedef struct mlstm_qkv_params {
  int32_t abi_version;                  /* MLSTM_B200_ABI_VERSION */
  int32_t B, GH, GW;                    /* batch, token grid (S = GH * GW) */
  int32_t D, NH;                        /* inner dim, projection blocks; d = D / NH in {64, 128} */
  int32_t rotate;
  int32_t x_dtype;                      /* 0 bf16, 1 fp16 */
  const void* x;   int64_t ld_x;
  const float* conv_w;                  /* (D, 3, 3) fp32 */
  const float* conv_b;                  /* (D) fp32 or NULL */
  const void *wq, *wk, *wv;             /* (NH, d, d) [out][in]; wq, wk bf16; wv in x_dtype */
  const float *bq, *bk, *bv;            /* (D) fp32, each may be NULL */
  void *c, *q, *k, *v;                  /* (B*S, D) bf16, dense */
  void* sp;                             /* optional (B*S, D) bf16, dense: silu'(conv(x)), what mlstm_b200_conv_bwd needs (training);
                                           NULL in inference */
} mlstm_qkv_params;

/* 1 when the producer handles the shape: d = D / NH in {64, 128}, GW <= 80 (halo rows staged on chip),
 * ld_x % 8 == 0. */
int mlstm_b200_qkv_supported(int D, int NH, int GH, int GW, int64_t ld_x);
int mlstm_b200_qkv_fwd(const mlstm_qkv_params* p, void* cuda_stream);
/* Backward of the three projections (ABI 5): the five GEMMs of LinearHeadwiseExpand's backward (vision_lstm2.py:1016-1021 under
 * autograd) and the bias sums in one kernel,
 *     dxc = dc + dq Wq + dk Wk            (gradient w.r.t. c = silu(conv(x)); dc: what reaches c from the layer tail's skip)
 *     dxv = dv Wv                         (the v projection's share of the gradient w.r.t. x)
 *     dWq = dq^T c,  dWk = dk^T c,  dWv = dv^T x            (per block, fp32, deterministic two-stage reduction over tiles)
 *     db  = column sums of dq | dk | dv
 * The depthwise conv's own backward (du = dxc * silu'(u), dx = conv^T(du) + dxv) stays with cuDNN.  All (T, D) operands dense
 * except x (row stride ld_x); bf16 except x (x_dtype). */
typedef struct mlstm_qkv_bwd_params {
  int32_t abi_version;                  /* MLSTM_B200_ABI_VERSION */
  int32_t T, D, NH;                     /* rows (B * S), inner dim, projection blocks; d = D / NH in {64, 128} */
  int32_t x_dtype;                      /* 0 bf16, 1 fp16 */
  int32_t reserved_;
  const void* x;   int64_t ld_x;
  const void* c;                        /* saved forward output c */
  const void *dq, *dk, *dv;
  const void* dc;                       /* or NULL */
  const void *wq, *wk, *wv;             /* (NH, d, d) [out][in], bf16 */
  void *dxc, *dxv;                      /* outputs (T, D) bf16 */
  float *dwq, *dwk, *dwv;               /* outputs (NH, d, d) fp32 */
  float* db;                            /* output (3, D) fp32, or NULL */
  void* workspace;                      /* >= mlstm_b200_qkv_bwd_workspace_bytes() */
  size_t workspace_bytes;
} mlstm_qkv_bwd_params;
size_t mlstm_b200_qkv_bwd_workspace_bytes(const mlstm_qkv_bwd_params* p);
int mlstm_b200_qkv_bwd(const mlstm_qkv_bwd_params* p, void* cuda_stream);

/* Backward of the depthwise conv + SiLU in front of the projections (ABI 5): with du = dxc * sp (sp = silu'(conv(x)) saved by
 * mlstm_b200_qkv_fwd),
 *     dx  = conv^T(du) + dxv             (the transposed depthwise 3x3 conv; dxv from mlstm_b200_qkv_bwd)
 *     dwc = sum over tokens of du (x) x  (per channel, 3 x 3),  dbc = sum over tokens of du
 * in one kernel: a tile of x and of dxc with one grid row + 1 of halo on each side is staged once, du is formed in place,
 * dx leaves in x's dtype; the weight gradients go through per-CTA partials reduced in fixed order (deterministic).
 * Replaces cuDNN's dgrad / wgrad, the conv recompute, silu_backward and the final add (and the channels-last copies
 * cuDNN makes of the strided x). */
typedef struct mlstm_conv_bwd_params {
  int32_t abi_version;                  /* MLSTM_B200_ABI_VERSION */
  int32_t B, GH, GW;                    /* batch, token grid (S = GH * GW) */
  int32_t D, NH;                        /* inner dim, channel blocks (d = D / NH in {64, 128}) */
  int32_t rotate;                       /* as in the forward */
  int32_t x_dtype;                      /* 0 bf16, 1 fp16: dtype of x and of dx */
  const void* x;   int64_t ld_x;
  const void *dxc, *dxv, *sp;           /* (B*S, D) bf16, dense */
  const float* conv_w;                  /* (D, 3, 3) fp32 */
  void* dx;                             /* output (B*S, D) in x_dtype, dense */
  float* dwc;                           /* output (D, 3, 3) fp32 */
  float* dbc;                           /* output (D) fp32, or NULL */
  void* workspace;                      /* >= mlstm_b200_conv_bwd_workspace_bytes() */
  size_t workspace_bytes;
} mlstm_conv_bwd_params;
size_t mlstm_b200_conv_bwd_workspace_bytes(const mlstm_conv_bwd_params* p);
int mlstm_b200_conv_bwd(const mlstm_conv_bwd_params* p, void* cuda_stream);

/* Bias gradients of the three projections (the backward of vision_lstm2.py:1016-1021's `+ bias`): out[j*D + col] = sum over
 * the T rows of src[j] (bf16, row stride ld elements, D % 8 == 0), j = 0..n_src-1 (n_src <= 3), in one streaming pass with a
 * fixed-order (deterministic) two-stage reduction.  workspace >= mlstm_b200_colsum_workspace_bytes(D, n_src) bytes. */
size_t mlstm_b200_colsum_workspace_bytes(int D, int n_src);
int mlstm_b200_colsum(const void* const* src, int n_src, int T, int D, int64_t ld, float* out, void* workspace,
                      size_t workspace_bytes, void* cuda_stream);

/* Library / ABI identification. */
int mlstm_b200_abi_version(void);

/* Scratch bytes the given call needs (0 is possible). is_backward: 0 fwd, 1 bwd. */
size_t mlstm_b200_workspace_bytes(const mlstm_params* p, int is_backward);

/* Bytes of the per-chunk state buffer `states` the given call needs (0 for the SIMT family). */
size_t mlstm_b200_state_bytes(const mlstm_params* p);

/* Forward: h = mLSTM(q,k,v,i,f[,C0,n0,m0]) (+ n_row, m_row, last states).
 * Replaces mLSTMBackend.forward at vision_lstm2.py:912-948 / chunkwise_simple backends.py:149. */
int mlstm_b200_fwd(const mlstm_params* p, void* cuda_stream);

/* Backward: (dq,dk,dv,di,df) from dh, recomputing the gate/decay matrices per chunk.
 * Replaces the autograd backward of the same backend call (trainer: engine/trainer.py:389). */
int mlstm_b200_bwd(const mlstm_params* p, void* cuda_stream);

/* Profiling aid: run only one kernel of the backward (part 0 = dq / forward-walk kernel,
 * part 1 = dk,dv,di,df / reverse-walk kernel; part 0 must have run before part 1 on the same
 * workspace).  mlstm_b200_bwd(p) == part 0 then part 1.  Used by bench.py to time each kernel
 * with CUDA events. */
int mlstm_b200_bwd_part(const mlstm_params* p, int part, void* cuda_stream);

/* Name of the kernel family the call would dispatch to: "tcgen05" or "simt" (or NULL). */
const char* mlstm_b200_kernel_name(const mlstm_params* p, int is_backward);

/* Variant inside the family for this shape on the current device.  Forward: "single_pass" (one CTA
 * walks all chunks of a (batch, head) pair, state on chip) or "two_phase" (light sequential state
 * kernel + persistent chunk-parallel kernel, chunk states in `states`).  Backward: "fused_walk" (one
 * CTA per (batch, head) pair walks the chunks in reverse from the chunk states in `states`) or
 * "chunk_parallel" (persistent chunk-parallel kernels around one sequential adjoint-state kernel).
 * "simt" for the SIMT family. */
const char* mlstm_b200_kernel_variant(const mlstm_params* p, int is_backward);

/* Kernels launched by this library in this process so far (for bench.py's gpu_launches). */
uint64_t mlstm_b200_launch_count(void);

/* Human-readable description of the last error on the calling thread ("" if none). */
const char* mlstm_b200_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* MLSTM_B200_H_ */
