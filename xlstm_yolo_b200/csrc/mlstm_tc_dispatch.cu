// Shape/dtype gate and kernel-variant selection of the tcgen05 family.
//   forward : single pass (mlstm_tc_fwd.cu) | two-phase (mlstm_tc_fwd2p.cu)
//   backward: fused single walk (mlstm_tc_bwd_fused.cu, DH = 64; mlstm_tc_bwd_fused128.cu, DH = 128) |
//             chunk-parallel two-phase (mlstm_tc_bwd.cu)
//   DH = 256: two-phase forward and chunk-parallel backward only (mlstm_tc_256.cu)
// The single-pass forward runs one CTA per (batch, head) with the state on chip: best when there are
// enough heads to fill the GPU or the per-head chunk chain is short.  The two-phase kernels spill
// per-chunk states to HBM and are chunk-parallel: best for long sequences / small batches.
#include <cstdlib>

#include "tc_common.cuh"
namespace mlstm {

bool tc_supported(const mlstm_params& p) {
  return p.dtype == MLSTM_BF16 && p.DHQK == p.DHV && (p.DHQK == 64 || p.DHQK == 128 || p.DHQK == 256);
}

// of the device that owns the tensors, not of whichever device is current when a size query is made
static int sm_count(const mlstm_params& p) { return sm_count_of(p.q.ptr); }

// MLSTM_FORCE_VARIANT="<f><b>" pins a variant whatever the shape (the tests run the wide-batch kernels on small
// shapes this way): f = 1 single-pass / 2 two-phase forward, b = 2 chunk-parallel / 3 fused-walk backward; any
// other character = automatic.
static int forced(int which) {
  static const char* env = getenv("MLSTM_FORCE_VARIANT");
  if (!env || !env[0] || !env[1]) return 0;
  const char c = env[which];
  if (which == 0) return c == '1' || c == '2' ? c - '0' : 0;
  return c == '2' || c == '3' ? c - '0' : 0;
}

bool tc_use_two_phase(const mlstm_params& p) {          // forward
  if (p.DHQK == 256) return true;                       // mlstm_tc_256.cu: chunk-parallel only
  if (forced(0)) return forced(0) == 2;
  return p.B * p.NH * 2 <= sm_count(p) && tc::num_chunks(p.S) >= 4;
}

// Enough (batch, head) pairs to fill the GPU: one reverse walk per (batch, head) producing dq, dk, dv together from the
// forward's chunk states, at any sequence length — it reads every tile once, so it also beats the chunk-parallel kernels on
// long sequences (B32 NH4 DH64: 244 vs 135 M tok/s at S=800, 309 vs 180 at S=1600).
bool tc_use_fused_bwd(const mlstm_params& p) {
  if (p.DHQK == 256) return false;
  if (forced(1)) return forced(1) == 3;
  return p.B * p.NH * 2 > sm_count(p);
}

// The chunk-state buffer is needed by the two-phase forward itself and by either backward whichever forward variant ran.
size_t tc_state_bytes(const mlstm_params& p) {
  // forward-only call (no saved rows => no backward will follow) through the single-pass forward: nothing reads the states
  if (!tc_use_two_phase(p) && p.n_row == nullptr) return 0;
  return tc::StateLayout(p.B, p.NH, p.S, p.DHQK).total;
}

}  // namespace mlstm
