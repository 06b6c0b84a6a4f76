// tcgen05 / TMEM / TMA forward kernel of the mLSTM cell for bf16 I/O, DH in {64, 128}.
//
// One CTA per (batch, head) walks the sequence in chunks of L = 128 tokens with the (C, n, m)
// state resident on chip.  18 warps in three roles:
//   16 compute warps  two groups of 8 (below); warp w owns tile rows / TMEM lanes 32*(w%4)..+31
//    1 control warp   lane 0 issues every TMA load/store and the S, H and C MMAs (pre-built descriptors),
//                     so no compute warp ever sits in an issue loop
//    1 gate warp      log-sigmoid cumsum / running-max scans of the gates, two chunks ahead
//   C  : fp32 accumulator in TMEM, updated by an accumulating MMA  C += Kbar^T V
//   Cb : bf16 copy of C in shared memory (MN-major B operand of  G = Q Cb)
//   n  : fp32 in TMEM (MMA against a ones tile) + an fp32 copy in shared memory
//   m  : scalar carried in shared memory
// Per chunk (reference: backends.py:149-263; variables as in DESIGN.md / oracle):
//   MMA1  S = Q K^T,  G = Q Cb                          (TMA-loaded swizzled tiles)
//   SIMT  gates of the NEXT chunk (log-sigmoid cumsum, running max) ; q.n_prev
//   SIMT  Kbar = kw * K in place;  MMA  C += Kbar^T V,  n += Kbar^T 1
//   SIMT  P = S * exp2(u - M) (causal) -> bf16 swizzled tile ; row sums
//   MMA2  H = P V   (into the TMEM columns S occupied)
//   SIMT  h = (H + w G) / (max(|n|, e^-m) + eps) -> bf16 staging tile -> TMA store
//   SIMT  Cb <- bf16(C),  C <- decay_next * C   (one TMEM pass per chunk)
// No intermediate (D matrix, gates, P) ever reaches HBM.  `reverse` walks the tokens from
// the end: tiles stay in memory order, the causal mask and the gate scans flip.
//
// The two compute groups work on the two dependency chains of a chunk concurrently:
//   group A (warps 0-7)   the score chain    wait S -> P = S * exp2(u - M) -> [MMA2 H = P V] -> h = (H + w G) / N
//   group B (warps 8-15)  the state chain    q . n_prev -> Kbar = kw K -> [state MMA] -> Cb <- bf16(C), C <- decay C, n
// A warp owns one half of the columns (two 32-column blocks).  The control lane polls the two hand-offs (P written, Kbar
// written) and issues MMA2 / the state MMA in whichever order they become ready; n += Kbar^T 1 goes out from a lane of
// group B, G = Q Cb from lane 0 of warp 1 once the state pass has refreshed Cb.  One CTA-wide barrier per chunk remains
// (gate ring, G of the next chunk after the state pass).  h is staged in its own tile (the state chain may still read K).
#include "tc_common.cuh"   // StateLayout / store_row32 (the per-chunk state buffer shared with the backward)

namespace mlstm {
namespace {

using namespace ptx;

constexpr int L = 128;                 // chunk rows
constexpr int CT = 512;                // compute threads (16 warps: 4 row groups x 4 column blocks)
constexpr int GT0 = CT + 32;           // first gate thread (after the control warp)
constexpr int NT = GT0 + 32;           // 576 threads = 18 warps
constexpr int TILE = L * 128;          // bytes of one [128 rows][64 bf16] swizzled tile
constexpr float LOG2E = 1.4426950408889634f;

struct FwdMaps { CUtensorMap q, k, v, h, cs; };   // cs: the per-chunk state buffer (2-D, rows of DH)

struct alignas(16) GateBuf {       // indexed by tile row
  float u2[L];         // u * log2e + log2(scale)   (exponent of P, scale folded in)
  float M2[L];         // M * log2e
  float wq[L];         // exp(m_prev - M) * scale   (row weight of the inter-chunk term)
  float mrow[L];       // m_t = b_t + M_t
  float kw[L];         // exp(u - M_L)              (key weight for the state update)
  float decay;         // exp(m_prev - M_L)
  float m_next;        // g + M_L
  float pad[2];
};

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void named_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
// log(sigmoid(x)) with fast intrinsics (abs error < 1e-7, enough for the bf16 path)
__device__ __forceinline__ float log_sigmoid_fast(float x) {
  return fminf(x, 0.f) - __logf(1.f + __expf(-fabsf(x)));
}

// Gate vectors of chunk `c` into `G`, computed by ONE warp (lane l owns scan-local indices
// 4l..4l+3), off the other warps' path.  Chunks are anchored at token 0 in both directions, so a
// partial chunk always has its invalid rows at the tile's end (TMA zero-fills / clips them); in
// reverse mode the partial chunk is simply the first one processed.
template <int DH>
__device__ __forceinline__ void compute_gates(GateBuf& G, const mlstm_params& p, int b, int h, int c, int lane,
                                              float m_prev, float scale) {
  if (p.gate_mode) m_prev = 0.f;   // sigmoid input gate: no stabiliser
  const int NCc = (p.S + L - 1) / L;
  const int mc = p.reverse ? (NCc - 1 - c) : c;
  const int tok0 = mc * L;
  const int nvalid = min(L, p.S - tok0);
  float ii[4], bs[4];
  int r[4];
  float run = 0.f;
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const int t = lane * 4 + e;
    const bool valid = t < nvalid;
    r[e] = (p.reverse && valid) ? (nvalid - 1 - t) : t;   // tile row of scan-local index t
    ii[e] = -INFINITY;
    float logf = 0.f;
    if (valid) {
      const int tok = tok0 + r[e];
      logf = log_sigmoid_fast(p.f.ptr[(int64_t)b * p.f.stride_b + (int64_t)h * p.f.stride_h + (int64_t)tok * p.f.stride_s]);
      ii[e] = igate_log(p, p.i.ptr[(int64_t)b * p.i.stride_b + (int64_t)h * p.i.stride_h + (int64_t)tok * p.i.stride_s]);
    }
    run += logf;
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
  const float l2s = log2f(scale);
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float M = p.gate_mode ? -bs[e] : fmaxf(m_prev, fmaxf(emax, cm[e]));   // sigmoid gate: m_t == 0
    G.u2[r[e]] = u[e] * LOG2E + l2s;
    G.M2[r[e]] = M * LOG2E;
    G.wq[r[e]] = __expf(m_prev - M) * scale;
    G.mrow[r[e]] = bs[e] + M;
    G.kw[r[e]] = __expf(u[e] - ML);
  }
  if (lane == 0) {
    G.decay = __expf(m_prev - ML);
    G.m_next = g_tot + ML;
  }
  __syncwarp();
}

template <int DH>
struct SmemWS {
  static constexpr int KT = DH / 64;
  static constexpr int TILE_C = DH * 128;
  alignas(1024) uint8_t q[KT * TILE];
  alignas(1024) uint8_t k[2][KT * TILE];
  alignas(1024) uint8_t v[KT * TILE];
  alignas(1024) uint8_t cb[KT * TILE_C];
  alignas(1024) uint8_t stage[KT * TILE];          // h of this chunk, for the TMA store
  alignas(1024) uint8_t ones[2048];
  GateBuf g[3];
  float n_prev[DH];
  float part_qn[2][L];                             // per column-half partials of q . n_prev (group B)
  float part_rs[2][L];                             // per column-half partials of the row sums of P (group A)
  uint64_t bar_q, bar_k[2], bar_v, bar_s, bar_g, bar_p, bar_h, bar_kb, bar_c, bar_qn;
  uint32_t tmem_base;
};

template <int DH>
__global__ void __launch_bounds__(NT, 1) tc_fwd_ws_kernel(const __grid_constant__ FwdMaps maps, const mlstm_params p,
                                                          const float scale) {
  constexpr int KT = DH / 64;
  constexpr int TILE_C = SmemWS<DH>::TILE_C;
  constexpr int NB = DH / 32;
  constexpr int GN = 256;                                    // threads per compute group
  constexpr uint32_t A_LBO_STATE = (DH == 128) ? TILE : 0;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  SmemWS<DH>& sm = *reinterpret_cast<SmemWS<DH>*>(smem_raw);
  if ((smem_u32(smem_raw) & 1023u) != 0) __trap();

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool compute = tid < CT;
  const bool grpA = tid < GN, grpB = compute && !grpA;
  const bool issuer = tid == CT;
  const bool gatew = tid >= GT0;
  const int rg = warp & 3;                                   // TMEM lane quadrant / row group
  const int ch = (warp >> 2) & 1;                            // column half of this warp inside its group
  const int cq = compute ? (warp >> 2) : 4;                  // prologue only: 16-warp (row group, column block) mapping
  const int row = rg * 32 + lane;
  const int bh = blockIdx.x, b = bh / p.NH, h = bh % p.NH;
  const int S = p.S, NC = (S + L - 1) / L;
  const bool has_init = p.c_initial != nullptr;
  const bool rev = p.reverse != 0;
  const bool save_states = p.states != nullptr && p.n_row != nullptr;
  const tc::StateLayout slay(p.B, p.NH, S, DH);
  __nv_bfloat16* Cs_g = reinterpret_cast<__nv_bfloat16*>(reinterpret_cast<uint8_t*>(p.states) + slay.cs_off) + (size_t)bh * NC * DH * DH;
  float* ns_g = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(p.states) + slay.ns_off) + (size_t)bh * NC * DH;
  float* ms_g = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(p.states) + slay.ms_off) + (size_t)bh * NC;

  if (issuer) {
    tma_prefetch_desc(&maps.q); tma_prefetch_desc(&maps.k); tma_prefetch_desc(&maps.v); tma_prefetch_desc(&maps.h);
    mbar_init(&sm.bar_q, 1); mbar_init(&sm.bar_k[0], 1); mbar_init(&sm.bar_k[1], 1); mbar_init(&sm.bar_v, 1);
    mbar_init(&sm.bar_s, 1); mbar_init(&sm.bar_g, 1); mbar_init(&sm.bar_p, GN); mbar_init(&sm.bar_h, 1); mbar_init(&sm.bar_kb, GN);
    mbar_init(&sm.bar_c, 2); mbar_init(&sm.bar_qn, GN);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(&sm.tmem_base, 512);
  for (int e = tid; e < 2048 / 4; e += NT) reinterpret_cast<uint32_t*>(sm.ones)[e] = 0x3F803F80u;
  if (!has_init) {
    for (int e = tid; e < KT * TILE_C / 16; e += NT) reinterpret_cast<uint4*>(sm.cb)[e] = make_uint4(0, 0, 0, 0);
    for (int e = tid; e < DH; e += NT) sm.n_prev[e] = 0.f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tm = sm.tmem_base;
  const uint32_t tS = tm, tG = tm + 128, tC = tm + 128 + DH, tN = tm + 128 + 2 * DH;
  const uint32_t tP = tm + 448;
  const uint32_t lane_sel = (uint32_t)(rg * 32) << 16;

  auto tok0_of = [&](int c) { return (rev ? (NC - 1 - c) : c) * L; };
  auto issue_loads = [&](uint8_t* dst, const CUtensorMap* map, uint64_t* bar, int c) {
    mbar_arrive_expect_tx(bar, KT * TILE);
    for (int kt = 0; kt < KT; ++kt) tma_load_4d(dst + kt * TILE, map, bar, kt * 64, tok0_of(c), h, b);
  };
  const uint64_t dQ = make_sdesc(smem_u32(sm.q), 16, 1024);
  const uint64_t dCbmn = make_sdesc(smem_u32(sm.cb), TILE_C, 1024), dVmn = make_sdesc(smem_u32(sm.v), TILE, 1024);
  const uint64_t dOnes = make_sdesc(smem_u32(sm.ones), 1024, 1024);
  const uint64_t dKk0 = make_sdesc(smem_u32(sm.k[0]), 16, 1024), dKmn0 = make_sdesc(smem_u32(sm.k[0]), A_LBO_STATE, 1024);
  constexpr uint64_t KBUF_STEP = (uint64_t)(KT * TILE) >> 4;
  auto kstep = [](int ks) { return (uint64_t)((((ks >> 2) * TILE) + (ks & 3) * 32) >> 4); };
  auto mnstep = [](int ks) { return (uint64_t)((ks * 2048) >> 4); };
  auto issue_mma1 = [&](int c, int part) {   // part 0: S = Q K^T (control lane), part 1: G = Q Cb (lane 0 of warp 1)
    if (part == 0) {
      const uint64_t dKk = dKk0 + (c & 1) * KBUF_STEP;
      constexpr uint32_t idS = make_idesc_bf16(128, 128, 0, 0);
#pragma unroll
      for (int ks = 0; ks < DH / 16; ++ks) umma_bf16_ss(tS, dQ + kstep(ks), dKk + kstep(ks), idS, ks > 0);
    } else {
      constexpr uint32_t idG = make_idesc_bf16(128, DH, 0, 1);
#pragma unroll
      for (int ks = 0; ks < DH / 16; ++ks) umma_bf16_ss(tG, dQ + kstep(ks), dCbmn + mnstep(ks), idG, ks > 0);
    }
    umma_commit(part == 0 ? &sm.bar_s : &sm.bar_g);
  };

  // ---- prologue: first loads, gates of chunk 0, initial state ------------------------------------------------------
  if (issuer) {
    issue_loads(sm.q, &maps.q, &sm.bar_q, 0);
    issue_loads(sm.k[0], &maps.k, &sm.bar_k[0], 0);
    issue_loads(sm.v, &maps.v, &sm.bar_v, 0);
  }
  if (gatew) compute_gates<DH>(sm.g[0], p, b, h, 0, lane, p.m_initial ? p.m_initial[bh] : 0.f, scale);
  __syncthreads();
  if (has_init) {
    const float d0 = sm.g[0].decay;
    if (row < DH && cq < NB) {
      const float* crow = p.c_initial + ((int64_t)bh * DH + row) * DH + cq * 32;
      float r[32];
#pragma unroll
      for (int x = 0; x < 32; ++x) r[x] = crow[x];
#pragma unroll
      for (int x = 0; x < 32; x += 8) {
        const int dv = cq * 32 + x;
        *reinterpret_cast<uint4*>(sm.cb + (dv >> 6) * TILE_C + swz128(row, dv & 63)) =
            make_uint4(pack_bf16x2(r[x], r[x + 1]), pack_bf16x2(r[x + 2], r[x + 3]), pack_bf16x2(r[x + 4], r[x + 5]),
                       pack_bf16x2(r[x + 6], r[x + 7]));
      }
#pragma unroll
      for (int x = 0; x < 32; ++x) r[x] *= d0;
      tmem_st32(tC + lane_sel + cq * 32, r);
      if (cq == 0) {
        const float n0 = p.n_initial[(int64_t)bh * DH + row];
        sm.n_prev[row] = n0;
#pragma unroll
        for (int x = 0; x < 32; ++x) r[x] = n0 * d0;
        tmem_st32(tN + lane_sel, r);
      }
      tmem_st_wait();
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
  }
  if (save_states && row < DH && cq < NB) {   // entry state of chunk 0
    uint32_t pk[16];
    const float* crow = has_init ? p.c_initial + ((int64_t)bh * DH + row) * DH + cq * 32 : nullptr;
#pragma unroll
    for (int x = 0; x < 32; x += 2) pk[x / 2] = has_init ? pack_bf16x2(crow[x], crow[x + 1]) : 0u;
    tc::store_row32(Cs_g + (size_t)row * DH + cq * 32, pk);
    if (cq == 0) ns_g[row] = has_init ? p.n_initial[(int64_t)bh * DH + row] : 0.f;
  }
  if (save_states && issuer) ms_g[0] = (p.m_initial && !p.gate_mode) ? p.m_initial[bh] : 0.f;
  if (issuer) {
    mbar_wait(&sm.bar_q, 0);
    mbar_wait(&sm.bar_k[0], 0);
    tc_fence_after();
    issue_mma1(0, 0);
  }
  if (tid == 32) {
    mbar_wait(&sm.bar_q, 0);
    tc_fence_after();
    issue_mma1(0, 1);
  }

  for (int c = 0; c < NC; ++c) {
    const uint32_t ph = c & 1;
    const bool last = (c + 1 == NC);
    const bool do_state = !last || p.c_last != nullptr;
    if (gatew) {
      if (c == 0 && NC > 1) {
        compute_gates<DH>(sm.g[1], p, b, h, 1, lane, sm.g[0].m_next, scale);
        named_sync(6, GN + 32);   // with group B, ahead of chunk 0's state pass (first reader: decay of chunk 1)
      }
      if (c + 2 < NC) compute_gates<DH>(sm.g[(c + 2) % 3], p, b, h, c + 2, lane, sm.g[(c + 1) % 3].m_next, scale);
      __syncthreads();
      continue;
    }
    GateBuf& G = sm.g[c % 3];
    const int tok0 = tok0_of(c);
    uint8_t* sk = sm.k[c & 1];

    if (issuer) {
      // ---- the control lane: loads as buffers die, MMA2 / state MMA as their operands are handed over ----------------------
      if (!last) issue_loads(sm.k[(c + 1) & 1], &maps.k, &sm.bar_k[(c + 1) & 1], c + 1);   // its last readers finished a chunk ago
      tma_store_wait_read<0>();                // h(c-1) has left the staging tile (group A restages behind bar_h)
      mbar_wait(&sm.bar_s, ph);                // S, G complete: Q's MMA readers are done
      mbar_wait(&sm.bar_g, ph);
      mbar_wait(&sm.bar_qn, ph);               // ... and so is group B's q . n_prev
      if (!last) issue_loads(sm.q, &maps.q, &sm.bar_q, c + 1);
      bool doneP = false, doneK = !do_state;
      mbar_wait(&sm.bar_v, ph);
      while (!(doneP && doneK)) {
        if (!doneP && mbar_try_wait(&sm.bar_p, ph)) {
          tc_fence_after();
          constexpr uint32_t idH = make_idesc_bf16(128, DH, 0, 1);
#pragma unroll
          for (int ks = 0; ks < L / 16; ++ks) umma_bf16_ts(tS, tP + ks * 8, dVmn + mnstep(ks), idH, ks > 0);
          umma_commit(&sm.bar_h);
          doneP = true;
        }
        if (!doneK && mbar_try_wait(&sm.bar_kb, ph)) {
          tc_fence_after();
          const uint64_t dKmn = dKmn0 + (c & 1) * KBUF_STEP;
          constexpr uint32_t idC = make_idesc_bf16(128, DH, 1, 1);
          const uint32_t acc0 = (c > 0 || has_init) ? 1u : 0u;
#pragma unroll
          for (int ks = 0; ks < L / 16; ++ks) umma_bf16_ss(tC, dKmn + mnstep(ks), dVmn + mnstep(ks), idC, (ks > 0) ? 1u : acc0);
          umma_commit(&sm.bar_c);              // (n += Kbar^T 1 goes out from a lane of group B: the second arrival)
          doneK = true;
        }
      }
      mbar_wait(&sm.bar_h, ph);
      if (do_state) mbar_wait(&sm.bar_c, ph);
      if (!last) issue_loads(sm.v, &maps.v, &sm.bar_v, c + 1);   // MMA2 and the state MMA were V's readers
      if (last && p.m_last) p.m_last[bh] = G.m_next;
      if (save_states && !last) ms_g[c + 1] = G.m_next;
    } else if (grpA) {
      // ---- group A: P, normaliser, h -----------------------------------------------------------------------------------
      mbar_wait(&sm.bar_s, ph);
      tc_fence_after();
      const float M2t = G.M2[row];
      float rowsum = 0.f;
#pragma unroll
      for (int bb = 0; bb < 2; ++bb) {
        const int cb_ = 2 * ch + bb;                       // 32-column block of the 128-wide S tile
        const bool full = rev ? (cb_ > rg) : (cb_ < rg);
        const bool diag = (cb_ == rg);
        uint32_t packed[16];
        if (full || diag) {
          float s[32];
          tmem_ld32(tS + lane_sel + cb_ * 32, s);
          const uint32_t cbits = causal_bits(full, !rev, lane);
          tmem_ld_wait();
#pragma unroll
          for (int x = 0; x < 32; x += 4) {
            const float4 u4 = *reinterpret_cast<const float4*>(&G.u2[cb_ * 32 + x]);
            const float uu[4] = {u4.x, u4.y, u4.z, u4.w};
            float pv[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const bool keep = (cbits >> (x + e)) & 1u;
              pv[e] = keep ? s[x + e] * ex2(uu[e] - M2t) : 0.f;
              rowsum += pv[e];
            }
            packed[x / 2] = pack_bf16x2(pv[0], pv[1]);
            packed[x / 2 + 1] = pack_bf16x2(pv[2], pv[3]);
          }
        } else {
#pragma unroll
          for (int x = 0; x < 16; ++x) packed[x] = 0u;
        }
        tmem_st16(tP + lane_sel + cb_ * 16, packed);
      }
      sm.part_rs[ch][row] = rowsum;
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(&sm.bar_p);
      named_sync(2, GN);                                   // both column halves' row sums are published
      mbar_wait(&sm.bar_qn, ph);
      const float wq = G.wq[row];
      const float mrow = G.mrow[row];
      const float nr = (sm.part_rs[0][row] + sm.part_rs[1][row]) + wq * (sm.part_qn[0][row] + sm.part_qn[1][row]);
      const float inv = 1.f / (fmaxf(fabsf(nr), __expf(-mrow)) + p.eps);   // backends.py:249-252
      if (ch == 0) {
        const int tok = tok0 + row;
        if (p.n_row && tok < S) {
          p.n_row[(int64_t)bh * S + tok] = nr;
          p.m_row[(int64_t)bh * S + tok] = mrow;
        }
      }
      mbar_wait(&sm.bar_h, ph);
      mbar_wait(&sm.bar_g, ph);
      tc_fence_after();
#pragma unroll
      for (int bb = 0; bb < 2; ++bb) {
        const int cb_ = 2 * ch + bb;
        if (cb_ < NB) {
          float hi[32], gg[32];
          tmem_ld32(tS + lane_sel + cb_ * 32, hi);
          tmem_ld32(tG + lane_sel + cb_ * 32, gg);
          tmem_ld_wait();
#pragma unroll
          for (int x = 0; x < 32; x += 8) {
            const int dv = cb_ * 32 + x;
            uint32_t w4[4];
#pragma unroll
            for (int e = 0; e < 4; ++e)
              w4[e] = pack_bf16x2((hi[x + 2 * e] + wq * gg[x + 2 * e]) * inv, (hi[x + 2 * e + 1] + wq * gg[x + 2 * e + 1]) * inv);
            *reinterpret_cast<uint4*>(sm.stage + (dv >> 6) * TILE + swz128(row, dv & 63)) = make_uint4(w4[0], w4[1], w4[2], w4[3]);
          }
        }
      }
    } else if (grpB) {
      // ---- group B: q . n_prev, Kbar, state pass (the control warp's other lanes go straight to the chunk-end barrier) ------
      const int tb = tid - GN;
      mbar_wait(&sm.bar_q, ph);
      {
        float qn = 0.f;
#pragma unroll
        for (int x = 0; x < DH / 2; x += 8) {
          const int col = ch * (DH / 2) + x;
          const uint4 w = *reinterpret_cast<const uint4*>(sm.q + (col >> 6) * TILE + swz128(row, col & 63));
          const float4 n0 = *reinterpret_cast<const float4*>(&sm.n_prev[col]);
          const float4 n1 = *reinterpret_cast<const float4*>(&sm.n_prev[col + 4]);
          const __nv_bfloat162* qq = reinterpret_cast<const __nv_bfloat162*>(&w);
          const float2 a = __bfloat1622float2(qq[0]), bq = __bfloat1622float2(qq[1]), cq_ = __bfloat1622float2(qq[2]),
                       dq = __bfloat1622float2(qq[3]);
          qn += a.x * n0.x + a.y * n0.y + bq.x * n0.z + bq.y * n0.w + cq_.x * n1.x + cq_.y * n1.y + dq.x * n1.z + dq.y * n1.w;
        }
        sm.part_qn[ch][row] = qn;
      }
      mbar_arrive(&sm.bar_qn);
      if (do_state) {
        mbar_wait(&sm.bar_k[c & 1], (c >> 1) & 1);
        mbar_wait(&sm.bar_s, ph);                          // S is complete: K may be rescaled in place
#pragma unroll
        for (int it = 0; it < KT * TILE / 16 / GN; ++it) {
          const uint32_t o = (uint32_t)(tb + it * GN) * 16u;
          const int krow = (o >> 7) & (L - 1);
          const float s_ = G.kw[krow];
          uint4 w = *reinterpret_cast<uint4*>(sk + o);
          __nv_bfloat162* kk = reinterpret_cast<__nv_bfloat162*>(&w);
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            float2 f2 = __bfloat1622float2(kk[e]);
            kk[e] = __floats2bfloat162_rn(f2.x * s_, f2.y * s_);
          }
          *reinterpret_cast<uint4*>(sk + o) = w;
        }
        fence_proxy_async_smem();
        mbar_arrive(&sm.bar_kb);
        if (tb == 32) {   // n += Kbar^T 1 from a second MMA lane (lane 0 of this group's warp 1), once the whole group has handed Kbar over
          mbar_wait(&sm.bar_kb, ph);
          tc_fence_after();
          const uint64_t dKmn = dKmn0 + (c & 1) * KBUF_STEP;
          constexpr uint32_t idN = make_idesc_bf16(128, 16, 1, 1);
          const uint32_t acc0 = (c > 0 || has_init) ? 1u : 0u;
#pragma unroll
          for (int ks = 0; ks < L / 16; ++ks) umma_bf16_ss(tN, dKmn + mnstep(ks), dOnes, idN, (ks > 0) ? 1u : acc0);
          umma_commit(&sm.bar_c);
        }
        if (c == 0 && NC > 1) named_sync(6, GN + 32);      // chunk 1's gates (gate warp) are complete
        const float dnext = last ? 1.f : sm.g[(c + 1) % 3].decay;
        mbar_wait(&sm.bar_c, ph);
        tc_fence_after();
        if (row < DH) {
#pragma unroll
          for (int bb = 0; bb < 2; ++bb) {
            const int cb_ = 2 * ch + bb;
            if (cb_ < NB) {
              float r[32];
              tmem_ld32(tC + lane_sel + cb_ * 32, r);
              tmem_ld_wait();
              if (last && p.c_last) {
                float* dst = p.c_last + ((int64_t)bh * DH + row) * DH + cb_ * 32;
#pragma unroll
                for (int x = 0; x < 32; x += 4) *reinterpret_cast<float4*>(dst + x) = make_float4(r[x], r[x + 1], r[x + 2], r[x + 3]);
              }
#pragma unroll
              for (int x = 0; x < 32; x += 8) {
                const int dv = cb_ * 32 + x;
                *reinterpret_cast<uint4*>(sm.cb + (dv >> 6) * TILE_C + swz128(row, dv & 63)) =
                    make_uint4(pack_bf16x2(r[x], r[x + 1]), pack_bf16x2(r[x + 2], r[x + 3]), pack_bf16x2(r[x + 4], r[x + 5]),
                               pack_bf16x2(r[x + 6], r[x + 7]));
              }
              if (!last) {
#pragma unroll
                for (int x = 0; x < 32; ++x) r[x] *= dnext;
                tmem_st32(tC + lane_sel + cb_ * 32, r);
              }
              if (cb_ == 0) {
                float rn[16];
                tmem_ld16(tN + lane_sel, rn);
                tmem_ld_wait();
                sm.n_prev[row] = rn[0];
                if (save_states && !last) ns_g[(size_t)(c + 1) * DH + row] = rn[0];
                if (last && p.n_last) p.n_last[(int64_t)bh * DH + row] = rn[0];
                if (!last) {
#pragma unroll
                  for (int x = 0; x < 32; ++x) r[x] = rn[0] * dnext;
                  tmem_st32(tN + lane_sel, r);
                }
              }
            }
          }
          if (!last) tmem_st_wait();
        }
      } else if (c == 0 && NC > 1) {
        named_sync(6, GN + 32);
      }
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();   // end of chunk: everybody, including the gate warp
    if (issuer) {
      for (int kt = 0; kt < KT; ++kt) tma_store_4d(&maps.h, sm.stage + kt * TILE, kt * 64, tok0, h, b);
      if (save_states && !last)
        for (int kt = 0; kt < KT; ++kt) tma_store_2d(&maps.cs, sm.cb + kt * TILE_C, kt * 64, (bh * NC + c + 1) * DH);
      tma_store_commit();
      if (!last) {   // S of the next chunk (issuing it before the barrier, as soon as group A has read H and G, measured slower)
        mbar_wait(&sm.bar_q, ph ^ 1);
        mbar_wait(&sm.bar_k[(c + 1) & 1], ((c + 1) >> 1) & 1);
        tc_fence_after();
        issue_mma1(c + 1, 0);
      }
    }
    if (tid == 32 && !last) {   // G of the next chunk (Cb was refreshed by the state pass above)
      mbar_wait(&sm.bar_q, ph ^ 1);
      tc_fence_after();
      issue_mma1(c + 1, 1);
    }
  }
  if (issuer) tma_store_wait_all<0>();
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tm, 512);
}

template <int DH>
int launch_fwd(const mlstm_params& p, cudaStream_t st) {
  FwdMaps maps;
  int r = 0;
  r |= make_act_tmap(&maps.q, p.q.ptr, p.B, p.NH, p.S, DH, p.q.stride_b, p.q.stride_h, p.q.stride_s, L);
  r |= make_act_tmap(&maps.k, p.k.ptr, p.B, p.NH, p.S, DH, p.k.stride_b, p.k.stride_h, p.k.stride_s, L);
  r |= make_act_tmap(&maps.v, p.v.ptr, p.B, p.NH, p.S, DH, p.v.stride_b, p.v.stride_h, p.v.stride_s, L);
  r |= make_act_tmap(&maps.h, p.h.ptr, p.B, p.NH, p.S, DH, p.h.stride_b, p.h.stride_h, p.h.stride_s, L);
  maps.cs = maps.h;   // placeholder when no state buffer is given (never dereferenced then)
  if (p.states) {
    const tc::StateLayout slay(p.B, p.NH, p.S, DH);
    if (p.states_bytes < slay.total) {
      set_error("chunk-state buffer too small: %zu < %zu bytes", p.states_bytes, slay.total);
      return MLSTM_ERR_WORKSPACE;
    }
    r |= tc::make_state_tmap(&maps.cs, reinterpret_cast<uint8_t*>(p.states) + slay.cs_off,
                             (size_t)p.B * p.NH * tc::num_chunks(p.S) * DH, DH);
  }
  if (r) {
    set_error("cuTensorMapEncodeTiled failed (%d): pointers must be 16-byte aligned, strides multiples of 8 elements", r);
    return r == -1 ? MLSTM_ERR_NO_DEVICE : MLSTM_ERR_INVALID_ARG;
  }
  const size_t smem = sizeof(SmemWS<DH>) + 1024;
  cudaError_t e = set_max_smem_once(reinterpret_cast<const void*>(tc_fwd_ws_kernel<DH>), smem);
  if (e != cudaSuccess) {
    set_error("cudaFuncSetAttribute(tc_fwd, %zu B): %s", smem, cudaGetErrorString(e));
    return MLSTM_ERR_CUDA;
  }
  tc_fwd_ws_kernel<DH><<<dim3(p.B * p.NH), dim3(NT), smem, st>>>(maps, p, resolve_scale(p));
  count_launch();
  e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("tc_fwd launch failed: %s", cudaGetErrorString(e));
    return MLSTM_ERR_CUDA;
  }
  return MLSTM_OK;
}

}  // namespace

bool tc_use_two_phase(const mlstm_params& p);
int tc_fwd_two_phase(const mlstm_params& p, cudaStream_t st);

int tc_fwd(const mlstm_params& p, cudaStream_t st) {
  if (tc_use_two_phase(p)) return tc_fwd_two_phase(p, st);
  if (p.DHQK == 64) return launch_fwd<64>(p, st);
  return launch_fwd<128>(p, st);
}

}  // namespace mlstm
