// tcgen05 / TMEM / TMA backward of the mLSTM cell for bf16 I/O, DH in {64, 128}.
//
// Everything of size S x S (gate/decay matrices, dS, E) is recomputed per 128-token chunk from
// q,k,v,i,f and the per-row (n_t, m_t) saved by the forward; the only stored intermediates are the
// per-chunk states: the forward's entry states Cs/ns (DH^2/128 bf16 per token-head) and their
// adjoints dCs/dns produced here.  With the states in HBM every chunk is independent, so all heavy
// kernels are chunk-parallel persistent kernels that fill the GPU whatever the batch size:
//
//   A   (par)  dn_t, dS = (dH V^T / N + dn) * D,  dq = s [ dS K + w (dH Cs^T / N + dn ns) ],  R_t = q.dq
//   SB  (seq)  dC <- decay dC + ((w s / N) Q)^T dH ;  dn_state <- decay dn_state + Q^T (w s dn)
//              one CTA per (batch, head), reverse chunk order, one MMA + one TMEM pass per chunk
//   B1  (par)  dv = (s S^T D / N) dH + kw (K dCs)
//   B2  (par)  dk = s [ dS^T Q + (kw/s) V dCs^T ] + kw dns ;  K_j = k_j . dk_j
//   DF  (seq)  di = K ;  df = sigmoid(-f) * suffix_sum(R - K)        (tiny scan kernel)
//
// (s = qk scale, N_t = max(|n_t|, e^-m_t) + eps, D_tj = exp(u_j - M_t) causal; derivation and
// CPU emulation in tests/emu_kernel_dataflow.py.)  The parallel kernels share one skeleton:
// MMA1 (128x128 tile product) -> SIMT gating into a bf16 tile -> MMA2, with 16 compute warps,
// one control warp issuing all TMA / tcgen05.mma, one gate warp preparing the next item.
#include "tc_common.cuh"

namespace mlstm {
namespace {

using namespace tc;

enum { MODE_A = 0, MODE_B1 = 1, MODE_B2 = 2 };

// Developer aid (-DMLSTM_TIMELINE): CTA 0 of kernel A dumps clock64() stamps per item into the
// (otherwise unused by A) K-partials region of the workspace; see tests/gpu_tools/timeline_bwd.py.
#ifdef MLSTM_TIMELINE
#ifndef MLSTM_TL_MODE
#define MLSTM_TL_MODE 0   // which kernel of the chunk-parallel family is stamped: 0 = A, 2 = B2 (stamps go to the R partials)
#endif
#define TLB(k) do { if (MODE == MLSTM_TL_MODE && blockIdx.x == 0 && n < 8) { \
    if (threadIdx.x == 0) tlb[n * 32 + (k)] = clock64(); \
    if (threadIdx.x == CT) tlb[n * 32 + 16 + (k)] = clock64(); } } while (0)
// state walk (tests/gpu_tools/timeline_state.py): CTA (bh 0, block 0) stamps its first 8 steps into the R partials
#define TLS(k) do { if (bh == 0 && by == 0 && pc < 8) { \
    if (threadIdx.x == 0) tls[pc * 32 + (k)] = clock64(); \
    if (threadIdx.x == CT) tls[pc * 32 + 16 + (k)] = clock64(); } } while (0)
#else
#define TLB(k) do { } while (0)
#define TLS(k) do { } while (0)
#endif

struct BwdMaps { CUtensorMap t0, t1, t2, st, t3, h, out; };   // t3: q (A) / k (B2) rows for R and K; h: A only

// backward scratch (p.workspace)
struct BwdLayout {
  size_t dn_off, rpart_off, kpart_off, dcs_off, dns_off, flow_off, total;
  int nparts, nblk;   // 32-column partial slots of R / K per row; 128 x 128 state blocks per chunk (flow partials)
  __host__ __device__ BwdLayout(int B, int NH, int S, int DH) {
    const size_t rows = (size_t)B * NH * S, items = (size_t)B * NH * num_chunks(S);
    nparts = DH > 128 ? DH / 32 : 4;
    nblk = DH > 128 ? (DH / 128) * (DH / 128) : 1;
    dn_off = 0;
    rpart_off = dn_off + rows * 4;
    kpart_off = rpart_off + nparts * rows * 4;
    dcs_off = (kpart_off + nparts * rows * 4 + 255) & ~(size_t)255;
    dns_off = dcs_off + items * DH * DH * 2;
    flow_off = (dns_off + items * DH * 4 + 255) & ~(size_t)255;   // fp32 per chunk (x nblk): <dC, C> + <dn, n> across its entry boundary
    total = (flow_off + items * nblk * 4 + 255) & ~(size_t)255;
  }
};

// 32 columns [32 cb, 32 cb + 32) of row `row` of a swizzled [128][DH] bf16 tile set -> fp32
template <int DH>
__device__ __forceinline__ void tile_row32(const uint8_t* tile, int row, int cb, float (&out)[32]) {
#pragma unroll
  for (int x = 0; x < 32; x += 8) {
    const int col = cb * 32 + x;
    const uint4 w = *reinterpret_cast<const uint4*>(tile + (col >> 6) * TILE + swz128(row, col & 63));
    const __nv_bfloat162* qq = reinterpret_cast<const __nv_bfloat162*>(&w);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 f2 = __bfloat1622float2(qq[e]);
      out[x + 2 * e] = f2.x;
      out[x + 2 * e + 1] = f2.y;
    }
  }
}

// =============================================================================================
// Chunk-parallel kernels A / B1 / B2
//   tiles:  A : t0 = dH, t1 = V, t2 = K, st = Cs     thread row = query t
//           B1: t0 = K,  t1 = Q, t2 = dH, st = dCs   thread row = key j
//           B2: t0 = V,  t1 = dH, t2 = Q, st = dCs   thread row = key j
//
// TMEM (512 columns): tS[2] (128 each)  MMA1 output S = t0 t1^T, double-buffered in A: the MMA1 of the next
//                                       item is issued right behind the MMA2 of the current one and runs
//                                       under its epilogue (A: MMA2 writes dQ over the consumed S)
//                     tO (128)          A: G = dH Cs^T          B: intra accumulator  X t2
//                     tP (64)           the gated tile (dS | E^T | dS^T) as packed bf16: the A operand of MMA2,
//                                       read by the tensor core straight from TMEM (no shared-memory round trip)
//                     tI (128, B only)  inter accumulator  t0 dCs(^T)  (row scale kw applied in the epilogue,
//                                       so K / V are never modified in shared memory).  B needs a single S
//                                       buffer: MMA2 writes tO, so S is free as soon as the gated tile is built
// =============================================================================================
template <int DH>
struct SmemB {
  static constexpr int KT = DH / 64;
  static constexpr int TILE_C = DH * 128;
  alignas(1024) uint8_t t0[KT * TILE];
  alignas(1024) uint8_t t1[KT * TILE];
  alignas(1024) uint8_t t2[KT * TILE];
  alignas(1024) uint8_t st[KT * TILE_C];
  alignas(1024) uint8_t x[2 * TILE];               // A: h tile | B: gated bf16 tile (K-major) -> output staging
  alignas(1024) uint8_t t3[KT * TILE];             // q (A) / k (B2): rows for R = q.dq / K = k.dk
  GateBuf g[3];                                    // ring: the gate warp runs two items ahead
  alignas(16) float vecf[3][DH];                   // ns (A) / dns (B2) of the item
  float part[4][L];
  uint64_t bar_t0, bar_t1, bar_t2, bar_st, bar_t3, bar_h, bar_m1, bar_i, bar_m2;
  uint32_t tmem_base;
};

// cta / ncta: this CTA's index and the number of CTAs sharing the item list (B1 and B2 run side by side
// in one launch, each on its own slice of the grid — see tc_bwd_b12_kernel)
template <int DH, int MODE>
__device__ __forceinline__ void par_body(const BwdMaps& maps, const mlstm_params& p, const float scale, const int n_items,
                                         const int cta, const int ncta, const bool write_dn = true) {
  constexpr int KT = DH / 64;
  constexpr int TILE_C = SmemB<DH>::TILE_C;
  constexpr int NB = DH / 32;
  constexpr bool IS_A = (MODE == MODE_A);
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  SmemB<DH>& sm = *reinterpret_cast<SmemB<DH>*>(smem_raw);
  if ((smem_u32(smem_raw) & 1023u) != 0) __trap();

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool compute = tid < CT, issuer = tid == CT, gatew = tid >= GT0;
  const int rg = warp & 3, cq = compute ? (warp >> 2) : 4, row = rg * 32 + lane;
  const int S = p.S, NC = num_chunks(S);
  const bool rev = p.reverse != 0;
  const size_t rows_total = (size_t)p.B * p.NH * S;
  const StateLayout slay(p.B, p.NH, S, DH);
  const BwdLayout blay(p.B, p.NH, S, DH);
  uint8_t* ws = reinterpret_cast<uint8_t*>(p.workspace);
  float* ws_dn = reinterpret_cast<float*>(ws + blay.dn_off);
  float* ws_rpart = reinterpret_cast<float*>(ws + blay.rpart_off);
  float* ws_kpart = reinterpret_cast<float*>(ws + blay.kpart_off);
  const float* ns_all = reinterpret_cast<const float*>(reinterpret_cast<const uint8_t*>(p.states) + slay.ns_off);
  const float* dns_all = reinterpret_cast<const float*>(ws + blay.dns_off);
  const float l2s = log2f(scale);

  if (issuer) {
    tma_prefetch_desc(&maps.t0); tma_prefetch_desc(&maps.t1); tma_prefetch_desc(&maps.t2); tma_prefetch_desc(&maps.st);
    mbar_init(&sm.bar_t0, 1); mbar_init(&sm.bar_t1, 1); mbar_init(&sm.bar_t2, 1); mbar_init(&sm.bar_st, 1);
    mbar_init(&sm.bar_t3, 1); mbar_init(&sm.bar_h, 1);
    mbar_init(&sm.bar_m1, 1); mbar_init(&sm.bar_i, 1); mbar_init(&sm.bar_m2, 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(&sm.tmem_base, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  // A: tS[0] tS[1] tO=G tP(64)        B: tS tI tO tP(64)
  const uint32_t tm = sm.tmem_base, tO = tm + 256, tP = tm + 384, tI = tm + 128;
  const uint32_t lane_sel = (uint32_t)(rg * 32) << 16;

  const uint64_t d0k = make_sdesc(smem_u32(sm.t0), 16, 1024), d1k = make_sdesc(smem_u32(sm.t1), 16, 1024);
  const uint64_t d2mn = make_sdesc(smem_u32(sm.t2), TILE, 1024);
  const uint64_t dStk = make_sdesc(smem_u32(sm.st), 16, 1024), dStmn = make_sdesc(smem_u32(sm.st), TILE_C, 1024);
  auto coords = [&](int item, int& b, int& h, int& tok0) {
    const int bh = item / NC, sc = item % NC;
    b = bh / p.NH; h = bh % p.NH; tok0 = mem_chunk(sc, NC, rev) * L;
  };
  auto load_act = [&](uint8_t* dst, const CUtensorMap* map, uint64_t* bar, int item) {
    int b, h, tok0; coords(item, b, h, tok0);
    mbar_arrive_expect_tx(bar, KT * TILE);
    for (int kt = 0; kt < KT; ++kt) tma_load_4d(dst + kt * TILE, map, bar, kt * 64, tok0, h, b);
  };
  auto load_st = [&](int item) {
    mbar_arrive_expect_tx(&sm.bar_st, KT * TILE_C);
    for (int kt = 0; kt < KT; ++kt) tma_load_2d(sm.st + kt * TILE_C, &maps.st, &sm.bar_st, kt * 64, item * DH);
  };
  auto issue_mma1 = [&](uint32_t tS) {   // tS = t0 t1^T
    constexpr uint32_t id1 = make_idesc_bf16(128, 128, 0, 0);
#pragma unroll
    for (int ks = 0; ks < DH / 16; ++ks) umma_bf16_ss(tS, d0k + kstep(ks), d1k + kstep(ks), id1, ks > 0);
    umma_commit(&sm.bar_m1);
  };
  auto issue_state_mma = [&]() {   // the product with the chunk state; its result is needed in the epilogue only
    if (IS_A) {                    // G = dH Cs^T : Cs read as a K-major operand
      constexpr uint32_t idG = make_idesc_bf16(128, DH, 0, 0);
#pragma unroll
      for (int ks = 0; ks < DH / 16; ++ks) umma_bf16_ss(tO, d0k + kstep(ks), dStk + kstep(ks, TILE_C), idG, ks > 0);
    } else if (MODE == MODE_B1) {  // K dCs : dCs as MN-major B operand [dk][dv]
      constexpr uint32_t idI = make_idesc_bf16(128, DH, 0, 1);
#pragma unroll
      for (int ks = 0; ks < DH / 16; ++ks) umma_bf16_ss(tI, d0k + kstep(ks), dStmn + mnstep(ks), idI, ks > 0);
    } else {                       // V dCs^T : dCs as K-major B operand (rows dk)
      constexpr uint32_t idI = make_idesc_bf16(128, DH, 0, 0);
#pragma unroll
      for (int ks = 0; ks < DH / 16; ++ks) umma_bf16_ss(tI, d0k + kstep(ks), dStk + kstep(ks, TILE_C), idI, ks > 0);
    }
    umma_commit(&sm.bar_i);
  };
  auto prep_item = [&](int item, int slot) {   // gate warp
    int b, h, tok0; coords(item, b, h, tok0);
    const int bh = item / NC, sc = item % NC;
    GateBuf& G = sm.g[slot];
    gates_warp_bwd(G, p, b, h, bh, mem_chunk(sc, NC, rev), lane, MODE == MODE_B2 ? ws_dn : nullptr);
    for (int d = lane; d < DH; d += 32)
      sm.vecf[slot][d] = IS_A ? ns_all[(size_t)item * DH + d] : (MODE == MODE_B2 ? dns_all[(size_t)item * DH + d] : 0.f);
    __syncwarp();
  };

  // Items are (batch*head, chunk) pairs with id bh*NC + sc, walked head-major: this CTA takes cta, cta + ncta, ...
  // (measured on B200: no chunk-major order beats it; the kernels are not DRAM-bound)
  const int item0 = cta;   // ncta is never larger than n_items
  if (issuer) {
    load_act(sm.t0, &maps.t0, &sm.bar_t0, item0); load_act(sm.t1, &maps.t1, &sm.bar_t1, item0);
    load_st(item0); load_act(sm.t2, &maps.t2, &sm.bar_t2, item0);
    if (MODE != MODE_B1) load_act(sm.t3, &maps.t3, &sm.bar_t3, item0);
    if (IS_A) load_act(sm.x, &maps.h, &sm.bar_h, item0);
  }
  if (gatew) {
    prep_item(item0, 0);
    if (cta + ncta < n_items) prep_item(cta + ncta, 1);
  }
  __syncthreads();
  if (issuer) {
    mbar_wait(&sm.bar_t0, 0); mbar_wait(&sm.bar_t1, 0);
    tc_fence_after();
    issue_mma1(tm);
    mbar_wait(&sm.bar_st, 0);
    tc_fence_after();
    issue_state_mma();
  }

#ifdef MLSTM_TIMELINE
  long long* tlb = reinterpret_cast<long long*>(MLSTM_TL_MODE == 0 ? ws_kpart : ws_rpart);
#endif
  int n = 0;
  for (int item = cta; item < n_items; item += ncta, ++n) {
    TLB(0);
    const uint32_t ph = n & 1;
    const uint32_t tS = IS_A ? tm + ph * 128 : tm;   // B: S is dead once the gated tile is built, one buffer suffices
    const int next = item + ncta;
    const bool has_next = next < n_items;
    if (gatew) {
      if (item + 2 * ncta < n_items) prep_item(item + 2 * ncta, (n + 2) % 3);
      __syncthreads();
      continue;
    }
    const GateBuf& G = sm.g[n % 3];
    const float* vecf = sm.vecf[n % 3];
    int b, h, tok0; coords(item, b, h, tok0);
    const int bh = item / NC;
    const int tok = tok0 + row;
    const bool row_ok = compute && tok < S;
    const size_t grow = (size_t)bh * S + tok;          // index into the per-row workspace arrays

    // ---- A: dn_t = dnf_t (dh_t . h_t): block partials from the h tile (x) and the dH tile --------
    float dn_row = 0.f;
    if (IS_A) {
      mbar_wait(&sm.bar_h, ph);
      mbar_wait(&sm.bar_t0, ph);
      float part = 0.f;
      if (cq < NB) {
#pragma unroll
        for (int x8 = 0; x8 < 32; x8 += 8) {
          const int col = cq * 32 + x8;
          const uint32_t off = (col >> 6) * TILE + swz128(row, col & 63);
          const uint4 wh = *reinterpret_cast<const uint4*>(sm.x + off);
          const uint4 wd = *reinterpret_cast<const uint4*>(sm.t0 + off);
          const __nv_bfloat162* hh = reinterpret_cast<const __nv_bfloat162*>(&wh);
          const __nv_bfloat162* dd = reinterpret_cast<const __nv_bfloat162*>(&wd);
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float2 a = __bfloat1622float2(hh[e]), c2 = __bfloat1622float2(dd[e]);
            part = fmaf(a.x, c2.x, fmaf(a.y, c2.y, part));
          }
        }
      }
      if (compute) sm.part[cq][row] = part;
      if (compute) named_sync(3, CT);
      if (compute) {
        dn_row = G.dnf[row] * ((sm.part[0][row] + sm.part[1][row]) + (sm.part[2][row] + sm.part[3][row]));
        if (write_dn && cq == 0 && row_ok) ws_dn[grow] = dn_row;
      }
    }
    TLB(1);
    mbar_wait(&sm.bar_m1, ph);
    tc_fence_after();
    TLB(2);
    if (issuer) {
      // MMA1 and the state product of this item are complete: t0, t1, st can take the next item's tiles
      mbar_wait(&sm.bar_i, ph);
      if (has_next) {
        load_act(sm.t1, &maps.t1, &sm.bar_t1, next);
        load_act(sm.t0, &maps.t0, &sm.bar_t0, next);
        load_st(next);
      }
      // The previous item's output store must have read its staging tile (A: t3, B: x) before it is
      // touched again.  A refills t3 (this item's q rows, needed in the epilogue) right behind the wait;
      // B's epilogue writes x after the barrier that ends the gated-tile phase, which this warp joins.
      tma_store_wait_read<0>();
      if (IS_A && n > 0) load_act(sm.t3, &maps.t3, &sm.bar_t3, item);
    }
    TLB(3);
    // ---- gated bf16 tile: one 32x32 block per warp ----------------------------------------------
    if (compute) {
      // A : row = query t, col = key j   : keep j <= t (forward) / j >= t (reverse)
      // B : row = key j,   col = query t : keep t >= j (forward) / t <= j (reverse)
      const bool full = IS_A ? (rev ? (cq > rg) : (cq < rg)) : (rev ? (cq < rg) : (cq > rg));
      const bool diag = (cq == rg);
      uint32_t packed[16];
      if (full || diag) {
        float a[32];
        tmem_ld32(tS + lane_sel + cq * 32, a);
        const uint32_t cbits = causal_bits(full, IS_A ? !rev : rev, lane);
        tmem_ld_wait();
        const float r0 = IS_A ? G.M2[row] : (MODE == MODE_B1 ? G.u2[row] + l2s : G.u2[row]);
        const float r1 = IS_A ? G.invN[row] : 0.f;
#pragma unroll
        for (int x = 0; x < 32; x += 4) {
          const int c0 = cq * 32 + x;
          const float4 e4 = *reinterpret_cast<const float4*>(IS_A ? &G.u2[c0] : (MODE == MODE_B1 ? &G.c2[c0] : &G.M2[c0]));
          const float ee[4] = {e4.x, e4.y, e4.z, e4.w};
          float in4[4] = {0.f, 0.f, 0.f, 0.f}, dn4[4] = {0.f, 0.f, 0.f, 0.f};
          if (MODE == MODE_B2) {
            const float4 i4 = *reinterpret_cast<const float4*>(&G.invN[c0]);
            const float4 d4 = *reinterpret_cast<const float4*>(&G.dn[c0]);
            in4[0] = i4.x; in4[1] = i4.y; in4[2] = i4.z; in4[3] = i4.w;
            dn4[0] = d4.x; dn4[1] = d4.y; dn4[2] = d4.z; dn4[3] = d4.w;
          }
          float pv[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const bool keep = (cbits >> (x + e)) & 1u;
            float val;
            if (IS_A) val = fmaf(a[x + e], r1, dn_row) * ex2(ee[e] - r0);
            else if (MODE == MODE_B1) val = a[x + e] * ex2(r0 - ee[e]);
            else val = fmaf(a[x + e], in4[e], dn4[e]) * ex2(r0 - ee[e]);
            pv[e] = keep ? val : 0.f;
          }
          packed[x / 2] = pack_bf16x2(pv[0], pv[1]);
          packed[x / 2 + 1] = pack_bf16x2(pv[2], pv[3]);
        }
      } else {
#pragma unroll
        for (int x = 0; x < 16; ++x) packed[x] = 0u;
      }
      // the gated tile stays on the tensor-core side: packed bf16x2 into TMEM, the A operand of MMA2
      tmem_st16(tP + lane_sel + cq * 16, packed);
      tmem_st_wait();
    }
    TLB(4);
    tc_fence_before();
    named_sync(2, GT0);
    TLB(5);

    // ---- MMA2, then the next item's MMA1 right behind it ------------------------------------------
    if (issuer) {
      mbar_wait(&sm.bar_t2, ph);
      tc_fence_after();
      constexpr uint32_t id2 = make_idesc_bf16(128, DH, 0, 1);
      // A: dQ = dS K over the consumed S | B: intra accumulator = X t2 ; X (dS | E^T | dS^T) read from TMEM
#pragma unroll
      for (int ks = 0; ks < L / 16; ++ks) umma_bf16_ts(IS_A ? tS : tO, tP + ks * 8, d2mn + mnstep(ks), id2, ks > 0);
      umma_commit(&sm.bar_m2);
      if (has_next) {
        // A: every warp is past its h-tile reads (named barrier 3 precedes the barrier this thread just left).
        // (Letting the control warp join barrier 3 to issue this earlier was measured slower: it is still
        // draining the previous item's output store when the compute warps get there.)
        if (IS_A) load_act(sm.x, &maps.h, &sm.bar_h, next);
        mbar_wait(&sm.bar_t0, ph ^ 1); mbar_wait(&sm.bar_t1, ph ^ 1);
        tc_fence_after();
        issue_mma1(IS_A ? tm + (ph ^ 1) * 128 : tm);
      }
    }
    TLB(6);
    mbar_wait(&sm.bar_m2, ph);
    tc_fence_after();
    TLB(7);
    if (issuer && has_next) load_act(sm.t2, &maps.t2, &sm.bar_t2, next);   // MMA2 was t2's last reader

    // ---- epilogue: outputs packed in registers --------------------------------------------------
    uint32_t opk[16];
    float psum = 0.f;
    if (cq < NB) {
      float acc[32], gg[32];
      tmem_ld32((IS_A ? tS : tO) + lane_sel + cq * 32, acc);
      tmem_ld32((IS_A ? tO : tI) + lane_sel + cq * 32, gg);    // state product (complete by MMA issue order)
      tmem_ld_wait();
      if (IS_A) {
        const float wt = G.w[row], invN = G.invN[row];
        float qr[32];
        mbar_wait(&sm.bar_t3, ph);
        tile_row32<DH>(sm.t3, row, cq, qr);
#pragma unroll
        for (int x = 0; x < 32; x += 2) {
          const float o0 = scale * (acc[x] + wt * fmaf(gg[x], invN, dn_row * vecf[cq * 32 + x]));
          const float o1 = scale * (acc[x + 1] + wt * fmaf(gg[x + 1], invN, dn_row * vecf[cq * 32 + x + 1]));
          if (row_ok) psum = fmaf(qr[x], o0, fmaf(qr[x + 1], o1, psum));
          opk[x / 2] = pack_bf16x2(o0, o1);
        }
      } else if (MODE == MODE_B1) {   // dv = E^T dH + kw (K dC)
        const float kwj = G.kw[row];
#pragma unroll
        for (int x = 0; x < 32; x += 2) opk[x / 2] = pack_bf16x2(fmaf(kwj, gg[x], acc[x]), fmaf(kwj, gg[x + 1], acc[x + 1]));
      } else {                        // dk = s dS^T Q + kw (V dC^T + dn_state)
        const float kwj = G.kw[row];
        float kr[32];
        mbar_wait(&sm.bar_t3, ph);
        tile_row32<DH>(sm.t3, row, cq, kr);
#pragma unroll
        for (int x = 0; x < 32; x += 2) {
          const float o0 = fmaf(kwj, gg[x] + vecf[cq * 32 + x], scale * acc[x]);
          const float o1 = fmaf(kwj, gg[x + 1] + vecf[cq * 32 + x + 1], scale * acc[x + 1]);
          if (row_ok) psum = fmaf(kr[x], o0, fmaf(kr[x + 1], o1, psum));
          opk[x / 2] = pack_bf16x2(o0, o1);
        }
      }
    }
    // stage the output rows for one coalesced TMA store.  A: in t3, over the q rows — each thread has just
    // read exactly the (row, 32-column) block it now overwrites, and t3 is the tile needed latest in the
    // next item, so its refill can wait for the store to drain without stalling anything.  B: in x.
    uint8_t* stage = IS_A ? sm.t3 : sm.x;
    if (cq < NB) {
#pragma unroll
      for (int x4 = 0; x4 < 4; ++x4) {
        const int col = cq * 32 + x4 * 8;
        *reinterpret_cast<uint4*>(stage + (col >> 6) * TILE + swz128(row, col & 63)) =
            make_uint4(opk[4 * x4], opk[4 * x4 + 1], opk[4 * x4 + 2], opk[4 * x4 + 3]);
      }
    }
    if (row_ok) {
      if (IS_A) ws_rpart[(size_t)cq * rows_total + grow] = psum;
      if (MODE == MODE_B2) ws_kpart[(size_t)cq * rows_total + grow] = psum;
    }
    TLB(8);
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();   // end of item: accumulators consumed, next gates published (the gate warp joins here)
    TLB(9);
    if (issuer) {
      for (int kt = 0; kt < KT; ++kt) tma_store_4d(&maps.out, stage + kt * TILE, kt * 64, tok0, h, b);
      tma_store_commit();
      if (has_next) {
        if (MODE == MODE_B2) load_act(sm.t3, &maps.t3, &sm.bar_t3, next);   // k rows were consumed in the epilogue
        mbar_wait(&sm.bar_st, ph ^ 1);
        tc_fence_after();
        issue_state_mma();   // t0 of the next item landed before its MMA1 was issued
      }
    }
    TLB(10);
  }
  if (issuer) tma_store_wait_all<0>();
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tm, 512);
}

template <int DH, int MODE>
__global__ void __launch_bounds__(NT, 1) tc_bwd_par_kernel(const __grid_constant__ BwdMaps maps, const mlstm_params p,
                                                           const float scale, const int n_items) {
  par_body<DH, MODE>(maps, p, scale, n_items, blockIdx.x, gridDim.x);
}

// B1 (dv) and B2 (dk) side by side in one launch: CTAs [0, n_b2) run B2, the rest run B1, both walking
// the same item list in the same order.  Four of the five input tiles of an item (q, dh, dCs, and k)
// are common to both; whichever CTA comes second finds them in the 126 MB L2, so DRAM sees them once —
// the traffic of a fused dk/dv kernel without its shared-memory and TMEM bill.
template <int DH>
__global__ void __launch_bounds__(NT, 1) tc_bwd_b12_kernel(const __grid_constant__ BwdMaps maps1, const __grid_constant__ BwdMaps maps2,
                                                           const mlstm_params p, const float scale, const int n_items,
                                                           const int n_b2) {
  if ((int)blockIdx.x < n_b2) par_body<DH, MODE_B2>(maps2, p, scale, n_items, blockIdx.x, n_b2);
  else par_body<DH, MODE_B1>(maps1, p, scale, n_items, blockIdx.x - n_b2, gridDim.x - n_b2);
}

// =============================================================================================
// SB: sequential adjoint-state kernel (reverse chunk order), one CTA per (batch, head)
// =============================================================================================
template <int DH>
struct SmemSB {
  static constexpr int KT = DH / 64;
  alignas(1024) uint8_t q[2][KT * TILE];
  alignas(1024) uint8_t dh[2][KT * TILE];
  alignas(1024) uint8_t vec[2][2 * 2048];          // K-major [16][128 t] bf16: (dn N)_t in every row
  alignas(1024) uint8_t stage[KT * DH * 128];      // bf16 dC tile staged for the TMA store
  alignas(1024) uint8_t cst[KT * DH * 128];        // forward entry state Cs[sc] (bf16), for the boundary flow <dC, C>
  GateBuf g[3];
  float fpart[16];
  uint64_t bar_q[2], bar_dh[2], bar_mma[2], bar_cs;
  uint32_t tmem_base;
};

// The recurrence  dC_{sc-1} = decay_{sc-1} dC_sc + Qtilde_sc^T dH_sc  is split so that the tensor-core half does
// not wait for the SIMT half: the per-chunk update U = Qtilde^T dH (and its n column) goes into one of two
// alternating TMEM buffers with a fresh accumulation, the running state lives in a third TMEM region that only
// the state pass touches.  U of step pc+1 is therefore computed while the state pass of step pc runs.
// Head dims above the template's DH (DHF = p.DHQK = 256, DH = 128): gridDim.y = (DHF / DH)^2 independent blocks
// dC[row0 .. +DH)[col0 .. +DH) = f(Q columns row0.., dH columns col0..); column block 0 also carries the dn state.
// bh: the (batch, head) pair of this CTA, by: its block of the state (0 unless DHF > DH)
template <int DH>
__device__ __forceinline__ void state_bwd_body(const BwdMaps& maps, const mlstm_params& p, const float scale, const int bh,
                                               const int by) {
  constexpr int KT = DH / 64;
  constexpr int NB = DH / 32;
  const int DHF = p.DHQK, ncb = DHF / DH, nblk = ncb * ncb;
  const int row0 = (by / ncb) * DH, col0 = (by % ncb) * DH;
  constexpr uint32_t A_LBO = (DH == 128) ? TILE : 0;
  constexpr uint32_t TCOLS = 512;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  SmemSB<DH>& sm = *reinterpret_cast<SmemSB<DH>*>(smem_raw);
  if ((smem_u32(smem_raw) & 1023u) != 0) __trap();

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool compute = tid < CT, issuer = tid == CT, gatew = tid >= GT0;
  const int rg = warp & 3, cq = compute ? (warp >> 2) : 4, row = rg * 32 + lane;
  const int b = bh / p.NH, h = bh % p.NH;
  const int S = p.S, NC = num_chunks(S);
  const bool rev = p.reverse != 0;
  const BwdLayout blay(p.B, p.NH, S, DHF);
  uint8_t* ws = reinterpret_cast<uint8_t*>(p.workspace);
  const float* ws_dn = reinterpret_cast<const float*>(ws + blay.dn_off);
  __nv_bfloat16* dCs = reinterpret_cast<__nv_bfloat16*>(ws + blay.dcs_off) + (size_t)bh * NC * DHF * DHF;
  float* dns = reinterpret_cast<float*>(ws + blay.dns_off) + (size_t)bh * NC * DHF;

  if (issuer) {
    tma_prefetch_desc(&maps.t0); tma_prefetch_desc(&maps.t1);
    mbar_init(&sm.bar_q[0], 1); mbar_init(&sm.bar_q[1], 1); mbar_init(&sm.bar_dh[0], 1); mbar_init(&sm.bar_dh[1], 1);
    mbar_init(&sm.bar_mma[0], 1); mbar_init(&sm.bar_mma[1], 1); mbar_init(&sm.bar_cs, 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(&sm.tmem_base, TCOLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  // tU[b] = tm + b*DH (update of a step), tC = running state, tUn[b] / tN: their n columns (16 wide)
  const uint32_t tm = sm.tmem_base, tC = tm + 2 * DH, tUn0 = tm + 3 * DH, tN = tm + 3 * DH + 32;
  const uint32_t lane_sel = (uint32_t)(rg * 32) << 16;
  const StateLayout slay(p.B, p.NH, S, DHF);
  const float* ns_f = reinterpret_cast<const float*>(reinterpret_cast<const uint8_t*>(p.states) + slay.ns_off) + (size_t)bh * NC * DHF;
  float* flow = reinterpret_cast<float*>(ws + blay.flow_off) + (size_t)bh * NC * nblk;
  auto load_cs = [&](int sc) {   // forward entry state of chunk sc (t2 map = the Cs buffer)
    mbar_arrive_expect_tx(&sm.bar_cs, KT * DH * 128);
    for (int kt = 0; kt < KT; ++kt)
      tma_load_2d(sm.cst + kt * (DH * 128), &maps.t2, &sm.bar_cs, col0 + kt * 64, (bh * NC + sc) * DHF + row0);
  };

  // processing step pc = 0..NC-1 handles scan chunk sc = NC-1-pc
  auto sc_of = [&](int pc) { return NC - 1 - pc; };
  auto load_qd = [&](int pc) {
    const int buf = pc & 1, tok0 = mem_chunk(sc_of(pc), NC, rev) * L;
    mbar_arrive_expect_tx(&sm.bar_q[buf], KT * TILE);
    for (int kt = 0; kt < KT; ++kt) tma_load_4d(sm.q[buf] + kt * TILE, &maps.t0, &sm.bar_q[buf], row0 + kt * 64, tok0, h, b);
    mbar_arrive_expect_tx(&sm.bar_dh[buf], KT * TILE);
    for (int kt = 0; kt < KT; ++kt) tma_load_4d(sm.dh[buf] + kt * TILE, &maps.t1, &sm.bar_dh[buf], col0 + kt * 64, tok0, h, b);
  };
  auto gates_of = [&](int pc) {   // gate warp: G.w <- (w s / N)_t, row scale of the Q tile
    GateBuf& G = sm.g[pc % 3];
    gates_warp_bwd(G, p, b, h, bh, mem_chunk(sc_of(pc), NC, rev), lane, ws_dn);
    for (int r = lane; r < L; r += 32) G.w[r] = G.w[r] * scale * G.invN[r];
    __syncwarp();
  };
  // Qtilde = (w s / N) Q in place and the (dn N) vector tile of step pc
  auto prep_operands = [&](int pc) {
    const GateBuf& G = sm.g[pc % 3];
    scale_rows<DH>(sm.q[pc & 1], G.w, tid);
    if (tid < L) {
      const float inv = G.invN[tid];
      const __nv_bfloat16 bv = __float2bfloat16_rn(inv > 0.f ? G.dn[tid] / inv : 0.f);
      uint8_t* base = sm.vec[pc & 1] + (tid >> 6) * 2048;
#pragma unroll
      for (int r = 0; r < 16; ++r) *reinterpret_cast<__nv_bfloat16*>(base + swz128(r, tid & 63)) = bv;
    }
  };
  const uint64_t dQ0 = make_sdesc(smem_u32(sm.q[0]), A_LBO, 1024), dH0 = make_sdesc(smem_u32(sm.dh[0]), TILE, 1024);
  const uint64_t dVec0 = make_sdesc(smem_u32(sm.vec[0]), 16, 1024);
  constexpr uint64_t BUF_STEP = (uint64_t)(KT * TILE) >> 4, VEC_STEP = (uint64_t)(2 * 2048) >> 4;

  auto issue_update = [&](int pc) {   // U(pc) = Qtilde^T dH and its n column, fresh accumulation into buffer pc & 1
    const int buf = pc & 1;
    const uint64_t dQ = dQ0 + buf * BUF_STEP, dH_ = dH0 + buf * BUF_STEP, dVec = dVec0 + buf * VEC_STEP;
    constexpr uint32_t idC = make_idesc_bf16(128, DH, 1, 1), idN = make_idesc_bf16(128, 16, 1, 0);
#pragma unroll
    for (int ks = 0; ks < L / 16; ++ks) umma_bf16_ss(tm + buf * DH, dQ + mnstep(ks), dH_ + mnstep(ks), idC, ks > 0);
#pragma unroll
    for (int ks = 0; ks < L / 16; ++ks) umma_bf16_ss(tUn0 + buf * 16, dQ + mnstep(ks), dVec + kstep(ks, 2048), idN, ks > 0);
    umma_commit(&sm.bar_mma[buf]);
  };

  if (issuer) { load_qd(0); if (NC > 1) { load_qd(1); load_cs(NC - 1); } }
  if (gatew) { gates_of(0); if (NC > 1) gates_of(1); }
  // adjoint state leaving the last chunk is zero (the last states carry no gradient)
  if (row < DH && cq < NB) {
    uint32_t z[16];
#pragma unroll
    for (int x = 0; x < 16; ++x) z[x] = 0u;
    store_row32(dCs + ((size_t)(NC - 1) * DHF + row0 + row) * DHF + col0 + cq * 32, z);
    if (cq == 0 && col0 == 0) dns[(size_t)(NC - 1) * DHF + row0 + row] = 0.f;
  }
  __syncthreads();
  if (!gatew) mbar_wait(&sm.bar_q[0], 0);
  if (compute) prep_operands(0);
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  if (issuer && NC > 1) {
    mbar_wait(&sm.bar_dh[0], 0);
    tc_fence_after();
    issue_update(0);
  }

#ifdef MLSTM_TIMELINE
  long long* tls = reinterpret_cast<long long*>(ws + blay.rpart_off);
#endif
  for (int pc = 0; pc < NC; ++pc) {
    const bool last = (pc + 1 == NC);
    const int buf = pc & 1, sc = sc_of(pc);
    if (gatew) {
      if (pc + 2 < NC) gates_of(pc + 2);
      __syncthreads();
      continue;
    }
    if (last) break;   // the state leaving chunk -1 is not needed (initial states carry no gradient)
    const bool more = pc + 2 < NC;   // step pc+1 still produces a state
    TLS(0);
    // ---- operands and update of the next step, under this step's MMA / state pass --------------
    if (more) {
      mbar_wait(&sm.bar_q[buf ^ 1], ((pc + 1) >> 1) & 1);
      if (compute) prep_operands(pc + 1);
      fence_proxy_async_smem();
    }
    TLS(1);
    if (issuer) tma_store_wait_read<0>();   // the previous step's staged dC tile has left shared memory
    tc_fence_before();
    named_sync(2, GT0);
    TLS(2);
    if (issuer && more) {
      mbar_wait(&sm.bar_dh[buf ^ 1], ((pc + 1) >> 1) & 1);
      tc_fence_after();
      issue_update(pc + 1);
    }
    TLS(3);
    mbar_wait(&sm.bar_mma[buf], (pc >> 1) & 1);
    tc_fence_after();
    TLS(4);
    if (issuer && more) load_qd(pc + 2);   // q / dh of this step are free: U(pc) is complete

    // ---- state pass: dC_{sc-1} = (decayed running state) + U -> workspace (bf16), running state <- decay dC_{sc-1}
    const float dnext = sm.g[(pc + 1) % 3].decay;
    float fl = 0.f;   // partial of the boundary flow <dC_{sc-1}, Cs[sc]> + <dn_{sc-1}, ns[sc]>
    mbar_wait(&sm.bar_cs, pc & 1);
    TLS(5);
    if (row < DH && cq < NB) {
      float r[32];
      tmem_ld32(tm + buf * DH + lane_sel + cq * 32, r);
      if (pc > 0) {
        float acc[32];
        tmem_ld32(tC + lane_sel + cq * 32, acc);
        tmem_ld_wait();
#pragma unroll
        for (int x = 0; x < 32; ++x) r[x] += acc[x];
      } else {
        tmem_ld_wait();
      }
#pragma unroll
      for (int x = 0; x < 32; x += 8) {
        const int dv = cq * 32 + x;
        const uint4 wc = *reinterpret_cast<const uint4*>(sm.cst + (dv >> 6) * (DH * 128) + swz128(row, dv & 63));
        const __nv_bfloat162* cc = reinterpret_cast<const __nv_bfloat162*>(&wc);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 c2 = __bfloat1622float2(cc[e]);
          fl = fmaf(r[x + 2 * e], c2.x, fmaf(r[x + 2 * e + 1], c2.y, fl));
        }
      }
#pragma unroll
      for (int x = 0; x < 32; x += 8) {
        const int dv = cq * 32 + x;
        *reinterpret_cast<uint4*>(sm.stage + (dv >> 6) * (DH * 128) + swz128(row, dv & 63)) =
            make_uint4(pack_bf16x2(r[x], r[x + 1]), pack_bf16x2(r[x + 2], r[x + 3]), pack_bf16x2(r[x + 4], r[x + 5]),
                       pack_bf16x2(r[x + 6], r[x + 7]));
      }
      if (more) {
#pragma unroll
        for (int x = 0; x < 32; ++x) r[x] *= dnext;
        tmem_st32(tC + lane_sel + cq * 32, r);
      }
      if (cq == 0 && col0 == 0) {
        float rn[16], an[16];
        tmem_ld16(tUn0 + buf * 16 + lane_sel, rn);
        if (pc > 0) {
          tmem_ld16(tN + lane_sel, an);
          tmem_ld_wait();
          rn[0] += an[0];
        } else {
          tmem_ld_wait();
        }
        dns[(size_t)(sc - 1) * DHF + row0 + row] = rn[0];
        fl = fmaf(rn[0], ns_f[(size_t)sc * DHF + row0 + row], fl);
        if (more) {
#pragma unroll
          for (int x = 0; x < 32; ++x) r[x] = rn[0] * dnext;
          tmem_st32(tN + lane_sel, r);   // 16 columns used; the next 16 are scratch
        }
      }
      if (more) tmem_st_wait();
    }
    TLS(6);
    if (compute) {
      fl = warp_sum(fl);
      if (lane == 0) sm.fpart[warp] = fl;
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    TLS(7);
    if (tid == 0) {
      float f_ = 0.f;
#pragma unroll
      for (int w = 0; w < 16; ++w) f_ += sm.fpart[w];
      flow[sc * nblk + by] = f_;
    }
    if (issuer && sc - 1 > 0) load_cs(sc - 1);   // (the boundary before chunk 0 is the initial state: not needed)
    if (issuer) {   // dC_{sc-1} tile -> workspace; its shared-memory copy is rewritten one step later
      for (int kt = 0; kt < KT; ++kt)
        tma_store_2d(&maps.st, sm.stage + kt * (DH * 128), col0 + kt * 64, (bh * NC + (sc - 1)) * DHF + row0);
      tma_store_commit();
    }
    TLS(8);
  }
  if (issuer) tma_store_wait_all<0>();
  if (!gatew) { tc_fence_before(); __syncthreads(); }   // matches the gate warp's last in-loop barrier
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tm, TCOLS);
}

template <int DH>
__global__ void __launch_bounds__(NT, 1) tc_state_bwd_kernel(const __grid_constant__ BwdMaps maps, const mlstm_params p,
                                                             const float scale) {
  // block launches (DHF > DH): block index in blockIdx.x, so the CTAs sharing a Q or dH tile run side by side (L2 reuse)
  const bool blocks = p.DHQK != DH;
  state_bwd_body<DH>(maps, p, scale, blocks ? blockIdx.y : blockIdx.x, blocks ? blockIdx.x : blockIdx.y);
}

// The adjoint-state walk occupies only B*NH SMs and kernel A (dq) does not depend on it: with few (batch, head) pairs
// the two share ONE launch — CTAs [0, n_state) walk the states, the rest run A's item list — so the walk's 30-50 us
// hide A entirely.  The walk's only input from A, dn_t, then comes from tc_dn_kernel (A keeps its own copy in
// registers and does not write it).
template <int DH>
__global__ void __launch_bounds__(NT, 1) tc_bwd_sa_kernel(const __grid_constant__ BwdMaps maps_s, const __grid_constant__ BwdMaps maps_a,
                                                          const mlstm_params p, const float scale, const int n_items,
                                                          const int n_state) {
  if ((int)blockIdx.x < n_state) state_bwd_body<DH>(maps_s, p, scale, blockIdx.x, 0);
  else par_body<DH, MODE_A>(maps_a, p, scale, n_items, blockIdx.x - n_state, gridDim.x - n_state, false);
}

// dn_t = dnf_t (dh_t . h_t) for every row (the same formula as kernel A and gates_warp_bwd): DH / 8 lanes per row, one 16-byte
// load per lane and operand, DN_U rows per lane group with all their loads in flight.
constexpr int DN_U = 4;
__global__ void __launch_bounds__(256) tc_dn_kernel(const mlstm_params p, float* __restrict__ ws_dn, const int DH, const int dv_true) {
  const int lpr = DH / 8, rpw = 32 / lpr;                 // lanes per row, rows per warp and pass
  const int lane = threadIdx.x & 31, sub = lane / lpr, l = lane % lpr;
  const int rows = p.B * p.NH * p.S;                      // < 2^31: checked by the launcher
  const int r0 = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * (rpw * DN_U) + sub;
  const __nv_bfloat16* hp = reinterpret_cast<const __nv_bfloat16*>(p.h.ptr) + l * 8;
  const __nv_bfloat16* dp = reinterpret_cast<const __nv_bfloat16*>(p.dh.ptr) + l * 8;
  uint4 wh[DN_U], wd[DN_U];
  float nr[DN_U], mr[DN_U];
#pragma unroll
  for (int u = 0; u < DN_U; ++u) {
    const int r = r0 + u * rpw;
    wh[u] = wd[u] = make_uint4(0, 0, 0, 0);
    nr[u] = mr[u] = 0.f;
    if (r < rows && l * 8 < dv_true) {   // (columns past dv_true: a zero-padded problem on the caller's narrow rows)
      const int bh = r / p.S, t = r - bh * p.S, b = bh / p.NH, h = bh - b * p.NH;
      wh[u] = *reinterpret_cast<const uint4*>(hp + (int64_t)b * p.h.stride_b + (int64_t)h * p.h.stride_h + (int64_t)t * p.h.stride_s);
      wd[u] = *reinterpret_cast<const uint4*>(dp + (int64_t)b * p.dh.stride_b + (int64_t)h * p.dh.stride_h + (int64_t)t * p.dh.stride_s);
    }
    if (r < rows && l == 0) { nr[u] = p.n_row[r]; mr[u] = p.m_row[r]; }
  }
#pragma unroll
  for (int u = 0; u < DN_U; ++u) {
    const int r = r0 + u * rpw;
    const __nv_bfloat162* hh = reinterpret_cast<const __nv_bfloat162*>(&wh[u]);
    const __nv_bfloat162* dd = reinterpret_cast<const __nv_bfloat162*>(&wd[u]);
    float part = 0.f;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 a = __bfloat1622float2(hh[e]), c2 = __bfloat1622float2(dd[e]);
      part = fmaf(a.x, c2.x, fmaf(a.y, c2.y, part));
    }
    for (int o = lpr >> 1; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if (r < rows && l == 0) {
      const float floor_ = __expf(-mr[u]);
      const float N = fmaxf(fabsf(nr[u]), floor_) + p.eps;
      ws_dn[r] = (fabsf(nr[u]) >= floor_) ? (-copysignf(1.f, nr[u]) / N) * part : 0.f;
    }
  }
}

// =============================================================================================
// DF: di = K, df = sigmoid(-f) * suffix_sum(R - K) in scan order.  One 128-thread CTA per chunk:
// the suffix sum inside the chunk is re-anchored on flow[sc+1] = <dC, C> + <dn, n> across the
// boundary to the next chunk (written by SB).  In exact arithmetic that flow equals the sum of
// R - K over all later chunks; taking it from the states keeps the rounding noise of a long
// sequence from accumulating in df.
// =============================================================================================
__global__ void __launch_bounds__(L) tc_dfscan_kernel(const mlstm_params p, const int DH) {
  __shared__ float wsum[L / 32];
  const int NC = num_chunks(p.S);
  const int bh = blockIdx.x / NC, sc = blockIdx.x % NC, b = bh / p.NH, h = bh % p.NH;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int S = p.S;
  const bool rev = p.reverse != 0;
  const size_t rows_total = (size_t)p.B * p.NH * S;
  const BwdLayout blay(p.B, p.NH, S, DH);
  const uint8_t* ws = reinterpret_cast<const uint8_t*>(p.workspace);
  const float* rp = reinterpret_cast<const float*>(ws + blay.rpart_off);
  const float* kp = reinterpret_cast<const float*>(ws + blay.kpart_off);
  const float* flow = reinterpret_cast<const float*>(ws + blay.flow_off) + (size_t)bh * NC * blay.nblk;
  const int nb = DH / 32;
  const int tok0 = mem_chunk(sc, NC, rev) * L, nvalid = min(L, S - tok0);
  const bool valid = t < nvalid;
  const int tok = tok0 + (rev ? (nvalid - 1 - t) : t);
  float dB = 0.f;
  if (valid) {
    const size_t g = (size_t)bh * S + tok;
    float R = 0.f, K = 0.f;
    for (int c = 0; c < nb; ++c) { R += rp[(size_t)c * rows_total + g]; K += kp[(size_t)c * rows_total + g]; }
    const float i_raw = p.i.ptr[(int64_t)b * p.i.stride_b + (int64_t)h * p.i.stride_h + (int64_t)tok * p.i.stride_s];
    p.di.ptr[(int64_t)b * p.di.stride_b + (int64_t)h * p.di.stride_h + (int64_t)tok * p.di.stride_s] = K * igate_dlog(p, i_raw);
    dB = R - K;
  }
  const float incl = warp_scan_add(dB, lane);
  if (lane == 31) wsum[warp] = incl;
  __syncthreads();
  float before = 0.f, all = 0.f;
#pragma unroll
  for (int w = 0; w < L / 32; ++w) { before += (w < warp) ? wsum[w] : 0.f; all += wsum[w]; }
  // inclusive suffix sum inside the chunk + the exact flow across the boundary to the next chunk
  float fnext = 0.f;
  if (sc + 1 < NC)
    for (int k = 0; k < blay.nblk; ++k) fnext += flow[(sc + 1) * blay.nblk + k];
  const float suffix = all - (incl + before) + dB + fnext;
  if (valid) {
    const float fi = p.f.ptr[(int64_t)b * p.f.stride_b + (int64_t)h * p.f.stride_h + (int64_t)tok * p.f.stride_s];
    p.df.ptr[(int64_t)b * p.df.stride_b + (int64_t)h * p.df.stride_h + (int64_t)tok * p.df.stride_s] = suffix / (1.f + __expf(fi));
  }
}

template <class K>
int prep(K kernel, size_t smem, const char* name) {
  cudaError_t e = set_max_smem_once(reinterpret_cast<const void*>(kernel), smem);
  if (e != cudaSuccess) {
    set_error("cudaFuncSetAttribute(%s, %zu B): %s", name, smem, cudaGetErrorString(e));
    return MLSTM_ERR_CUDA;
  }
  return MLSTM_OK;
}
int launched(const char* name) {
  count_launch();
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s launch failed: %s", name, cudaGetErrorString(e));
    return MLSTM_ERR_CUDA;
  }
  return MLSTM_OK;
}

template <int DH>
int launch_bwd(const mlstm_params& p, cudaStream_t st, int part) {
  const StateLayout slay(p.B, p.NH, p.S, DH);
  const BwdLayout blay(p.B, p.NH, p.S, DH);
  if (!p.states || p.states_bytes < slay.total) {
    set_error("backward needs the forward's chunk-state buffer (%zu bytes)", slay.total);
    return MLSTM_ERR_WORKSPACE;
  }
  const int NC = num_chunks(p.S), n_items = p.B * p.NH * NC;
  CUtensorMap mq, mk, mv, mdh, mcs, mdcs, mh, mdq, mdk, mdv;
  int r = 0;
  r |= make_act_tmap(&mh, p.h.ptr, p.B, p.NH, p.S, DH, p.h.stride_b, p.h.stride_h, p.h.stride_s, L);
  r |= make_act_tmap(&mdq, p.dq.ptr, p.B, p.NH, p.S, DH, p.dq.stride_b, p.dq.stride_h, p.dq.stride_s, L);
  r |= make_act_tmap(&mdk, p.dk.ptr, p.B, p.NH, p.S, DH, p.dk.stride_b, p.dk.stride_h, p.dk.stride_s, L);
  r |= make_act_tmap(&mdv, p.dv.ptr, p.B, p.NH, p.S, DH, p.dv.stride_b, p.dv.stride_h, p.dv.stride_s, L);
  r |= make_act_tmap(&mq, p.q.ptr, p.B, p.NH, p.S, DH, p.q.stride_b, p.q.stride_h, p.q.stride_s, L);
  r |= make_act_tmap(&mk, p.k.ptr, p.B, p.NH, p.S, DH, p.k.stride_b, p.k.stride_h, p.k.stride_s, L);
  r |= make_act_tmap(&mv, p.v.ptr, p.B, p.NH, p.S, DH, p.v.stride_b, p.v.stride_h, p.v.stride_s, L);
  r |= make_act_tmap(&mdh, p.dh.ptr, p.B, p.NH, p.S, DH, p.dh.stride_b, p.dh.stride_h, p.dh.stride_s, L);
  r |= make_state_tmap(&mcs, reinterpret_cast<uint8_t*>(p.states) + slay.cs_off, (size_t)n_items * DH, DH);
  r |= make_state_tmap(&mdcs, reinterpret_cast<uint8_t*>(p.workspace) + blay.dcs_off, (size_t)n_items * DH, DH);
  if (r) {
    set_error("cuTensorMapEncodeTiled failed (%d)", r);
    return r == -1 ? MLSTM_ERR_NO_DEVICE : MLSTM_ERR_INVALID_ARG;
  }
  const int sms = sm_count_of(p.q.ptr);
  const int grid = n_items < sms ? n_items : sms;
  const float scale = resolve_scale(p);
  const size_t smB = sizeof(SmemB<DH>), smSB = sizeof(SmemSB<DH>);
  int rc;
  // whole backward in one call with few (batch, head) pairs: the state walk and kernel A share a launch (tc_bwd_sa_kernel)
  const int n_state = p.B * p.NH;
  const bool merged = part != 0 && part != 1 && 2 * n_state <= sms && NC > 1 && (int64_t)n_state * p.S < (1ll << 31);
  if (merged) {
    const int64_t rows = (int64_t)n_state * p.S;
    const int rows_per_cta = 8 * (32 / (DH / 8)) * DN_U;
    tc_dn_kernel<<<dim3((unsigned)((rows + rows_per_cta - 1) / rows_per_cta)), dim3(256), 0, st>>>(
        p, reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(p.workspace) + blay.dn_off), DH, true_extent(p.h.ptr, DH));
    if ((rc = launched("tc_dn"))) return rc;
    BwdMaps ma{mdh, mv, mk, mcs, mq, mh, mdq};
    BwdMaps ms{mq, mdh, mcs, mdcs, mq, mh, mdq};
    const size_t smSA = smB > smSB ? smB : smSB;
    const int n_a = n_items < sms - n_state ? n_items : sms - n_state;
    if ((rc = prep(tc_bwd_sa_kernel<DH>, smSA, "tc_bwd_state_dq"))) return rc;
    tc_bwd_sa_kernel<DH><<<dim3(n_state + n_a), dim3(NT), smSA, st>>>(ms, ma, p, scale, n_items, n_state);
    if ((rc = launched("tc_bwd_state_dq"))) return rc;
  }
  if (part != 1 && !merged) {
    BwdMaps m{mdh, mv, mk, mcs, mq, mh, mdq};
    if ((rc = prep(tc_bwd_par_kernel<DH, MODE_A>, smB, "tc_bwd_dq"))) return rc;
    tc_bwd_par_kernel<DH, MODE_A><<<dim3(grid), dim3(NT), smB, st>>>(m, p, scale, n_items);
    if ((rc = launched("tc_bwd_dq"))) return rc;
  }
  if (part != 0) {
    if (!merged) {
      BwdMaps ms{mq, mdh, mcs, mdcs, mq, mh, mdq};
      if ((rc = prep(tc_state_bwd_kernel<DH>, smSB, "tc_state_bwd"))) return rc;
      tc_state_bwd_kernel<DH><<<dim3(p.B * p.NH), dim3(NT), smSB, st>>>(ms, p, scale);
      if ((rc = launched("tc_state_bwd"))) return rc;
    }
    BwdMaps m1{mk, mq, mdh, mdcs, mq, mh, mdv};
    BwdMaps m2{mv, mdh, mq, mdcs, mk, mh, mdk};
    if (n_items < 4 * sms) {
      // few items per CTA: two full-width launches balance better than two half-width groups
      if ((rc = prep(tc_bwd_par_kernel<DH, MODE_B1>, smB, "tc_bwd_dv"))) return rc;
      tc_bwd_par_kernel<DH, MODE_B1><<<dim3(grid), dim3(NT), smB, st>>>(m1, p, scale, n_items);
      if ((rc = launched("tc_bwd_dv"))) return rc;
      if ((rc = prep(tc_bwd_par_kernel<DH, MODE_B2>, smB, "tc_bwd_dk"))) return rc;
      tc_bwd_par_kernel<DH, MODE_B2><<<dim3(grid), dim3(NT), smB, st>>>(m2, p, scale, n_items);
      if ((rc = launched("tc_bwd_dk"))) return rc;
    } else {
      // B2 costs ~1.2x B1 per item: it gets the larger share of the CTAs
      const int n_b2 = (sms * 6 + 5) / 11;
      if ((rc = prep(tc_bwd_b12_kernel<DH>, smB, "tc_bwd_dkdv"))) return rc;
      tc_bwd_b12_kernel<DH><<<dim3(sms), dim3(NT), smB, st>>>(m1, m2, p, scale, n_items, n_b2);
      if ((rc = launched("tc_bwd_dkdv"))) return rc;
    }
    tc_dfscan_kernel<<<dim3(n_items), dim3(L), 0, st>>>(p, DH);
    if ((rc = launched("tc_dfscan"))) return rc;
  }
  return MLSTM_OK;
}

}  // namespace

// Pieces shared with the head-dim-256 family (mlstm_tc_256.cu): the adjoint-state walk over (DHF/128)^2 independent
// 128 x 128 blocks per (batch, head) (`mcs`, `mdcs`: state maps with a box of 128 rows), the di / df scan, the scratch layout.
int tc_state_bwd_blocks(const mlstm_params& p, cudaStream_t st, const CUtensorMap& mq, const CUtensorMap& mdh,
                        const CUtensorMap& mcs, const CUtensorMap& mdcs) {
  BwdMaps ms{mq, mdh, mcs, mdcs, mq, mq, mq};
  int rc;
  const size_t smSB = sizeof(SmemSB<128>);
  if ((rc = prep(tc_state_bwd_kernel<128>, smSB, "tc_state_bwd"))) return rc;
  const int ncb = p.DHQK / 128;
  tc_state_bwd_kernel<128><<<dim3(ncb * ncb, p.B * p.NH), dim3(NT), smSB, st>>>(ms, p, resolve_scale(p));
  return launched("tc_state_bwd");
}
int tc_dfscan_launch(const mlstm_params& p, cudaStream_t st) {
  tc_dfscan_kernel<<<dim3(p.B * p.NH * num_chunks(p.S)), dim3(L), 0, st>>>(p, p.DHQK);
  return launched("tc_dfscan");
}
void tc_bwd_layout(const mlstm_params& p, size_t* dn_off, size_t* rpart_off, size_t* kpart_off, size_t* dcs_off, size_t* dns_off,
                   size_t* total) {
  const BwdLayout b(p.B, p.NH, p.S, p.DHQK);
  *dn_off = b.dn_off; *rpart_off = b.rpart_off; *kpart_off = b.kpart_off; *dcs_off = b.dcs_off; *dns_off = b.dns_off;
  *total = b.total;
}

size_t tc_bwd_fused_workspace(const mlstm_params& p);
int tc_bwd_fused(const mlstm_params& p, cudaStream_t st, int part);
size_t tc_bwd_fused128_workspace(const mlstm_params& p);
int tc_bwd_fused128(const mlstm_params& p, cudaStream_t st, int part);

size_t tc_bwd_workspace(const mlstm_params& p) {
  if (tc_use_fused_bwd(p)) return p.DHQK == 64 ? tc_bwd_fused_workspace(p) : tc_bwd_fused128_workspace(p);
  return BwdLayout(p.B, p.NH, p.S, p.DHQK).total;
}

int tc256_bwd(const mlstm_params& p, cudaStream_t st, int part);

int tc_bwd(const mlstm_params& p, cudaStream_t st, int part) {
  if (p.DHQK == 256) return tc256_bwd(p, st, part);
  if (tc_use_fused_bwd(p)) return p.DHQK == 64 ? tc_bwd_fused(p, st, part) : tc_bwd_fused128(p, st, part);
  if (p.DHQK == 64) return launch_bwd<64>(p, st, part);
  return launch_bwd<128>(p, st, part);
}

}  // namespace mlstm
