// Bulk-copy pipelined variants of the throughput-mode agent kernels (included by gj_kernels.cu after gj_lean.cuh).
//
// The register-batched kernels of gj_lean.cuh are latency-bound: every streaming operand is an LDG whose latency a
// thread has to sit out with at most two agents in flight (ncu, profiles/r1_lean_v3_56M_*: 40-65 % of the stall
// samples are long-scoreboard waits at the first use of a loaded value, 35-47 % occupancy).  Here a persistent
// CTA of 512 threads walks its run of agent tiles (<= 1024 agents each) with a two-stage shared-memory pipeline:
// one elected thread issues, per tile, one `cp.async.bulk` (TMA 1-D bulk copy, completion counted in bytes on an
// mbarrier) for each per-agent array of the tile — state, tapes, index words, class bytes, and the member values
// of the range-tier (household) network with a halo for the neighbours — while all warps compute the previous tile
// out of shared memory, two agents per thread.  Memory-level parallelism is then set by the bytes in flight per SM
// (2 CTAs x 1-2 tiles x 30-43 KB), not by registers x occupancy; the global loads left in the agent loops are the
// L2-resident gathers of the generic groups' sums and a few arrays that stream through registers because staging
// them would cost the second CTA per SM (the backward's six cotangents, the gather's packed profile).  The
// arithmetic is lean_forward_core() / lean_backward_agent() / lean_gather_agent() of gj_lean.cuh: trajectories are
// bit-identical to the register-batched kernels (tests/test_gpu_scale.py::test_pipelined_kernels_are_bit_identical).
//
// Requirements checked by the launcher (else the gj_lean.cuh kernels run): every per-agent array 16-byte aligned.
// Bulk copies move 16-byte granules, so a tile's copy starts at the preceding and ends at the following multiple of
// four agents (sixteen for the class bytes); at the end of an array this reads up to 12 bytes past its last
// element — inside the allocation granule of every allocator we are called with (documented in the header).
#pragma once
#include "gj_lean.cuh"

namespace gj {

constexpr int kPipeThreads = 512;
constexpr int kPipeTile = GJ_TILE_AGENTS;  // agents per stage (a world tile)
constexpr int kPipeHalo = 64;              // >= RANGE_MAX_GROUP - 1 of the world builder
constexpr int kPipeStages = 2;
constexpr int kPipeWarps = kPipeThreads / 32;
constexpr int kPipePer = kPipeTile / kPipeThreads;  // agents per thread and tile, processed interleaved (ILP)
static_assert(kPipePer * kPipeThreads == kPipeTile, "tile = whole agents per thread");

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// global -> shared bulk copy of `bytes` (multiple of 16; both addresses 16-byte aligned), completion on `bar`
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// ---- the copies of one tile ---------------------------------------------------------------------------------
// 4-byte arrays: agents [lo4, hi4) (multiples of four around [a0, a1)); element a sits at index a - lo4
struct TileSpan {
  uint32_t a0, a1, lo4, hi4, n4;   // n4 = bytes of a 4-byte array's copy
  uint32_t tlo, thi;               // window of the range-tier member values (halo on both sides)
  uint32_t lo16, hi16;             // class bytes
};
__device__ __forceinline__ TileSpan tile_span(const gj_world_desc& w, int64_t tile) {
  TileSpan t;
  t.a0 = w.tile_begin[tile];
  t.a1 = w.tile_begin[tile + 1];
  t.lo4 = t.a0 & ~3u;
  t.hi4 = (t.a1 + 3u) & ~3u;
  t.n4 = (t.hi4 - t.lo4) * 4u;
  const uint32_t nmax = (uint32_t)((w.n_agents + 3) & ~(int64_t)3);
  t.tlo = (t.a0 > (uint32_t)kPipeHalo ? t.a0 - kPipeHalo : 0u) & ~3u;
  t.thi = (t.a1 + kPipeHalo + 3u) & ~3u;
  if (t.thi > nmax) t.thi = nmax;
  t.lo16 = t.a0 & ~15u;
  t.hi16 = (t.a1 + 15u) & ~15u;
  return t;
}
__device__ __forceinline__ uint32_t halo_lo(uint32_t a0) { return (a0 > (uint32_t)kPipeHalo ? a0 - kPipeHalo : 0u) & ~3u; }

struct Copier {   // one elected thread: sums the bytes first (expect_tx must precede the copies' completion)
  uint64_t* bar;
  __device__ __forceinline__ void f4(void* dst, const void* base, const TileSpan& t) const {
    bulk_g2s(dst, reinterpret_cast<const char*>(base) + (size_t)t.lo4 * 4u, t.n4, bar);
  }
};

// sum of the member values of agent a's range-tier group out of the staged window (same order as
// lean_range_issue / lean_range_finish)
__device__ __forceinline__ float pipe_range_sum(const float* __restrict__ Ts, uint32_t tlo, uint32_t a, uint32_t slot) {
  if (slot == kNoSlot) return 0.0f;
  const uint32_t b0 = a - (slot >> 16) - tlo;
  const int nb = (int)(slot & 0xFFFFu);
  float x[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) x[j] = (j < nb) ? Ts[b0 + j] : 0.0f;
  float S = ((x[0] + x[1]) + (x[2] + x[3])) + ((x[4] + x[5]) + (x[6] + x[7]));
  for (int j = 8; j < nb; ++j) S += Ts[b0 + j];
  return S;
}

// Tile bounds and cell flags of the tile a CTA computes, fetched ONE TILE AHEAD: read at the top of a tile they were
// CTA-uniform dependent global loads that every warp sat out right after the barrier (ncu: 10-14 % of the stall
// samples of the three kernels); issued a tile early, their latency hides behind the tile's arithmetic.
struct TileWalk {
  uint32_t a1;       // end of the current tile (= start of the following one)
  // prefetched RAW, consumed one tile later (no compare or select at load time: that would wait for the load right
  // away, which is what made these CTA-uniform loads 17 % of the forward kernel's stall samples and 11 % of its
  // instructions in profiles/r2_56M_stalls_k_pipe_forward.txt):
  uint32_t nxt_a1;   // end of the following tile
  uint32_t nxt_flag; // gj_world_desc.tile_flags of the following tile (bit 0: it starts a new cell)
};
__device__ __forceinline__ TileWalk tile_walk_begin(const gj_world_desc& w, const LeanPlan& lp, const TileRun& run) {
  TileWalk t;
  t.a1 = t.nxt_a1 = 0;
  t.nxt_flag = 1u;                      // the run's first tile always builds its class table
  if (run.t0 < run.t1) {
    t.a1 = w.tile_begin[run.t0];
    t.nxt_a1 = w.tile_begin[run.t0 + 1];
  }
  return t;
}
// top of tile `tile`: take the facts prefetched a tile ago, issue the loads of the following tile's.  Both arrays carry
// readable slack behind their last element, so the loads need no bounds branch (past the run's end they are unused).
#define PIPE_TILE_FACTS                                                   \
  const uint32_t a0 = tw.a1, a1 = tw.nxt_a1;                              \
  const bool new_cell = lp.n_cell > 0 && (tw.nxt_flag & 1u);              \
  (void)new_cell;                                                         \
  tw.a1 = a1;                                                             \
  tw.nxt_flag = w.tile_flags[tile + 1];                                   \
  tw.nxt_a1 = w.tile_begin[tile + 2]
// does the current tile end a cell (or the run)?  Evaluated at the END of the tile, from the flag loaded at its top.
#define PIPE_FLUSH(tw, lp) ((lp).n_cell > 0 && (tile + 1 == run.t1 || ((tw).nxt_flag & 1u)))

// end of a tile: every warp is done with the stage, one thread refills it with the tile kPipeStages ahead.
// (Letting the last warp to finish do the refill instead of a CTA barrier, and shipping the tile facts with the
// stage, were both measured: no gain / a loss — see DESIGN.md.)
__device__ __forceinline__ bool pipe_release() {
  __syncthreads();
  return threadIdx.x == 0;
}

// contact probability of a range-tier group from its size (gj_world_desc.range_pc_from_size): the same fp32 formula
// as the world builders' p_contact, so the table entries are bit-identical to the per-agent array they replace
constexpr int kPcLut = kPipeHalo + 8;
__device__ __forceinline__ void pipe_fill_pc_lut(float* lut) {
  for (int n = threadIdx.x; n < kPcLut; n += blockDim.x) lut[n] = fmaxf(fminf(1.0f / (float)(n - 1), 1.0f), 0.0f);
}

constexpr int kPipeF = kPipeTile + 8;                     // floats of a staged 4-byte array
constexpr int kPipeH = kPipeTile + 2 * kPipeHalo + 8;     // ... with the halo

__device__ __forceinline__ void pipe_init_barriers(uint64_t* full) {
  if (threadIdx.x == 0) {
    for (int i = 0; i < kPipeStages; ++i) mbar_init(&full[i], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
}

// =====================================================================================================
// K3p  forward (+ optionally the transmission pass of the FOLLOWING step, from the state just written)
// =====================================================================================================
// what the forward has to know about the step after this one to run its transmission pass (K1 of gj_lean.cuh)
struct NextStep {
  int on;
  float now;
  int day_type;
  int n_quar;
  float quar_thr[GJ_MAX_QUAR];
  int n_cell;                       // cell channels of the next step and their attendance tables
  int c_row[GJ_MAX_CHANNELS];
  int n_tc;                         // its distinct tile -> cell maps
  const uint32_t* tc[GJ_MAX_CHANNELS];
  float* T;
  float* Tq;                        // may alias T when n_quar <= 0
  float* tile_part;
  int has_generic;                  // the next step has generic-tier networks: scatter into their accumulators
  Scatter sct;
};
__device__ __forceinline__ float quar_mask_next(const NextStep& nx, float cur) {
  bool ok = true;
#pragma unroll
  for (int i = 0; i < GJ_MAX_QUAR; ++i)
    if (i < nx.n_quar) ok = ok && (cur < nx.quar_thr[i]);
  return ok ? 1.0f : 0.0f;
}
__device__ __forceinline__ bool next_new_cell(const NextStep& nx, int64_t a, int64_t b) {
  bool changed = false;
  for (int i = 0; i < nx.n_tc; ++i) changed = changed || (nx.tc[i][a] != nx.tc[i][b]);
  return changed;
}
template <bool kBatch>
struct alignas(16) PipeFwdStageT {
  float s[kPipeF], inf[kPipeF], tinf[kPipeF], cur[kPipeF], nxt[kPipeF], ttn[kPipeF], rpc[kPipeF];
  uint32_t ent[kPipeF], slot[kPipeF], oid[kPipeF];
  float T[kPipeH];
  uint8_t cls[kPipeTile + 32];
  float dE[kBatch ? kPipeF : 4];   // batched ensemble: the draw's noise, shared by the samples (Batch::noise)
};
template <bool kNext, bool kBatch>
struct PipeFwdSharedT {
  PipeFwdStageT<kBatch> st[kPipeStages];
  ProbRow prob[200];
  ProbRow prob_next[kNext ? 200 : 1];   // transmission-side tables of the next step (look-ahead only)
  float L[2][200];
  float beta[GJ_MAX_NETS];
  float hist[100];
  float deaths;
  float pc_lut[kPcLut];
  alignas(8) uint64_t full[kPipeStages];
};

// so: batched ensemble — this sample's offset into the per-sample arrays (a multiple of four agents: the copies stay
// 16-byte aligned); the world's arrays are shared
// kRegion: also the region codes (gj_fwd_io.region) into `reg`, the stage's slice of the region staging area
template <bool kBatch, bool kRegion = false>
__device__ __forceinline__ void pipe_fwd_issue(PipeFwdStageT<kBatch>& sg, uint64_t* bar, const gj_world_desc& w,
                                               const LeanPlan& lp, const gj_fwd_io& io, const float* Tr, int64_t tile,
                                               bool has_gen, bool has_range, uint32_t so = 0u,
                                               const float* noise = nullptr, int32_t* reg = nullptr) {
  const TileSpan t = tile_span(w, tile);
  uint32_t total = 6u * t.n4 + (t.hi16 - t.lo16);
  if (kRegion) total += t.n4;
  if (kBatch && noise) total += t.n4;
  if (has_gen) total += t.n4;
  if (w.orig_id) total += t.n4;
  if (has_range) total += (lp.r_pc_lut ? 1u : 2u) * t.n4 + (t.thi - t.tlo) * 4u;
  mbar_expect_tx(bar, total);
  const Copier c{bar};
  if (kRegion) c.f4(reg, io.region, t);
  if (kBatch && noise) c.f4(sg.dE, noise, t);
  if (w.orig_id) c.f4(sg.oid, w.orig_id, t);
  c.f4(sg.s, io.s + so, t);
  c.f4(sg.inf, io.inf + so, t);
  c.f4(sg.tinf, io.tinf + so, t);
  c.f4(sg.cur, io.cur + so, t);
  c.f4(sg.nxt, io.nxt + so, t);
  c.f4(sg.ttn, io.ttn + so, t);
  if (has_gen) c.f4(sg.ent, w.ent1, t);
  if (has_range) {
    c.f4(sg.slot, lp.r_slot, t);
    if (!lp.r_pc_lut) c.f4(sg.rpc, lp.r_pc, t);
    bulk_g2s(sg.T, Tr + so + t.tlo, (t.thi - t.tlo) * 4u, bar);
  }
  bulk_g2s(sg.cls, w.cls + t.lo16, t.hi16 - t.lo16, bar);
}

// region staging (kRegion): kPipeStages slices of kPipeF region codes, in the dynamic shared memory right after the
// kernel's shared struct (whose size is a multiple of 16), so the other instantiations keep their layout
constexpr size_t kPipeRegionBytes = sizeof(int32_t) * kPipeStages * kPipeF;

// kRegion: regional transmission factor (gj_fwd_io.region): the code is staged with the tile's other operands and the
// factor gathered from region_factor (R floats, cached)
template <bool kQuar, bool kDiag, bool kNext, bool kBatch, bool kLabel, bool kRegion>
__device__ __forceinline__ void pipe_forward_body(const gj_world_desc& w, const gj_step_params& p, const LeanPlan& lp,
                                                  const gj_fwd_io& io, const float* __restrict__ cell_buf,
                                                  double* __restrict__ red_part, unsigned int* __restrict__ ticket,
                                                  NextStep nx, const Batch& bt) {
  static_assert(!(kNext && kBatch), "the look-ahead transmission pass is not batched");
  static_assert(!(kNext && kLabel), "a step with a label table runs without the look-ahead");
  static_assert(!(kNext && kRegion), "a step with a regional factor runs without the look-ahead");
  extern __shared__ __align__(128) unsigned char pipe_smem[];
  PipeFwdSharedT<kNext, kBatch>& sh = *reinterpret_cast<PipeFwdSharedT<kNext, kBatch>*>(pipe_smem);
  int32_t* const reg_st = reinterpret_cast<int32_t*>(pipe_smem + sizeof(PipeFwdSharedT<kNext, kBatch>));
  const BatchCta bc = batch_cta<kBatch>(bt);
  const float* noise = kBatch ? bt.noise : nullptr;
  const uint32_t so = bc.so;
  float* __restrict__ red_out = io.red;
  const float* __restrict__ beta_in = io.beta;
  uint32_t* __restrict__ lacc = io.label_acc;
  const float* __restrict__ rfac = io.region_factor;
  if (kBatch) {   // this sample's slices of the scratch and of the small per-sample arrays
    cell_buf = scr_shift(cell_buf, bt, bc.s);
    red_part = scr_shift(red_part, bt, bc.s);
    ticket = scr_shift(ticket, bt, bc.s);
    if (red_out) red_out += (int64_t)bc.s * bt.sRed;
    if (kLabel) lacc += bc.s * bt.sLab;
    if (kRegion) rfac += bc.s * bt.sReg;
    beta_in += (int64_t)bc.s * bt.sBeta;
  }
  const TileRun run = lean_tiles(w, bc);
  const float* __restrict__ Tr = (kQuar && !lp.r_house) ? io.Tq : io.T;
  const bool has_gen = lp.has_generic != 0, has_range = lp.n_range > 0;
  pdl_launch();
  pipe_init_barriers(sh.full);
  lean_load_prob<true>(sh.prob, p, lp, io.leisure_prob);
  pipe_fill_pc_lut(sh.pc_lut);
  if (kNext) {
    for (int i = threadIdx.x; i < GJ_MAX_CHANNELS * 200; i += blockDim.x) {
      const int j = i / 200, c = i - j * 200;
      sh.prob_next[c].v[j] = j < nx.n_cell ? io.leisure_prob[(size_t)(nx.c_row[j] * 2 + nx.day_type) * 200 + c] : 0.0f;
    }
  }
  pdl_wait();   // everything below reads what earlier kernels of the stream wrote
  if (threadIdx.x < p.n_nets) sh.beta[threadIdx.x] = beta_in[threadIdx.x];
  if (threadIdx.x < 100) sh.hist[threadIdx.x] = 0.0f;
  if (threadIdx.x == 0) sh.deaths = 0.0f;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 0; i < kPipeStages; ++i)
      if (run.t0 + i < run.t1)
        pipe_fwd_issue<kBatch, kRegion>(sh.st[i], &sh.full[i], w, lp, io, Tr, run.t0 + i, has_gen, has_range, so,
                                        noise, reg_st + i * kPipeF);
  }
  const float* __restrict__ SP = io.S_scaled + lp.gen_base + (kBatch ? (int64_t)bc.s * bt.sG : (int64_t)0);
  const float dead = (float)(p.n_stages - 1);
  const float inv_tau = 1.0f / p.tau;
  const float beta_r = lp.n_range > 0 ? sh.beta[lp.r_net] : 0.0f;

  const float4* __restrict__ prof = reinterpret_cast<const float4*>(io.prof4);
  float acc[GJ_MAX_CHANNELS];   // look-ahead: partial sums of the next step's cell channels
#pragma unroll
  for (int j = 0; j < GJ_MAX_CHANNELS; ++j) acc[j] = 0.0f;
  int nbuild = 0, stg = 0;
  uint32_t parity = 0;
  const float* L = sh.L[0];
  TileWalk tw = tile_walk_begin(w, lp, run);
  for (int64_t tile = run.t0; tile < run.t1; ++tile) {
    PipeFwdStageT<kBatch>& sg = sh.st[stg];
    PIPE_TILE_FACTS;
    mbar_wait(&sh.full[stg], parity);
    if (new_cell) {
      // rebuilt in the other buffer: a buffer is rewritten two rebuilds later, after the barriers in between
      lean_class_table(sh.L[nbuild & 1], sh.prob, lp, cell_buf, tile);
      L = sh.L[nbuild & 1];
      ++nbuild;
      __syncthreads();
    }
    const uint32_t sk = a0 & 3u, sk16 = a0 & 15u, tlo = halo_lo(a0);
    uint32_t ent[kPipePer];
    float gen[kPipePer];
    float4 pfe[kPipePer];   // look-ahead: packed profile of the agents that are already infected (issued early)
#pragma unroll
    for (int h = 0; h < kPipePer; ++h) {   // the L2 gathers first, for all of this thread's agents
      const uint32_t j = threadIdx.x + h * kPipeThreads;
      ent[h] = (has_gen && a0 + j < a1) ? sg.ent[j + sk] : kEntNone;
      gen[h] = lean_generic_issue(SP, ent[h]);
      if (kNext) {
        pfe[h] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        if (a0 + j < a1 && sg.inf[j + sk] != 0.0f) pfe[h] = prof[a0 + j];
      }
    }
#pragma unroll
    for (int h = 0; h < kPipePer; ++h) {
      const uint32_t j = threadIdx.x + h * kPipeThreads;
      const uint32_t a = a0 + j, i = j + sk;
      if (a >= a1) break;
      const float hs = has_range ? pipe_range_sum(sg.T, tlo, a, sg.slot[i]) : 0.0f;
      const int cls = sg.cls[j + sk16];
      const float Lc = lp.n_cell > 0 ? L[cls] : 0.0f;
      const float gv = lean_generic_finish(w, SP, ent[h], a, gen[h]);
      const uint64_t ga = w.orig_id ? (uint64_t)sg.oid[i] : p.agent_offset + a;
      const float rpc = !has_range ? 0.0f : (lp.r_pc_lut ? ((sg.slot[i] == kNoSlot) ? 0.0f : sh.pc_lut[sg.slot[i] & 0xFFFFu])
                                                         : sg.rpc[i]);
      const float mreg = kRegion ? __ldg(rfac + reg_st[stg * kPipeF + i]) : 1.0f;
      const FwdOut o = lean_forward_agent<kQuar, kDiag, kRegion>(p, lp, io, a + so, ga, hs, gv, Lc, beta_r, rpc,
                                                        sg.s[i], sg.inf[i], sg.tinf[i], sg.cur[i], sg.nxt[i], sg.ttn[i], cls,
                                                        inv_tau, dead, sh.hist, &sh.deaths, kBatch && noise != nullptr,
                                                        (kBatch && noise) ? sg.dE[i] : 0.0f, mreg);
      if (kLabel) label_add(lacc, io.label, a, (uint32_t)o.inf, o.cur == dead ? 1u : 0u);
      if (kNext) {   // TransmissionUpdater of the next step (same arithmetic as k_lean_transmission)
        float T = 0.0f;
        if (o.inf != 0.0f) {
          const float4 pf = (sg.inf[i] != 0.0f) ? pfe[h] : prof[a];   // newly infected: fetched now (rare)
          T = lean_transmission<false>(nx.now, o.tinf, pf).coef * o.inf;
        }
        nx.T[a] = T;
        float Tq = T;
        if (nx.n_quar > 0) {
          Tq = quar_mask_next(nx, o.cur) * T;
          nx.Tq[a] = Tq;
        }
        if (Tq != 0.0f) {
          if (nx.n_cell > 0) lean_channel_fma(acc, sh.prob_next, cls, Tq, nx.n_cell);
          if (nx.has_generic) lean_scatter(w, nx.sct, has_gen ? ent[h] : w.ent1[a], a, Tq);
        }
      }
    }
    if (pipe_release() && tile + kPipeStages < run.t1)
      pipe_fwd_issue<kBatch, kRegion>(sg, &sh.full[stg], w, lp, io, Tr, tile + kPipeStages, has_gen, has_range, so,
                                      noise, reg_st + stg * kPipeF);
    if (++stg == kPipeStages) {
      stg = 0;
      parity ^= 1u;
    }
    if (kNext && nx.n_cell > 0) {   // as in B1p: a cell run's sums go to its last tile, zeros to the others
      if (tile + 1 == run.t1 || next_new_cell(nx, tile, tile + 1)) {
        block_sums<float, GJ_MAX_CHANNELS, kPipeWarps>(acc, nx.n_cell, nx.tile_part + tile * GJ_MAX_CHANNELS);
#pragma unroll
        for (int j = 0; j < GJ_MAX_CHANNELS; ++j) acc[j] = 0.0f;
      } else if ((int)threadIdx.x < nx.n_cell) {
        nx.tile_part[tile * GJ_MAX_CHANNELS + threadIdx.x] = 0.0f;
      }
    }
  }
  if (red_out) {
    __syncthreads();
    const int nr = 2 + p.n_age_bins;
    if ((int)threadIdx.x < nr) {
      double v = 0.0;
      if (threadIdx.x == 0) {
        for (int c = 0; c < 100; ++c) v += (double)sh.hist[c];
      } else if (threadIdx.x == 1) {
        v = (double)sh.deaths;
      } else {
        const int b = threadIdx.x - 2;
        for (int c = max(p.age_bins[b] + 1, 0); c < p.age_bins[b + 1] && c < 100; ++c) v += (double)sh.hist[c];
      }
      red_part[(int64_t)bc.bx * kMaxRed + threadIdx.x] = v;
    }
    finish_partials<kMaxRed>(nr, red_part, bc.gx, ticket, red_out);
  }
}

template <bool kQuar, bool kDiag, bool kNext, bool kBatch, bool kLabel>
__global__ void __launch_bounds__(kPipeThreads, 2) k_pipe_forward(gj_world_desc w, gj_step_params p, LeanPlan lp,
                                                                 gj_fwd_io io, const float* __restrict__ cell_buf,
                                                                 double* __restrict__ red_part,
                                                                 unsigned int* __restrict__ ticket, NextStep nx,
                                                                 Batch bt) {
  pipe_forward_body<kQuar, kDiag, kNext, kBatch, kLabel, false>(w, p, lp, io, cell_buf, red_part, ticket, nx, bt);
}

// the same with the regional transmission factor (gj_fwd_io.region); dynamic shared memory + kPipeRegionBytes
template <bool kQuar, bool kDiag, bool kBatch, bool kLabel>
__global__ void __launch_bounds__(kPipeThreads, 2) k_pipe_forward_region(gj_world_desc w, gj_step_params p, LeanPlan lp,
                                                                        gj_fwd_io io, const float* __restrict__ cell_buf,
                                                                        double* __restrict__ red_part,
                                                                        unsigned int* __restrict__ ticket, NextStep nx,
                                                                        Batch bt) {
  pipe_forward_body<kQuar, kDiag, false, kBatch, kLabel, true>(w, p, lp, io, cell_buf, red_part, ticket, nx, bt);
}

// =====================================================================================================
// B1p  backward, per agent
// =====================================================================================================
struct alignas(16) PipeBwdStage {
  float s[kPipeF], tinf[kPipeF], cur[kPipeF], nxt[kPipeF], ttn[kPipeF], ty[kPipeF], v[kPipeF];
  uint8_t cls[kPipeTile + 32];
};
struct PipeBwdShared {
  PipeBwdStage st[kPipeStages];
  ProbRow prob[200];
  float gred_age[100];
  uint32_t next_flag[kPipeStages];   // tile_flags of the tile AFTER the one in the stage (thread 0 fetches it at the
                                     // tile's top; read after the end-of-tile barrier: no register, no exposed load)
  alignas(8) uint64_t full[kPipeStages];
};
struct BwdCot {
  const float* p[6];
};

template <bool kRegion = false>
__device__ __forceinline__ void pipe_bwd_issue(PipeBwdStage& sg, uint64_t* bar, const gj_world_desc& w,
                                               const gj_bwd_io& io, int64_t tile, uint32_t so = 0u,
                                               int32_t* reg = nullptr) {
  const TileSpan t = tile_span(w, tile);
  const uint32_t total = (kRegion ? 8u : 7u) * t.n4 + (t.hi16 - t.lo16);
  mbar_expect_tx(bar, total);
  const Copier c{bar};
  if (kRegion) c.f4(reg, io.region, t);
  c.f4(sg.s, io.s + so, t);
  c.f4(sg.tinf, io.tinf + so, t);
  c.f4(sg.cur, io.cur + so, t);
  c.f4(sg.nxt, io.nxt + so, t);
  c.f4(sg.ttn, io.ttn + so, t);
  c.f4(sg.ty, io.tape_y0 + so, t);
  c.f4(sg.v, io.tape_v + so, t);
  bulk_g2s(sg.cls, w.cls + t.lo16, t.hi16 - t.lo16, bar);
}

#ifndef GJ_PIPE_BWD_THREADS
#define GJ_PIPE_BWD_THREADS 512
#endif
constexpr int kBwdThreads = GJ_PIPE_BWD_THREADS;
constexpr int kBwdPer = kPipeTile / kBwdThreads;
constexpr int kBwdCtas = kBwdThreads == 256 ? 3 : 2;
// kRegion: regional transmission factor; the region codes are staged like in the forward (after PipeBwdShared)
template <bool kQuar, bool kBatch, bool kLabel, bool kRegion>
__device__ __forceinline__ void pipe_backward_body(const gj_world_desc& w, const gj_step_params& p, const LeanPlan& lp,
                                                   const gj_bwd_io& io, float* __restrict__ tile_part, const Batch& bt) {
  extern __shared__ __align__(128) unsigned char pipe_smem[];
  PipeBwdShared& sh = *reinterpret_cast<PipeBwdShared*>(pipe_smem);
  int32_t* const reg_st = reinterpret_cast<int32_t*>(pipe_smem + sizeof(PipeBwdShared));
  const BatchCta bc = batch_cta<kBatch>(bt);
  const uint32_t so = bc.so;
  const float* __restrict__ g_red = io.g_red;
  const float* __restrict__ g_lab = io.g_red_label;
  const float* __restrict__ rfac = io.region_factor;
  if (kBatch) {
    tile_part = scr_shift(tile_part, bt, bc.s);
    if (g_red) g_red += (int64_t)bc.s * bt.sRed;
    if (kLabel) g_lab += bc.s * bt.sLab;
    if (kRegion) rfac += bc.s * bt.sReg;
  }
  const TileRun run = lean_tiles(w, bc);
  const BwdCot cot{{io.g_s_o, io.g_inf_o, io.g_tinf_o, io.g_cur_o, io.g_nxt_o, io.g_ttn_o}};
  pdl_launch();
  pipe_init_barriers(sh.full);
  lean_load_prob<true>(sh.prob, p, lp, io.leisure_prob);
  pdl_wait();   // everything below reads what earlier kernels of the stream wrote
  if (threadIdx.x < 100) {
    float g = 0.0f;
    if (g_red) {
      g = g_red[0];
      const int age = threadIdx.x;
      for (int b = 0; b < p.n_age_bins; ++b)
        if (age > p.age_bins[b] && age < p.age_bins[b + 1]) g += g_red[2 + b];
    }
    sh.gred_age[threadIdx.x] = g;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 0; i < kPipeStages; ++i)
      if (run.t0 + i < run.t1) pipe_bwd_issue<kRegion>(sh.st[i], &sh.full[i], w, io, run.t0 + i, so, reg_st + i * kPipeF);
  }
  const float dead = (float)(p.n_stages - 1);
  const float g_deaths = g_red ? g_red[1] / dead : 0.0f;
  const float inv_tau = 1.0f / p.tau;
  float acc[GJ_MAX_CHANNELS];
#pragma unroll
  for (int j = 0; j < GJ_MAX_CHANNELS; ++j) acc[j] = 0.0f;
  int stg = 0;
  uint32_t parity = 0;
  // this kernel runs at its register cap: the tile bounds are prefetched raw as in the other two kernels, the cell flag
  // of the following tile goes through shared memory instead of living in a register across the tile
  uint32_t w_a1 = run.t0 < run.t1 ? w.tile_begin[run.t0] : 0u, w_nxt = run.t0 < run.t1 ? w.tile_begin[run.t0 + 1] : 0u;
  for (int64_t tile = run.t0; tile < run.t1; ++tile) {
    PipeBwdStage& sg = sh.st[stg];
    const uint32_t a0 = w_a1, a1 = w_nxt;
    w_a1 = a1;
    w_nxt = w.tile_begin[tile + 2];
    if (threadIdx.x == 0 && lp.n_cell > 0) sh.next_flag[stg] = w.tile_flags[tile + 1];
    mbar_wait(&sh.full[stg], parity);
    // the cotangents of the state outputs stream through registers
    float c[kBwdPer][6];
    int32_t lab[kBwdPer];   // label codes (kLabel), fetched with the cotangents
#pragma unroll
    for (int h = 0; h < kBwdPer; ++h) {
      const uint32_t a = a0 + threadIdx.x + h * kBwdThreads;
      const uint32_t al = a < a1 ? a : a0;
#pragma unroll
      for (int k = 0; k < 6; ++k) c[h][k] = cot.p[k] ? cot.p[k][al + so] : 0.0f;
      if (kLabel) lab[h] = io.label[al];
    }
    const uint32_t sk = a0 & 3u, sk16 = a0 & 15u;
#pragma unroll
    for (int h = 0; h < kBwdPer; ++h) {
      const uint32_t j = threadIdx.x + h * kBwdThreads;
      const uint32_t a = a0 + j, i = j + sk;
      if (a >= a1) break;
      const float glab_i = kLabel ? g_lab[2 * (int64_t)lab[h]] : 0.0f;
      const float glab_d = kLabel ? g_lab[2 * (int64_t)lab[h] + 1] / dead : 0.0f;
      const float mreg = kRegion ? __ldg(rfac + reg_st[stg * kPipeF + i]) : 1.0f;
      lean_backward_agent<kQuar, kLabel, kRegion>(p, lp, io, a, sg.s[i], sg.tinf[i], sg.cur[i], sg.nxt[i], sg.ttn[i],
                                                  sg.ty[i], sg.v[i], sg.cls[j + sk16], c[h][0], c[h][1], c[h][2], c[h][3],
                                                  c[h][4], c[h][5], inv_tau, dead, g_deaths, sh.gred_age, sh.prob, acc,
                                                  w.orig_id, so, glab_i, glab_d, mreg);
    }
    if (pipe_release() && tile + kPipeStages < run.t1)
      pipe_bwd_issue<kRegion>(sg, &sh.full[stg], w, io, tile + kPipeStages, so, reg_st + stg * kPipeF);
    const bool ends_cell = lp.n_cell > 0 && (tile + 1 == run.t1 || (sh.next_flag[stg] & 1u));   // after the barrier
    if (++stg == kPipeStages) {
      stg = 0;
      parity ^= 1u;
    }
    if (lp.n_cell > 0) {   // partial sums of the cell channels: written at the last tile of a cell run (see K1)
      if (ends_cell) {
        block_sums<float, GJ_MAX_CHANNELS, (kBwdThreads / 32)>(acc, lp.n_cell, tile_part + tile * GJ_MAX_CHANNELS);
#pragma unroll
        for (int j = 0; j < GJ_MAX_CHANNELS; ++j) acc[j] = 0.0f;
      } else if ((int)threadIdx.x < lp.n_cell) {
        tile_part[tile * GJ_MAX_CHANNELS + threadIdx.x] = 0.0f;
      }
    }
  }
}

template <bool kQuar, bool kBatch, bool kLabel>
__global__ void __launch_bounds__(kBwdThreads, kBwdCtas) k_pipe_backward(gj_world_desc w, gj_step_params p, LeanPlan lp,
                                                                  gj_bwd_io io, float* __restrict__ tile_part,
                                                                  Batch bt) {
  pipe_backward_body<kQuar, kBatch, kLabel, false>(w, p, lp, io, tile_part, bt);
}

// the same with the regional transmission factor (gj_bwd_io.region); dynamic shared memory + kPipeRegionBytes
template <bool kQuar, bool kBatch, bool kLabel>
__global__ void __launch_bounds__(kBwdThreads, kBwdCtas) k_pipe_backward_region(gj_world_desc w, gj_step_params p,
                                                                         LeanPlan lp, gj_bwd_io io,
                                                                         float* __restrict__ tile_part, Batch bt) {
  pipe_backward_body<kQuar, kBatch, kLabel, true>(w, p, lp, io, tile_part, bt);
}

// =====================================================================================================
// B3p  backward gather
// =====================================================================================================
struct alignas(16) PipeGatStage {
  float rpc[kPipeF], Tm[kPipeF], cur[kPipeF], inf[kPipeF], tinf[kPipeF], gi[kPipeF], gt[kPipeF];
  uint32_t ent[kPipeF], slot[kPipeF];
  float wr[kPipeH];
  uint8_t cls[kPipeTile + 32];
};
struct PipeGatShared {
  PipeGatStage st[kPipeStages];
  ProbRow prob[200];
  float L[2][200];
  float beta[GJ_MAX_NETS];
  float pc_lut[kPcLut];
  alignas(8) uint64_t full[kPipeStages];
};

template <bool kQuar>
__device__ __forceinline__ void pipe_gat_issue(PipeGatStage& sg, uint64_t* bar, const gj_world_desc& w,
                                               const LeanPlan& lp, const gj_bwd_io& io, const float* wr, int64_t tile,
                                               bool has_gen, bool has_range, uint32_t so = 0u) {
  const TileSpan t = tile_span(w, tile);
  uint32_t total = 4u * t.n4 + (t.hi16 - t.lo16);
  if (kQuar) total += t.n4;
  if (has_gen) total += t.n4;
  if (has_range) total += (lp.r_pc_lut ? 2u : 3u) * t.n4 + (t.thi - t.tlo) * 4u;
  mbar_expect_tx(bar, total);
  const Copier c{bar};
  c.f4(sg.inf, io.inf + so, t);
  c.f4(sg.tinf, io.tinf + so, t);
  c.f4(sg.gi, io.g_inf + so, t);
  c.f4(sg.gt, io.g_tinf + so, t);
  if (kQuar) c.f4(sg.cur, io.cur + so, t);
  if (has_gen) c.f4(sg.ent, w.ent1, t);
  if (has_range) {
    c.f4(sg.slot, lp.r_slot, t);
    if (!lp.r_pc_lut) c.f4(sg.rpc, lp.r_pc, t);
    c.f4(sg.Tm, io.T_in + so, t);
    bulk_g2s(sg.wr, wr + so + t.tlo, (t.thi - t.tlo) * 4u, bar);
  }
  bulk_g2s(sg.cls, w.cls + t.lo16, t.hi16 - t.lo16, bar);
}

template <bool kQuar, bool kBatch>
__global__ void __launch_bounds__(kPipeThreads, 2) k_pipe_backward_gather(gj_world_desc w, gj_step_params p,
                                                                         LeanPlan lp, gj_bwd_io io,
                                                                         const float* __restrict__ cell_buf,
                                                                         double* __restrict__ dbeta_part, Batch bt) {
  extern __shared__ __align__(128) unsigned char pipe_smem[];
  PipeGatShared& sh = *reinterpret_cast<PipeGatShared*>(pipe_smem);
  const BatchCta bc = batch_cta<kBatch>(bt);
  const uint32_t so = bc.so;
  const float* __restrict__ beta_in = io.beta;
  if (kBatch) {
    cell_buf = scr_shift(cell_buf, bt, bc.s);
    dbeta_part = scr_shift(dbeta_part, bt, bc.s);
    beta_in += (int64_t)bc.s * bt.sBeta;
  }
  const TileRun run = lean_tiles(w, bc);
  const float* __restrict__ wr = (kQuar && !lp.r_house) ? io.wq : io.w;  // member values of the range network
  const bool has_gen = lp.has_generic != 0, has_range = lp.n_range > 0;
  pdl_launch();
  pipe_init_barriers(sh.full);
  lean_load_prob<false>(sh.prob, p, lp, io.leisure_prob);
  pipe_fill_pc_lut(sh.pc_lut);
  pdl_wait();   // everything below reads what earlier kernels of the stream wrote
  if (threadIdx.x < p.n_nets) sh.beta[threadIdx.x] = beta_in[threadIdx.x];
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 0; i < kPipeStages; ++i)
      if (run.t0 + i < run.t1)
        pipe_gat_issue<kQuar>(sh.st[i], &sh.full[i], w, lp, io, wr, run.t0 + i, has_gen, has_range, so);
  }
  const float* __restrict__ cRP = io.cR + lp.gen_base + (kBatch ? (int64_t)bc.s * bt.sG : (int64_t)0);
  const float4* __restrict__ prof = reinterpret_cast<const float4*>(io.prof4);
  const float beta_r = lp.n_range > 0 ? sh.beta[lp.r_net] : 0.0f;
  double db[1] = {0.0};
  int nbuild = 0, stg = 0;
  uint32_t parity = 0;
  const float* L = sh.L[0];
  TileWalk tw = tile_walk_begin(w, lp, run);
  for (int64_t tile = run.t0; tile < run.t1; ++tile) {
    PipeGatStage& sg = sh.st[stg];
    PIPE_TILE_FACTS;
    mbar_wait(&sh.full[stg], parity);
    if (new_cell) {
      lean_class_table(sh.L[nbuild & 1], sh.prob, lp, cell_buf, tile);
      L = sh.L[nbuild & 1];
      ++nbuild;
      __syncthreads();
    }
    float4 pf[kPipePer];   // the packed profile streams through registers
#pragma unroll
    for (int h = 0; h < kPipePer; ++h) {
      const uint32_t a = a0 + threadIdx.x + h * kPipeThreads;
      pf[h] = prof[a < a1 ? a : a0];
    }
    const uint32_t sk = a0 & 3u, sk16 = a0 & 15u, tlo = halo_lo(a0);
    uint32_t ent[kPipePer];
    float gen[kPipePer];
#pragma unroll
    for (int h = 0; h < kPipePer; ++h) {
      const uint32_t j = threadIdx.x + h * kPipeThreads;
      ent[h] = (has_gen && a0 + j < a1) ? sg.ent[j + sk] : kEntNone;
      gen[h] = lean_generic_issue(cRP, ent[h]);
    }
#pragma unroll
    for (int h = 0; h < kPipePer; ++h) {
      const uint32_t j = threadIdx.x + h * kPipeThreads;
      const uint32_t a = a0 + j, i = j + sk;
      if (a >= a1) break;
      const float R = has_range ? pipe_range_sum(sg.wr, tlo, a, sg.slot[i]) : 0.0f;
      const int cls = sg.cls[j + sk16];
      const float Lc = lp.n_cell > 0 ? L[cls] : 0.0f;
      const float gv = lean_generic_finish(w, cRP, ent[h], a, gen[h]);
      const float rpc = !has_range ? 0.0f : (lp.r_pc_lut ? ((sg.slot[i] == kNoSlot) ? 0.0f : sh.pc_lut[sg.slot[i] & 0xFFFFu])
                                                         : sg.rpc[i]);
      lean_gather_agent<kQuar>(p, lp, io, a + so, R, gv, Lc, beta_r, rpc,
                               has_range ? sg.Tm[i] : 0.0f, kQuar ? sg.cur[i] : 0.0f, sg.inf[i], sg.tinf[i], pf[h],
                               sg.gi[i], sg.gt[i], db[0]);
    }
    if (pipe_release() && tile + kPipeStages < run.t1)
      pipe_gat_issue<kQuar>(sg, &sh.full[stg], w, lp, io, wr, tile + kPipeStages, has_gen, has_range, so);
    if (++stg == kPipeStages) {
      stg = 0;
      parity ^= 1u;
    }
  }
  if (lp.n_range > 0)
    block_sums<double, 1, kPipeWarps>(db, 1, dbeta_part + (int64_t)bc.bx * GJ_MAX_RANGE_NETS);
}

}  // namespace gj
