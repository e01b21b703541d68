// Throughput-mode kernels of the fused step (included by gj_kernels.cu after gj_tiled.cuh).
//
// Same step as the reference-order kernels of gj_tiled.cuh, written for HBM throughput:
//   * every kernel is a persistent grid (a few CTAs per SM); each CTA walks a contiguous run of agent tiles, so
//     tables are loaded once per CTA, per-cell work (class table, partial sums of the cell channels) is redone only
//     when the run enters a new cell, and reductions are combined once per CTA;
//   * a thread keeps a batch of agents in flight: all their streaming loads are issued first, then the dependent
//     gathers (group value from L2, household neighbours from L1 with predicated, unrolled loads), then arithmetic;
//   * the per-agent instruction count is small: the eleven-network loop collapses to
//         pressure = s * (range + mq * (generic + L[class]))
//     with ONE shared-memory lookup L[class] = sum_k V_k * p_k(class) for all cell-tier (leisure) networks, ONE
//     combined value per generic group (all generic networks of a type are PLAIN, so they share the group sum)
//     fetched through the one-entry-per-agent ELL word `ent1`, and the household re-sum over neighbouring agents;
//   * the infectiousness profile is read as one packed float4 per agent and evaluated with ex2/lg2;
//   * the Gumbel-softmax decision uses six hardware log2 and one exp2; q itself stays the IEEE expf so that
//     (1 - q) rounds like the reference's;
//   * result reductions go through a shared-memory age histogram (small integers: exact in any order).
// The kernels run when the noise is the in-kernel Philox stream and the step is "simple" (lean_plan() in
// gj_kernels.cu): at most one range-tier network (HOUSEHOLD or PLAIN kind), cell-tier networks with an
// attendance table, generic-tier networks of PLAIN kind.  Anything else, and every call with injected noise
// (parity tests), runs the reference-order kernels.  Results agree with those to ~1e-6 on q (fp32 re-association)
// and differ in masks only at near-ties (tests/test_gpu_scale.py::test_throughput_mode_*).
#pragma once
#include "gj_tiled.cuh"

namespace gj {

constexpr int kLeanThreads = 256;
// resident CTAs per SM the agent kernels are compiled for (register budget): measured best on B200
#ifndef GJ_LEAN_MINB_FWD
#define GJ_LEAN_MINB_FWD 3
#endif
#ifndef GJ_LEAN_MINB_BWD
#define GJ_LEAN_MINB_BWD 4
#endif
#ifndef GJ_LEAN_MINB_GATHER
#define GJ_LEAN_MINB_GATHER 3
#endif
constexpr uint32_t kEntNone = 0xFFFFFFFFu;   // ent1: no generic edge
constexpr uint32_t kEntMulti = 0xFFFFFFFEu;  // ent1: several generic edges -> agent-major CSR
constexpr uint32_t kEntGiant = 0x80000000u;  // ent1 bit 31: the group has more than GJ_SCATTER_MAX_GROUP members
constexpr uint32_t kEntId = 0x7FFFFFFFu;

// ---- forward sums of the generic tier by scatter -----------------------------------------------------------
// Only infectious agents transmit (a few per cent of the world): instead of a group-major pass that gathers every
// member's transmission (a 32-byte DRAM sector per 4-byte member: 2.7x the algorithmic traffic, r1 profile), the
// transmission pass lets each infectious agent ADD its value to its group's accumulator.  The accumulators are
// 64-bit FIXED-POINT integers (GJ_SCATTER_FRAC fractional bits): integer addition is exact and order-independent,
// so the sums are bit-reproducible whatever order the atomics land in — and more accurate than an fp32 sum.  A value
// outside [0, 2^GJ_SCATTER_CAP_LOG2) (never seen with the reference's profiles; non-finite included) marks its group
// dirty: the finalize pass re-sums such a group from its member list.  k_lean_scatter_finalize turns accumulators
// into the fp32 group sums and leaves them zero.
struct Scatter {
  unsigned long long* acc;   // [n_groups] zero between steps
  uint8_t* dirty;            // [n_groups]
};
constexpr float kScatterScale = (float)(1ull << GJ_SCATTER_FRAC);
constexpr float kScatterCap = (float)(1u << GJ_SCATTER_CAP_LOG2);
__device__ __forceinline__ void scatter_one(const Scatter& sc, uint32_t g, float v) {
  if (v > 0.0f && v < kScatterCap) atomicAdd(&sc.acc[g], (unsigned long long)__float2ll_rn(v * kScatterScale));
  else sc.dirty[g] = 1;
}
// v != 0: add it to every scatter-tier group of agent a (ent = its ent1 word)
__device__ __forceinline__ void lean_scatter(const gj_world_desc& w, const Scatter& sc, uint32_t ent, uint32_t a,
                                             float v) {
  if (ent < kEntGiant) {
    scatter_one(sc, ent, v);
  } else if (ent == kEntMulti) {
    for (uint32_t j = w.am_ptr[a]; j < w.am_ptr[a + 1]; ++j) {
      const uint32_t e = w.am_ent[j];
      const uint32_t g = (uint32_t)w.type_group_off[e >> 28] + (e & 0x0FFFFFFFu);
      if (w.gm_ptr[g + 1] - w.gm_ptr[g] <= (uint32_t)GJ_SCATTER_MAX_GROUP) scatter_one(sc, g, v);
    }
  }
}

struct LeanPlan {
  int n_range;                              // networks on RANGE-tier types: 0 or 1
  const uint32_t* r_slot;                   // per agent (offset << 16) | size, kNoSlot = not a member
  const float* r_pc;                        // per agent contact probability of its group
  int r_pc_lut;                             // 1: it equals clamp(1/(size-1), 0, 1): the pipelined kernels use a table
  int r_net;                                // index of the network (beta)
  int r_house;                              // 1: HOUSEHOLD kind (ignores quarantine), 0: PLAIN
  int n_cell;                               // networks on CELL-tier types, same order as Plan::t2_net
  int c_row[GJ_MAX_CHANNELS];               // attendance table row
  int c_care[GJ_MAX_CHANNELS];              // CARE_VISIT: susceptible side masked by age > 75
  int64_t c_cell_off[GJ_MAX_CHANNELS];
  const uint32_t* c_tile_cell[GJ_MAX_CHANNELS];
  int n_tc;                                 // distinct tile -> cell maps among the channels
  const uint32_t* tc[GJ_MAX_CHANNELS];
  const uint32_t* ctp[GJ_MAX_CHANNELS];     // their cell -> first tile maps (cell_tile_ptr)
  int has_generic;
  int64_t gen_base;                         // offset of the per-global-group buffers inside the S / R arrays
};

__device__ __forceinline__ float lg2_fast(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float ex2_fast(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_fast(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ int age_of(int cls) { return cls >= 100 ? cls - 100 : cls; }  // cls = sex * 100 + age

// packed profile {A = maxinf * k0 * rate, rate, e = shape - 1, shift}: T / is_infected and d/d infection_time
// (transmission.py:38-51; same function as transmission_terms, evaluated as A * 2^(e*log2(x) - x*log2(e)))
template <bool kGrad>
__device__ __forceinline__ TransTerms lean_transmission(float now, float tinf, float4 pf) {
  const float d = (now - tinf) - pf.w;
  const float sg = d + 1e-10f;
  const float sign01 = (sg > 0.0f) ? 1.0f : ((sg == 0.0f) ? 0.5f : 0.0f);
  const float x = d * pf.y;
  const float pe = ex2_fast(fmaf(pf.z, lg2_fast(x), -x * 1.4426950408889634f));
  TransTerms r;
  r.coef = (pf.x * sign01) * pe;
  r.dcoef = 0.0f;
  if (kGrad) r.dcoef = r.coef * pf.y * (1.0f - pf.z * rcp_fast(x));  // d/dtinf = -d/dt
  return r;
}

__global__ void __launch_bounds__(kBlock) k_profile_pack(int64_t n, const float* __restrict__ maxinf,
                                                         const float* __restrict__ shape,
                                                         const float* __restrict__ rate,
                                                         const float* __restrict__ shift, const float* __restrict__ k0,
                                                         float4* __restrict__ out) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; a < n; a += stride)
    out[a] = make_float4((maxinf[a] * k0[a]) * rate[a], rate[a], shape[a] - 1.0f, shift[a]);
}

// ---- the CTA's run of tiles -------------------------------------------------------------------------------
struct TileRun {
  int64_t t0, t1;
};
__device__ __forceinline__ TileRun lean_tiles(const gj_world_desc& w) {
  TileRun r;
  r.t0 = w.n_tiles * (int64_t)blockIdx.x / gridDim.x;
  r.t1 = w.n_tiles * ((int64_t)blockIdx.x + 1) / gridDim.x;
  return r;
}
// ... of a batched launch: the run of this CTA among its sample's CTAs
__device__ __forceinline__ TileRun lean_tiles(const gj_world_desc& w, const BatchCta& bc) {
  TileRun r;
  r.t0 = w.n_tiles * (int64_t)bc.bx / bc.gx;
  r.t1 = w.n_tiles * ((int64_t)bc.bx + 1) / bc.gx;
  return r;
}
// first tile after `tile` that lies in another cell (of any cell-tier type), clipped to the run  (CTA-uniform)
__device__ __forceinline__ int64_t lean_segment_end(const LeanPlan& lp, int64_t tile, int64_t t1) {
  int64_t e = t1;
  for (int i = 0; i < lp.n_tc; ++i) {
    const int64_t c = lp.ctp[i][lp.tc[i][tile] + 1];
    e = c < e ? c : e;
  }
  return e;
}
// does tile b lie in another cell (of any cell-tier type) than tile a?  (CTA-uniform)
__device__ __forceinline__ bool lean_new_cell(const LeanPlan& lp, int64_t a, int64_t b) {
  bool changed = false;
  for (int i = 0; i < lp.n_tc; ++i) changed = changed || (lp.tc[i][a] != lp.tc[i][b]);
  return changed;
}

// attendance tables of the cell-tier channels for today's day type, one row of GJ_MAX_CHANNELS per class;
// kCareSide folds the (age > 75) mask of care visits into the table (susceptible side of the forward, member side
// of the backward)
struct alignas(16) ProbRow {
  float v[GJ_MAX_CHANNELS];
};
template <bool kCareSide>
__device__ __forceinline__ void lean_load_prob(ProbRow* prob, const gj_step_params& p, const LeanPlan& lp,
                                               const float* __restrict__ lprob) {
  for (int i = threadIdx.x; i < GJ_MAX_CHANNELS * 200; i += blockDim.x) {
    const int j = i / 200, c = i - j * 200;
    float v = 0.0f;
    if (j < lp.n_cell) {
      v = lprob[(size_t)(lp.c_row[j] * 2 + p.day_type) * 200 + c];
      if (kCareSide && lp.c_care[j] && age_of(c) <= 75) v = 0.0f;
    }
    prob[c].v[j] = v;
  }
}

// acc[j] += prob[cls][j] * x for the cell channels (two 16-byte shared loads)
__device__ __forceinline__ void lean_channel_fma(float (&acc)[GJ_MAX_CHANNELS], const ProbRow* prob, int cls, float x,
                                                 int n_cell) {
  const float4 lo = *reinterpret_cast<const float4*>(&prob[cls].v[0]);
  acc[0] = fmaf(lo.x, x, acc[0]);
  acc[1] = fmaf(lo.y, x, acc[1]);
  acc[2] = fmaf(lo.z, x, acc[2]);
  acc[3] = fmaf(lo.w, x, acc[3]);
  if (n_cell > 4) {
    const float4 hi = *reinterpret_cast<const float4*>(&prob[cls].v[4]);
    acc[4] = fmaf(hi.x, x, acc[4]);
    acc[5] = fmaf(hi.y, x, acc[5]);
    acc[6] = fmaf(hi.z, x, acc[6]);
    acc[7] = fmaf(hi.w, x, acc[7]);
  }
}

// L[class] = sum_j V_j * prob[class][j] from the per-cell values of `tile`'s cell: lane j of every warp fetches
// V_j, the warp shares it by shuffles
__device__ __forceinline__ void lean_class_table(float* __restrict__ L, const ProbRow* prob, const LeanPlan& lp,
                                                 const float* __restrict__ cell_buf, int64_t tile) {
  const int lane = threadIdx.x & 31;
  float mine = 0.0f;
  if (lane < lp.n_cell)
    mine = cell_buf[(lp.c_cell_off[lane] + lp.c_tile_cell[lane][tile]) * GJ_MAX_CHANNELS + lane];
  float acc = 0.0f;
  const int c = threadIdx.x < 200 ? threadIdx.x : 0;
#pragma unroll
  for (int j = 0; j < GJ_MAX_CHANNELS; ++j) {
    const float v = __shfl_sync(0xffffffffu, mine, j);
    acc = fmaf(v, prob[c].v[j], acc);  // channels >= n_cell hold zeros
  }
  if (threadIdx.x < 200) L[threadIdx.x] = acc;
}

// generic tier: combined value of the agent's group(s): the single-entry gather is issued early, the (rare)
// several-entries case walks the agent-major CSR afterwards
__device__ __forceinline__ float lean_generic_issue(const float* __restrict__ buf, uint32_t ent) {
  return (ent < kEntMulti) ? buf[ent & kEntId] : 0.0f;
}
__device__ __forceinline__ float lean_generic_finish(const gj_world_desc& w, const float* __restrict__ buf, uint32_t ent,
                                                     uint32_t a, float v) {
  if (ent == kEntMulti) {
    for (uint32_t j = w.am_ptr[a]; j < w.am_ptr[a + 1]; ++j) {
      const uint32_t e = w.am_ent[j];
      v += buf[w.type_group_off[e >> 28] + (e & 0x0FFFFFFFu)];
    }
  }
  return v;
}

// range-tier network: (offset, size) word -> the group's member values (members = neighbouring agents).  The
// first eight members are fetched with predicated loads that are all in flight together (households); the sum is
// formed later, after the other loads of the batch have been issued.
struct RangeLoads {
  float x[8];
};
__device__ __forceinline__ RangeLoads lean_range_issue(const float* __restrict__ v, uint32_t a, uint32_t slot) {
  RangeLoads r;
  const uint32_t b0 = a - (slot >> 16);
  const int nb = (slot == kNoSlot) ? 0 : (int)(slot & 0xFFFFu);
#pragma unroll
  for (int j = 0; j < 8; ++j) r.x[j] = (j < nb) ? v[b0 + j] : 0.0f;
  return r;
}
__device__ __forceinline__ float lean_range_finish(const RangeLoads& r, const float* __restrict__ v, uint32_t a,
                                                   uint32_t slot) {
  float S = ((r.x[0] + r.x[1]) + (r.x[2] + r.x[3])) + ((r.x[4] + r.x[5]) + (r.x[6] + r.x[7]));
  if (slot != kNoSlot && (slot & 0xFFFFu) > 8u) {
    const uint32_t b0 = a - (slot >> 16), nb = slot & 0xFFFFu;
    for (uint32_t b = b0 + 8; b < b0 + nb; ++b) S += v[b];
  }
  return S;
}

__device__ __forceinline__ float quar_mask(const gj_step_params& p, float cur) {
  bool ok = true;
#pragma unroll
  for (int i = 0; i < GJ_MAX_QUAR; ++i)
    if (i < p.n_quar) ok = ok && (cur < p.quar_thr[i]);
  return ok ? 1.0f : 0.0f;
}

// =====================================================================================================
// K1  transmissions (+ quarantine-masked copy) and the partial sums of the cell channels.  A CTA's run of tiles
//     is walked cell by cell ("segments"); a segment's partial sums are written to its first tile and zeros to its
//     other tiles: k_cell_groups adds a cell's tiles, so the per-cell totals are unchanged.
// =====================================================================================================
#ifndef GJ_K1_BATCH
#define GJ_K1_BATCH 2   // measured on B200 (56 M agents): batch x CTAs/SM = 2x7 0.208 ms, 2x8 0.208, 4x4 0.236, 1x8 0.244, 8x3 0.273
#endif
#ifndef GJ_K1_MINB
#define GJ_K1_MINB 7
#endif
constexpr int kK1Batch = GJ_K1_BATCH;

template <bool kQuar, bool kBatch>
__global__ void __launch_bounds__(kLeanThreads, GJ_K1_MINB) k_lean_transmission(gj_world_desc w, gj_step_params p, LeanPlan lp,
                                                                    gj_fwd_io io, float* __restrict__ tile_part,
                                                                    Scatter sct, Batch bt) {
  __shared__ ProbRow prob[200];
  pdl_launch();
  lean_load_prob<false>(prob, p, lp, io.leisure_prob);
  pdl_wait();
  __syncthreads();
  const BatchCta bc = batch_cta<kBatch>(bt);
  const uint32_t so = bc.so;   // batched ensemble: this sample's offset into the per-agent arrays (else 0)
  if (kBatch) {
    tile_part = scr_shift(tile_part, bt, bc.s);
    sct.acc = scr_shift(sct.acc, bt, bc.s);
    sct.dirty = scr_shift(sct.dirty, bt, bc.s);
  }
  const float4* __restrict__ prof = reinterpret_cast<const float4*>(io.prof4);
  const float* __restrict__ g_inf = io.inf;
  const float* __restrict__ g_cur = io.cur;
  const TileRun run = lean_tiles(w, bc);
  for (int64_t tile = run.t0; tile < run.t1;) {
    const int64_t tend = lp.n_cell > 0 ? lean_segment_end(lp, tile, run.t1) : run.t1;
    const uint32_t a0 = w.tile_begin[tile], a1 = w.tile_begin[tend];
    float acc[GJ_MAX_CHANNELS];
#pragma unroll
    for (int j = 0; j < GJ_MAX_CHANNELS; ++j) acc[j] = 0.0f;
    for (uint32_t base = a0 + threadIdx.x; base < a1; base += kK1Batch * kLeanThreads) {
      float inf[kK1Batch], cur[kK1Batch];
#pragma unroll
      for (int h = 0; h < kK1Batch; ++h) {  // the batch's streaming loads first
        const uint32_t a = base + h * kLeanThreads;
        inf[h] = (a < a1) ? g_inf[a + so] : 0.0f;
        cur[h] = (kQuar && a < a1) ? g_cur[a + so] : 0.0f;
      }
      // the infectious few: ALL their dependent loads (infection time, packed profile, group word, class) are issued
      // before the first use — one exposed DRAM latency per batch instead of one per infectious agent
      float tinf[kK1Batch];
      float4 pf[kK1Batch];
      uint32_t ent[kK1Batch];
      int cls[kK1Batch];
#pragma unroll
      for (int h = 0; h < kK1Batch; ++h) {
        const uint32_t a = base + h * kLeanThreads;
        const bool on = inf[h] != 0.0f;   // false beyond a1
        tinf[h] = on ? io.tinf[a + so] : 0.0f;
        pf[h] = on ? prof[a] : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        ent[h] = (on && lp.has_generic) ? w.ent1[a] : kEntNone;
        cls[h] = (on && lp.n_cell > 0) ? (int)w.cls[a] : 0;
      }
#pragma unroll
      for (int h = 0; h < kK1Batch; ++h) {
        const uint32_t a = base + h * kLeanThreads;
        if (a >= a1) break;
        float T = 0.0f;
        if (inf[h] != 0.0f) T = lean_transmission<false>(p.now, tinf[h], pf[h]).coef * inf[h];
        io.T[a + so] = T;
        float Tq = T;
        if (kQuar) {
          Tq = quar_mask(p, cur[h]) * T;
          io.Tq[a + so] = Tq;
        }
        if (Tq != 0.0f) {   // cell-channel partial sums and the generic groups' accumulators
          if (lp.n_cell > 0) lean_channel_fma(acc, prob, cls[h], Tq, lp.n_cell);
          if (lp.has_generic) lean_scatter(w, sct, ent[h], a, Tq);
        }
      }
    }
    if (lp.n_cell > 0) {
      block_sums<float, GJ_MAX_CHANNELS>(acc, lp.n_cell, tile_part + tile * GJ_MAX_CHANNELS);
      for (int64_t i = threadIdx.x; i < (tend - tile - 1) * GJ_MAX_CHANNELS; i += kLeanThreads)
        tile_part[(tile + 1) * GJ_MAX_CHANNELS + i] = 0.0f;
    }
    tile = tend;
  }
}

// =====================================================================================================
// K1c  the same pass with the infectious agents COMPACTED per warp.  K1 above is latency-bound: a warp keeps 64 agents
//      in flight and sits out two dependent DRAM round trips per batch (is_infected, then the profile of the few
//      infectious lanes) however few those lanes are.  Here a warp streams a chunk of 32 x GJ_K1C_PER agents with that
//      many independent loads per lane, writes the zeros of everybody who is not infectious straight away, ballots, and then hands the
//      chunk's infectious agents out densely, one per lane: ONE exposed round trip for the dependent loads of up to 32
//      infectious agents.  Same arithmetic per agent (T is bit-identical to K1's); the per-thread partial sums of the
//      cell channels are associated differently (another agent -> lane map).  The quarantine stage is read for the
//      infectious agents only.
// =====================================================================================================
#ifndef GJ_K1C_MINB
#define GJ_K1C_MINB 4
#endif
#ifndef GJ_K1C_PER
#define GJ_K1C_PER 16   // measured on B200 (56 M agents): per x CTAs/SM = 16x4 0.152 ms, 8x5 0.161, 8x6 0.166, 12x5 0.165, 16x3 0.169, 16x5 0.168, 24x3 0.195, 4x8 0.188; K1: 0.208
#endif
constexpr int kK1cPer = GJ_K1C_PER;   // agents per lane and chunk

template <bool kQuar, bool kBatch>
__global__ void __launch_bounds__(kLeanThreads, GJ_K1C_MINB) k_lean_transmission_c(gj_world_desc w, gj_step_params p,
                                                                                  LeanPlan lp, gj_fwd_io io,
                                                                                  float* __restrict__ tile_part,
                                                                                  Scatter sct, Batch bt) {
  __shared__ ProbRow prob[200];
  pdl_launch();
  lean_load_prob<false>(prob, p, lp, io.leisure_prob);
  pdl_wait();
  __syncthreads();
  const BatchCta bc = batch_cta<kBatch>(bt);
  const uint32_t so = bc.so;
  if (kBatch) {
    tile_part = scr_shift(tile_part, bt, bc.s);
    sct.acc = scr_shift(sct.acc, bt, bc.s);
    sct.dirty = scr_shift(sct.dirty, bt, bc.s);
  }
  const float4* __restrict__ prof = reinterpret_cast<const float4*>(io.prof4);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  constexpr uint32_t kChunk = 32u * kK1cPer;
  constexpr uint32_t kWarps = kLeanThreads / 32;
  const TileRun run = lean_tiles(w, bc);
  for (int64_t tile = run.t0; tile < run.t1;) {
    const int64_t tend = lp.n_cell > 0 ? lean_segment_end(lp, tile, run.t1) : run.t1;
    const uint32_t a0 = w.tile_begin[tile], a1 = w.tile_begin[tend];
    float acc[GJ_MAX_CHANNELS];
#pragma unroll
    for (int j = 0; j < GJ_MAX_CHANNELS; ++j) acc[j] = 0.0f;
    for (uint32_t cb = a0 + wid * kChunk; cb < a1; cb += kWarps * kChunk) {
      float inf[kK1cPer];
      unsigned int mask[kK1cPer];
#pragma unroll
      for (int j = 0; j < kK1cPer; ++j) {   // the chunk's streaming loads, all in flight
        const uint32_t a = cb + j * 32 + lane;
        inf[j] = (a < a1) ? io.inf[a + so] : 0.0f;
      }
      int total = 0;
#pragma unroll
      for (int j = 0; j < kK1cPer; ++j) {   // zeros for everybody who is not infectious; who is, by ballot
        const uint32_t a = cb + j * 32 + lane;
        const bool on = inf[j] != 0.0f;
        mask[j] = __ballot_sync(0xffffffffu, on);
        total += __popc(mask[j]);
        if (a < a1 && !on) {
          io.T[a + so] = 0.0f;
          if (kQuar) io.Tq[a + so] = 0.0f;
        }
      }
      for (int k0 = 0; k0 < total; k0 += 32) {   // the infectious agents, one per lane
        int rem = k0 + lane, jsel = 0;
        unsigned int m = 0u;
        bool found = false;
#pragma unroll
        for (int j = 0; j < kK1cPer; ++j) {
          const int c = __popc(mask[j]);
          if (!found) {
            if (rem < c) {
              found = true;
              m = mask[j];
              jsel = j;
            } else {
              rem -= c;
            }
          }
        }
        if (!found) continue;
        const uint32_t a = cb + jsel * 32 + __fns(m, 0u, rem + 1);
        // every dependent load of the agent is issued before the first use
        const float infv = io.inf[a + so];
        const float tinf = io.tinf[a + so];
        const float4 pf = prof[a];
        const uint32_t ent = lp.has_generic ? w.ent1[a] : kEntNone;
        const int cls = lp.n_cell > 0 ? (int)w.cls[a] : 0;
        const float cur = kQuar ? io.cur[a + so] : 0.0f;
        const float T = lean_transmission<false>(p.now, tinf, pf).coef * infv;
        io.T[a + so] = T;
        float Tq = T;
        if (kQuar) {
          Tq = quar_mask(p, cur) * T;
          io.Tq[a + so] = Tq;
        }
        if (Tq != 0.0f) {
          if (lp.n_cell > 0) lean_channel_fma(acc, prob, cls, Tq, lp.n_cell);
          if (lp.has_generic) lean_scatter(w, sct, ent, a, Tq);
        }
      }
    }
    if (lp.n_cell > 0) {
      block_sums<float, GJ_MAX_CHANNELS>(acc, lp.n_cell, tile_part + tile * GJ_MAX_CHANNELS);
      for (int64_t i = threadIdx.x; i < (tend - tile - 1) * GJ_MAX_CHANNELS; i += kLeanThreads)
        tile_part[(tile + 1) * GJ_MAX_CHANNELS + i] = 0.0f;
    }
    tile = tend;
  }
}

// =====================================================================================================
// K2  generic-tier group sums, one value per global group: plain = sum of member values,
//     scaled = (sum of the betas of the type's networks) * pc_g * plain.  Forward: in = Tq; backward: in = wq.
// =====================================================================================================
struct LeanGroupShared {
  float bsum[GJ_MAX_TYPES];     // sum of the betas of the type's generic networks; NaN = no active network
  uint32_t toff[GJ_MAX_TYPES];  // first global group id of each type (32-bit: n_groups < 2^32 is checked on entry)
};
__device__ __forceinline__ void lean_beta_sums(LeanGroupShared& sh, const gj_world_desc& w, const gj_step_params& p,
                                               const Plan& pl, const float* __restrict__ beta) {
  if (threadIdx.x < GJ_MAX_TYPES) {
    float b = 0.0f;
    bool any = false;
    for (int k = 0; k < p.n_nets; ++k)
      if (pl.tier[k] == GJ_TIER_GENERIC && p.nets[k].type == (int)threadIdx.x) {
        b += beta[k];
        any = true;
      }
    sh.bsum[threadIdx.x] = any ? b : nanf("");
    sh.toff[threadIdx.x] = (int)threadIdx.x < w.n_types ? (uint32_t)w.type_group_off[threadIdx.x] : 0xFFFFFFFFu;
  }
  __syncthreads();
}
// beta sum of group g's type (type_of_group() with 32-bit compares against shared memory)
__device__ __forceinline__ float lean_group_beta(const LeanGroupShared& sh, uint32_t g) {
  int t = 0;
#pragma unroll
  for (int i = 1; i < GJ_MAX_TYPES; ++i) t += (g >= sh.toff[i]) ? 1 : 0;
  return sh.bsum[t];
}
// regional venue factor: the generic networks of each type (ascending k, the order of lean_beta_sums) and their betas
struct LeanVenueShared {
  int nk[GJ_MAX_TYPES];
  int k[GJ_MAX_TYPES][GJ_MAX_CHANNELS];
  float beta[GJ_MAX_NETS];
};
__device__ __forceinline__ void lean_venue_nets(LeanVenueShared& vs, const gj_step_params& p, const Plan& pl,
                                                const float* __restrict__ beta) {
  if (threadIdx.x < GJ_MAX_TYPES) {
    int n = 0;
    for (int k = 0; k < p.n_nets; ++k)
      if (pl.tier[k] == GJ_TIER_GENERIC && p.nets[k].type == (int)threadIdx.x && n < GJ_MAX_CHANNELS)
        vs.k[threadIdx.x][n++] = k;
    vs.nk[threadIdx.x] = n;
  }
  if (threadIdx.x < GJ_MAX_NETS) vs.beta[threadIdx.x] = (int)threadIdx.x < p.n_nets ? beta[threadIdx.x] : 0.0f;
  // the caller's lean_beta_sums synchronises
}
// the value that replaces the type's beta sum for group g: sum_k beta_k * f_k[region(g)] (NaN = no active network);
// a factor of 1 gives the beta sum bit for bit
__device__ __forceinline__ float lean_venue_beta(const LeanGroupShared& sh, const LeanVenueShared& vs, const Venue& v,
                                                 uint32_t g) {
  int t = 0;
#pragma unroll
  for (int i = 1; i < GJ_MAX_TYPES; ++i) t += (g >= sh.toff[i]) ? 1 : 0;
  float b = sh.bsum[t];
  if (b == b) {
    const int64_t r = __ldg(v.region + g);
    b = 0.0f;
    for (int i = 0; i < vs.nk[t]; ++i) {
      const int k = vs.k[t][i];
      b += vs.beta[k] * __ldg(v.factor + (int64_t)k * v.n + r);
    }
  }
  return b;
}
template <bool kVenue>
__device__ __forceinline__ float lean_beta_of(const LeanGroupShared& sh, const LeanVenueShared* vs, const Venue& v,
                                              uint32_t g) {
  return kVenue ? lean_venue_beta(sh, *vs, v, g) : lean_group_beta(sh, g);
}

// one group of <= GJ_SMALL_GROUP members per thread
template <bool kVenue = false>
__device__ __forceinline__ void lean_group_small_body(const gj_world_desc& w, const LeanGroupShared& gs, int64_t i,
                                                      const float* __restrict__ in, float* __restrict__ out_scaled,
                                                      float* __restrict__ out_plain,
                                                      const LeanVenueShared* vs = nullptr, const Venue& v = Venue{}) {
  if (i >= w.n_small) return;
  const uint32_t g = w.small_groups[i];
  const float b = lean_beta_of<kVenue>(gs, vs, v, g);
  float S = 0.0f;
  if (b == b) {
    const uint32_t j0 = w.gm_ptr[g], j1 = w.gm_ptr[g + 1];
    for (uint32_t j = j0; j < j1; j += 4) {  // four member gathers in flight (same summation order)
      uint32_t m[4];
      float x[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) m[k] = (j + k < j1) ? w.gm_agent[j + k] : 0u;
#pragma unroll
      for (int k = 0; k < 4; ++k) x[k] = (j + k < j1) ? in[m[k]] : 0.0f;
#pragma unroll
      for (int k = 0; k < 4; ++k) S += x[k];
    }
  }
  out_plain[g] = S;
  out_scaled[g] = (b == b) ? (b * w.pc[g]) * S : 0.0f;
}

// one chunk of <= GJ_CHUNK members per warp
template <bool kVenue = false>
__device__ __forceinline__ void lean_group_chunk_body(const gj_world_desc& w, const LeanGroupShared& gs, int64_t ci,
                                                      const float* __restrict__ in, float* __restrict__ out_scaled,
                                                      float* __restrict__ out_plain, float* __restrict__ part,
                                                      const LeanVenueShared* vs = nullptr, const Venue& v = Venue{}) {
  const int lane = threadIdx.x & 31;
  if (ci >= w.n_chunks) return;
  const uint32_t g = w.chunk_group[ci];
  const float b = lean_beta_of<kVenue>(gs, vs, v, g);
  float S = 0.0f;
  if (b == b) {
    const uint32_t j0 = w.chunk_begin[ci], j1 = w.chunk_end[ci];
    constexpr int kDeep = 4;  // member gathers per lane in flight (16 was measured slower); the summation order is
                              // that of a sequential walk of the lane's members
    for (uint32_t j = j0 + lane; j < j1; j += 32 * kDeep) {
      uint32_t m[kDeep];
      float x[kDeep];
#pragma unroll
      for (int k = 0; k < kDeep; ++k) m[k] = (j + 32 * k < j1) ? w.gm_agent[j + 32 * k] : 0u;
#pragma unroll
      for (int k = 0; k < kDeep; ++k) x[k] = (j + 32 * k < j1) ? in[m[k]] : 0.0f;
#pragma unroll
      for (int k = 0; k < kDeep; ++k) S += x[k];
    }
    S = warp_sum(S);
  }
  if (lane != 0) return;
  const int pi = w.chunk_part[ci];
  if (pi < 0) {
    out_plain[g] = S;
    out_scaled[g] = (b == b) ? (b * w.pc[g]) * S : 0.0f;
  } else {
    part[pi] = S;
  }
}

// ONE launch for both group-size classes: blocks [0, chunk_blocks) take the chunks (the longer work first), the rest
// the small groups.  Both are latency-bound gathers, so they overlap almost perfectly (measured: 0.058 + 0.166 ms as
// two launches at 56 M agents).
__global__ void __launch_bounds__(kBlock) k_lean_group_sums(gj_world_desc w, gj_step_params p, Plan pl,
                                                            const float* __restrict__ beta,
                                                            const float* __restrict__ in, float* __restrict__ out_scaled,
                                                            float* __restrict__ out_plain, float* __restrict__ part,
                                                            int chunk_blocks, Batch bt) {
  __shared__ LeanGroupShared gs;
  pdl_launch();
  pdl_wait();
  uint32_t bx = blockIdx.x;
  if (bt.nb > 1) {   // batched ensemble: block = unit * nb + sample (the samples share the member lists through L2)
    const int s = (int)(bx % (uint32_t)bt.nb);
    bx /= (uint32_t)bt.nb;
    beta += (int64_t)s * bt.sBeta;
    in += (int64_t)s * bt.sN;
    out_scaled += (int64_t)s * bt.sG;
    out_plain += (int64_t)s * bt.sG;
    part = scr_shift(part, bt, s);
  }
  lean_beta_sums(gs, w, p, pl, beta);
  if ((int)bx < chunk_blocks)
    lean_group_chunk_body(w, gs, ((int64_t)bx * blockDim.x + threadIdx.x) >> 5, in, out_scaled, out_plain, part);
  else
    lean_group_small_body(w, gs, (int64_t)(bx - chunk_blocks) * blockDim.x + threadIdx.x, in, out_scaled,
                          out_plain);
}
// k_lean_group_sums with the regional venue factor
__global__ void __launch_bounds__(kBlock) k_lean_group_sums_venue(gj_world_desc w, gj_step_params p, Plan pl,
                                                                  const float* __restrict__ beta,
                                                                  const float* __restrict__ in,
                                                                  float* __restrict__ out_scaled,
                                                                  float* __restrict__ out_plain,
                                                                  float* __restrict__ part, int chunk_blocks, Batch bt,
                                                                  Venue v) {
  __shared__ LeanGroupShared gs;
  __shared__ LeanVenueShared vs;
  pdl_launch();
  pdl_wait();
  uint32_t bx = blockIdx.x;
  if (bt.nb > 1) {
    const int s = (int)(bx % (uint32_t)bt.nb);
    bx /= (uint32_t)bt.nb;
    beta += (int64_t)s * bt.sBeta;
    in += (int64_t)s * bt.sN;
    out_scaled += (int64_t)s * bt.sG;
    out_plain += (int64_t)s * bt.sG;
    part = scr_shift(part, bt, s);
    v.factor += (int64_t)s * bt.sVen;
  }
  lean_venue_nets(vs, p, pl, beta);
  lean_beta_sums(gs, w, p, pl, beta);
  if ((int)bx < chunk_blocks)
    lean_group_chunk_body<true>(w, gs, ((int64_t)bx * blockDim.x + threadIdx.x) >> 5, in, out_scaled, out_plain, part,
                                &vs, v);
  else
    lean_group_small_body<true>(w, gs, (int64_t)(bx - chunk_blocks) * blockDim.x + threadIdx.x, in, out_scaled,
                                out_plain, &vs, v);
}

// groups spanning several chunks: one WARP per group adds the chunk partials (lanes stride over them, then the fixed
// shuffle tree): a handful of groups, so the kernel is pure latency — a serial walk per thread measured 8.6 us
template <bool kVenue>
__device__ __forceinline__ void lean_group_fix_body(const gj_world_desc& w, const gj_step_params& p, const Plan& pl,
                                                    const float* __restrict__ beta, const float* __restrict__ part,
                                                    float* __restrict__ out_scaled, float* __restrict__ out_plain,
                                                    const Batch& bt, LeanGroupShared& gs, LeanVenueShared* vs,
                                                    Venue v) {
  pdl_launch();
  pdl_wait();
  uint32_t bx = blockIdx.x;
  if (bt.nb > 1) {
    const int s = (int)(bx % (uint32_t)bt.nb);
    bx /= (uint32_t)bt.nb;
    beta += (int64_t)s * bt.sBeta;
    out_scaled += (int64_t)s * bt.sG;
    out_plain += (int64_t)s * bt.sG;
    part = scr_shift(part, bt, s);
    if (kVenue) v.factor += (int64_t)s * bt.sVen;
  }
  if (kVenue) lean_venue_nets(*vs, p, pl, beta);
  lean_beta_sums(gs, w, p, pl, beta);
  const int lane = threadIdx.x & 31;
  const int64_t i = ((int64_t)bx * blockDim.x + threadIdx.x) >> 5;
  if (i >= w.n_big) return;
  const uint32_t g = w.big_groups[i];
  const float b = lean_beta_of<kVenue>(gs, vs, v, g);
  float S = 0.0f;
  for (uint32_t j = w.big_part_ptr[i] + lane; j < w.big_part_ptr[i + 1]; j += 32) S += part[j];
  S = warp_sum(S);
  if (lane != 0) return;
  out_plain[g] = S;
  out_scaled[g] = (b == b) ? (b * w.pc[g]) * S : 0.0f;
}
__global__ void __launch_bounds__(kBlock) k_lean_group_fix(gj_world_desc w, gj_step_params p, Plan pl,
                                                           const float* __restrict__ beta,
                                                           const float* __restrict__ part,
                                                           float* __restrict__ out_scaled,
                                                           float* __restrict__ out_plain, Batch bt) {
  __shared__ LeanGroupShared gs;
  lean_group_fix_body<false>(w, p, pl, beta, part, out_scaled, out_plain, bt, gs, nullptr, Venue{nullptr, nullptr, 0});
}
__global__ void __launch_bounds__(kBlock) k_lean_group_fix_venue(gj_world_desc w, gj_step_params p, Plan pl,
                                                                 const float* __restrict__ beta,
                                                                 const float* __restrict__ part,
                                                                 float* __restrict__ out_scaled,
                                                                 float* __restrict__ out_plain, Batch bt, Venue v) {
  __shared__ LeanGroupShared gs;
  __shared__ LeanVenueShared vs;
  lean_group_fix_body<true>(w, p, pl, beta, part, out_scaled, out_plain, bt, gs, &vs, v);
}

// the generic-tier types' global group id ranges, concatenated: thread i -> group (host-built, passed by value)
struct GenericRanges {
  int n;
  int64_t first[GJ_MAX_TYPES];   // first global group id of the range
  int64_t start[GJ_MAX_TYPES + 1];   // first linear index of the range
};
template <bool kVenue>
__device__ __forceinline__ void lean_scatter_finalize_body(const gj_world_desc& w, const gj_step_params& p,
                                                           const Plan& pl, const GenericRanges& gr,
                                                           const float* __restrict__ beta, const float* __restrict__ in,
                                                           Scatter sct, float* __restrict__ out_scaled,
                                                           float* __restrict__ out_plain, const Batch& bt,
                                                           LeanGroupShared& gs, LeanVenueShared* vs, Venue v) {
  pdl_launch();
  pdl_wait();
  uint32_t bx = blockIdx.x;
  if (bt.nb > 1) {
    const int s = (int)(bx % (uint32_t)bt.nb);
    bx /= (uint32_t)bt.nb;
    beta += (int64_t)s * bt.sBeta;
    in += (int64_t)s * bt.sN;
    out_scaled += (int64_t)s * bt.sG;
    out_plain += (int64_t)s * bt.sG;
    sct.acc = scr_shift(sct.acc, bt, s);
    sct.dirty = scr_shift(sct.dirty, bt, s);
    if (kVenue) v.factor += (int64_t)s * bt.sVen;
  }
  if (kVenue) lean_venue_nets(*vs, p, pl, beta);
  lean_beta_sums(gs, w, p, pl, beta);
  const int64_t i = (int64_t)bx * blockDim.x + threadIdx.x;
  if (i >= gr.start[gr.n]) return;
  int r = 0;
#pragma unroll
  for (int k = 1; k < GJ_MAX_TYPES; ++k) r += (k < gr.n && i >= gr.start[k]) ? 1 : 0;
  const int64_t g = gr.first[r] + (i - gr.start[r]);
  const uint32_t j0 = w.gm_ptr[g], j1 = w.gm_ptr[g + 1];
  if (j1 - j0 > (uint32_t)GJ_SCATTER_MAX_GROUP) return;                 // giant: the chunk kernels wrote it
  const unsigned long long acc = sct.acc[g];
  const bool dirty = sct.dirty[g] != 0;
  if (acc != 0ull) sct.acc[g] = 0ull;
  const float b = lean_beta_of<kVenue>(gs, vs, v, (uint32_t)g);
  float S = (float)((double)(long long)acc * (1.0 / (double)(1ull << GJ_SCATTER_FRAC)));
  if (dirty) {
    sct.dirty[g] = 0;
    S = 0.0f;
    for (uint32_t j = j0; j < j1; ++j) S += in[w.gm_agent[j]];
  }
  out_plain[g] = S;
  out_scaled[g] = (b == b) ? (b * w.pc[g]) * S : 0.0f;
}
__global__ void __launch_bounds__(kBlock) k_lean_scatter_finalize(gj_world_desc w, gj_step_params p, Plan pl,
                                                                  GenericRanges gr, const float* __restrict__ beta,
                                                                  const float* __restrict__ in, Scatter sct,
                                                                  float* __restrict__ out_scaled,
                                                                  float* __restrict__ out_plain, Batch bt) {
  __shared__ LeanGroupShared gs;
  lean_scatter_finalize_body<false>(w, p, pl, gr, beta, in, sct, out_scaled, out_plain, bt, gs, nullptr,
                                    Venue{nullptr, nullptr, 0});
}
__global__ void __launch_bounds__(kBlock) k_lean_scatter_finalize_venue(gj_world_desc w, gj_step_params p, Plan pl,
                                                                        GenericRanges gr,
                                                                        const float* __restrict__ beta,
                                                                        const float* __restrict__ in, Scatter sct,
                                                                        float* __restrict__ out_scaled,
                                                                        float* __restrict__ out_plain, Batch bt,
                                                                        Venue v) {
  __shared__ LeanGroupShared gs;
  __shared__ LeanVenueShared vs;
  lean_scatter_finalize_body<true>(w, p, pl, gr, beta, in, sct, out_scaled, out_plain, bt, gs, &vs, v);
}

// per-agent arithmetic of the forward pass, shared by the register-batched kernel below and the bulk-copy pipelined
// kernel of gj_pipe.cuh (identical results): pressure -> q -> Gumbel-softmax draw -> infect -> symptoms -> reductions.
// hs = sum of the member values of the agent's range-tier group, gv = combined value of its generic groups,
// Lc = class-table value of the cell channels
struct FwdOut {
  float inf, tinf, cur;   // post-step is_infected, infection_time, current_stage
};
struct FwdRes {   // everything one agent's forward produces
  float tape_v, tape_y0, q, lam, n;
  float s_o, inf_o, tinf_o, cur_o, nxt_o, ttn_o;
};
// Gumbel noise of the draw from the agent's Philox2x32 pair (philox_step_pair): lg2 E0 - lg2 E1, E = -lg2 u
__device__ __forceinline__ float lean_noise_dE(uint32_t r0, uint32_t r1) {
  return lg2_fast(fmaxf(-lg2_fast(u01_open(r0)), kMinE2)) - lg2_fast(fmaxf(-lg2_fast(u01_open(r1)), kMinE2));
}
// dE: lean_noise_dE of the agent's Philox pair; ga = its id in the noise stream
// kRegion: the pressure is multiplied by the agent's regional factor mreg before the clamp (the tape keeps lam)
template <bool kQuar, bool kRegion = false>
__device__ __forceinline__ FwdRes lean_forward_core(const gj_step_params& p, const LeanPlan& lp,
                                                    const float* __restrict__ stage_prob, uint64_t ga, float dE,
                                                    float hs, float gv, float Lc, float beta_r, float rpc,
                                                    float s, float inf, float tinf, float cur, float nxt, float ttn,
                                                    int cls, float inv_tau, float dead, float* __restrict__ hist,
                                                    float* __restrict__ deaths, float q_seed = -1.0f,
                                                    float mreg = 1.0f) {
  FwdRes o;
  const float rv = (beta_r * rpc) * hs;
  const float house = lp.r_house ? rv : 0.0f;
  const float plain = (gv + Lc) + (lp.r_house ? 0.0f : rv);
  const float mq = kQuar ? quar_mask(p, cur) : 1.0f;
  const float X = fmaf(mq, plain, house);  // pressure per unit susceptibility
  const float lam0 = X * s;
  const float lam = kRegion ? lam0 * mreg : lam0;
  // q_seed >= 0: the seeding step (infect_fraction_of_people, infection.py:31-42): a uniform q = 1 - fraction
  const float q = (q_seed >= 0.0f) ? q_seed : not_infected_prob(lam, p.dt);
  o.tape_v = (s == 0.0f) ? X : lam0;
  // Gumbel-softmax hard draw from Philox bits (same stream as draw_step_noise):
  // x0 - x1 = (ln2 / tau) * d,  d = lg2 q - lg2(1-q) - lg2 E0 + lg2 E1, E = -ln u (the ln2 factors cancel)
  const float d = (lg2_fast(q) - lg2_fast(1.0f - q)) - dE;
  const float e = ex2_fast(-fabsf(d) * inv_tau);  // exp(x_small - x_big) <= 1
  const float ys = e * rcp_fast(1.0f + e);        // the smaller soft probability
  const bool hit = (d < 0.0f) && (e < 1.0f);      // argmax of the softmax; ties -> not infected
  const float n = hit ? 1.0f : 0.0f;
  o.tape_y0 = hit ? -ys : ys;
  o.q = q;
  o.lam = lam;
  o.n = n;
  // infect (model.py:103-110)
  o.inf_o = inf + n;
  o.s_o = fmaxf(0.0f, s - n);
  o.tinf_o = tinf + n * (p.now - tinf);
  // symptoms (symptoms.py:204-247); its draws are needed by the few agents whose stage changes
  const uint64_t seed = p.seed;
  const uint32_t call = p.call_index;
  const int age = age_of(cls);
  const SympOut so = symptoms_forward(p, stage_prob, cur, nxt, ttn, n, age,
                                      [&]() { return draw_step_uniform(seed, call, (int64_t)ga); },
                                      [&](int) { return draw_step_normal(seed, call, (int64_t)ga); });
  o.cur_o = so.cur;
  o.nxt_o = so.nxt;
  o.ttn_o = so.ttn;
  // reductions (runner.py:167-171,198-224): small integers, exact in any order
  if (o.inf_o != 0.0f) atomicAdd(&hist[age], o.inf_o);
  if (so.cur == dead) atomicAdd(deaths, so.cur / dead);
  return o;
}

// one agent: noise, core, stores
template <bool kQuar, bool kDiag, bool kRegion = false>
__device__ __forceinline__ FwdOut lean_forward_agent(const gj_step_params& p, const LeanPlan& lp, const gj_fwd_io& io,
                                                   uint32_t a, uint64_t ga, float hs, float gv, float Lc, float beta_r, float rpc,
                                                   float s, float inf, float tinf, float cur, float nxt, float ttn,
                                                   int cls, float inv_tau, float dead, float* __restrict__ hist,
                                                   float* __restrict__ deaths, bool noise_given = false,
                                                   float dE_given = 0.0f, float mreg = 1.0f) {
  float dE = dE_given;   // batched ensemble: evaluated once for all samples (k_batch_noise)
  if (!noise_given) {
    uint32_t r[2];
    philox_step_pair(p.seed, p.call_index, ga, r);   // ga: the agent's id in the noise stream (noise_agent())
    dE = lean_noise_dE(r[0], r[1]);
  }
  const FwdRes o = lean_forward_core<kQuar, kRegion>(p, lp, io.stage_prob, ga, dE, hs, gv, Lc, beta_r, rpc, s, inf,
                                                     tinf, cur, nxt, ttn, cls, inv_tau, dead, hist, deaths, -1.0f,
                                                     mreg);
  io.tape_v[a] = o.tape_v;
  io.tape_y0[a] = o.tape_y0;
  if (kDiag) {
    if (io.q) io.q[a] = o.q;
    if (io.lam) io.lam[a] = o.lam;
    if (io.n) io.n[a] = o.n;
  }
  io.s_o[a] = o.s_o;
  io.inf_o[a] = o.inf_o;
  io.tinf_o[a] = o.tinf_o;
  io.cur_o[a] = o.cur_o;
  io.nxt_o[a] = o.nxt_o;
  io.ttn_o[a] = o.ttn_o;
  FwdOut out;
  out.inf = o.inf_o;
  out.tinf = o.tinf_o;
  out.cur = o.cur_o;
  return out;
}

// batched ensemble: the draw's noise of every agent, once for all samples of the batch (gj_batch.noise)
__global__ void __launch_bounds__(kBlock) k_batch_noise(gj_world_desc w, gj_step_params p, float* __restrict__ dE) {
  pdl_launch();
  pdl_wait();
  const uint32_t N = (uint32_t)w.n_agents;
  for (uint32_t a = blockIdx.x * blockDim.x + threadIdx.x; a < N; a += gridDim.x * blockDim.x) {
    const uint64_t ga = w.orig_id ? (uint64_t)w.orig_id[a] : p.agent_offset + a;
    uint32_t r[2];
    philox_step_pair(p.seed, p.call_index, ga, r);
    dE[a] = lean_noise_dE(r[0], r[1]);
  }
}

// =====================================================================================================
// K3  forward: pressure -> q -> draw -> state update -> symptoms -> reductions
// =====================================================================================================
struct LeanFwdShared {
  ProbRow prob[200];
  float L[2][200];
  float beta[GJ_MAX_NETS];
  float hist[100];  // sum of post-step is_infected by age
  float deaths;
};

constexpr int kLeanBatch = 2;  // agents a thread keeps in flight: their loads are issued before any arithmetic

// kRegion: regional transmission factor (gj_fwd_io.region): the code is loaded with the batch's other per-agent
// operands, the factor gathered (R floats, L1/L2-resident) before the arithmetic
template <bool kQuar, bool kDiag, bool kLabel, bool kRegion>
__device__ __forceinline__ void lean_forward_body(const gj_world_desc& w, const gj_step_params& p, const LeanPlan& lp,
                                                  const gj_fwd_io& io, const float* __restrict__ cell_buf,
                                                  double* __restrict__ red_part, unsigned int* __restrict__ ticket) {
  __shared__ LeanFwdShared sh;
  lean_load_prob<true>(sh.prob, p, lp, io.leisure_prob);
  if (threadIdx.x < p.n_nets) sh.beta[threadIdx.x] = io.beta[threadIdx.x];
  if (threadIdx.x < 100) sh.hist[threadIdx.x] = 0.0f;
  if (threadIdx.x == 0) sh.deaths = 0.0f;
  __syncthreads();
  const float* __restrict__ Tr = (kQuar && !lp.r_house) ? io.Tq : io.T;  // member values of the range network
  const float* __restrict__ SP = io.S_scaled + lp.gen_base;
  const float* __restrict__ i_s = io.s;
  const float* __restrict__ i_inf = io.inf;
  const float* __restrict__ i_tinf = io.tinf;
  const float* __restrict__ i_cur = io.cur;
  const float* __restrict__ i_nxt = io.nxt;
  const float* __restrict__ i_ttn = io.ttn;
  const uint32_t* __restrict__ i_ent = w.ent1;
  const uint32_t* __restrict__ i_slot = lp.r_slot;
  const float dead = (float)(p.n_stages - 1);
  const float inv_tau = 1.0f / p.tau;
  const float beta_r = lp.n_range > 0 ? sh.beta[lp.r_net] : 0.0f;
  const bool has_gen = lp.has_generic != 0, has_range = lp.n_range > 0;

  const TileRun run = lean_tiles(w);
  int nbuild = 0;
  for (int64_t tile = run.t0; tile < run.t1;) {
    // ---- one segment = the part of the CTA's run that lies in one cell: one class table -----------------
    const int64_t tend = lp.n_cell > 0 ? lean_segment_end(lp, tile, run.t1) : run.t1;
    const uint32_t a0 = w.tile_begin[tile], a1 = w.tile_begin[tend];
    const float* __restrict__ L = sh.L[nbuild & 1];
    if (lp.n_cell > 0) {
      // rebuilt in the other buffer; one barrier per rebuild is enough: a buffer is rewritten only two rebuilds
      // later, after every warp has passed the barrier in between
      lean_class_table(sh.L[nbuild & 1], sh.prob, lp, cell_buf, tile);
      ++nbuild;
      __syncthreads();
    }
    // index words (generic entry, household slot) are fetched one batch ahead, so that the gathers they
    // address are issued together with the batch's streaming loads
    uint32_t ent_n[kLeanBatch], slot_n[kLeanBatch];
#pragma unroll
    for (int h = 0; h < kLeanBatch; ++h) {
      const uint32_t a = a0 + threadIdx.x + h * kLeanThreads;
      const uint32_t al = (a < a1) ? a : a0;
      ent_n[h] = has_gen ? i_ent[al] : kEntNone;
      slot_n[h] = has_range ? i_slot[al] : kNoSlot;
    }
    for (uint32_t base = a0 + threadIdx.x; base < a1; base += kLeanBatch * kLeanThreads) {
      float s[kLeanBatch], inf[kLeanBatch], tinf[kLeanBatch], cur[kLeanBatch], nxt[kLeanBatch], ttn[kLeanBatch];
      float rpc[kLeanBatch], gen[kLeanBatch];
      RangeLoads rl[kLeanBatch];
      uint32_t ent[kLeanBatch], slot[kLeanBatch], oid[kLeanBatch];
      int cls[kLeanBatch];
      int32_t reg[kLeanBatch];
      // ---- issue every load of the batch: gathers (addresses known from the previous iteration), streaming
      //      loads, and the next batch's index words --------------------------------------------------------
#pragma unroll
      for (int h = 0; h < kLeanBatch; ++h) {
        const uint32_t a = base + h * kLeanThreads;
        const uint32_t al = (a < a1) ? a : a0;  // dead slots re-read the segment's first agent (no branches)
        ent[h] = ent_n[h];
        slot[h] = slot_n[h];
        gen[h] = lean_generic_issue(SP, ent[h]);
        rl[h] = lean_range_issue(Tr, al, slot[h]);
        s[h] = i_s[al];
        inf[h] = i_inf[al];
        tinf[h] = i_tinf[al];
        cur[h] = i_cur[al];
        nxt[h] = i_nxt[al];
        ttn[h] = i_ttn[al];
        cls[h] = w.cls[al];
        rpc[h] = has_range ? lp.r_pc[al] : 0.0f;
        oid[h] = w.orig_id ? w.orig_id[al] : 0u;
        if (kRegion) reg[h] = io.region[al];
        const uint32_t an = a + kLeanBatch * kLeanThreads;
        const uint32_t anl = (an < a1) ? an : a0;
        ent_n[h] = has_gen ? i_ent[anl] : kEntNone;
        slot_n[h] = has_range ? i_slot[anl] : kNoSlot;
      }
      float mreg[kLeanBatch];
#pragma unroll
      for (int h = 0; h < kLeanBatch; ++h) mreg[h] = kRegion ? __ldg(io.region_factor + reg[h]) : 1.0f;
      // ---- arithmetic and stores ------------------------------------------------------------------------------
#pragma unroll
      for (int h = 0; h < kLeanBatch; ++h) {
        const uint32_t a = base + h * kLeanThreads;
        if (a >= a1) break;
        const float hs = lean_range_finish(rl[h], Tr, a, slot[h]);
        const float gv = lean_generic_finish(w, SP, ent[h], a, gen[h]);
        const float Lc = lp.n_cell > 0 ? L[cls[h]] : 0.0f;
        const uint64_t ga = w.orig_id ? (uint64_t)oid[h] : p.agent_offset + a;
        const FwdOut o = lean_forward_agent<kQuar, kDiag, kRegion>(p, lp, io, a, ga, hs, gv, Lc, beta_r, rpc[h], s[h],
                                                                   inf[h], tinf[h], cur[h], nxt[h], ttn[h], cls[h], inv_tau,
                                                                   dead, sh.hist, &sh.deaths, false, 0.0f, mreg[h]);
        if (kLabel) label_add(io.label_acc, io.label, a, (uint32_t)o.inf, o.cur == dead ? 1u : 0u);
      }
    }
    tile = tend;
  }
  if (io.red) {
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
      red_part[(int64_t)blockIdx.x * kMaxRed + threadIdx.x] = v;
    }
    finish_partials<kMaxRed>(nr, red_part, gridDim.x, ticket, io.red);
  }
}

template <bool kQuar, bool kDiag, bool kLabel>
__global__ void __launch_bounds__(kLeanThreads, GJ_LEAN_MINB_FWD) k_lean_forward(gj_world_desc w, gj_step_params p, LeanPlan lp,
                                                                  gj_fwd_io io, const float* __restrict__ cell_buf,
                                                                  double* __restrict__ red_part,
                                                                  unsigned int* __restrict__ ticket) {
  lean_forward_body<kQuar, kDiag, kLabel, false>(w, p, lp, io, cell_buf, red_part, ticket);
}

// the same with the regional transmission factor (gj_fwd_io.region)
template <bool kQuar, bool kDiag, bool kLabel>
__global__ void __launch_bounds__(kLeanThreads, GJ_LEAN_MINB_FWD) k_lean_forward_region(gj_world_desc w, gj_step_params p,
                                                                  LeanPlan lp, gj_fwd_io io,
                                                                  const float* __restrict__ cell_buf,
                                                                  double* __restrict__ red_part,
                                                                  unsigned int* __restrict__ ticket) {
  lean_forward_body<kQuar, kDiag, kLabel, true>(w, p, lp, io, cell_buf, red_part, ticket);
}

// =====================================================================================================
// seeding step in throughput mode (GJ_MODE_SEED with in-kernel noise): sample with q = 1 - fraction, infect (clamp
// variant: same values), first symptoms update, reductions — the arithmetic of lean_forward_core without networks.
// Replaces the generic k_agent_forward (IEEE libm, 1.45 ms per window at 56 M agents) for Runner.set_initial_cases.
// kSeed: seeding by label, q = 1 - seed_fraction[seed_label[a]]; the code and the region's fraction are loaded with the
// other per-agent operands of the batch, outside the draw loop.
// =====================================================================================================
template <bool kDiag, bool kLabel, bool kSeed>
__device__ __forceinline__ void lean_seed_body(const gj_world_desc& w, const gj_step_params& p, const gj_fwd_io& io,
                                               double* __restrict__ red_part, unsigned int* __restrict__ ticket) {
  __shared__ float hist[100];
  __shared__ float deaths;
  pdl_launch();
  if (threadIdx.x < 100) hist[threadIdx.x] = 0.0f;
  if (threadIdx.x == 0) deaths = 0.0f;
  pdl_wait();
  __syncthreads();
  LeanPlan lp;
  lp.r_house = 0;
  const float q_seed = 1.0f - io.seed_fraction[0] * 1.0f;
  const float dead = (float)(p.n_stages - 1);
  const float inv_tau = 1.0f / p.tau;
  const uint32_t N = (uint32_t)w.n_agents;
  const uint32_t stride = gridDim.x * kLeanThreads * kLeanBatch;
  for (uint32_t base = blockIdx.x * kLeanThreads * kLeanBatch + threadIdx.x; base < N; base += stride) {
    float s[kLeanBatch], inf[kLeanBatch], tinf[kLeanBatch], cur[kLeanBatch], nxt[kLeanBatch], ttn[kLeanBatch];
    uint32_t oid[kLeanBatch];
    int cls[kLeanBatch];
    int32_t lab[kLeanBatch];
    float qs[kLeanBatch];
#pragma unroll
    for (int h = 0; h < kLeanBatch; ++h) {
      const uint32_t a = base + h * kLeanThreads;
      const uint32_t al = a < N ? a : 0u;
      s[h] = io.s[al];
      inf[h] = io.inf[al];
      tinf[h] = io.tinf[al];
      cur[h] = io.cur[al];
      nxt[h] = io.nxt[al];
      ttn[h] = io.ttn[al];
      cls[h] = w.cls ? w.cls[al] : 0;
      oid[h] = w.orig_id ? w.orig_id[al] : 0u;
      if (kSeed) lab[h] = io.seed_label[al];
    }
    if (kSeed) {
#pragma unroll
      for (int h = 0; h < kLeanBatch; ++h) qs[h] = 1.0f - io.seed_fraction[lab[h]] * 1.0f;
    }
#pragma unroll
    for (int h = 0; h < kLeanBatch; ++h) {
      const uint32_t a = base + h * kLeanThreads;
      if (a >= N) break;
      const uint64_t ga = w.orig_id ? (uint64_t)oid[h] : p.agent_offset + a;
      uint32_t r[2];
      philox_step_pair(p.seed, p.call_index, ga, r);
      const FwdRes o = lean_forward_core<false>(p, lp, io.stage_prob, ga, lean_noise_dE(r[0], r[1]), 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, s[h],
                                                inf[h], tinf[h], cur[h], nxt[h], ttn[h], cls[h], inv_tau, dead, hist,
                                                &deaths, kSeed ? qs[h] : q_seed);
      io.tape_y0[a] = o.tape_y0;
      if (kDiag && io.n) io.n[a] = o.n;
      io.s_o[a] = o.s_o;
      io.inf_o[a] = o.inf_o;
      io.tinf_o[a] = o.tinf_o;
      io.cur_o[a] = o.cur_o;
      io.nxt_o[a] = o.nxt_o;
      io.ttn_o[a] = o.ttn_o;
      if (kLabel) label_add(io.label_acc, io.label, a, (uint32_t)o.inf_o, o.cur_o == dead ? 1u : 0u);
    }
  }
  if (io.red) {
    __syncthreads();
    const int nr = 2 + p.n_age_bins;
    if ((int)threadIdx.x < nr) {
      double v = 0.0;
      if (threadIdx.x == 0) {
        for (int c = 0; c < 100; ++c) v += (double)hist[c];
      } else if (threadIdx.x == 1) {
        v = (double)deaths;
      } else {
        const int b = threadIdx.x - 2;
        for (int c = max(p.age_bins[b] + 1, 0); c < p.age_bins[b + 1] && c < 100; ++c) v += (double)hist[c];
      }
      red_part[(int64_t)blockIdx.x * kMaxRed + threadIdx.x] = v;
    }
    finish_partials<kMaxRed>(nr, red_part, gridDim.x, ticket, io.red);
  }
}

template <bool kDiag, bool kLabel>
__global__ void __launch_bounds__(kLeanThreads, 4) k_lean_seed(gj_world_desc w, gj_step_params p, gj_fwd_io io,
                                                              double* __restrict__ red_part,
                                                              unsigned int* __restrict__ ticket) {
  lean_seed_body<kDiag, kLabel, false>(w, p, io, red_part, ticket);
}

// the same with seeding by label (gj_fwd_io.seed_label)
template <bool kDiag, bool kLabel>
__global__ void __launch_bounds__(kLeanThreads, 4) k_lean_seed_by(gj_world_desc w, gj_step_params p, gj_fwd_io io,
                                                                 double* __restrict__ red_part,
                                                                 unsigned int* __restrict__ ticket) {
  lean_seed_body<kDiag, kLabel, true>(w, p, io, red_part, ticket);
}

// per-agent arithmetic of the backward pass (shared with gj_pipe.cuh): symptoms^T, infect^T, sampler^T, clamp/exp
// chain -> cotangents of the state, w = dL/dLambda * s (and its quarantine-masked copy), cell-channel sums in acc
// kLabel: glab_i / glab_d are the cotangents of the agent's column of the label table (cases, and deaths / dead)
// kRegion: the forward multiplied the pressure by the regional factor mreg before the clamp: the clamp gates d/dlam',
// d/dlam' * lam goes to io.region_work and d/dlam' * mreg down the chain
template <bool kQuar, bool kLabel = false, bool kRegion = false>
__device__ __forceinline__ void lean_backward_agent(const gj_step_params& p, const LeanPlan& lp, const gj_bwd_io& io,
                                                    uint32_t a, float s, float tinf, float cur, float nxt, float ttn,
                                                    float ty, float v, int cls, float gs_o, float ginf_o, float gtinf_o,
                                                    float gcur_o, float gnxt_o, float gttn_o, float inv_tau, float dead,
                                                    float g_deaths, const float* __restrict__ gred_age,
                                                    const ProbRow* __restrict__ prob, float (&acc)[GJ_MAX_CHANNELS],
                                                    const uint32_t* __restrict__ orig_id, uint32_t soff = 0u,
                                                    float glab_i = 0.0f, float glab_d = 0.0f, float mreg = 1.0f) {
    // soff: batched ensemble — this sample's offset into the per-sample arrays (outputs below); the agent's id in the
    // world and in the noise stream stays `a`
    const int age = age_of(cls);
    const float n = signbit(ty) ? 1.0f : 0.0f;  // the tape's sign bit is the draw
    // symptoms^T: the draws (and the agent's id in the noise stream) are fetched only by the few agents whose
    // stage actually updates
    const uint64_t seed = p.seed;
    const uint32_t call = p.call_index;
    auto ga = [&]() { return orig_id ? (int64_t)orig_id[a] : (int64_t)p.agent_offset + a; };
    const SympOut so = symptoms_forward(p, io.stage_prob, cur, nxt, ttn, n, age,
                                        [&]() { return draw_step_uniform(seed, call, ga()); },
                                        [&](int) { return draw_step_normal(seed, call, ga()); });
    float gc = gcur_o;
    if (so.cur == dead) gc += g_deaths;
    if (kLabel && so.cur == dead) gc += glab_d;
    float gcur1 = gc, gnxt1 = gnxt_o;
    if (so.branch == 1) {
      gcur1 += (gnxt_o + gttn_o * so.dwell) / (float)so.stage;
    } else if (so.branch == 2) {
      gcur1 += (gttn_o * so.dwell - gnxt_o * so.nxt1) / (float)so.stage;
      gnxt1 = 0.0f;
    }
    const float g_cur = gcur1 * (1.0f - so.tr);
    gnxt1 += gcur1 * so.tr;
    const float g_nxt = gnxt1 * (1.0f - n);
    const float g_ttn = gttn_o * (1.0f - n);
    float gn = gnxt1 * (2.0f - nxt) + gttn_o * (p.now - ttn);
    // reductions and infect^T
    float gi = ginf_o + gred_age[age];
    if (kLabel) gi += glab_i;
    const float dd = s - n;
    const float wgt = (dd > 0.0f) ? 1.0f : ((dd == 0.0f) ? 0.5f : 0.0f);  // maximum(0, x): ties split 1/2
    float g_s = gs_o * wgt;
    gn += -(gs_o * wgt) + gi + gtinf_o * (p.now - tinf);
    const float g_tinf = gtinf_o * (1.0f - n);
    // sampler^T and the clamp / exp chain: dL/dq = gl0/q - gl1/(1-q), dL/dLambda = dL/dq * q * (-dt)
    // evaluated as (gl1 * q/(1-q) - gl0) * dt
    const float lam0 = (s == 0.0f) ? 0.0f : v;
    const float lam = kRegion ? lam0 * mreg : lam0;
    const float q = not_infected_prob(lam, p.dt);
    float y0, y1;
    decode_soft(ty, y0, y1);
    const float gret0 = -gn;
    const float dot = gret0 * y0;
    const float gl0 = ((gret0 - dot) * y0) * inv_tau, gl1 = ((0.0f - dot) * y1) * inv_tau;
    float glam = 0.0f;
    if (lam >= 1e-6f && lam <= 100.0f) glam = (gl1 * (q * rcp_fast(1.0f - q)) - gl0) * p.dt;
    const uint32_t ao = a + soff;
    if (kRegion) {
      io.region_work[ao] = glam * lam0;
      glam = glam * mreg;
    }
    const float X = (s == 0.0f) ? v : ((s == 1.0f) ? v : v * rcp_fast(s));
    g_s += glam * X;
    // outputs
    const float wv = glam * s;
    io.w[ao] = wv;
    float wqv = wv;
    if (kQuar) {
      wqv = glam * (quar_mask(p, cur) * s);
      io.wq[ao] = wqv;
    }
    if (wqv != 0.0f && lp.n_cell > 0) lean_channel_fma(acc, prob, cls, wqv, lp.n_cell);
    if (io.g_s) io.g_s[ao] = g_s;
    io.g_inf[ao] = gi;
    io.g_tinf[ao] = g_tinf;
    if (io.g_cur) io.g_cur[ao] = g_cur;
    if (io.g_nxt) io.g_nxt[ao] = g_nxt;
    if (io.g_ttn) io.g_ttn[ao] = g_ttn;
}

// =====================================================================================================
// B1  backward, per agent: symptoms^T, infect^T, sampler^T, clamp/exp chain -> cotangents of the state,
//     w = dL/dLambda * s (and its quarantine-masked copy), partial sums of the cell channels (as in K1)
// =====================================================================================================
template <bool kQuar, bool kLabel, bool kRegion>
__device__ __forceinline__ void lean_backward_body(const gj_world_desc& w, const gj_step_params& p, const LeanPlan& lp,
                                                   const gj_bwd_io& io, float* __restrict__ tile_part) {
  __shared__ ProbRow prob[200];
  __shared__ float gred_age[100];  // cotangent of is_infected from the cases / cases-by-age reductions
  lean_load_prob<true>(prob, p, lp, io.leisure_prob);
  if (threadIdx.x < 100) {
    float g = 0.0f;
    if (io.g_red) {
      g = io.g_red[0];
      const int age = threadIdx.x;
      for (int b = 0; b < p.n_age_bins; ++b)
        if (age > p.age_bins[b] && age < p.age_bins[b + 1]) g += io.g_red[2 + b];
    }
    gred_age[threadIdx.x] = g;
  }
  __syncthreads();
  const float dead = (float)(p.n_stages - 1);
  const float g_deaths = io.g_red ? io.g_red[1] / dead : 0.0f;
  const float inv_tau = 1.0f / p.tau;
  const float* __restrict__ i_s = io.s;
  const float* __restrict__ i_tinf = io.tinf;
  const float* __restrict__ i_cur = io.cur;
  const float* __restrict__ i_nxt = io.nxt;
  const float* __restrict__ i_ttn = io.ttn;
  const float* __restrict__ i_ty = io.tape_y0;
  const float* __restrict__ i_v = io.tape_v;
  const float* __restrict__ c_s = io.g_s_o;
  const float* __restrict__ c_inf = io.g_inf_o;
  const float* __restrict__ c_tinf = io.g_tinf_o;
  const float* __restrict__ c_cur = io.g_cur_o;
  const float* __restrict__ c_nxt = io.g_nxt_o;
  const float* __restrict__ c_ttn = io.g_ttn_o;

  const TileRun run = lean_tiles(w);
  float acc[GJ_MAX_CHANNELS];
#pragma unroll
  for (int j = 0; j < GJ_MAX_CHANNELS; ++j) acc[j] = 0.0f;
  uint32_t a1 = run.t0 < run.t1 ? w.tile_begin[run.t0] : 0;
  for (int64_t tile = run.t0; tile < run.t1; ++tile) {
    const uint32_t a0 = a1;
    a1 = w.tile_begin[tile + 1];
    for (uint32_t base = a0 + threadIdx.x; base < a1; base += kLeanBatch * kLeanThreads) {
      float s[kLeanBatch], tinf[kLeanBatch], cur[kLeanBatch], nxt[kLeanBatch], ttn[kLeanBatch], ty[kLeanBatch],
          v[kLeanBatch];
      float gs_o[kLeanBatch], ginf_o[kLeanBatch], gtinf_o[kLeanBatch], gcur_o[kLeanBatch], gnxt_o[kLeanBatch],
          gttn_o[kLeanBatch];
      int cls[kLeanBatch];
      int32_t reg[kLeanBatch];
#pragma unroll
      for (int h = 0; h < kLeanBatch; ++h) {
        const uint32_t a = base + h * kLeanThreads;
        const uint32_t al = (a < a1) ? a : a0;
        if (kRegion) reg[h] = io.region[al];
        s[h] = i_s[al];
        tinf[h] = i_tinf[al];
        cur[h] = i_cur[al];
        nxt[h] = i_nxt[al];
        ttn[h] = i_ttn[al];
        ty[h] = i_ty[al];
        v[h] = i_v[al];
        cls[h] = w.cls[al];
        gs_o[h] = c_s ? c_s[al] : 0.0f;
        ginf_o[h] = c_inf ? c_inf[al] : 0.0f;
        gtinf_o[h] = c_tinf ? c_tinf[al] : 0.0f;
        gcur_o[h] = c_cur ? c_cur[al] : 0.0f;
        gnxt_o[h] = c_nxt ? c_nxt[al] : 0.0f;
        gttn_o[h] = c_ttn ? c_ttn[al] : 0.0f;
      }
#pragma unroll
      for (int h = 0; h < kLeanBatch; ++h) {
        const uint32_t a = base + h * kLeanThreads;
        if (a >= a1) break;
        float glab_i = 0.0f, glab_d = 0.0f;
        if (kLabel) {
          const int64_t l = io.label[a];
          glab_i = io.g_red_label[2 * l];
          glab_d = io.g_red_label[2 * l + 1] / dead;
        }
        const float mreg = kRegion ? __ldg(io.region_factor + reg[h]) : 1.0f;
        lean_backward_agent<kQuar, kLabel, kRegion>(p, lp, io, a, s[h], tinf[h], cur[h], nxt[h], ttn[h], ty[h], v[h],
                                                    cls[h], gs_o[h], ginf_o[h], gtinf_o[h], gcur_o[h], gnxt_o[h],
                                                    gttn_o[h], inv_tau, dead, g_deaths, gred_age, prob, acc, w.orig_id,
                                                    0u, glab_i, glab_d, mreg);
      }
    }
    if (lp.n_cell > 0) {
      const bool flush = (tile + 1 == run.t1) || lean_new_cell(lp, tile, tile + 1);
      if (flush) {
        block_sums<float, GJ_MAX_CHANNELS>(acc, lp.n_cell, tile_part + tile * GJ_MAX_CHANNELS);
#pragma unroll
        for (int j = 0; j < GJ_MAX_CHANNELS; ++j) acc[j] = 0.0f;
      } else if ((int)threadIdx.x < lp.n_cell) {
        tile_part[tile * GJ_MAX_CHANNELS + threadIdx.x] = 0.0f;
      }
    }
  }
}

template <bool kQuar, bool kLabel>
__global__ void __launch_bounds__(kLeanThreads, GJ_LEAN_MINB_BWD) k_lean_backward(gj_world_desc w, gj_step_params p, LeanPlan lp,
                                                                   gj_bwd_io io, float* __restrict__ tile_part) {
  lean_backward_body<kQuar, kLabel, false>(w, p, lp, io, tile_part);
}

// the same with the regional transmission factor (gj_bwd_io.region)
template <bool kQuar, bool kLabel>
__global__ void __launch_bounds__(kLeanThreads, GJ_LEAN_MINB_BWD) k_lean_backward_region(gj_world_desc w, gj_step_params p,
                                                                   LeanPlan lp, gj_bwd_io io,
                                                                   float* __restrict__ tile_part) {
  lean_backward_body<kQuar, kLabel, true>(w, p, lp, io, tile_part);
}

// per-agent arithmetic of the backward gather (shared with gj_pipe.cuh): dL/dT from the three tiers ->
// cotangents of (is_infected, infection_time); db accumulates the range-tier network's d/dbeta terms.
// R = sum of w over the agent's range-tier group, gv = combined cR of its generic groups, Lc = class-table value
template <bool kQuar>
__device__ __forceinline__ void lean_gather_agent(const gj_step_params& p, const LeanPlan& lp, const gj_bwd_io& io,
                                                  uint32_t a, float R, float gv, float Lc, float beta_r, float rpc,
                                                  float Tm, float cur, float inf, float tinf, float4 pf, float gi,
                                                  float gt, double& db) {
    const float mq = kQuar ? quar_mask(p, cur) : 1.0f;
    const float pr = rpc * R;
    if (pr != 0.0f) db += (double)((kQuar && !lp.r_house) ? mq * Tm : Tm) * (double)pr;
    const float rv = beta_r * pr;
    const float house = lp.r_house ? rv : 0.0f;
    const float plain = (gv + Lc) + (lp.r_house ? 0.0f : rv);
    const float gT = fmaf(mq, plain, house);
    if (gT != 0.0f) {
      const TransTerms tt = lean_transmission<true>(p.now, tinf, pf);
      io.g_inf[a] = gi + gT * tt.coef;
      io.g_tinf[a] = gt + gT * (tt.dcoef * inf);
    }
}

// =====================================================================================================
// B3  backward gather: dL/dT from the three tiers -> (is_infected, infection_time); d/dbeta partial of the
//     range-tier network: sum_g pc_g S_g R_g = sum over agents of T_a * pc_g(a) * R_g(a)
// =====================================================================================================
template <bool kQuar>
__global__ void __launch_bounds__(kLeanThreads, GJ_LEAN_MINB_GATHER) k_lean_backward_gather(gj_world_desc w, gj_step_params p,
                                                                          LeanPlan lp, gj_bwd_io io,
                                                                          const float* __restrict__ cell_buf,
                                                                          double* __restrict__ dbeta_part) {
  __shared__ ProbRow prob[200];
  __shared__ float Ls[2][200];
  __shared__ float beta_s[GJ_MAX_NETS];
  lean_load_prob<false>(prob, p, lp, io.leisure_prob);
  if (threadIdx.x < p.n_nets) beta_s[threadIdx.x] = io.beta[threadIdx.x];
  __syncthreads();
  const float* __restrict__ cRP = io.cR + lp.gen_base;
  const float* __restrict__ wr = (kQuar && !lp.r_house) ? io.wq : io.w;  // member values of the range network
  const float* __restrict__ T = io.T_in;
  const float* __restrict__ i_cur = io.cur;
  const float* __restrict__ i_inf = io.inf;
  const float* __restrict__ i_tinf = io.tinf;
  const uint32_t* __restrict__ i_ent = w.ent1;
  const uint32_t* __restrict__ i_slot = lp.r_slot;
  const float4* __restrict__ prof = reinterpret_cast<const float4*>(io.prof4);
  const float beta_r = lp.n_range > 0 ? beta_s[lp.r_net] : 0.0f;
  const bool has_gen = lp.has_generic != 0, has_range = lp.n_range > 0;
  double db[1] = {0.0};

  const TileRun run = lean_tiles(w);
  int nbuild = 0;
  for (int64_t tile = run.t0; tile < run.t1;) {
    const int64_t tend = lp.n_cell > 0 ? lean_segment_end(lp, tile, run.t1) : run.t1;
    const uint32_t a0 = w.tile_begin[tile], a1 = w.tile_begin[tend];
    const float* __restrict__ L = Ls[nbuild & 1];
    if (lp.n_cell > 0) {
      lean_class_table(Ls[nbuild & 1], prob, lp, cell_buf, tile);
      ++nbuild;
      __syncthreads();
    }
    uint32_t ent_n[kLeanBatch], slot_n[kLeanBatch];
#pragma unroll
    for (int h = 0; h < kLeanBatch; ++h) {
      const uint32_t a = a0 + threadIdx.x + h * kLeanThreads;
      const uint32_t al = (a < a1) ? a : a0;
      ent_n[h] = has_gen ? i_ent[al] : kEntNone;
      slot_n[h] = has_range ? i_slot[al] : kNoSlot;
    }
    for (uint32_t base = a0 + threadIdx.x; base < a1; base += kLeanBatch * kLeanThreads) {
      float rpc[kLeanBatch], cur[kLeanBatch], inf[kLeanBatch], tinf[kLeanBatch], gen[kLeanBatch], gi[kLeanBatch],
          gt[kLeanBatch], Tm[kLeanBatch];
      RangeLoads rl[kLeanBatch];
      float4 pf[kLeanBatch];
      uint32_t ent[kLeanBatch], slot[kLeanBatch];
      int cls[kLeanBatch];
#pragma unroll
      for (int h = 0; h < kLeanBatch; ++h) {
        const uint32_t a = base + h * kLeanThreads;
        const uint32_t al = (a < a1) ? a : a0;
        ent[h] = ent_n[h];
        slot[h] = slot_n[h];
        gen[h] = lean_generic_issue(cRP, ent[h]);
        rl[h] = lean_range_issue(wr, al, slot[h]);
        cls[h] = w.cls[al];
        rpc[h] = has_range ? lp.r_pc[al] : 0.0f;
        Tm[h] = has_range ? T[al] : 0.0f;
        cur[h] = kQuar ? i_cur[al] : 0.0f;
        inf[h] = i_inf[al];
        tinf[h] = i_tinf[al];
        pf[h] = prof[al];
        gi[h] = io.g_inf[al];
        gt[h] = io.g_tinf[al];
        const uint32_t an = a + kLeanBatch * kLeanThreads;
        const uint32_t anl = (an < a1) ? an : a0;
        ent_n[h] = has_gen ? i_ent[anl] : kEntNone;
        slot_n[h] = has_range ? i_slot[anl] : kNoSlot;
      }
#pragma unroll
      for (int h = 0; h < kLeanBatch; ++h) {
        const uint32_t a = base + h * kLeanThreads;
        if (a >= a1) break;
        const float R = lean_range_finish(rl[h], wr, a, slot[h]);
        const float gv = lean_generic_finish(w, cRP, ent[h], a, gen[h]);
        lean_gather_agent<kQuar>(p, lp, io, a, R, gv, lp.n_cell > 0 ? L[cls[h]] : 0.0f, beta_r, rpc[h], Tm[h], cur[h],
                                 inf[h], tinf[h], pf[h], gi[h], gt[h], db[0]);
      }
    }
    tile = tend;
  }
  if (lp.n_range > 0) block_sums<double, 1>(db, 1, dbeta_part + (int64_t)blockIdx.x * GJ_MAX_RANGE_NETS);
}

}  // namespace gj
