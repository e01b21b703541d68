// Kernels + C ABI of the B200-native infection step (see include/gradjune_b200.h).
//
// One timestep forward = passes over HBM-resident arrays:
//   K1  transmission   agent tiles   state -> T (and quarantine-masked Tq); tile partials of CELL types
//   K2  group sums     group-major   CSR-sorted members -> per-group sums S (GENERIC types only)
//        (+ a fix-up for groups that span several chunks); k_cell_groups/k_cell_gather for CELL types
//   K3  forward        agent tiles   pressure from RANGE / CELL / GENERIC tiers -> q -> Gumbel-softmax
//                                    draw -> state + symptoms update -> reductions
// and backward mirrors it (per-agent backward, the same group/cell kernels on cotangents, backward gather,
// k_dbeta).  Two implementations of every pass: the reference-order kernels (gj_tiled.cuh: the reference's
// summation order and IEEE libm, used with injected noise) and the throughput-mode kernels (gj_lean.cuh).
// No global atomics on data: every sum has a fixed order, so results are bit-reproducible run to run.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "gj_device.cuh"
#include "gj_tiled.cuh"
#include "gj_lean.cuh"
#include "gj_pipe.cuh"

namespace gj {

static thread_local char g_err[512] = "";

static int fail(const char* what, cudaError_t e) {
  snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
  return -2;
}
static int bad(const char* what) {
  snprintf(g_err, sizeof(g_err), "invalid argument: %s", what);
  return -1;
}
#define GJ_CHECK_LAUNCH(name)                         \
  do {                                                \
    cudaError_t _e = cudaGetLastError();              \
    if (_e != cudaSuccess) return fail(name, _e);     \
  } while (0)

// ---- optional per-kernel timing with CUDA events on the launching stream (gj_profile_*) -------------
enum KernelId {
  K_TRANSMISSION = 0, K_GROUP_SMALL_F, K_GROUP_CHUNK_F, K_GROUP_FIX_F, K_AGENT_FWD,
  K_AGENT_BWD, K_GROUP_SMALL_B, K_GROUP_CHUNK_B, K_GROUP_FIX_B, K_DBETA, K_AGENT_BWD_GATHER, K_CELL, K_OTHER, K_SEED,
  K_EXCHANGE, K_SEED_GRAD, K_REGION_GRAD, K_VENUE_GRAD, K_COUNT
};
static const char* kKernelNames[K_COUNT] = {
  "transmission", "group_small<fwd>", "group_chunk<fwd>", "group_fix<fwd>", "agent_forward",
  "agent_backward", "group_small<bwd>", "group_chunk<bwd>", "group_fix<bwd>", "dbeta",
  "backward_gather", "cell_groups+gather", "other", "seeding", "boundary_exchange", "seed_label_grad",
  "region_factor_grad", "venue_factor_grad"};
constexpr int kMaxProfiled = 16384;
struct Profiler {
  bool on = false;
  int n = 0;
  int64_t launches[K_COUNT] = {0};
  cudaEvent_t ev[kMaxProfiled][2];
  int id[kMaxProfiled];
  bool created = false;
};
static Profiler g_prof;
struct ProfScope {
  int slot = -1;
  cudaStream_t st;
  ProfScope(int kid, cudaStream_t s) : st(s) {
    g_prof.launches[kid]++;
    if (g_prof.on && g_prof.n < kMaxProfiled) {
      slot = g_prof.n++;
      g_prof.id[slot] = kid;
      cudaEventRecord(g_prof.ev[slot][0], st);
    }
  }
  ~ProfScope() {
    if (slot >= 0) cudaEventRecord(g_prof.ev[slot][1], st);
  }
};

// launch with the programmatic-stream-serialization attribute (see pdl_wait / pdl_launch in gj_device.cuh): only for
// kernels that call pdl_wait() before touching anything an earlier kernel wrote.  OFF by default — measured on B200
// with the window replayed as a graph: 56 M agents 2.721 -> 2.740 ms per step, 9 M agents 0.501 -> 0.510 (the successor's
// CTAs that become resident early take issue slots and L2 from the predecessor's tail; the launch latency they save
// is already hidden inside the graph).  GJ_PDL=1 in the environment turns it on; without the attribute both device
// calls are no-ops.
static bool pdl_enabled() {
  static int on = -1;
  if (on < 0) {
    const char* e = getenv("GJ_PDL");
    on = (e && e[0] == '1') ? 1 : 0;
  }
  return on != 0;
}
template <typename... KArgs, typename... Args>
static void launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

static inline int blocks_for(int64_t n, int per_block) {
  int64_t b = (n + per_block - 1) / per_block;
  return (int)(b < 1 ? 1 : b);
}
static inline int agent_grid(int64_t n) {
  int64_t b = (n + kBlock - 1) / kBlock;
  if (b > kRedBlocks) b = kRedBlocks;
  return (int)(b < 1 ? 1 : b);
}

// scratch layout: tickets | reduction partials | d/dbeta partials | chunk partial sums (generic tier) |
//                 tile partial sums + per-cell values (cell tier) | per-tile d/dbeta partials (range tier)
struct Scratch {
  unsigned int* tickets;
  double* red_part;    // [max(n_tiles, kRedBlocks)][kMaxRed]
  double* dbeta_part;  // [GJ_MAX_NETS][kRedBlocks]
  float* part_a;       // [GJ_MAX_CHANNELS][n_parts]
  float* part_b;
  float* tile_part;    // [n_tiles][GJ_MAX_CHANNELS]
  float* cell_buf;     // [n_cells_total][GJ_MAX_CHANNELS]
  double* dbeta_tile;  // [n_tiles][GJ_MAX_RANGE_NETS]
  unsigned long long* sct_acc;  // [n_groups] fixed-point accumulators of the scatter tier (zero between steps)
  uint8_t* sct_dirty;           // [n_groups]
};
static inline int64_t align256(int64_t b) { return (b + 255) / 256 * 256; }
static inline Scratch carve(const gj_world_desc* w, void* base, int64_t* total) {
  Scratch s;
  int64_t off = 0;
  char* p = (char*)base;
  const int64_t n_tiles = w->n_tiles > 0 ? w->n_tiles : 1;
  const int64_t n_red = n_tiles > kRedBlocks ? n_tiles : kRedBlocks;
  const int64_t n_parts = w->n_parts > 0 ? w->n_parts : 1;
  const int64_t n_cells = w->n_cells_total > 0 ? w->n_cells_total : 1;
  auto take = [&](int64_t bytes) {
    char* r = p ? p + off : nullptr;
    off += align256(bytes);
    return r;
  };
  s.tickets = (unsigned int*)take(256);
  s.red_part = (double*)take((int64_t)sizeof(double) * n_red * kMaxRed);
  s.dbeta_part = (double*)take((int64_t)sizeof(double) * GJ_MAX_NETS * kRedBlocks);
  s.part_a = (float*)take((int64_t)sizeof(float) * GJ_MAX_CHANNELS * n_parts);
  s.part_b = (float*)take((int64_t)sizeof(float) * GJ_MAX_CHANNELS * n_parts);
  s.tile_part = (float*)take((int64_t)sizeof(float) * GJ_MAX_CHANNELS * n_tiles);
  s.cell_buf = (float*)take((int64_t)sizeof(float) * GJ_MAX_CHANNELS * n_cells);
  s.dbeta_tile = (double*)take((int64_t)sizeof(double) * GJ_MAX_RANGE_NETS * n_tiles);
  const int64_t n_groups = w->n_groups > 0 ? w->n_groups : 1;
  s.sct_acc = (unsigned long long*)take((int64_t)sizeof(unsigned long long) * n_groups);
  s.sct_dirty = (uint8_t*)take(n_groups);
  if (total) *total = off;
  return s;
}
static inline int64_t scratch_bytes(const gj_world_desc* w) {
  int64_t total = 0;
  carve(w, nullptr, &total);
  return total;
}

// per-type channel table derived from the net list (host, passed by value)
struct Channels {
  int nch[GJ_MAX_TYPES];
  int net[GJ_MAX_TYPES][GJ_MAX_CHANNELS];
};

// ================================================================================================
// F1  transmission
// ================================================================================================
__global__ void __launch_bounds__(kBlock) k_transmission(int64_t n, float now, const float* __restrict__ tinf,
                                                         const float* __restrict__ inf,
                                                         const float* __restrict__ maxinf,
                                                         const float* __restrict__ shape,
                                                         const float* __restrict__ rate,
                                                         const float* __restrict__ shift,
                                                         const float* __restrict__ k0, float* __restrict__ T) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; a < n; a += stride) {
    const TransTerms tt = transmission_terms<false>(now, tinf[a], maxinf[a], shape[a], rate[a], shift[a], k0[a]);
    T[a] = tt.coef * inf[a];
  }
}

__global__ void __launch_bounds__(kBlock) k_transmission_bwd(int64_t n, float now, const float* __restrict__ tinf,
                                                             const float* __restrict__ inf,
                                                             const float* __restrict__ maxinf,
                                                             const float* __restrict__ shape,
                                                             const float* __restrict__ rate,
                                                             const float* __restrict__ shift,
                                                             const float* __restrict__ k0,
                                                             const float* __restrict__ gT, float* __restrict__ g_tinf,
                                                             float* __restrict__ g_inf) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; a < n; a += stride) {
    const TransTerms tt = transmission_terms<true>(now, tinf[a], maxinf[a], shape[a], rate[a], shift[a], k0[a]);
    const float g = gT[a];
    if (g_inf) g_inf[a] = g * tt.coef;
    if (g_tinf) g_tinf[a] = g * (tt.dcoef * inf[a]);
  }
}

__global__ void __launch_bounds__(kBlock) k_profile_prepare(int64_t n, const float* __restrict__ shape,
                                                            float* __restrict__ k0) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; a < n; a += stride)
    k0[a] = expf(-lgammaf(shape[a]));
}

// ================================================================================================
// F2 / B2  group-major segmented sums
//   forward : in0 = T,  in1 = Tq -> out_a = S_scaled (sum of v*c_g), out_b = S_unscaled (sum of v)
//   backward: in0 = w,  in1 = wq -> out_a = cR (c_g * sum v),        out_b = R (sum v)
// v per member and channel (network sharing the edge type):
//   HOUSEHOLD in0 ; PLAIN in1 ; LEISURE p*in1 ; CARE_VISIT p*in1 (forward) / p*in1*(age>75) (backward)
// ================================================================================================
struct GroupAcc {
  float a[GJ_MAX_CHANNELS];
  float b[GJ_MAX_CHANNELS];
};

template <bool kBwd>
__device__ __forceinline__ void group_member(const gj_step_params& p, const Channels& ch, int type, int nch,
                                             const float* __restrict__ beta_c, float pcg, uint32_t agent,
                                             const float* __restrict__ in0, const float* __restrict__ in1,
                                             const uint8_t* __restrict__ cls, const float* __restrict__ lprob,
                                             GroupAcc& acc) {
  const float v0 = in0[agent];
  const float v1 = (in1 == in0) ? v0 : in1[agent];
  int c8 = -1;
#pragma unroll
  for (int c = 0; c < GJ_MAX_CHANNELS; ++c) {
    if (c < nch) {
      const gj_net& net = p.nets[ch.net[type][c]];
      float v;
      if (net.kind == GJ_KIND_HOUSEHOLD) {
        v = v0;
      } else if (net.kind == GJ_KIND_PLAIN) {
        v = v1;
      } else {
        if (c8 < 0) c8 = cls[agent];
        v = leisure_prob(lprob, net.prob_row, p.day_type, c8) * v1;
        if (kBwd && net.kind == GJ_KIND_CARE_VISIT) v = v * (((c8 % 100) > 75) ? 1.0f : 0.0f);
      }
      if (!kBwd) acc.a[c] += v * (beta_c[c] * pcg);  // message = T' * (beta * p_contact)   base.py:70,86-87
      acc.b[c] += v;
    }
  }
}

template <bool kBwd>
__device__ __forceinline__ void group_store(const gj_world_desc& w, const gj_step_params& p, const Channels& ch,
                                            int type, int nch, const float* __restrict__ beta_c, float pcg, uint32_t g,
                                            const GroupAcc& acc, float* __restrict__ out_a,
                                            float* __restrict__ out_b) {
  const int64_t lg = (int64_t)g - w.type_group_off[type];
#pragma unroll
  for (int c = 0; c < GJ_MAX_CHANNELS; ++c) {
    if (c < nch) {
      const int64_t o = (int64_t)p.nets[ch.net[type][c]].s_off + lg;
      out_a[o] = kBwd ? (beta_c[c] * pcg) * acc.b[c] : acc.a[c];
      out_b[o] = acc.b[c];
    }
  }
}

// per-channel beta of group g; kVenue: times the venue factor of the group's region
template <bool kVenue>
__device__ __forceinline__ void group_betas(const Channels& ch, int type, int nch, const float* __restrict__ beta,
                                            const Venue& v, uint32_t g, float (&beta_c)[GJ_MAX_CHANNELS]) {
#pragma unroll
  for (int c = 0; c < GJ_MAX_CHANNELS; ++c)
    beta_c[c] = (c < nch) ? (kVenue ? beta[ch.net[type][c]] * venue_factor(v, ch.net[type][c], g)
                                    : beta[ch.net[type][c]])
                          : 0.0f;
}

template <bool kBwd, bool kVenue>
__device__ __forceinline__ void group_small_body(const gj_world_desc& w, const gj_step_params& p, const Channels& ch,
                                                 const float* __restrict__ beta, const float* __restrict__ lprob,
                                                 const float* __restrict__ in0, const float* __restrict__ in1,
                                                 float* __restrict__ out_a, float* __restrict__ out_b, const Venue& v) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= w.n_small) return;
  const uint32_t g = w.small_groups[i];
  const int type = type_of_group(w, g);
  const int nch = ch.nch[type];
  if (nch == 0) return;
  float beta_c[GJ_MAX_CHANNELS];
  group_betas<kVenue>(ch, type, nch, beta, v, g, beta_c);
  const float pcg = w.pc[g];
  GroupAcc acc;
#pragma unroll
  for (int c = 0; c < GJ_MAX_CHANNELS; ++c) acc.a[c] = acc.b[c] = 0.0f;
  const uint32_t b = w.gm_ptr[g], e = w.gm_ptr[g + 1];
  for (uint32_t j = b; j < e; ++j)  // sequential in the reference's edge order (bit-exact small groups)
    group_member<kBwd>(p, ch, type, nch, beta_c, pcg, w.gm_agent[j], in0, in1, w.cls, lprob, acc);
  group_store<kBwd>(w, p, ch, type, nch, beta_c, pcg, g, acc, out_a, out_b);
}
template <bool kBwd>
__global__ void __launch_bounds__(kBlock) k_group_small(gj_world_desc w, gj_step_params p, Channels ch,
                                                        const float* __restrict__ beta,
                                                        const float* __restrict__ lprob,
                                                        const float* __restrict__ in0,
                                                        const float* __restrict__ in1, float* __restrict__ out_a,
                                                        float* __restrict__ out_b) {
  group_small_body<kBwd, false>(w, p, ch, beta, lprob, in0, in1, out_a, out_b, Venue{nullptr, nullptr, 0});
}
template <bool kBwd>
__global__ void __launch_bounds__(kBlock) k_group_small_venue(gj_world_desc w, gj_step_params p, Channels ch,
                                                              const float* __restrict__ beta,
                                                              const float* __restrict__ lprob,
                                                              const float* __restrict__ in0,
                                                              const float* __restrict__ in1, float* __restrict__ out_a,
                                                              float* __restrict__ out_b, Venue v) {
  group_small_body<kBwd, true>(w, p, ch, beta, lprob, in0, in1, out_a, out_b, v);
}

// one warp per chunk (<= GJ_CHUNK members): lanes stride over the member list, then a fixed shuffle tree
template <bool kBwd, bool kVenue>
__device__ __forceinline__ void group_chunk_body(const gj_world_desc& w, const gj_step_params& p, const Channels& ch,
                                                 const float* __restrict__ beta, const float* __restrict__ lprob,
                                                 const float* __restrict__ in0, const float* __restrict__ in1,
                                                 float* __restrict__ out_a, float* __restrict__ out_b,
                                                 float* __restrict__ part_a, float* __restrict__ part_b,
                                                 const Venue& v) {
  const int lane = threadIdx.x & 31;
  const int64_t ci = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (ci >= w.n_chunks) return;
  const uint32_t g = w.chunk_group[ci];
  const int type = type_of_group(w, g);
  const int nch = ch.nch[type];
  if (nch == 0) return;
  float beta_c[GJ_MAX_CHANNELS];
  group_betas<kVenue>(ch, type, nch, beta, v, g, beta_c);
  const float pcg = w.pc[g];
  GroupAcc acc;
#pragma unroll
  for (int c = 0; c < GJ_MAX_CHANNELS; ++c) acc.a[c] = acc.b[c] = 0.0f;
  const uint32_t b = w.chunk_begin[ci], e = w.chunk_end[ci];
  for (uint32_t j = b + lane; j < e; j += 32)
    group_member<kBwd>(p, ch, type, nch, beta_c, pcg, w.gm_agent[j], in0, in1, w.cls, lprob, acc);
#pragma unroll
  for (int c = 0; c < GJ_MAX_CHANNELS; ++c) {
    if (c < nch) {
      if (!kBwd) acc.a[c] = warp_sum(acc.a[c]);
      acc.b[c] = warp_sum(acc.b[c]);
    }
  }
  if (lane != 0) return;
  const int part = w.chunk_part[ci];
  if (part < 0) {
    group_store<kBwd>(w, p, ch, type, nch, beta_c, pcg, g, acc, out_a, out_b);
  } else {
#pragma unroll
    for (int c = 0; c < GJ_MAX_CHANNELS; ++c) {
      if (c < nch) {
        part_a[(int64_t)c * w.n_parts + part] = acc.a[c];
        part_b[(int64_t)c * w.n_parts + part] = acc.b[c];
      }
    }
  }
}
template <bool kBwd>
__global__ void __launch_bounds__(kBlock) k_group_chunk(gj_world_desc w, gj_step_params p, Channels ch,
                                                        const float* __restrict__ beta,
                                                        const float* __restrict__ lprob,
                                                        const float* __restrict__ in0,
                                                        const float* __restrict__ in1, float* __restrict__ out_a,
                                                        float* __restrict__ out_b, float* __restrict__ part_a,
                                                        float* __restrict__ part_b) {
  group_chunk_body<kBwd, false>(w, p, ch, beta, lprob, in0, in1, out_a, out_b, part_a, part_b,
                                Venue{nullptr, nullptr, 0});
}
template <bool kBwd>
__global__ void __launch_bounds__(kBlock) k_group_chunk_venue(gj_world_desc w, gj_step_params p, Channels ch,
                                                              const float* __restrict__ beta,
                                                              const float* __restrict__ lprob,
                                                              const float* __restrict__ in0,
                                                              const float* __restrict__ in1, float* __restrict__ out_a,
                                                              float* __restrict__ out_b, float* __restrict__ part_a,
                                                              float* __restrict__ part_b, Venue v) {
  group_chunk_body<kBwd, true>(w, p, ch, beta, lprob, in0, in1, out_a, out_b, part_a, part_b, v);
}

// groups spanning several chunks: add the chunk partials in chunk order
template <bool kBwd, bool kVenue>
__device__ __forceinline__ void group_fix_body(const gj_world_desc& w, const gj_step_params& p, const Channels& ch,
                                               const float* __restrict__ beta, const float* __restrict__ part_a,
                                               const float* __restrict__ part_b, float* __restrict__ out_a,
                                               float* __restrict__ out_b, const Venue& v) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= w.n_big) return;
  const uint32_t g = w.big_groups[i];
  const int type = type_of_group(w, g);
  const int nch = ch.nch[type];
  if (nch == 0) return;
  float beta_c[GJ_MAX_CHANNELS];
  group_betas<kVenue>(ch, type, nch, beta, v, g, beta_c);
  GroupAcc acc;
#pragma unroll
  for (int c = 0; c < GJ_MAX_CHANNELS; ++c) acc.a[c] = acc.b[c] = 0.0f;
  for (uint32_t j = w.big_part_ptr[i]; j < w.big_part_ptr[i + 1]; ++j) {
#pragma unroll
    for (int c = 0; c < GJ_MAX_CHANNELS; ++c) {
      if (c < nch) {
        acc.a[c] += part_a[(int64_t)c * w.n_parts + j];
        acc.b[c] += part_b[(int64_t)c * w.n_parts + j];
      }
    }
  }
  group_store<kBwd>(w, p, ch, type, nch, beta_c, w.pc[g], g, acc, out_a, out_b);
}
template <bool kBwd>
__global__ void __launch_bounds__(kBlock) k_group_fix(gj_world_desc w, gj_step_params p, Channels ch,
                                                      const float* __restrict__ beta,
                                                      const float* __restrict__ part_a,
                                                      const float* __restrict__ part_b, float* __restrict__ out_a,
                                                      float* __restrict__ out_b) {
  group_fix_body<kBwd, false>(w, p, ch, beta, part_a, part_b, out_a, out_b, Venue{nullptr, nullptr, 0});
}
template <bool kBwd>
__global__ void __launch_bounds__(kBlock) k_group_fix_venue(gj_world_desc w, gj_step_params p, Channels ch,
                                                            const float* __restrict__ beta,
                                                            const float* __restrict__ part_a,
                                                            const float* __restrict__ part_b, float* __restrict__ out_a,
                                                            float* __restrict__ out_b, Venue v) {
  group_fix_body<kBwd, true>(w, p, ch, beta, part_a, part_b, out_a, out_b, v);
}

// ================================================================================================
// block reduction of a few doubles + "last block finishes" (fixed summation order -> deterministic)
// ================================================================================================
template <int kR>
__device__ __forceinline__ void block_reduce_finish(double (&v)[kR], int nr, double* __restrict__ partials,
                                                    unsigned int* __restrict__ ticket, float* __restrict__ out) {
  __shared__ double sm[kBlock / 32][kR];
  __shared__ bool last;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int r = 0; r < kR; ++r)
    if (r < nr) v[r] = warp_sum(v[r]);
  if (lane == 0)
    for (int r = 0; r < nr; ++r) sm[wid][r] = v[r];
  __syncthreads();
  if (threadIdx.x < nr) {
    double s = 0.0;
    for (int k = 0; k < kBlock / 32; ++k) s += sm[k][threadIdx.x];
    partials[(int64_t)blockIdx.x * kR + threadIdx.x] = s;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int t = atomicAdd(ticket, 1u);
    last = (t == gridDim.x - 1);
  }
  __syncthreads();
  if (last) {
    __threadfence();
    if (threadIdx.x < nr) {
      double s = 0.0;
      for (unsigned int b = 0; b < gridDim.x; ++b) s += partials[(int64_t)b * kR + threadIdx.x];
      out[threadIdx.x] = (float)s;
    }
    if (threadIdx.x == 0) *ticket = 0u;  // leave the scratch zeroed for the next launch
  }
}

// ================================================================================================
// agent-major kernels for calls WITHOUT the networks phase (stand-alone sampler / infect / symptoms and the
// seeding step): persistent grid-stride loop, reductions finished by the last CTA
// ================================================================================================
// kSeed: seeding by label (gj_fwd_io.seed_label / gj_bwd_io.seed_label)
template <bool kLabel, bool kSeed>
__device__ __forceinline__ void agent_forward_body(const gj_world_desc& w, const gj_step_params& p, const gj_fwd_io& io,
                                                   double* __restrict__ red_part, unsigned int* __restrict__ ticket) {
  const int64_t N = w.n_agents;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  float redf[kMaxRed];   // per-thread sums of small integers (<= 2 per agent, < 2^24 agents per thread): exact in fp32
#pragma unroll
  for (int r = 0; r < kMaxRed; ++r) redf[r] = 0.0f;
  for (int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; a < N; a += stride) {
    const int cls = w.cls ? w.cls[a] : 0;
    AgentState st;
    st.s = io.s ? io.s[a] : 0.0f;
    st.inf = io.inf ? io.inf[a] : 0.0f;
    st.tinf = io.tinf ? io.tinf[a] : 0.0f;
    st.cur = io.cur ? io.cur[a] : 1.0f;
    st.nxt = io.nxt ? io.nxt[a] : 1.0f;
    st.ttn = io.ttn ? io.ttn[a] : 0.0f;
    const float q = io.q_in ? io.q_in[a] : 1.0f;
    forward_tail<kLabel, kSeed>(p, io, N, a, noise_agent(w, p, a), cls % 100, q, st, redf, io.label_acc);
  }
  if (io.red) {
    double red[kMaxRed];
#pragma unroll
    for (int r = 0; r < kMaxRed; ++r) red[r] = (double)redf[r];
    block_reduce_finish<kMaxRed>(red, 2 + p.n_age_bins, red_part, ticket, io.red);
  }
}

template <bool kLabel>
__global__ void __launch_bounds__(kBlock) k_agent_forward(gj_world_desc w, gj_step_params p, gj_fwd_io io,
                                                          double* __restrict__ red_part,
                                                          unsigned int* __restrict__ ticket) {
  agent_forward_body<kLabel, false>(w, p, io, red_part, ticket);
}

template <bool kLabel>
__global__ void __launch_bounds__(kBlock) k_agent_seed_forward(gj_world_desc w, gj_step_params p, gj_fwd_io io,
                                                               double* __restrict__ red_part,
                                                               unsigned int* __restrict__ ticket) {
  agent_forward_body<kLabel, true>(w, p, io, red_part, ticket);
}

// kSeed: each agent's d/dseed_fraction goes to the scratch row io.seed_work (reduced per label by k_seed_label_grad)
// instead of the single fp64 sum
template <bool kLabel, bool kSeed>
__device__ __forceinline__ void agent_backward_body(const gj_world_desc& w, const gj_step_params& p, const gj_bwd_io& io,
                                                    double* __restrict__ red_part, unsigned int* __restrict__ ticket) {
  const int64_t N = w.n_agents;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  double gfrac[1] = {0.0};
  const bool seed_mode = p.mode == GJ_MODE_SEED;
  for (int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; a < N; a += stride) {
    const int cls = w.cls ? w.cls[a] : 0;
    AgentState st;
    st.s = io.s ? io.s[a] : 0.0f;
    st.inf = io.inf ? io.inf[a] : 0.0f;
    st.tinf = io.tinf ? io.tinf[a] : 0.0f;
    st.cur = io.cur ? io.cur[a] : 1.0f;
    st.nxt = io.nxt ? io.nxt[a] : 1.0f;
    st.ttn = io.ttn ? io.ttn[a] : 0.0f;
    const BackAgent r = backward_agent<kLabel, kSeed>(p, io, N, a, noise_agent(w, p, a), cls % 100, st, false);
    if (io.g_q_out) io.g_q_out[a] = r.gq;
    if (io.g_n_out) io.g_n_out[a] = r.gn;
    if (kSeed) io.seed_work[a] = -r.gq;
    else if (seed_mode) gfrac[0] += (double)(-r.gq);  // q = 1 - fraction
    if (io.g_s) io.g_s[a] = r.gs;
    if (io.g_inf) io.g_inf[a] = r.ginf;
    if (io.g_tinf) io.g_tinf[a] = r.gtinf;
    if (io.g_cur) io.g_cur[a] = r.gcur;
    if (io.g_nxt) io.g_nxt[a] = r.gnxt;
    if (io.g_ttn) io.g_ttn[a] = r.gttn;
  }
  if (!kSeed && seed_mode && io.g_seed_fraction) block_reduce_finish<1>(gfrac, 1, red_part, ticket, io.g_seed_fraction);
}

template <bool kLabel>
__global__ void __launch_bounds__(kBlock) k_agent_backward(gj_world_desc w, gj_step_params p, gj_bwd_io io,
                                                           double* __restrict__ red_part,
                                                           unsigned int* __restrict__ ticket) {
  agent_backward_body<kLabel, false>(w, p, io, red_part, ticket);
}

template <bool kLabel>
__global__ void __launch_bounds__(kBlock) k_agent_seed_backward(gj_world_desc w, gj_step_params p, gj_bwd_io io,
                                                                double* __restrict__ red_part,
                                                                unsigned int* __restrict__ ticket) {
  agent_backward_body<kLabel, true>(w, p, io, red_part, ticket);
}

// ================================================================================================
// seeding by label: g_seed_fraction[l] = sum of seed_work over the agents of label l, deterministically.
// seed_order lists the agents stably sorted by label; label l owns positions [offsets[l], offsets[l+1]).  The positions
// are cut into fixed chunks of `chunk` (a power of two that depends on the world only).  One warp per chunk sums, in
// fp64 with a fixed lane order and shuffle tree, each label's piece of the chunk: a label that lies inside the chunk is
// finished there; a label that crosses a chunk boundary leaves its piece in one of the chunk's two partial slots —
// slot 0 for the label that holds the chunk's first position, slot 1 for a label that starts inside the chunk and
// runs past its end.  k_seed_label_fix then adds a crossing label's pieces in chunk order.  Nothing depends on the
// launch grid, and there are no floating-point atomics.
// ================================================================================================
__global__ void __launch_bounds__(kBlock) k_seed_label_grad(int64_t N, int64_t chunk, const int32_t* __restrict__ order,
                                                            const int32_t* __restrict__ offsets, int n_labels,
                                                            const float* __restrict__ work, double* __restrict__ part,
                                                            float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t n_chunks = (N + chunk - 1) / chunk;
  const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t c = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; c < n_chunks; c += warps) {
    const int64_t lo = c * chunk, hi = lo + chunk < N ? lo + chunk : N;
    int l0 = 0, l1 = n_labels;   // the label holding position lo: the last l with offsets[l] <= lo
    while (l1 - l0 > 1) {
      const int m = (l0 + l1) >> 1;
      if ((int64_t)offsets[m] <= lo) l0 = m;
      else l1 = m;
    }
    int l = l0;
    int64_t pos = lo;
    while (pos < hi) {
      while ((int64_t)offsets[l + 1] <= pos) ++l;   // skip empty labels
      const int64_t b = offsets[l], e = offsets[l + 1];
      const int64_t end = e < hi ? e : hi;
      double v = 0.0;
      for (int64_t j = pos + lane; j < end; j += 32) v += (double)work[order[j]];
      v = warp_sum(v);
      if (lane == 0) {
        if (b >= lo && e <= hi) out[l] = (float)v;
        else part[2 * c + (b <= lo ? 0 : 1)] = v;
      }
      pos = end;
    }
  }
}

// one warp per label that crosses a chunk boundary: its pieces in chunk order; empty labels get 0
__global__ void __launch_bounds__(kBlock) k_seed_label_fix(int64_t chunk, const int32_t* __restrict__ offsets,
                                                           int n_labels, const double* __restrict__ part,
                                                           float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t l = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; l < n_labels; l += warps) {
    const int64_t b = offsets[l], e = offsets[l + 1];
    if (b == e) {
      if (lane == 0) out[l] = 0.0f;
      continue;
    }
    const int64_t c0 = b / chunk, c1 = (e - 1) / chunk;
    if (c0 == c1) continue;   // finished by k_seed_label_grad
    double v = 0.0;
    for (int64_t c = c0 + lane; c <= c1; c += 32) v += part[2 * c + ((c == c0 && b != c0 * chunk) ? 1 : 0)];
    v = warp_sum(v);
    if (lane == 0) out[l] = (float)v;
  }
}

// results by label: the step's integer accumulator -> fp32 table, and back to zero for the next step (sample blockIdx.z)
__global__ void __launch_bounds__(kBlock) k_label_finish(int64_t n, uint32_t* __restrict__ acc, float* __restrict__ out,
                                                         int64_t stride) {
  pdl_launch();
  pdl_wait();
  acc += (int64_t)blockIdx.z * stride;
  out += (int64_t)blockIdx.z * stride;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    out[i] = (float)acc[i];
    acc[i] = 0u;
  }
}

// dL/dbeta_k = sum_g pc_g * S~_g * R_g   (fixed-order two-level sum in fp64)
struct DbetaPlan {
  int64_t soff[GJ_MAX_NETS];  // where network k's plain group sums / R live inside S_unscaled / R
  int64_t n_range_parts;      // partials written by the backward gather (tiles, or CTAs of the persistent grid)
};

// kVenue: dL/dbeta_k = sum_g ((own * pc_g) * f) * S~_g * R_g, and (work != NULL) the per-group terms of
// dL/df = beta_k * own * pc_g * S~_g * R_g go to work, laid out like S_un / R
template <bool kVenue>
__device__ __forceinline__ void dbeta_body(const gj_world_desc& w, const gj_step_params& p, const Plan& pl,
                                           const DbetaPlan& dp, const float* __restrict__ S_un,
                                           const float* __restrict__ R, const double* __restrict__ dbeta_tile,
                                           double* __restrict__ partials, unsigned int* __restrict__ tickets,
                                           float* __restrict__ g_beta, const Batch& bt, const float* __restrict__ beta,
                                           Venue v, float* __restrict__ work) {
  pdl_launch();
  pdl_wait();
  if (bt.nb > 1) {   // batched ensemble: sample blockIdx.z
    const int s = blockIdx.z;
    S_un += (int64_t)s * bt.sG;
    R += (int64_t)s * bt.sG;
    dbeta_tile = scr_shift(dbeta_tile, bt, s);
    partials = scr_shift(partials, bt, s);
    tickets = scr_shift(tickets, bt, s);
    g_beta += (int64_t)s * bt.sBeta;
    if (kVenue) {
      beta += (int64_t)s * bt.sBeta;
      v.factor += (int64_t)s * bt.sVen;
      if (work) work += (int64_t)s * bt.sG;
    }
  }
  const int k = blockIdx.y;
  const gj_net net = p.nets[k];
  double acc[1] = {0.0};
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  if (w.type_tier[net.type] == GJ_TIER_RANGE) {  // partials written by the backward gather
    const int i = pl.net_t1[k];
    for (int64_t tl = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; tl < dp.n_range_parts; tl += stride)
      acc[0] += dbeta_tile[tl * GJ_MAX_RANGE_NETS + i];
  } else {
    const int64_t g0 = w.type_group_off[net.type];
    const int64_t G = w.type_group_off[net.type + 1] - g0;
    const int64_t so = dp.soff[k];
    const float bk = kVenue ? beta[k] : 0.0f;
    // network k's own work row (nets[k].s_off): generic networks sharing an edge type share `so` on the throughput
    // path, but each has its own beta_k and its own row of d/df
    const int64_t wo = net.s_off;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < G; i += stride) {
      const float own = w.dbeta_w ? w.dbeta_w[g0 + i] : 1.0f;  // partitioned worlds: every group counted by one rank
      if (kVenue) {
        const float opc = own * w.pc[g0 + i];
        const float Sg = S_un[so + i], Rg = R[so + i];
        acc[0] += (double)((opc * venue_factor(v, k, (uint32_t)(g0 + i))) * Sg) * (double)Rg;
        if (work) work[wo + i] = (float)((double)((bk * opc) * Sg) * (double)Rg);
      } else {
        acc[0] += (double)((own * w.pc[g0 + i]) * S_un[so + i]) * (double)R[so + i];
      }
    }
  }
  block_reduce_finish<1>(acc, 1, partials + (int64_t)k * kRedBlocks, tickets + 1 + k, g_beta + k);
}
__global__ void __launch_bounds__(kBlock) k_dbeta(gj_world_desc w, gj_step_params p, Plan pl, DbetaPlan dp,
                                                  const float* __restrict__ S_un, const float* __restrict__ R,
                                                  const double* __restrict__ dbeta_tile, double* __restrict__ partials,
                                                  unsigned int* __restrict__ tickets, float* __restrict__ g_beta,
                                                  Batch bt) {
  dbeta_body<false>(w, p, pl, dp, S_un, R, dbeta_tile, partials, tickets, g_beta, bt, nullptr,
                    Venue{nullptr, nullptr, 0}, nullptr);
}
__global__ void __launch_bounds__(kBlock) k_dbeta_venue(gj_world_desc w, gj_step_params p, Plan pl, DbetaPlan dp,
                                                        const float* __restrict__ S_un, const float* __restrict__ R,
                                                        const double* __restrict__ dbeta_tile,
                                                        double* __restrict__ partials,
                                                        unsigned int* __restrict__ tickets, float* __restrict__ g_beta,
                                                        Batch bt, const float* __restrict__ beta, Venue v,
                                                        float* __restrict__ work) {
  dbeta_body<true>(w, p, pl, dp, S_un, R, dbeta_tile, partials, tickets, g_beta, bt, beta, v, work);
}

__global__ void k_philox_fill(uint64_t seed, uint32_t call, int64_t first, int64_t n, float* __restrict__ E,
                              float* __restrict__ u, float* __restrict__ z) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; a < n; a += stride) {
    const StepNoise nz = draw_step_noise(seed, call, first + a);
    if (E) {
      E[a] = nz.E0;
      E[n + a] = nz.E1;
    }
    if (u) u[a] = nz.u;
    if (z) z[a] = draw_step_normal(seed, call, first + a);
  }
}

// ================================================================================================
// host side
// ================================================================================================
static int build_channels(const gj_world_desc* w, const gj_step_params* p, Channels* ch, Plan* pl) {
  memset(ch, 0, sizeof(*ch));
  memset(pl, 0, sizeof(*pl));
  if (p->n_nets < 0 || p->n_nets > GJ_MAX_NETS) return bad("n_nets");
  for (int k = 0; k < p->n_nets; ++k) {
    const int t = p->nets[k].type;
    if (t < 0 || t >= w->n_types) return bad("net.type");
    pl->net_t1[k] = pl->net_t2[k] = pl->net_lei[k] = -1;
    const int kind = p->nets[k].kind;
    if (kind == GJ_KIND_LEISURE || kind == GJ_KIND_CARE_VISIT) {
      if (pl->n_lei >= GJ_MAX_CHANNELS) return bad("too many networks with attendance tables");
      if (p->nets[k].prob_row < 0) return bad("leisure network without a table row");
      pl->net_lei[k] = pl->n_lei;
      pl->lei_net[pl->n_lei++] = k;
    }
    const int tier = w->type_tier[t];
    pl->tier[k] = tier;
    pl->slot[k] = w->range_slot[t];
    pl->rpc[k] = w->range_pc[t];
    if (tier == GJ_TIER_RANGE) {
      if (!w->range_slot[t] || !w->range_pc[t]) return bad("range-tier type without slot arrays");
      if (pl->n_t1 >= GJ_MAX_RANGE_NETS) return bad("too many networks on range-tier edge types");
      pl->net_t1[k] = pl->n_t1;
      pl->t1_net[pl->n_t1++] = k;
    } else if (tier == GJ_TIER_CELL) {
      if (pl->n_t2 >= GJ_MAX_CHANNELS) return bad("too many networks on cell-tier edge types");
      pl->net_t2[k] = pl->n_t2;
      pl->t2_net[pl->n_t2++] = k;
    } else {
      if (ch->nch[t] >= GJ_MAX_CHANNELS) return bad("too many networks share one edge type");
      ch->net[t][ch->nch[t]++] = k;
      pl->n_generic++;
    }
  }
  return 0;
}

static const Batch kNoBatch = {1, 0u, 0, 0, 0, 0, nullptr, 0, 0, 0};
static const Venue kNoVenue = {nullptr, nullptr, 0};
// grid of a persistent kernel in a batched launch: the resident wave is split between the samples (block = run * nb +
// sample), at least one CTA and at most one per tile for each
static inline int batch_grid(const gj_world_desc* w, int64_t resident, const Batch& bt) {
  int64_t per = resident / bt.nb;
  if (per < 1) per = 1;
  if (per > w->n_tiles) per = w->n_tiles;
  return (int)(per * bt.nb);
}

// persistent grids of the throughput-mode kernels.  Occupancy, the SM count and the opt-in to large dynamic
// shared memory are properties of (kernel, device): the caches are per device (a process may drive several GPUs,
// `system.device: cuda:1` — ADVICE r1), indexed by the CURRENT device, which the caller has made the one that owns
// the stream and the pointers (grad_june.ops wraps every call in torch.cuda.device).
constexpr int kMaxDevices = 32;
struct OccCache {
  int v[kMaxDevices];
};
static int current_device() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) dev = 0;
  return dev;
}
static int sm_count() {
  static int n[kMaxDevices] = {0};
  const int dev = current_device();
  if (n[dev] == 0) {
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    n[dev] = sms;
  }
  return n[dev];
}
// one resident wave: SMs x (CTAs of this kernel that fit on an SM), at most one CTA per tile
template <typename K>
static int lean_grid(const gj_world_desc* w, K kernel, OccCache* cache, const Batch& bt = kNoBatch) {
  int& c = cache->v[current_device()];
  if (c == 0) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kLeanThreads, 0) != cudaSuccess || per_sm < 1)
      per_sm = 1;
    c = per_sm;
  }
  const int64_t g = (int64_t)sm_count() * c;
  if (bt.nb > 1) return batch_grid(w, g, bt);
  return (int)(w->n_tiles < g ? w->n_tiles : g);
}

// bulk-copy pipelined kernels (gj_pipe.cuh): on unless GJ_PIPE=0; they need 16-byte aligned per-agent arrays
static int g_pipe_on = -1;   // bit 0: pipelined agent kernels, bit 1: look-ahead transmission pass,
                             // bit 2: the UNCOMPACTED transmission pass (k_lean_transmission instead of _c)
static int pipe_flags() {
  if (g_pipe_on < 0) {
    const char* e = getenv("GJ_PIPE");
    g_pipe_on = (e && e[0] >= '0' && e[0] <= '7') ? (e[0] - '0') : 1;   // look-ahead off: measured neutral
    const char* c = getenv("GJ_K1C");
    if (c && c[0] == '0') g_pipe_on |= 4;
  }
  return g_pipe_on;
}
static bool pipe_enabled() { return (pipe_flags() & 1) != 0; }
static bool lookahead_enabled() { return (pipe_flags() & 3) == 3; }
static bool aligned16(const void* p) { return (((uintptr_t)p) & 15u) == 0; }
static bool pipe_aligned_fwd(const gj_world_desc* w, const LeanPlan& lp, const gj_fwd_io* io) {
  return aligned16(io->s) && aligned16(io->inf) && aligned16(io->tinf) && aligned16(io->cur) && aligned16(io->nxt) &&
         aligned16(io->ttn) && aligned16(io->T) && aligned16(io->Tq) && aligned16(w->ent1) && aligned16(w->cls) &&
         aligned16(w->orig_id) &&
         aligned16(lp.r_slot) && aligned16(lp.r_pc) && aligned16(io->region);
}
static bool pipe_aligned_bwd(const gj_world_desc* w, const LeanPlan& lp, const gj_bwd_io* io) {
  const void* ptrs[] = {io->s, io->inf, io->tinf, io->cur, io->nxt, io->ttn, io->tape_y0, io->tape_v, io->g_s_o,
                        io->g_inf_o, io->g_tinf_o, io->g_cur_o, io->g_nxt_o, io->g_ttn_o, io->prof4, io->g_inf,
                        io->g_tinf, io->T_in, io->w, io->wq, w->ent1, w->cls, lp.r_slot, lp.r_pc, io->region};
  for (const void* q : ptrs)
    if (!aligned16(q)) return false;   // NULL counts as aligned
  return true;
}
// one resident wave of a kernel with dynamic shared memory
template <typename K>
static int pipe_grid(const gj_world_desc* w, K kernel, int threads, size_t smem, OccCache* cache,
                     const Batch& bt = kNoBatch) {
  int& c = cache->v[current_device()];
  if (c == 0) {
    int per_sm = 0;
    cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem) != cudaSuccess || per_sm < 1)
      per_sm = 1;
    c = per_sm;
  }
  const int64_t g = (int64_t)sm_count() * c;
  if (bt.nb > 1) return batch_grid(w, g, bt);
  return (int)(w->n_tiles < g ? w->n_tiles : g);
}

static int check_world(const gj_world_desc* w) {
  if (!w) return bad("world is NULL");
  if (w->n_agents < 0 || w->n_types < 0 || w->n_types > GJ_MAX_TYPES) return bad("world sizes");
  if (w->n_edges >= ((int64_t)1 << 32) || w->n_agents >= ((int64_t)1 << 32)) return bad("world too large for 32-bit CSR");
  for (int t = 0; t < w->n_types; ++t)
    if (w->type_group_off[t + 1] - w->type_group_off[t] >= ((int64_t)1 << 28)) return bad("too many groups in one type");
  return 0;
}

template <bool kBwd>
static int launch_group_pass(const gj_world_desc* w, const gj_step_params* p, const Channels& ch, const float* beta,
                             const float* lprob, const float* in0, const float* in1, float* out_a, float* out_b,
                             const Scratch& sc, cudaStream_t st, const Venue& v = kNoVenue) {
  const bool venue = v.region != nullptr;
  if (w->n_small > 0) {
    ProfScope ps(kBwd ? K_GROUP_SMALL_B : K_GROUP_SMALL_F, st);
    if (venue)
      k_group_small_venue<kBwd><<<blocks_for(w->n_small, kBlock), kBlock, 0, st>>>(*w, *p, ch, beta, lprob, in0, in1,
                                                                                 out_a, out_b, v);
    else
      k_group_small<kBwd><<<blocks_for(w->n_small, kBlock), kBlock, 0, st>>>(*w, *p, ch, beta, lprob, in0, in1, out_a,
                                                                           out_b);
    GJ_CHECK_LAUNCH("k_group_small");
  }
  if (w->n_chunks > 0) {
    ProfScope ps(kBwd ? K_GROUP_CHUNK_B : K_GROUP_CHUNK_F, st);
    if (venue)
      k_group_chunk_venue<kBwd><<<blocks_for(w->n_chunks * 32, kBlock), kBlock, 0, st>>>(
          *w, *p, ch, beta, lprob, in0, in1, out_a, out_b, sc.part_a, sc.part_b, v);
    else
      k_group_chunk<kBwd><<<blocks_for(w->n_chunks * 32, kBlock), kBlock, 0, st>>>(*w, *p, ch, beta, lprob, in0, in1,
                                                                                out_a, out_b, sc.part_a, sc.part_b);
    GJ_CHECK_LAUNCH("k_group_chunk");
  }
  if (w->n_big > 0) {
    ProfScope ps(kBwd ? K_GROUP_FIX_B : K_GROUP_FIX_F, st);
    if (venue)
      k_group_fix_venue<kBwd><<<blocks_for(w->n_big, kBlock), kBlock, 0, st>>>(*w, *p, ch, beta, sc.part_a, sc.part_b,
                                                                             out_a, out_b, v);
    else
      k_group_fix<kBwd><<<blocks_for(w->n_big, kBlock), kBlock, 0, st>>>(*w, *p, ch, beta, sc.part_a, sc.part_b, out_a,
                                                                       out_b);
    GJ_CHECK_LAUNCH("k_group_fix");
  }
  return 0;
}

// cell tier, part 1: tile partials -> per-group sums (plain + beta*pc-scaled)
static int launch_cell_groups(const gj_world_desc* w, const gj_step_params* p, const Plan& pl, const float* beta,
                              float* out_scaled, float* out_plain, const Scratch& sc, cudaStream_t st,
                              const Batch& bt = kNoBatch, const Venue& v = kNoVenue) {
  if (pl.n_t2 == 0) return 0;
  int64_t maxG = 1;
  for (int j = 0; j < pl.n_t2; ++j) {
    const int t = p->nets[pl.t2_net[j]].type;
    const int64_t G = w->type_group_off[t + 1] - w->type_group_off[t];
    if (G > maxG) maxG = G;
  }
  ProfScope ps(K_CELL, st);
  if (v.region)
    launch_pdl(k_cell_groups_venue, dim3(blocks_for(maxG, kBlock), pl.n_t2, bt.nb), dim3(kBlock), 0, st, *w, *p, pl,
               beta, (const float*)sc.tile_part, out_scaled, out_plain, bt, v);
  else
    launch_pdl(k_cell_groups, dim3(blocks_for(maxG, kBlock), pl.n_t2, bt.nb), dim3(kBlock), 0, st, *w, *p, pl, beta,
               (const float*)sc.tile_part, out_scaled, out_plain, bt);
  GJ_CHECK_LAUNCH("k_cell_groups");
  return 0;
}

// cell tier, part 2: per-cell sum of the scaled group sums (after the sums of straddling groups were exchanged)
static int launch_cell_gather(const gj_world_desc* w, const gj_step_params* p, const Plan& pl, const float* in_scaled,
                              const Scratch& sc, cudaStream_t st, const Batch& bt = kNoBatch) {
  if (pl.n_t2 == 0) return 0;
  int64_t maxC = 1;
  for (int j = 0; j < pl.n_t2; ++j) {
    const int t = p->nets[pl.t2_net[j]].type;
    if (w->n_cells[t] > maxC) maxC = w->n_cells[t];
  }
  ProfScope ps(K_CELL, st);
  launch_pdl(k_cell_gather, dim3(blocks_for(maxC, kBlock), pl.n_t2, bt.nb), dim3(kBlock), 0, st, *w, *p, pl, in_scaled,
             sc.cell_buf, bt);
  GJ_CHECK_LAUNCH("k_cell_gather");
  return 0;
}

// ---- throughput mode (gj_lean.cuh) ---------------------------------------------------------------------------
// A step runs on the throughput-mode kernels when it is the whole fused step with in-kernel Philox noise and every
// network is of the kind its layout tier handles in closed form; forward and backward take the same decision
// from (world, params, prof4), so the group-sum buffers they exchange have the same layout.
static bool lean_plan(const gj_world_desc* w, const gj_step_params* p, const Plan& pl, LeanPlan* lp) {
  memset(lp, 0, sizeof(*lp));
  if (p->mode != GJ_MODE_STEP || p->phases != GJ_PHASE_ALL || p->exact_order) return false;
  if (p->n_nets <= 0 || pl.n_t1 > 1) return false;
  if (pl.n_generic > 0 && !w->ent1) return false;
  int64_t total = 0;
  for (int k = 0; k < p->n_nets; ++k) {
    const int kind = p->nets[k].kind, t = p->nets[k].type;
    total += w->type_group_off[t + 1] - w->type_group_off[t];
    if (pl.tier[k] == GJ_TIER_RANGE) {
      if (kind != GJ_KIND_HOUSEHOLD && kind != GJ_KIND_PLAIN) return false;
      lp->n_range = 1;
      lp->r_slot = w->range_slot[t];
      lp->r_pc = w->range_pc[t];
      lp->r_pc_lut = w->range_pc_from_size[t] != 0;
      lp->r_net = k;
      lp->r_house = kind == GJ_KIND_HOUSEHOLD;
    } else if (pl.tier[k] == GJ_TIER_CELL) {
      if (kind != GJ_KIND_LEISURE && kind != GJ_KIND_CARE_VISIT) return false;
      const int j = pl.net_t2[k];
      lp->c_row[j] = p->nets[k].prob_row;
      lp->c_care[j] = kind == GJ_KIND_CARE_VISIT;
      lp->c_cell_off[j] = w->cell_off[t];
      lp->c_tile_cell[j] = w->tile_cell[t];
      bool seen = false;
      for (int i = 0; i < lp->n_tc; ++i) seen = seen || lp->tc[i] == w->tile_cell[t];
      if (!seen) {
        lp->ctp[lp->n_tc] = w->cell_tile_ptr[t];
        lp->tc[lp->n_tc++] = w->tile_cell[t];
      }
    } else if (kind == GJ_KIND_HOUSEHOLD) {
      // generic-tier household (giant or non-contiguous groups, e.g. the two-group world of utils.py:97-133): its
      // members are summed unmasked, which is the PLAIN sum exactly when no quarantine mask is active
      if (p->n_quar > 0) return false;
    } else if (kind != GJ_KIND_PLAIN) {
      return false;
    }
  }
  lp->n_cell = pl.n_t2;
  lp->has_generic = pl.n_generic > 0;
  lp->gen_base = total;
  return true;
}

// forward: the scatter tier was accumulated by the transmission pass; giant groups are summed group-major (the first
// n_giant_chunks chunks / n_giant_big multi-chunk groups of the lists), then the accumulators become fp32 sums
static int launch_lean_group_pass(const gj_world_desc* w, const gj_step_params* p, const Plan& pl, const float* beta,
                                  const float* in, float* out_scaled, float* out_plain, const Scratch& sc, bool bwd,
                                  cudaStream_t st, const Batch& bt, const Venue& v);
static int launch_lean_forward_sums(const gj_world_desc* w, const gj_step_params* p, const Plan& pl, const float* beta,
                                    const float* in, float* out_scaled, float* out_plain, const Scratch& sc,
                                    cudaStream_t st, const Batch& bt, const Venue& v) {
  if (w->n_giant_chunks > 0) {
    gj_world_desc wg = *w;
    wg.n_small = 0;
    wg.n_chunks = w->n_giant_chunks;
    wg.n_big = w->n_giant_big;
    if (int e = launch_lean_group_pass(&wg, p, pl, beta, in, out_scaled, out_plain, sc, false, st, bt, v)) return e;
  }
  {
    ProfScope ps(K_GROUP_SMALL_F, st);
    Scatter sct{sc.sct_acc, sc.sct_dirty};
    GenericRanges gr;
    memset(&gr, 0, sizeof(gr));
    for (int t = 0; t < w->n_types; ++t)
      if (w->type_tier[t] == GJ_TIER_GENERIC && w->type_group_off[t + 1] > w->type_group_off[t]) {
        gr.first[gr.n] = w->type_group_off[t];
        gr.start[gr.n + 1] = gr.start[gr.n] + (w->type_group_off[t + 1] - w->type_group_off[t]);
        ++gr.n;
      }
    if (gr.n == 0) return 0;
    if (v.region)
      launch_pdl(k_lean_scatter_finalize_venue, dim3(blocks_for(gr.start[gr.n], kBlock) * bt.nb), dim3(kBlock), 0, st,
                 *w, *p, pl, gr, beta, in, sct, out_scaled, out_plain, bt, v);
    else
      launch_pdl(k_lean_scatter_finalize, dim3(blocks_for(gr.start[gr.n], kBlock) * bt.nb), dim3(kBlock), 0, st, *w, *p,
                 pl, gr, beta, in, sct, out_scaled, out_plain, bt);
    GJ_CHECK_LAUNCH("k_lean_scatter_finalize");
  }
  return 0;
}

static int launch_lean_group_pass(const gj_world_desc* w, const gj_step_params* p, const Plan& pl, const float* beta,
                                  const float* in, float* out_scaled, float* out_plain, const Scratch& sc, bool bwd,
                                  cudaStream_t st, const Batch& bt, const Venue& v) {
  if (w->n_small > 0 || w->n_chunks > 0) {
    ProfScope ps(bwd ? K_GROUP_CHUNK_B : K_GROUP_CHUNK_F, st);
    const int chunk_blocks = w->n_chunks > 0 ? blocks_for(w->n_chunks * 32, kBlock) : 0;
    const int small_blocks = w->n_small > 0 ? blocks_for(w->n_small, kBlock) : 0;
    if (v.region)
      launch_pdl(k_lean_group_sums_venue, dim3((chunk_blocks + small_blocks) * bt.nb), dim3(kBlock), 0, st, *w, *p, pl,
                 beta, in, out_scaled, out_plain, sc.part_a, chunk_blocks, bt, v);
    else
      launch_pdl(k_lean_group_sums, dim3((chunk_blocks + small_blocks) * bt.nb), dim3(kBlock), 0, st, *w, *p, pl, beta,
                 in, out_scaled, out_plain, sc.part_a, chunk_blocks, bt);
    GJ_CHECK_LAUNCH("k_lean_group_sums");
  }
  if (w->n_big > 0) {
    ProfScope ps(bwd ? K_GROUP_FIX_B : K_GROUP_FIX_F, st);
    if (v.region)
      launch_pdl(k_lean_group_fix_venue, dim3(blocks_for(w->n_big * 32, kBlock) * bt.nb), dim3(kBlock), 0, st, *w, *p,
                 pl, beta, (const float*)sc.part_a, out_scaled, out_plain, bt, v);
    else
      launch_pdl(k_lean_group_fix, dim3(blocks_for(w->n_big * 32, kBlock) * bt.nb), dim3(kBlock), 0, st, *w, *p, pl,
                 beta, (const float*)sc.part_a, out_scaled, out_plain, bt);
    GJ_CHECK_LAUNCH("k_lean_group_fix");
  }
  return 0;
}

// `next` != NULL: also run the transmission pass of the following step inside the agent kernel (pipelined family
// only); returns 1 when it did.  bt.nb > 1: a batched ensemble (pipelined kernels only; the caller has checked).
static int lean_forward(const gj_world_desc* w, const gj_step_params* p, const Plan& pl, const LeanPlan& lp,
                        const gj_fwd_io* io, const Scratch& sc, cudaStream_t st, const NextStep* next,
                        const Batch& bt = kNoBatch) {
  const bool quar = p->n_quar > 0;
  const bool batch = bt.nb > 1;
  if (p->stage != GJ_STAGE_REST) {
    if (!p->t_ready) {
      ProfScope ps(K_TRANSMISSION, st);
      static OccCache occ[4];
      const Scatter sct{sc.sct_acc, sc.sct_dirty};
#define GJ_K1(Q, B, I)                                                                                               \
  launch_pdl(k_lean_transmission<Q, B>, dim3(lean_grid(w, k_lean_transmission<Q, B>, &occ[I], bt)), dim3(kLeanThreads), \
             0, st, *w, *p, lp, *io, sc.tile_part, sct, bt)
#define GJ_K1C(Q, B, I)                                                                                              \
  launch_pdl(k_lean_transmission_c<Q, B>, dim3(lean_grid(w, k_lean_transmission_c<Q, B>, &occ_c[I], bt)),              \
             dim3(kLeanThreads), 0, st, *w, *p, lp, *io, sc.tile_part, sct, bt)
      static OccCache occ_c[4];
      const bool compact = (pipe_flags() & 4) == 0;   // gj_pipeline_enable bit 2 / GJ_K1C=0: the uncompacted pass
      if (compact) {
        if (batch) {
          if (quar) GJ_K1C(true, true, 3);
          else GJ_K1C(false, true, 2);
        } else {
          if (quar) GJ_K1C(true, false, 1);
          else GJ_K1C(false, false, 0);
        }
      } else if (batch) {
        if (quar) GJ_K1(true, true, 3);
        else GJ_K1(false, true, 2);
      } else {
        if (quar) GJ_K1(true, false, 1);
        else GJ_K1(false, false, 0);
      }
#undef GJ_K1
#undef GJ_K1C
      GJ_CHECK_LAUNCH("k_lean_transmission");
    }
    const Venue v{io->venue_region, io->venue_factor, io->n_venue_regions};
    if (lp.has_generic)
      if (int e = launch_lean_forward_sums(w, p, pl, io->beta, quar ? io->Tq : io->T, io->S_scaled + lp.gen_base,
                                           io->S_unscaled + lp.gen_base, sc, st, bt, v))
        return e;
    if (int e = launch_cell_groups(w, p, pl, io->beta, io->S_scaled, io->S_unscaled, sc, st, bt, v)) return e;
  }
  if (p->stage == GJ_STAGE_SUMS) return 0;
  if (int e = launch_cell_gather(w, p, pl, io->S_scaled, sc, st, bt)) return e;
  if (batch && bt.noise && pipe_enabled() && pipe_aligned_fwd(w, lp, io)) {   // the draw's noise, once for all samples
    ProfScope pn(K_OTHER, st);
    launch_pdl(k_batch_noise, dim3(agent_grid(w->n_agents)), dim3(kBlock), 0, st, *w, *p, const_cast<float*>(bt.noise));
    GJ_CHECK_LAUNCH("k_batch_noise");
  }
  if (pipe_enabled() && pipe_aligned_fwd(w, lp, io)) {
    ProfScope ps(K_AGENT_FWD, st);
    static OccCache occ[20];
    const bool diag = io->q || io->n;
    const bool lab = io->label != nullptr;
    const bool region = io->region != nullptr;   // a step with a regional factor never gets a look-ahead
    const size_t smem = next ? sizeof(PipeFwdSharedT<true, false>)
                             : (batch ? sizeof(PipeFwdSharedT<false, true>) : sizeof(PipeFwdSharedT<false, false>)) +
                                   (region ? kPipeRegionBytes : 0);
    NextStep nx;
    memset(&nx, 0, sizeof(nx));
    if (next) {
      nx = *next;
      nx.tile_part = sc.tile_part;   // consumed by this step's k_cell_groups before the agent kernel runs
      nx.sct = Scatter{sc.sct_acc, sc.sct_dirty};   // zeroed by this step's finalize pass, which has already run
    }
#define GJ_PIPE_FWD(Q, D, X, B, L, I)                                                                                 \
  launch_pdl(k_pipe_forward<Q, D, X, B, L>,                                                                           \
             dim3(pipe_grid(w, k_pipe_forward<Q, D, X, B, L>, kPipeThreads, smem, &occ[I], bt)), dim3(kPipeThreads),    \
             smem, st, *w, *p, lp, *io, (const float*)sc.cell_buf, sc.red_part, sc.tickets, nx, bt)
#define GJ_PIPE_FWD_R(Q, D, B, L, I)                                                                                  \
  launch_pdl(k_pipe_forward_region<Q, D, B, L>,                                                                       \
             dim3(pipe_grid(w, k_pipe_forward_region<Q, D, B, L>, kPipeThreads, smem, &occ_r[I], bt)),                \
             dim3(kPipeThreads), smem, st, *w, *p, lp, *io, (const float*)sc.cell_buf, sc.red_part, sc.tickets, nx, bt)
    static OccCache occ_r[16];
    if (region) {
      const int i = (quar ? 8 : 0) | (diag ? 4 : 0) | (batch ? 2 : 0) | (lab ? 1 : 0);
      switch (i) {
        case 0: GJ_PIPE_FWD_R(false, false, false, false, 0); break;
        case 1: GJ_PIPE_FWD_R(false, false, false, true, 1); break;
        case 2: GJ_PIPE_FWD_R(false, false, true, false, 2); break;
        case 3: GJ_PIPE_FWD_R(false, false, true, true, 3); break;
        case 4: GJ_PIPE_FWD_R(false, true, false, false, 4); break;
        case 5: GJ_PIPE_FWD_R(false, true, false, true, 5); break;
        case 6: GJ_PIPE_FWD_R(false, true, true, false, 6); break;
        case 7: GJ_PIPE_FWD_R(false, true, true, true, 7); break;
        case 8: GJ_PIPE_FWD_R(true, false, false, false, 8); break;
        case 9: GJ_PIPE_FWD_R(true, false, false, true, 9); break;
        case 10: GJ_PIPE_FWD_R(true, false, true, false, 10); break;
        case 11: GJ_PIPE_FWD_R(true, false, true, true, 11); break;
        case 12: GJ_PIPE_FWD_R(true, true, false, false, 12); break;
        case 13: GJ_PIPE_FWD_R(true, true, false, true, 13); break;
        case 14: GJ_PIPE_FWD_R(true, true, true, false, 14); break;
        default: GJ_PIPE_FWD_R(true, true, true, true, 15); break;
      }
    } else if (lab && batch) {   // a step with a label table never gets a look-ahead (step_forward_impl)
      if (quar && diag) GJ_PIPE_FWD(true, true, false, true, true, 19);
      else if (quar) GJ_PIPE_FWD(true, false, false, true, true, 18);
      else if (diag) GJ_PIPE_FWD(false, true, false, true, true, 17);
      else GJ_PIPE_FWD(false, false, false, true, true, 16);
    } else if (lab) {
      if (quar && diag) GJ_PIPE_FWD(true, true, false, false, true, 15);
      else if (quar) GJ_PIPE_FWD(true, false, false, false, true, 14);
      else if (diag) GJ_PIPE_FWD(false, true, false, false, true, 13);
      else GJ_PIPE_FWD(false, false, false, false, true, 12);
    } else if (batch) {
      if (quar && diag) GJ_PIPE_FWD(true, true, false, true, false, 11);
      else if (quar) GJ_PIPE_FWD(true, false, false, true, false, 10);
      else if (diag) GJ_PIPE_FWD(false, true, false, true, false, 9);
      else GJ_PIPE_FWD(false, false, false, true, false, 8);
    } else if (next) {
      if (quar && diag) GJ_PIPE_FWD(true, true, true, false, false, 7);
      else if (quar) GJ_PIPE_FWD(true, false, true, false, false, 6);
      else if (diag) GJ_PIPE_FWD(false, true, true, false, false, 5);
      else GJ_PIPE_FWD(false, false, true, false, false, 4);
    } else {
      if (quar && diag) GJ_PIPE_FWD(true, true, false, false, false, 3);
      else if (quar) GJ_PIPE_FWD(true, false, false, false, false, 2);
      else if (diag) GJ_PIPE_FWD(false, true, false, false, false, 1);
      else GJ_PIPE_FWD(false, false, false, false, false, 0);
    }
#undef GJ_PIPE_FWD
#undef GJ_PIPE_FWD_R
    GJ_CHECK_LAUNCH("k_pipe_forward");
    return next ? 1 : 0;
  }
  if (batch) return bad("batched step: the pipelined kernels are off or an array is not 16-byte aligned");
  {
    ProfScope ps(K_AGENT_FWD, st);
    static OccCache occ[8];
    const bool diag = io->q || io->n;
#define GJ_LEAN_FWD(Q, D, L, I)                                                                                       \
  k_lean_forward<Q, D, L><<<lean_grid(w, k_lean_forward<Q, D, L>, &occ[I]), kLeanThreads, 0, st>>>(                   \
      *w, *p, lp, *io, sc.cell_buf, sc.red_part, sc.tickets)
#define GJ_LEAN_FWD_R(Q, D, L, I)                                                                                     \
  k_lean_forward_region<Q, D, L><<<lean_grid(w, k_lean_forward_region<Q, D, L>, &occ_r[I]), kLeanThreads, 0, st>>>(     \
      *w, *p, lp, *io, sc.cell_buf, sc.red_part, sc.tickets)
    static OccCache occ_r[8];
    if (io->region) {
      if (io->label) {
        if (quar && diag) GJ_LEAN_FWD_R(true, true, true, 7);
        else if (quar) GJ_LEAN_FWD_R(true, false, true, 6);
        else if (diag) GJ_LEAN_FWD_R(false, true, true, 5);
        else GJ_LEAN_FWD_R(false, false, true, 4);
      } else {
        if (quar && diag) GJ_LEAN_FWD_R(true, true, false, 3);
        else if (quar) GJ_LEAN_FWD_R(true, false, false, 2);
        else if (diag) GJ_LEAN_FWD_R(false, true, false, 1);
        else GJ_LEAN_FWD_R(false, false, false, 0);
      }
    } else if (io->label) {
      if (quar && diag) GJ_LEAN_FWD(true, true, true, 7);
      else if (quar) GJ_LEAN_FWD(true, false, true, 6);
      else if (diag) GJ_LEAN_FWD(false, true, true, 5);
      else GJ_LEAN_FWD(false, false, true, 4);
    } else {
      if (quar && diag) GJ_LEAN_FWD(true, true, false, 3);
      else if (quar) GJ_LEAN_FWD(true, false, false, 2);
      else if (diag) GJ_LEAN_FWD(false, true, false, 1);
      else GJ_LEAN_FWD(false, false, false, 0);
    }
#undef GJ_LEAN_FWD
#undef GJ_LEAN_FWD_R
    GJ_CHECK_LAUNCH("k_lean_forward");
  }
  return 0;
}

// seeding by label, backward: the per-agent pass writes d/dseed_fraction to seed_work, then the per-label reduction.
// The reduction's chunk partials live in the scratch's reduction partials (free once the agent pass is done); the chunk
// is the smallest power of two >= kSeedChunk whose partials fit there, so it depends on the world only.
// Venue regions hold few groups each (a leisure venue is often a region of its own): a warp walks its chunk's labels
// one after the other, so the groups' reduction uses short chunks to spread them over many warps.
constexpr int64_t kSeedChunk = 2048;
constexpr int64_t kVenueChunk = 32;
static int64_t seed_chunk(const gj_world_desc* w, int64_t N, int64_t min_chunk = kSeedChunk) {
  const int64_t n_tiles = w->n_tiles > 0 ? w->n_tiles : 1;
  const int64_t slots = (n_tiles > kRedBlocks ? n_tiles : kRedBlocks) * kMaxRed;   // doubles in Scratch::red_part
  int64_t chunk = min_chunk;
  while (2 * ((N + chunk - 1) / chunk) > slots) chunk *= 2;
  return chunk;
}
// out[l] = sum of work over the N items (agents, or the groups of one edge type) of label l (order / offsets: the
// items stably sorted by label), in fp64 over fixed chunks combined in chunk order: bit-reproducible and independent
// of the launch grid
static int label_sums(const gj_world_desc* w, int64_t N, const int32_t* order, const int32_t* offsets, int n_labels,
                      const float* work, const Scratch& sc, float* out, cudaStream_t st,
                      int64_t min_chunk = kSeedChunk) {
  const int64_t chunk = seed_chunk(w, N, min_chunk);
  const int64_t n_chunks = (N + chunk - 1) / chunk;
  k_seed_label_grad<<<blocks_for(n_chunks * 32, kBlock), kBlock, 0, st>>>(N, chunk, order, offsets, n_labels, work,
                                                                         sc.red_part, out);
  GJ_CHECK_LAUNCH("k_seed_label_grad");
  k_seed_label_fix<<<blocks_for((int64_t)n_labels * 32, kBlock), kBlock, 0, st>>>(chunk, offsets, n_labels, sc.red_part,
                                                                                  out);
  GJ_CHECK_LAUNCH("k_seed_label_fix");
  return 0;
}

// regional venue factor, backward: k_dbeta_venue wrote network k's per-group terms of dL/df to its own row of
// venue_work (at nets[k].s_off); the per-label reduction sums them over the groups of the network's edge type, region by region, per network
// and sample.  A RANGE-tier network has no group terms: its row is 0.
static int venue_backward(const gj_world_desc* w, const gj_step_params* p, const Plan& pl, const gj_bwd_io* io,
                          const Scratch& sc, const Batch& bt, cudaStream_t st) {
  if (!io->venue_region || !io->g_venue_factor) return 0;
  ProfScope ps(K_VENUE_GRAD, st);
  const int n = io->n_venue_regions;
  for (int s = 0; s < bt.nb; ++s) {
    for (int k = 0; k < p->n_nets; ++k) {
      float* out = io->g_venue_factor + (int64_t)s * bt.sVen + (int64_t)k * n;
      const int t = p->nets[k].type;
      if (pl.tier[k] == GJ_TIER_RANGE) {
        const cudaError_t e = cudaMemsetAsync(out, 0, sizeof(float) * (size_t)n, st);
        if (e != cudaSuccess) return fail("cudaMemsetAsync (g_venue_factor)", e);
        continue;
      }
      const int64_t g0 = w->type_group_off[t];
      if (int e = label_sums(w, w->type_group_off[t + 1] - g0, io->venue_order + g0,
                             io->venue_offsets + (int64_t)t * (n + 1), n,
                             io->venue_work + (int64_t)s * bt.sG + p->nets[k].s_off, sc, out, st, kVenueChunk))
        return e;
    }
  }
  return 0;
}

static int lean_backward(const gj_world_desc* w, const gj_step_params* p, const Plan& pl, LeanPlan lp,
                         const gj_bwd_io* io, const Scratch& sc, cudaStream_t st, const Batch& bt = kNoBatch) {
  const bool quar = p->n_quar > 0;
  const bool batch = bt.nb > 1;
  static OccCache occ_b[4], occ_g[2];
  const bool lab = io->label && io->g_red_label;
  const bool region = io->region != nullptr;
  int gather_grid = 1;
  const bool pipe = pipe_enabled() && pipe_aligned_bwd(w, lp, io);
  if (batch && !pipe) return bad("batched step: the pipelined kernels are off or an array is not 16-byte aligned");
  if (p->stage != GJ_STAGE_REST) {
    if (pipe) {
      ProfScope ps(K_AGENT_BWD, st);
      static OccCache occ[8];
      const size_t smem = sizeof(PipeBwdShared) + (region ? kPipeRegionBytes : 0);
#define GJ_PIPE_BWD(Q, B, L, I)                                                                                       \
  launch_pdl(k_pipe_backward<Q, B, L>, dim3(pipe_grid(w, k_pipe_backward<Q, B, L>, kBwdThreads, smem, &occ[I], bt)),    \
             dim3(kBwdThreads), smem, st, *w, *p, lp, *io, sc.tile_part, bt)
#define GJ_PIPE_BWD_R(Q, B, L, I)                                                                                     \
  launch_pdl(k_pipe_backward_region<Q, B, L>,                                                                         \
             dim3(pipe_grid(w, k_pipe_backward_region<Q, B, L>, kBwdThreads, smem, &occ_r[I], bt)), dim3(kBwdThreads), \
             smem, st, *w, *p, lp, *io, sc.tile_part, bt)
      static OccCache occ_r[8];
      if (region) {
        const int i = (quar ? 4 : 0) | (batch ? 2 : 0) | (lab ? 1 : 0);
        switch (i) {
          case 0: GJ_PIPE_BWD_R(false, false, false, 0); break;
          case 1: GJ_PIPE_BWD_R(false, false, true, 1); break;
          case 2: GJ_PIPE_BWD_R(false, true, false, 2); break;
          case 3: GJ_PIPE_BWD_R(false, true, true, 3); break;
          case 4: GJ_PIPE_BWD_R(true, false, false, 4); break;
          case 5: GJ_PIPE_BWD_R(true, false, true, 5); break;
          case 6: GJ_PIPE_BWD_R(true, true, false, 6); break;
          default: GJ_PIPE_BWD_R(true, true, true, 7); break;
        }
      } else if (lab && batch) {
        if (quar) GJ_PIPE_BWD(true, true, true, 7);
        else GJ_PIPE_BWD(false, true, true, 6);
      } else if (lab) {
        if (quar) GJ_PIPE_BWD(true, false, true, 5);
        else GJ_PIPE_BWD(false, false, true, 4);
      } else if (batch) {
        if (quar) GJ_PIPE_BWD(true, true, false, 3);
        else GJ_PIPE_BWD(false, true, false, 2);
      } else {
        if (quar) GJ_PIPE_BWD(true, false, false, 1);
        else GJ_PIPE_BWD(false, false, false, 0);
      }
#undef GJ_PIPE_BWD
#undef GJ_PIPE_BWD_R
      GJ_CHECK_LAUNCH("k_pipe_backward");
    } else {
      ProfScope ps(K_AGENT_BWD, st);
#define GJ_LEAN_BWD(Q, L, I) \
  k_lean_backward<Q, L><<<lean_grid(w, k_lean_backward<Q, L>, &occ_b[I]), kLeanThreads, 0, st>>>(*w, *p, lp, *io, sc.tile_part)
#define GJ_LEAN_BWD_R(Q, L, I)                                                                                        \
  k_lean_backward_region<Q, L><<<lean_grid(w, k_lean_backward_region<Q, L>, &occ_br[I]), kLeanThreads, 0, st>>>(        \
      *w, *p, lp, *io, sc.tile_part)
      static OccCache occ_br[4];
      if (region) {
        if (lab) {
          if (quar) GJ_LEAN_BWD_R(true, true, 3);
          else GJ_LEAN_BWD_R(false, true, 2);
        } else {
          if (quar) GJ_LEAN_BWD_R(true, false, 1);
          else GJ_LEAN_BWD_R(false, false, 0);
        }
      } else if (lab) {
        if (quar) GJ_LEAN_BWD(true, true, 3);
        else GJ_LEAN_BWD(false, true, 2);
      } else {
        if (quar) GJ_LEAN_BWD(true, false, 1);
        else GJ_LEAN_BWD(false, false, 0);
      }
#undef GJ_LEAN_BWD
#undef GJ_LEAN_BWD_R
      GJ_CHECK_LAUNCH("k_lean_backward");
    }
    const Venue v{io->venue_region, io->venue_factor, io->n_venue_regions};
    if (lp.has_generic)
      if (int e = launch_lean_group_pass(w, p, pl, io->beta, quar ? io->wq : io->w, io->cR + lp.gen_base,
                                         io->R + lp.gen_base, sc, true, st, bt, v))
        return e;
    if (int e = launch_cell_groups(w, p, pl, io->beta, io->cR, io->R, sc, st, bt, v)) return e;
  }
  if (p->stage == GJ_STAGE_SUMS) return 0;
  if (int e = launch_cell_gather(w, p, pl, io->cR, sc, st, bt)) return e;
  if (pipe) {
    ProfScope ps(K_AGENT_BWD_GATHER, st);
    static OccCache occ[4];
    const size_t smem = sizeof(PipeGatShared);
#define GJ_PIPE_GAT(Q, B, I)                                                                                          \
  launch_pdl(k_pipe_backward_gather<Q, B>,                                                                            \
             dim3(gather_grid = pipe_grid(w, k_pipe_backward_gather<Q, B>, kPipeThreads, smem, &occ[I], bt)),          \
             dim3(kPipeThreads), smem, st, *w, *p, lp, *io, (const float*)sc.cell_buf, sc.dbeta_tile, bt)
    if (batch) {
      if (quar) GJ_PIPE_GAT(true, true, 3);
      else GJ_PIPE_GAT(false, true, 2);
    } else {
      if (quar) GJ_PIPE_GAT(true, false, 1);
      else GJ_PIPE_GAT(false, false, 0);
    }
#undef GJ_PIPE_GAT
    GJ_CHECK_LAUNCH("k_pipe_backward_gather");
    gather_grid /= bt.nb;   // the partials of ONE sample
  } else {
    ProfScope ps(K_AGENT_BWD_GATHER, st);
    if (quar) k_lean_backward_gather<true><<<(gather_grid = lean_grid(w, k_lean_backward_gather<true>, &occ_g[1])), kLeanThreads, 0, st>>>(*w, *p, lp, *io, sc.cell_buf, sc.dbeta_tile);
    else k_lean_backward_gather<false><<<(gather_grid = lean_grid(w, k_lean_backward_gather<false>, &occ_g[0])), kLeanThreads, 0, st>>>(*w, *p, lp, *io, sc.cell_buf, sc.dbeta_tile);
    GJ_CHECK_LAUNCH("k_lean_backward_gather");
  }
  if (io->g_beta) {
    ProfScope ps(K_DBETA, st);
    DbetaPlan dp;
    for (int k = 0; k < GJ_MAX_NETS; ++k) {
      dp.soff[k] = 0;
      if (k < p->n_nets)
        dp.soff[k] = pl.tier[k] == GJ_TIER_GENERIC ? lp.gen_base + w->type_group_off[p->nets[k].type] : p->nets[k].s_off;
    }
    dp.n_range_parts = gather_grid;
    dim3 grid2(kRedBlocks / 8, p->n_nets, bt.nb);
    if (io->venue_region)
      launch_pdl(k_dbeta_venue, grid2, dim3(kBlock), 0, st, *w, *p, pl, dp, io->S_unscaled, (const float*)io->R,
                 (const double*)sc.dbeta_tile, sc.dbeta_part, sc.tickets, io->g_beta, bt, io->beta,
                 Venue{io->venue_region, io->venue_factor, io->n_venue_regions},
                 io->g_venue_factor ? io->venue_work : nullptr);
    else
      launch_pdl(k_dbeta, grid2, dim3(kBlock), 0, st, *w, *p, pl, dp, io->S_unscaled, (const float*)io->R,
                 (const double*)sc.dbeta_tile, sc.dbeta_part, sc.tickets, io->g_beta, bt);
    GJ_CHECK_LAUNCH("k_dbeta");
    if (int e = venue_backward(w, p, pl, io, sc, bt, st)) return e;
  }
  return 0;
}

// ---- boundary exchange of a partitioned world: pack / unpack of the straddling groups' sums -------------------
// pack position q holds the sum of boundary group q (all edge types of the step concatenated); inv[q] = index of
// that group's entry in this rank's group-sum buffers, or -1 if the rank does not attend the group (contributes 0)
__global__ void __launch_bounds__(kBlock) k_boundary_pack(int64_t n, const int32_t* __restrict__ inv,
                                                          const float* __restrict__ a, const float* __restrict__ b,
                                                          float* __restrict__ pack) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += stride) {
    const int32_t j = inv[q];
    pack[q] = j >= 0 ? a[j] : 0.0f;
    pack[n + q] = j >= 0 ? b[j] : 0.0f;
  }
}
__global__ void __launch_bounds__(kBlock) k_boundary_unpack(int64_t n, const int32_t* __restrict__ inv,
                                                            const float* __restrict__ pack, float* __restrict__ a,
                                                            float* __restrict__ b) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += stride) {
    const int32_t j = inv[q];
    if (j >= 0) {
      a[j] = pack[q];
      b[j] = pack[n + q];
    }
  }
}

// ---- peer-memory exchange (see gradjune_b200.h) -----------------------------------------------------------
// receive buffer of one rank: [2 sets][world_size sources][2 arrays][capacity] floats, then the flags
// [2 sets][world_size] uint32, then {exchange counter, ticket A, ticket B, error} uint32
constexpr int kPeerBlocks = 148;     // co-resident by construction: blocks wait on flags other GPUs raise
constexpr int kPeerThreads = 1024;   // one CTA per SM: the SMs are idle between the two stages of a step anyway
constexpr int kPeerBatch = 4;        // packed groups a thread keeps in flight (the loop is a chain of dependent loads:
                                     // inv -> a[j], b[j] -> remote store; 256 threads x 1 in flight measured 61 us per
                                     // exchange of 655 k groups at 8 GPUs, profiles/r2_bench_56M_n8_strong_run14.json)
struct PeerView {
  int rank, world;
  int64_t cap;
  float* recv[32];       // every rank's receive buffer (own included), mapped into this process
  uint32_t* flags[32];   // every rank's flag array
  uint32_t* ctl;         // own {counter, ticket A, ticket B, error}
};
__device__ __forceinline__ float* peer_slot(const PeerView& v, int dst, uint32_t set, int src, int arr) {
  return v.recv[dst] + (((int64_t)set * v.world + src) * 2 + arr) * v.cap;
}
// n_mine / mine: the packed positions this rank attends (inv[q] >= 0), ascending; NULL = walk all n positions
__global__ void __launch_bounds__(kPeerThreads) k_peer_exchange(PeerView v, int64_t n_all, const int32_t* __restrict__ inv,
                                                                 const uint32_t* __restrict__ attend,
                                                                 float* __restrict__ a, float* __restrict__ b,
                                                                 int64_t n_mine, const int32_t* __restrict__ mine) {
  const int64_t n = mine ? n_mine : n_all;
  __shared__ uint32_t s_epoch;
  __shared__ bool s_last;
  pdl_launch();
  pdl_wait();
  if (threadIdx.x == 0) s_epoch = *(volatile uint32_t*)&v.ctl[0] + 1u;   // bumped by the last block at the very end
  __syncthreads();
  const uint32_t e = s_epoch, set = e & 1u;
  const uint32_t me = 1u << v.rank;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t q0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  // ---- push: my partial sums into the receive buffers of the other ranks attending each group ---------------
  for (int64_t base = q0; base < n; base += stride * kPeerBatch) {
    int32_t j[kPeerBatch];
    uint32_t m[kPeerBatch];
    float va[kPeerBatch], vb[kPeerBatch];
    int64_t qq[kPeerBatch];
#pragma unroll
    for (int h = 0; h < kPeerBatch; ++h) {
      const int64_t i = base + h * stride;
      qq[h] = i < n ? (mine ? (int64_t)mine[i] : i) : -1;
    }
#pragma unroll
    for (int h = 0; h < kPeerBatch; ++h) {
      j[h] = qq[h] >= 0 ? inv[qq[h]] : -1;
      m[h] = qq[h] >= 0 ? (attend[qq[h]] & ~me) : 0u;
    }
#pragma unroll
    for (int h = 0; h < kPeerBatch; ++h) {
      va[h] = j[h] >= 0 ? a[j[h]] : 0.0f;
      vb[h] = j[h] >= 0 ? b[j[h]] : 0.0f;
    }
#pragma unroll
    for (int h = 0; h < kPeerBatch; ++h) {
      if (j[h] < 0) continue;
      const int64_t q = qq[h];
      uint32_t mm = m[h];
      while (mm) {
        const int dst = __ffs(mm) - 1;
        mm &= mm - 1;
        peer_slot(v, dst, set, v.rank, 0)[q] = va[h];
        peer_slot(v, dst, set, v.rank, 1)[q] = vb[h];
      }
    }
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(&v.ctl[1], 1u) == gridDim.x - 1;
  __syncthreads();
  if (s_last) {   // every block of this rank has pushed (and fenced): tell the peers
    __threadfence_system();
    if ((int)threadIdx.x < v.world && (int)threadIdx.x != v.rank)
      *(volatile uint32_t*)&v.flags[threadIdx.x][set * v.world + v.rank] = e;
    if (threadIdx.x == 0) v.ctl[1] = 0u;
    __threadfence_system();
  }
  // ---- wait for every peer's flag in my own memory ----------------------------------------------------------
  if ((int)threadIdx.x < v.world && (int)threadIdx.x != v.rank) {
    volatile uint32_t* f = (volatile uint32_t*)&v.flags[v.rank][set * v.world + threadIdx.x];
    unsigned long long t0 = 0, t1 = 0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    while (*f != e) {
      __nanosleep(32);
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
      if (t1 - t0 > 10000000000ull) {   // ~10 s: a peer is gone; give up rather than hang the GPU
        v.ctl[3] = 1u;
        break;
      }
    }
  }
  __threadfence_system();
  __syncthreads();
  // ---- reduce in ascending rank order (my own term in its place): identical on every rank -------------------
  for (int64_t base = q0; base < n; base += stride * kPeerBatch) {
    int32_t j[kPeerBatch];
    uint32_t m[kPeerBatch];
    float oa[kPeerBatch], ob[kPeerBatch];
    int64_t qq[kPeerBatch];
#pragma unroll
    for (int h = 0; h < kPeerBatch; ++h) {
      const int64_t i = base + h * stride;
      qq[h] = i < n ? (mine ? (int64_t)mine[i] : i) : -1;
    }
#pragma unroll
    for (int h = 0; h < kPeerBatch; ++h) {
      j[h] = qq[h] >= 0 ? inv[qq[h]] : -1;
      m[h] = qq[h] >= 0 ? attend[qq[h]] : 0u;
    }
#pragma unroll
    for (int h = 0; h < kPeerBatch; ++h) {
      oa[h] = j[h] >= 0 ? a[j[h]] : 0.0f;
      ob[h] = j[h] >= 0 ? b[j[h]] : 0.0f;
    }
#pragma unroll
    for (int h = 0; h < kPeerBatch; ++h) {
      if (j[h] < 0) continue;
      const int64_t q = qq[h];
      uint32_t mm = m[h];
      float sa = 0.0f, sb = 0.0f;
      while (mm) {
        const int src = __ffs(mm) - 1;
        mm &= mm - 1;
        if (src == v.rank) {
          sa += oa[h];
          sb += ob[h];
        } else {
          sa += __ldcg(peer_slot(v, v.rank, set, src, 0) + q);
          sb += __ldcg(peer_slot(v, v.rank, set, src, 1) + q);
        }
      }
      a[j[h]] = sa;
      b[j[h]] = sb;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0 && atomicAdd(&v.ctl[2], 1u) == gridDim.x - 1) {   // the last block closes the exchange
    v.ctl[2] = 0u;
    *(volatile uint32_t*)&v.ctl[0] = e;
  }
}

}  // namespace gj

using namespace gj;

struct gj_peer {
  int rank, world, device;
  int64_t cap;
  size_t bytes, flag_off, ctl_off;
  char* own;           // cudaMalloc'ed
  char* mapped[32];    // every rank's buffer in this process (own = own)
  bool connected;
};

extern "C" {

int gj_abi_version(void) { return GJ_ABI_VERSION; }
const char* gj_last_error(void) { return g_err; }

int gj_config(int64_t* out, int n) {
  const int64_t v[10] = {GJ_SMALL_GROUP,      GJ_CHUNK,          (int64_t)sizeof(gj_world_desc), (int64_t)sizeof(gj_step_params),
                         (int64_t)sizeof(gj_fwd_io), (int64_t)sizeof(gj_bwd_io), kRedBlocks, GJ_TILE_AGENTS,
                         GJ_SCATTER_MAX_GROUP, (int64_t)sizeof(gj_batch)};
  for (int i = 0; i < n && i < 10; ++i) out[i] = v[i];
  return 10;
}

int64_t gj_scratch_bytes(const gj_world_desc* w) { return w ? scratch_bytes(w) : -1; }

int gj_boundary_pack(int64_t n_pack, const int32_t* inv, const float* a, const float* b, float* pack, void* stream) {
  if (n_pack <= 0) return 0;
  if (!inv || !a || !b || !pack) return bad("NULL array");
  k_boundary_pack<<<agent_grid(n_pack), kBlock, 0, (cudaStream_t)stream>>>(n_pack, inv, a, b, pack);
  GJ_CHECK_LAUNCH("k_boundary_pack");
  return 0;
}

int gj_boundary_unpack(int64_t n_pack, const int32_t* inv, const float* pack, float* a, float* b, void* stream) {
  if (n_pack <= 0) return 0;
  if (!inv || !a || !b || !pack) return bad("NULL array");
  k_boundary_unpack<<<agent_grid(n_pack), kBlock, 0, (cudaStream_t)stream>>>(n_pack, inv, pack, a, b);
  GJ_CHECK_LAUNCH("k_boundary_unpack");
  return 0;
}

int gj_peer_create(int rank, int world_size, int64_t capacity, gj_peer** out) {
  if (!out || rank < 0 || world_size < 1 || world_size > 32 || rank >= world_size || capacity < 0) return bad("gj_peer_create arguments");
  gj_peer* p = new gj_peer();
  p->rank = rank;
  p->world = world_size;
  p->cap = capacity > 0 ? (capacity + 63) / 64 * 64 : 64;
  p->connected = false;
  cudaGetDevice(&p->device);
  const size_t data = sizeof(float) * 2ull * world_size * 2ull * (size_t)p->cap;
  p->flag_off = (data + 255) / 256 * 256;
  p->ctl_off = p->flag_off + 256 * ((sizeof(uint32_t) * 2 * world_size + 255) / 256);
  p->bytes = p->ctl_off + 256;
  for (int i = 0; i < 32; ++i) p->mapped[i] = nullptr;
  cudaError_t e = cudaMalloc((void**)&p->own, p->bytes);
  if (e != cudaSuccess) {
    delete p;
    return fail("cudaMalloc (peer buffer)", e);
  }
  e = cudaMemset(p->own, 0, p->bytes);
  if (e != cudaSuccess) return fail("cudaMemset (peer buffer)", e);
  p->mapped[rank] = p->own;
  *out = p;
  return 0;
}

int gj_peer_handle(gj_peer* p, void* handle) {
  if (!p || !handle) return bad("gj_peer_handle arguments");
  static_assert(sizeof(cudaIpcMemHandle_t) == GJ_IPC_HANDLE_BYTES, "IPC handle size");
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, p->own);
  if (e != cudaSuccess) return fail("cudaIpcGetMemHandle", e);
  memcpy(handle, &h, sizeof(h));
  return 0;
}

int gj_peer_connect(gj_peer* p, const void* handles) {
  if (!p || !handles) return bad("gj_peer_connect arguments");
  for (int r = 0; r < p->world; ++r) {
    if (r == p->rank) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, (const char*)handles + (size_t)r * GJ_IPC_HANDLE_BYTES, sizeof(h));
    void* ptr = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) return fail("cudaIpcOpenMemHandle", e);
    p->mapped[r] = (char*)ptr;
  }
  p->connected = true;
  return 0;
}

int gj_peer_exchange(gj_peer* p, int64_t n_pack, const int32_t* inv, const uint32_t* attend, float* a, float* b,
                     int64_t n_mine, const int32_t* mine, void* stream) {
  if (!p || !p->connected) return bad("peer context is not connected");
  if (n_pack > p->cap) return bad("n_pack exceeds the peer buffers' capacity");
  if (n_pack > 0 && (!inv || !attend || !a || !b)) return bad("NULL array");
  PeerView v;
  v.rank = p->rank;
  v.world = p->world;
  v.cap = p->cap;
  for (int r = 0; r < 32; ++r) {
    v.recv[r] = r < p->world ? (float*)p->mapped[r] : nullptr;
    v.flags[r] = r < p->world ? (uint32_t*)(p->mapped[r] + p->flag_off) : nullptr;
  }
  v.ctl = (uint32_t*)(p->own + p->ctl_off);
  ProfScope ps(K_EXCHANGE, (cudaStream_t)stream);
  launch_pdl(k_peer_exchange, dim3(kPeerBlocks), dim3(kPeerThreads), 0, (cudaStream_t)stream, v, n_pack, inv, attend, a, b, n_mine,
             mine);
  GJ_CHECK_LAUNCH("k_peer_exchange");
  return 0;
}

int gj_peer_status(gj_peer* p) {
  if (!p) return bad("peer is NULL");
  uint32_t err = 0;
  cudaError_t e = cudaMemcpy(&err, p->own + p->ctl_off + 3 * sizeof(uint32_t), sizeof(err), cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) return fail("cudaMemcpy (peer status)", e);
  if (err) {
    cudaMemset(p->own + p->ctl_off + 3 * sizeof(uint32_t), 0, sizeof(uint32_t));
    snprintf(g_err, sizeof(g_err), "a peer did not arrive at a boundary exchange within 10 s");
  }
  return err ? 1 : 0;
}

int gj_peer_destroy(gj_peer* p) {
  if (!p) return 0;
  for (int r = 0; r < p->world; ++r)
    if (r != p->rank && p->mapped[r]) cudaIpcCloseMemHandle(p->mapped[r]);
  cudaFree(p->own);
  delete p;
  return 0;
}

int gj_pipeline_enable(int on) {
  const int prev = pipe_flags();
  if (on >= 0) g_pipe_on = on & 7;
  return prev;
}

int gj_profile_enable(int on) {
  if (on && !g_prof.created) {
    for (int i = 0; i < kMaxProfiled; ++i) {
      if (cudaEventCreate(&g_prof.ev[i][0]) != cudaSuccess || cudaEventCreate(&g_prof.ev[i][1]) != cudaSuccess)
        return fail("cudaEventCreate", cudaGetLastError());
    }
    g_prof.created = true;
  }
  g_prof.on = on != 0;
  g_prof.n = 0;
  for (int i = 0; i < K_COUNT; ++i) g_prof.launches[i] = 0;
  return 0;
}

int gj_profile_read(double* ms, int64_t* timed, int64_t* launches, int n) {
  for (int i = 0; i < n && i < K_COUNT; ++i) {
    ms[i] = 0.0;
    timed[i] = 0;
    launches[i] = g_prof.launches[i];
  }
  for (int s = 0; s < g_prof.n; ++s) {
    if (cudaEventSynchronize(g_prof.ev[s][1]) != cudaSuccess) return fail("cudaEventSynchronize", cudaGetLastError());
    float t = 0.f;
    if (cudaEventElapsedTime(&t, g_prof.ev[s][0], g_prof.ev[s][1]) != cudaSuccess)
      return fail("cudaEventElapsedTime", cudaGetLastError());
    if (g_prof.id[s] < n) {
      ms[g_prof.id[s]] += t;
      timed[g_prof.id[s]]++;
    }
  }
  return K_COUNT;
}

const char* gj_profile_kernel_name(int i) { return (i >= 0 && i < K_COUNT) ? kKernelNames[i] : ""; }

int gj_profile_prepare(int64_t n, const float* shape, float* k0, void* stream) {
  if (n <= 0) return 0;
  k_profile_prepare<<<agent_grid(n), kBlock, 0, (cudaStream_t)stream>>>(n, shape, k0);
  GJ_CHECK_LAUNCH("k_profile_prepare");
  return 0;
}

int gj_profile_pack(int64_t n, const float* maxinf, const float* shape, const float* rate, const float* shift,
                    const float* k0, float* prof4, void* stream) {
  if (n <= 0) return 0;
  if (!maxinf || !shape || !rate || !shift || !k0 || !prof4) return bad("NULL array");
  if (((uintptr_t)prof4) & 15) return bad("prof4 must be 16-byte aligned");
  k_profile_pack<<<agent_grid(n), kBlock, 0, (cudaStream_t)stream>>>(n, maxinf, shape, rate, shift, k0,
                                                                    reinterpret_cast<float4*>(prof4));
  GJ_CHECK_LAUNCH("k_profile_pack");
  return 0;
}

int gj_transmission_forward(int64_t n, float now, const float* tinf, const float* inf, const float* maxinf,
                            const float* shape, const float* rate, const float* shift, const float* k0, float* T,
                            void* stream) {
  if (n <= 0) return 0;
  if (!tinf || !inf || !maxinf || !shape || !rate || !shift || !k0 || !T) return bad("NULL array");
  k_transmission<<<agent_grid(n), kBlock, 0, (cudaStream_t)stream>>>(n, now, tinf, inf, maxinf, shape, rate, shift, k0,
                                                                    T);
  GJ_CHECK_LAUNCH("k_transmission");
  return 0;
}

int gj_transmission_backward(int64_t n, float now, const float* tinf, const float* inf, const float* maxinf,
                             const float* shape, const float* rate, const float* shift, const float* k0,
                             const float* g_T, float* g_tinf, float* g_inf, void* stream) {
  if (n <= 0) return 0;
  if (!tinf || !inf || !maxinf || !shape || !rate || !shift || !k0 || !g_T) return bad("NULL array");
  k_transmission_bwd<<<agent_grid(n), kBlock, 0, (cudaStream_t)stream>>>(n, now, tinf, inf, maxinf, shape, rate, shift,
                                                                        k0, g_T, g_tinf, g_inf);
  GJ_CHECK_LAUNCH("k_transmission_bwd");
  return 0;
}

// gj_batch -> the kernels' Batch, with the checks of the header
static int make_batch(const gj_world_desc* w, const gj_step_params* p, const gj_batch* b, Batch* bt) {
  if (!b) return bad("batch is NULL");
  if (b->n_samples < 1 || b->n_samples > 1024) return bad("batch: n_samples out of range");
  if (b->agent_stride < w->n_agents || (b->agent_stride & 3)) return bad("batch: agent_stride must be >= n_agents and a multiple of 4");
  if ((int64_t)b->n_samples * b->agent_stride >= ((int64_t)1 << 32)) return bad("batch: n_samples * agent_stride must stay below 2^32");
  if (b->scratch_stride < scratch_bytes(w) || (b->scratch_stride & 255)) return bad("batch: scratch_stride must be >= gj_scratch_bytes and a multiple of 256");
  if (b->group_stride < 0 || b->beta_stride < 0 || b->red_stride < 0 || b->beta_stride > (1 << 20) || b->red_stride > (1 << 20))
    return bad("batch: strides");
  if (p->mode != GJ_MODE_STEP || p->stage != GJ_STAGE_ALL || p->phases != GJ_PHASE_ALL)
    return bad("batch: only the whole fused step (GJ_MODE_STEP, GJ_PHASE_ALL, GJ_STAGE_ALL) is batched");
  bt->nb = b->n_samples;
  bt->sN = (uint32_t)b->agent_stride;
  bt->sG = b->group_stride;
  bt->sScr = b->scratch_stride;
  bt->sBeta = (int)b->beta_stride;
  bt->sRed = (int)b->red_stride;
  bt->noise = b->noise;
  bt->sLab = b->label_stride;
  bt->sReg = b->region_stride;
  bt->sVen = b->venue_stride;
  if (b->region_stride < 0) return bad("batch: region_stride must be >= 0");
  if (b->venue_stride < 0) return bad("batch: venue_stride must be >= 0");
  if (b->noise && !aligned16(b->noise)) return bad("batch: noise must be 16-byte aligned");
  return 0;
}

// results by label: the checks of the header, and the conversion of the step's integer sums
static int check_labels(const gj_fwd_io* io, const Batch& bt) {
  if (!io->label) return 0;
  if (io->n_labels < 1 || io->n_labels > (1 << 30)) return bad("n_labels must lie in [1, 2^30]");
  if (!io->red_label || !io->label_acc) return bad("label given without red_label / label_acc");
  if (bt.nb > 1 && bt.sLab < 2 * (int64_t)io->n_labels) return bad("batch: label_stride must be >= 2 * n_labels");
  return 0;
}
// regional transmission factor: the checks of the header (the codes and factors themselves are not checked)
static int check_region(const int32_t* region, int n_regions, const float* factor, const Batch& bt) {
  if (!region) return 0;
  if (n_regions < 1 || n_regions > (1 << 30)) return bad("n_regions must lie in [1, 2^30]");
  if (!factor) return bad("region given without region_factor");
  if (bt.nb > 1 && bt.sReg < (int64_t)n_regions) return bad("batch: region_stride must be >= n_regions");
  return 0;
}
// regional venue factor: the checks of the header (codes and factors are not checked)
static int check_venue(const gj_step_params* p, const int32_t* region, int n, const float* factor, const Batch& bt) {
  if (!region) return 0;
  if (n < 1 || n > (1 << 30)) return bad("n_venue_regions must lie in [1, 2^30]");
  if (!factor) return bad("venue_region given without venue_factor");
  if (bt.nb > 1 && bt.sVen < (int64_t)p->n_nets * n) return bad("batch: venue_stride must be >= n_nets * n_venue_regions");
  return 0;
}
static int finish_labels(const gj_fwd_io* io, cudaStream_t st, const Batch& bt) {
  if (!io->label) return 0;
  ProfScope ps(K_OTHER, st);
  const int64_t n = 2 * (int64_t)io->n_labels;
  const int64_t blocks = (n + kBlock - 1) / kBlock;
  launch_pdl(k_label_finish, dim3((int)(blocks < kRedBlocks ? blocks : kRedBlocks), 1, bt.nb), dim3(kBlock), 0, st, n,
             io->label_acc, io->red_label, bt.sLab);
  GJ_CHECK_LAUNCH("k_label_finish");
  return 0;
}

static int step_forward_run(const gj_world_desc* w, const gj_step_params* p, const gj_step_params* next,
                            const gj_fwd_io* io, void* stream, const gj_batch* batch);
// the agent kernels accumulate the label table as integers; one small kernel then converts it (and re-zeroes)
static int step_forward_impl(const gj_world_desc* w, const gj_step_params* p, const gj_step_params* next,
                             const gj_fwd_io* io, void* stream, const gj_batch* batch = nullptr) {
  if (int e = check_world(w)) return e;
  if (!p || !io) return bad("params/io is NULL");
  Batch bt = kNoBatch;
  if (batch)
    if (int e = make_batch(w, p, batch, &bt)) return e;
  if (int e = check_labels(io, bt)) return e;
  if (int e = check_region(io->region, io->n_regions, io->region_factor, bt)) return e;
  if (int e = check_venue(p, io->venue_region, io->n_venue_regions, io->venue_factor, bt)) return e;
  const int rc = step_forward_run(w, p, next, io, stream, batch);
  if (rc < 0 || p->stage == GJ_STAGE_SUMS) return rc;
  if (int e = finish_labels(io, (cudaStream_t)stream, bt)) return e;
  return rc;
}

static int step_forward_run(const gj_world_desc* w, const gj_step_params* p, const gj_step_params* next,
                            const gj_fwd_io* io, void* stream, const gj_batch* batch) {
  Batch bt = kNoBatch;
  if (batch)
    if (int e = make_batch(w, p, batch, &bt)) return e;
  if (p->n_stages > GJ_MAX_STAGES || p->n_age_bins > GJ_MAX_AGE_BINS || p->n_quar > GJ_MAX_QUAR) return bad("params sizes");
  if (!io->scratch) return bad("scratch is NULL");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t N = w->n_agents;
  if (N == 0) return 0;
  const Scratch sc = carve(w, io->scratch, nullptr);
  if (p->reset_scatter && w->n_groups > 0) {   // an unused look-ahead left its transmissions in the accumulators
    if (batch) return bad("batch: reset_scatter is not supported (no look-ahead in batched steps)");
    cudaMemsetAsync(sc.sct_acc, 0, sizeof(unsigned long long) * (size_t)w->n_groups, st);
    cudaMemsetAsync(sc.sct_dirty, 0, (size_t)w->n_groups, st);
  }
  Channels ch;
  Plan pl;
  if (int e = build_channels(w, p, &ch, &pl)) return e;
  gj_step_params pp = *p;
  if (p->mode == GJ_MODE_SEED) {
    pp.phases &= ~GJ_PHASE_NETWORKS;
    if (!io->seed_fraction) return bad("seed_fraction is NULL");
    if (io->seed_label && (io->n_seed_labels < 1 || io->n_seed_labels > (1 << 30)))
      return bad("n_seed_labels must lie in [1, 2^30]");
  }
  const bool seed_by = p->mode == GJ_MODE_SEED && io->seed_label != nullptr;
  if (p->mode == GJ_MODE_SEED && pp.phases == (GJ_PHASE_SAMPLE | GJ_PHASE_INFECT | GJ_PHASE_SYMPTOMS) &&
      !p->exact_order && !io->inj_E && !io->inj_u && !io->inj_z && io->s && io->inf && io->tinf && io->cur && io->nxt &&
      io->ttn && io->tape_y0 && io->stage_prob && io->s_o && io->inf_o && io->tinf_o && io->cur_o && io->nxt_o &&
      io->ttn_o) {   // Runner.set_initial_cases with in-kernel noise: the throughput-mode seeding kernel
    ProfScope ps(K_SEED, st);
    static OccCache occ[4];
    const bool diag = io->n != nullptr;
    int64_t g = (N + (int64_t)kLeanThreads * kLeanBatch - 1) / ((int64_t)kLeanThreads * kLeanBatch);
    gj_world_desc wt = *w;
    wt.n_tiles = g;   // lean_grid clips the persistent grid to the work available
#define GJ_SEED(K, C, D, L, I) \
  launch_pdl(K<D, L>, dim3(lean_grid(&wt, K<D, L>, &C[I])), dim3(kLeanThreads), 0, st, *w, pp, *io, sc.red_part, \
             sc.tickets)
    if (io->seed_label) {   // seeding by label
      static OccCache occ_by[4];
      if (io->label) {
        if (diag) GJ_SEED(k_lean_seed_by, occ_by, true, true, 3);
        else GJ_SEED(k_lean_seed_by, occ_by, false, true, 2);
      } else {
        if (diag) GJ_SEED(k_lean_seed_by, occ_by, true, false, 1);
        else GJ_SEED(k_lean_seed_by, occ_by, false, false, 0);
      }
    } else if (io->label) {
      if (diag) GJ_SEED(k_lean_seed, occ, true, true, 3);
      else GJ_SEED(k_lean_seed, occ, false, true, 2);
    } else {
      if (diag) GJ_SEED(k_lean_seed, occ, true, false, 1);
      else GJ_SEED(k_lean_seed, occ, false, false, 0);
    }
#undef GJ_SEED
    GJ_CHECK_LAUNCH("k_lean_seed");
    return 0;
  }
  if (!(pp.phases & GJ_PHASE_NETWORKS)) {  // stand-alone sampler / infect / symptoms, seeding
    ProfScope ps(K_AGENT_FWD, st);
    if (seed_by) {
      if (io->label) k_agent_seed_forward<true><<<agent_grid(N), kBlock, 0, st>>>(*w, pp, *io, sc.red_part, sc.tickets);
      else k_agent_seed_forward<false><<<agent_grid(N), kBlock, 0, st>>>(*w, pp, *io, sc.red_part, sc.tickets);
    } else if (io->label) {
      k_agent_forward<true><<<agent_grid(N), kBlock, 0, st>>>(*w, pp, *io, sc.red_part, sc.tickets);
    } else {
      k_agent_forward<false><<<agent_grid(N), kBlock, 0, st>>>(*w, pp, *io, sc.red_part, sc.tickets);
    }
    GJ_CHECK_LAUNCH("k_agent_forward");
    return 0;
  }
  // ---- networks phase (fused step or stand-alone InfectionNetworks): tile kernels ----------------------
  if (w->n_tiles <= 0 || !w->tile_begin) return bad("world has no tiles");
  if (!io->beta || !io->S_scaled || !io->S_unscaled || !io->s || !io->tape_v) return bad("beta / S / state buffers are NULL");
  if (!io->T_in && (!io->T || !io->tinf || !io->inf || !io->maxinf || !io->shape || !io->rate || !io->shift || !io->k0))
    return bad("state / T buffers are NULL");
  if (p->n_quar > 0 && (!io->Tq || !io->cur)) return bad("Tq / cur are NULL with an active quarantine");
  if ((pp.phases & ~GJ_PHASE_NETWORKS) && (!io->inf || !io->tinf || !io->cur || !io->nxt || !io->ttn))
    return bad("state arrays are NULL");
  if (pl.n_lei > 0 && !io->leisure_prob) return bad("leisure_prob is NULL");
  {
    LeanPlan lp;
    const bool no_injection = !io->inj_E && !io->inj_u && !io->inj_z;
    if (no_injection && !io->T_in && !io->lam && io->prof4 && lean_plan(w, &pp, pl, &lp)) {
      if (!io->inf || !io->tinf || !io->cur || !io->nxt || !io->ttn || !io->T || !io->tape_y0 || !io->stage_prob ||
          !io->s_o || !io->inf_o || !io->tinf_o || !io->cur_o || !io->nxt_o || !io->ttn_o)
        return bad("fused step: state / tape arrays are NULL");
      // look-ahead: the following step must itself run on the throughput-mode kernels (it then honours t_ready)
      NextStep nx;
      bool have_next = false;
      if (next && !io->label && !io->region && lookahead_enabled() && io->T_next && next->mode == GJ_MODE_STEP && next->phases == GJ_PHASE_ALL &&
          (next->n_quar <= 0 || io->Tq_next)) {
        Channels chn;
        Plan pln;
        LeanPlan lpn;
        if (build_channels(w, next, &chn, &pln) == 0 && lean_plan(w, next, pln, &lpn)) {
          memset(&nx, 0, sizeof(nx));
          nx.on = 1;
          nx.now = next->now;
          nx.day_type = next->day_type;
          nx.n_quar = next->n_quar > 0 ? next->n_quar : 0;
          for (int i = 0; i < GJ_MAX_QUAR; ++i) nx.quar_thr[i] = next->quar_thr[i];
          nx.n_cell = lpn.n_cell;
          for (int j = 0; j < GJ_MAX_CHANNELS; ++j) nx.c_row[j] = lpn.c_row[j];
          nx.n_tc = lpn.n_tc;
          for (int j = 0; j < GJ_MAX_CHANNELS; ++j) nx.tc[j] = lpn.tc[j];
          nx.has_generic = lpn.has_generic;
          nx.T = io->T_next;
          nx.Tq = nx.n_quar > 0 ? io->Tq_next : io->T_next;
          have_next = aligned16(io->T_next) && aligned16(io->Tq_next);
        }
      }
      if (batch) {
        if (io->S_scaled && batch->n_samples > 1 && batch->group_stride < lp.gen_base + w->n_groups)
          return bad("batch: group_stride smaller than the group-sum buffers");
        if (p->t_ready) return bad("batch: t_ready (look-ahead) is not supported");
        return lean_forward(w, &pp, pl, lp, io, sc, st, nullptr, bt);
      }
      return lean_forward(w, &pp, pl, lp, io, sc, st, have_next ? &nx : nullptr);
    }
  }
  if (batch) return bad("batch: this step does not run on the throughput-mode kernels (gj_step_plan = 0, injected noise, or no packed profile)");
  const int grid = (int)w->n_tiles;
  if (pp.stage != GJ_STAGE_REST) {
    {
      ProfScope ps(K_TRANSMISSION, st);
      k_tile_transmission<<<grid, kBlock, 0, st>>>(*w, pp, pl, *io, sc.tile_part);
      GJ_CHECK_LAUNCH("k_tile_transmission");
    }
    const float* T = io->T_in ? io->T_in : io->T;
    const float* Tq = (p->n_quar > 0) ? io->Tq : T;
    const Venue v{io->venue_region, io->venue_factor, io->n_venue_regions};
    if (pl.n_generic > 0)
      if (int e = launch_group_pass<false>(w, &pp, ch, io->beta, io->leisure_prob, T, Tq, io->S_scaled, io->S_unscaled,
                                           sc, st, v))
        return e;
    if (int e = launch_cell_groups(w, &pp, pl, io->beta, io->S_scaled, io->S_unscaled, sc, st, kNoBatch, v)) return e;
  }
  if (pp.stage == GJ_STAGE_SUMS) return 0;
  if (int e = launch_cell_gather(w, &pp, pl, io->S_scaled, sc, st)) return e;
  {
    ProfScope ps(K_AGENT_FWD, st);
    if (io->region && io->label)
      k_tile_forward_region<true><<<grid, kBlock, 0, st>>>(*w, pp, pl, *io, sc.cell_buf, sc.red_part, sc.tickets);
    else if (io->region)
      k_tile_forward_region<false><<<grid, kBlock, 0, st>>>(*w, pp, pl, *io, sc.cell_buf, sc.red_part, sc.tickets);
    else if (io->label) k_tile_forward<true><<<grid, kBlock, 0, st>>>(*w, pp, pl, *io, sc.cell_buf, sc.red_part, sc.tickets);
    else k_tile_forward<false><<<grid, kBlock, 0, st>>>(*w, pp, pl, *io, sc.cell_buf, sc.red_part, sc.tickets);
    GJ_CHECK_LAUNCH("k_tile_forward");
  }
  return 0;
}

int gj_step_forward(const gj_world_desc* w, const gj_step_params* p, const gj_fwd_io* io, void* stream) {
  const int rc = step_forward_impl(w, p, nullptr, io, stream);
  return rc > 0 ? 0 : rc;
}

int gj_step_forward_next(const gj_world_desc* w, const gj_step_params* p, const gj_step_params* next,
                         const gj_fwd_io* io, void* stream) {
  if (!next) return bad("next params is NULL");
  return step_forward_impl(w, p, next, io, stream);
}

int gj_step_forward_batch(const gj_world_desc* w, const gj_step_params* p, const gj_fwd_io* io, const gj_batch* batch,
                          void* stream) {
  if (!batch) return bad("batch is NULL");
  const int rc = step_forward_impl(w, p, nullptr, io, stream, batch);
  return rc > 0 ? 0 : rc;
}

static int seed_backward(const gj_world_desc* w, const gj_step_params& pp, const gj_bwd_io* io, const Scratch& sc,
                         cudaStream_t st) {
  if (io->n_seed_labels < 1 || io->n_seed_labels > (1 << 30)) return bad("n_seed_labels must lie in [1, 2^30]");
  if (!io->seed_order || !io->seed_offsets || !io->seed_work) return bad("seed_label given without seed_order / seed_offsets / seed_work");
  const int64_t N = w->n_agents;
  {
    ProfScope ps(K_AGENT_BWD, st);
    if (io->label && io->g_red_label)
      k_agent_seed_backward<true><<<agent_grid(N), kBlock, 0, st>>>(*w, pp, *io, sc.red_part, sc.tickets);
    else k_agent_seed_backward<false><<<agent_grid(N), kBlock, 0, st>>>(*w, pp, *io, sc.red_part, sc.tickets);
    GJ_CHECK_LAUNCH("k_agent_seed_backward");
  }
  if (!io->g_seed_fraction) return 0;
  ProfScope ps(K_SEED_GRAD, st);
  return label_sums(w, w->n_agents, io->seed_order, io->seed_offsets, io->n_seed_labels, io->seed_work, sc,
                    io->g_seed_fraction, st);
}

// regional transmission factor, backward: the agent kernels wrote d/dlam' * lam to region_work; the same per-label
// reduction as seeding by label sums it per region, once per sample (after the agent pass, so sample 0's reduction
// partials are free).  With a partitioned world it runs in the second stage, after every agent has written its term.
static int region_backward(const gj_world_desc* w, const gj_bwd_io* io, const Scratch& sc, const Batch& bt,
                           cudaStream_t st) {
  if (!io->region || !io->g_region_factor) return 0;
  ProfScope ps(K_REGION_GRAD, st);
  for (int s = 0; s < bt.nb; ++s)
    if (int e = label_sums(w, w->n_agents, io->region_order, io->region_offsets, io->n_regions,
                           io->region_work + (int64_t)s * bt.sN, sc, io->g_region_factor + (int64_t)s * bt.sReg, st))
      return e;
  return 0;
}

static int step_backward_impl(const gj_world_desc* w, const gj_step_params* p, const gj_bwd_io* io, void* stream,
                              const gj_batch* batch) {
  if (int e = check_world(w)) return e;
  if (!p || !io) return bad("params/io is NULL");
  if (!io->scratch) return bad("scratch is NULL");
  Batch bt = kNoBatch;
  if (batch)
    if (int e = make_batch(w, p, batch, &bt)) return e;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t N = w->n_agents;
  if (N == 0) return 0;
  const Scratch sc = carve(w, io->scratch, nullptr);
  Channels ch;
  Plan pl;
  if (int e = build_channels(w, p, &ch, &pl)) return e;
  gj_step_params pp = *p;
  if (p->mode == GJ_MODE_SEED) pp.phases &= ~GJ_PHASE_NETWORKS;
  if ((pp.phases & GJ_PHASE_SAMPLE) && !io->tape_y0) return bad("tape_y0 is NULL");
  if (!(pp.phases & GJ_PHASE_NETWORKS)) {
    if (p->mode == GJ_MODE_SEED && io->seed_label) return seed_backward(w, pp, io, sc, st);
    ProfScope ps(K_AGENT_BWD, st);
    if (io->label && io->g_red_label)
      k_agent_backward<true><<<agent_grid(N), kBlock, 0, st>>>(*w, pp, *io, sc.red_part, sc.tickets);
    else k_agent_backward<false><<<agent_grid(N), kBlock, 0, st>>>(*w, pp, *io, sc.red_part, sc.tickets);
    GJ_CHECK_LAUNCH("k_agent_backward");
    return 0;
  }
  if (w->n_tiles <= 0 || !w->tile_begin) return bad("world has no tiles");
  if (!io->w || !io->wq || !io->R || !io->cR || !io->tape_v || !io->S_unscaled || !io->beta || !io->s || !io->T_in)
    return bad("backward workspaces are NULL");
  if (p->n_quar > 0 && !io->cur) return bad("cur is NULL with an active quarantine");
  if (int e = check_region(io->region, io->n_regions, io->region_factor, bt)) return e;
  if (io->region && !io->region_work) return bad("region given without region_work");
  if (io->region && io->g_region_factor && (!io->region_order || !io->region_offsets))
    return bad("g_region_factor given without region_order / region_offsets");
  if (int e = check_venue(p, io->venue_region, io->n_venue_regions, io->venue_factor, bt)) return e;
  if (io->venue_region && io->g_venue_factor && (!io->venue_order || !io->venue_offsets || !io->venue_work || !io->g_beta))
    return bad("g_venue_factor given without venue_order / venue_offsets / venue_work / g_beta");
  const bool region_last = io->region && pp.stage != GJ_STAGE_SUMS;   // the per-region reduction ends the call
  if (!io->g_T && (!io->tinf || !io->inf || !io->maxinf || !io->k0 || !io->g_inf || !io->g_tinf))
    return bad("state arrays are NULL");
  {
    LeanPlan lp;
    const bool no_injection = !io->inj_E && !io->inj_u && !io->inj_z;
    if (no_injection && !io->g_T && !io->g_lam && !io->g_q && !io->g_n && io->prof4 && lean_plan(w, &pp, pl, &lp)) {
      if (!io->tinf || !io->inf || !io->cur || !io->nxt || !io->ttn || !io->tape_y0 || !io->stage_prob || !io->g_inf ||
          !io->g_tinf)
        return bad("fused step backward: state / tape arrays are NULL");
      if (batch && batch->n_samples > 1 && batch->group_stride < lp.gen_base + w->n_groups)
        return bad("batch: group_stride smaller than the group-sum buffers");
      if (int e = lean_backward(w, &pp, pl, lp, io, sc, st, bt)) return e;
      return region_last ? region_backward(w, io, sc, bt, st) : 0;
    }
  }
  if (batch) return bad("batch: this step does not run on the throughput-mode kernels (gj_step_plan = 0, injected noise, or no packed profile)");
  const int grid = (int)w->n_tiles;
  if (pp.stage != GJ_STAGE_REST) {
    {
      ProfScope ps(K_AGENT_BWD, st);
      const bool lab = io->label && io->g_red_label;
      if (io->region && lab) k_tile_backward_region<true><<<grid, kBlock, 0, st>>>(*w, pp, pl, *io, sc.tile_part);
      else if (io->region) k_tile_backward_region<false><<<grid, kBlock, 0, st>>>(*w, pp, pl, *io, sc.tile_part);
      else if (lab) k_tile_backward<true><<<grid, kBlock, 0, st>>>(*w, pp, pl, *io, sc.tile_part);
      else k_tile_backward<false><<<grid, kBlock, 0, st>>>(*w, pp, pl, *io, sc.tile_part);
      GJ_CHECK_LAUNCH("k_tile_backward");
    }
    const Venue v{io->venue_region, io->venue_factor, io->n_venue_regions};
    if (pl.n_generic > 0)
      if (int e = launch_group_pass<true>(w, &pp, ch, io->beta, io->leisure_prob, io->w, io->wq, io->cR, io->R, sc, st,
                                          v))
        return e;
    if (int e = launch_cell_groups(w, &pp, pl, io->beta, io->cR, io->R, sc, st, kNoBatch, v)) return e;
  }
  if (pp.stage == GJ_STAGE_SUMS) return 0;
  if (int e = launch_cell_gather(w, &pp, pl, io->cR, sc, st)) return e;
  {
    ProfScope ps(K_AGENT_BWD_GATHER, st);
    k_tile_backward_gather<<<grid, kBlock, 0, st>>>(*w, pp, pl, *io, sc.cell_buf, sc.dbeta_tile);
    GJ_CHECK_LAUNCH("k_tile_backward_gather");
  }
  if (io->g_beta && pp.n_nets > 0) {
    ProfScope ps(K_DBETA, st);
    DbetaPlan dp;
    for (int k = 0; k < GJ_MAX_NETS; ++k) dp.soff[k] = k < pp.n_nets ? pp.nets[k].s_off : 0;
    dp.n_range_parts = w->n_tiles;
    dim3 grid2(kRedBlocks / 8, pp.n_nets);
    if (io->venue_region)
      k_dbeta_venue<<<grid2, kBlock, 0, st>>>(*w, pp, pl, dp, io->S_unscaled, io->R, sc.dbeta_tile, sc.dbeta_part,
                                              sc.tickets, io->g_beta, kNoBatch, io->beta,
                                              Venue{io->venue_region, io->venue_factor, io->n_venue_regions},
                                              io->g_venue_factor ? io->venue_work : nullptr);
    else
      k_dbeta<<<grid2, kBlock, 0, st>>>(*w, pp, pl, dp, io->S_unscaled, io->R, sc.dbeta_tile, sc.dbeta_part,
                                        sc.tickets, io->g_beta, kNoBatch);
    GJ_CHECK_LAUNCH("k_dbeta");
    if (int e = venue_backward(w, &pp, pl, io, sc, kNoBatch, st)) return e;
  }
  return region_last ? region_backward(w, io, sc, bt, st) : 0;
}

int gj_step_backward(const gj_world_desc* w, const gj_step_params* p, const gj_bwd_io* io, void* stream) {
  return step_backward_impl(w, p, io, stream, nullptr);
}

int gj_step_backward_batch(const gj_world_desc* w, const gj_step_params* p, const gj_bwd_io* io, const gj_batch* batch,
                           void* stream) {
  if (!batch) return bad("batch is NULL");
  return step_backward_impl(w, p, io, stream, batch);
}

int gj_philox_fill_at(uint64_t seed, uint32_t call_index, uint64_t first_agent, int64_t n, float* E, float* u, float* z,
                      void* stream) {
  if (n <= 0) return 0;
  k_philox_fill<<<agent_grid(n), kBlock, 0, (cudaStream_t)stream>>>(seed, call_index, (int64_t)first_agent, n, E, u, z);
  GJ_CHECK_LAUNCH("k_philox_fill");
  return 0;
}

int gj_philox_fill(uint64_t seed, uint32_t call_index, int64_t n, float* E, float* u, float* z, void* stream) {
  return gj_philox_fill_at(seed, call_index, 0, n, E, u, z, stream);
}

int gj_step_plan(const gj_world_desc* w, const gj_step_params* p, int64_t* out, int n) {
  if (int e = check_world(w)) return e;
  if (!p) return bad("params is NULL");
  Channels ch;
  Plan pl;
  if (int e = build_channels(w, p, &ch, &pl)) return e;
  LeanPlan lp;
  const bool lean = lean_plan(w, p, pl, &lp);
  if (out && n > 0) out[0] = lean ? lp.gen_base : 0;
  return lean ? 1 : 0;
}

void gj_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
  philox4x32_10(ctr[0], ctr[1], ctr[2], ctr[3], key[0], key[1], out);
}

void gj_philox2x32_10(const uint32_t ctr[2], uint32_t key, uint32_t out[2]) { philox2x32_10(ctr[0], ctr[1], key, out); }

}  // extern "C"
