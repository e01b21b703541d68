// Tile-based kernels of the fused step (included by gj_kernels.cu).
//
// One CTA owns one tile of <= GJ_TILE_AGENTS consecutive agents (never straddling a cell of a CELL-tier
// edge type).  Per network the pressure on an agent comes from the layout tier of its edge type:
//   RANGE   the group is a contiguous run of agents -> each agent re-sums its few neighbours' T (L1 hits),
//           no group buffer, no group-major pass (households);
//   CELL    every agent of the tile attends the same groups -> agents -> tile partial sums -> cell sums ->
//           group sums -> one per-cell value broadcast from shared memory (leisure);
//   GENERIC CSR gather of per-group sums produced by the group-major segmented-sum kernels.
// All sums have a fixed order (tile -> cell -> group; shuffle trees inside a CTA): bit-reproducible.
#pragma once
#include "gj_device.cuh"

namespace gj {

constexpr uint32_t kNoSlot = 0xFFFFFFFFu;

struct Plan {
  int n_t2;                         // networks on CELL-tier types ("cell channels"), in network order
  int t2_net[GJ_MAX_CHANNELS];
  int net_t2[GJ_MAX_NETS];
  int n_t1;                         // networks on RANGE-tier types
  int t1_net[GJ_MAX_RANGE_NETS];
  int net_t1[GJ_MAX_NETS];
  int n_lei;                        // networks with an attendance table (LEISURE / CARE_VISIT)
  int lei_net[GJ_MAX_CHANNELS];
  int net_lei[GJ_MAX_NETS];
  int n_generic;                    // networks on GENERIC types
  int tier[GJ_MAX_NETS];            // layout tier of each network's edge type
  const uint32_t* slot[GJ_MAX_NETS];  // RANGE networks: the type's per-agent (offset, size) words
  const float* rpc[GJ_MAX_NETS];      //                 and per-agent contact probability
};

// ---- batched ensemble (gj_step_forward_batch / gj_step_backward_batch) ------------------------------------------
// b independent samples on one world: sample s of a batched launch reads and writes every per-sample array at a fixed
// stride behind sample 0's (gj_batch).  Persistent and 1-D kernels interleave the samples in the block index
// (block = unit * nb + sample), so the CTAs that walk the same agent tiles / group lists run next to each other and
// share the world's index data through L2; kernels with a 2-D grid take the sample from blockIdx.z.
struct Batch {
  int nb;          // samples
  uint32_t sN;     // stride of the per-agent arrays (elements; nb * sN < 2^32)
  int64_t sG;      // stride of the group-sum buffers (elements)
  int64_t sScr;    // stride of the scratch buffers (bytes, multiple of 256)
  int sBeta, sRed; // strides of beta / g_beta and red / g_red (elements)
  const float* noise;  // [n_agents] the draw's Gumbel noise difference, evaluated once for all samples; NULL = in-kernel
  int64_t sLab;        // stride of red_label / g_red_label / label_acc (elements)
};
struct BatchCta {
  int s;           // sample of this CTA
  uint32_t bx, gx; // its block index among the sample's CTAs, and how many those are
  uint32_t so;     // s * sN: added to agent indices of per-sample arrays
};
template <bool kBatch>
__device__ __forceinline__ BatchCta batch_cta(const Batch& bt) {
  BatchCta c;
  if (kBatch) {
    c.s = (int)(blockIdx.x % (uint32_t)bt.nb);
    c.bx = blockIdx.x / (uint32_t)bt.nb;
    c.gx = gridDim.x / (uint32_t)bt.nb;
    c.so = (uint32_t)c.s * bt.sN;
  } else {
    c.s = 0;
    c.bx = blockIdx.x;
    c.gx = gridDim.x;
    c.so = 0u;
  }
  return c;
}
template <typename T>
__device__ __forceinline__ T* scr_shift(T* p, const Batch& bt, int s) {
  return reinterpret_cast<T*>(reinterpret_cast<char*>(p) + (int64_t)s * bt.sScr);
}
template <typename T>
__device__ __forceinline__ const T* scr_shift(const T* p, const Batch& bt, int s) {
  return reinterpret_cast<const T*>(reinterpret_cast<const char*>(p) + (int64_t)s * bt.sScr);
}

// ---- shared-memory tables ---------------------------------------------------------------------------
struct TileTables {
  float prob[GJ_MAX_CHANNELS][200];  // attendance probability by (sex, age) class for today's day type
  float beta[GJ_MAX_NETS];
  float cellv[GJ_MAX_CHANNELS];      // per cell-channel value of this tile's cell
};

__device__ __forceinline__ void load_tables(TileTables& tb, const gj_step_params& p, const Plan& pl,
                                            const float* __restrict__ lprob, const float* __restrict__ beta) {
  for (int i = threadIdx.x; i < pl.n_lei * 200; i += blockDim.x) {
    const int j = i / 200, c = i - j * 200;
    tb.prob[j][c] = lprob[(size_t)(p.nets[pl.lei_net[j]].prob_row * 2 + p.day_type) * 200 + c];
  }
  if (threadIdx.x < p.n_nets) tb.beta[threadIdx.x] = beta ? beta[threadIdx.x] : 0.0f;
}

__device__ __forceinline__ void load_cell_values(TileTables& tb, const gj_world_desc& w, const gj_step_params& p,
                                                 const Plan& pl, const float* __restrict__ cell_buf, int64_t tile) {
  if (threadIdx.x < pl.n_t2) {
    const int t = p.nets[pl.t2_net[threadIdx.x]].type;
    const uint32_t cell = w.tile_cell[t][tile];
    tb.cellv[threadIdx.x] = cell_buf[(w.cell_off[t] + cell) * GJ_MAX_CHANNELS + threadIdx.x];
  }
}

// value an agent contributes to a group sum of network `net` (forward: from T / Tq; backward: from w / wq)
__device__ __forceinline__ float member_value(const TileTables& tb, const Plan& pl, int k, int kind, float v0, float v1,
                                              int cls) {
  if (kind == GJ_KIND_HOUSEHOLD) return v0;
  if (kind == GJ_KIND_PLAIN) return v1;
  return tb.prob[pl.net_lei[k]][cls] * v1;
}

// block-wide sums of up to kR values; result valid in threads [0, nr) of warp 0 ... written by the caller's lambda
template <typename T, int kR, int kWarps = kBlock / 32>
__device__ __forceinline__ void block_sums(T (&v)[kR], int nr, T* __restrict__ out /* [nr] global */) {
  __shared__ T sm[kWarps][kR];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int r = 0; r < kR; ++r)
    if (r < nr) v[r] = warp_sum(v[r]);
  if (lane == 0) {
#pragma unroll
    for (int r = 0; r < kR; ++r)
      if (r < nr) sm[wid][r] = v[r];
  }
  __syncthreads();
  if (threadIdx.x < nr) {
    T s = (T)0;
#pragma unroll
    for (int k = 0; k < kWarps; ++k) s += sm[k][threadIdx.x];
    out[threadIdx.x] = s;
  }
  __syncthreads();
}

// the last CTA to finish adds the per-CTA partials in a fixed order (strided per thread, then a tree)
template <int kR>
__device__ __forceinline__ void finish_partials(int nr, const double* __restrict__ partials, int64_t n_part,
                                                unsigned int* __restrict__ ticket, float* __restrict__ out) {
  // n_part = number of CTAs taking a ticket (the whole grid, or one sample's CTAs of a batched launch)
  __shared__ bool last;
  __shared__ double sm[32];
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = (atomicAdd(ticket, 1u) == (unsigned int)n_part - 1u);
  __syncthreads();
  if (!last) return;
  __threadfence();
  for (int r = 0; r < nr; ++r) {
    double s = 0.0;
    for (int64_t b = threadIdx.x; b < n_part; b += blockDim.x) s += partials[b * kR + r];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
      double tsum = 0.0;
      for (int k = 0; k < (int)(blockDim.x / 32); ++k) tsum += sm[k];
      out[r] = (float)tsum;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) *ticket = 0u;
}

// =====================================================================================================
// K1'  transmissions + tile partial sums of the cell channels
// =====================================================================================================
__global__ void __launch_bounds__(kBlock) k_tile_transmission(gj_world_desc w, gj_step_params p, Plan pl, gj_fwd_io io,
                                                              float* __restrict__ tile_part) {
  __shared__ TileTables tb;
  const int64_t tile = blockIdx.x;
  const uint32_t a0 = w.tile_begin[tile], a1 = w.tile_begin[tile + 1];
  if (pl.n_t2 > 0) load_tables(tb, p, pl, io.leisure_prob, nullptr);
  __syncthreads();
  float acc[GJ_MAX_CHANNELS];
#pragma unroll
  for (int j = 0; j < GJ_MAX_CHANNELS; ++j) acc[j] = 0.0f;
  const bool quar = p.n_quar > 0;
  for (uint32_t a = a0 + threadIdx.x; a < a1; a += kBlock) {
    float T = 0.0f;
    if (io.T_in) {  // stand-alone InfectionNetworks: transmissions are given
      T = io.T_in[a];
    } else {
      const float inf = io.inf[a];
      if (inf != 0.0f) {  // never-infected agents transmit nothing: skip their profile (most of the world early on)
        const TransTerms tt =
            transmission_terms<false>(p.now, io.tinf[a], io.maxinf[a], io.shape[a], io.rate[a], io.shift[a], io.k0[a]);
        T = tt.coef * inf;
      }
      io.T[a] = T;
    }
    float Tq = T;
    if (quar) {
      Tq = quarantine_mask(p, io.cur[a]) * T;
      io.Tq[a] = Tq;
    }
    if (pl.n_t2 > 0 && T != 0.0f) {
      const int cls = w.cls[a];
#pragma unroll
      for (int j = 0; j < GJ_MAX_CHANNELS; ++j)
        if (j < pl.n_t2) acc[j] += member_value(tb, pl, pl.t2_net[j], p.nets[pl.t2_net[j]].kind, T, Tq, cls);
    }
  }
  if (pl.n_t2 > 0) block_sums<float, GJ_MAX_CHANNELS>(acc, pl.n_t2, tile_part + tile * GJ_MAX_CHANNELS);
}

// =====================================================================================================
// cell tier: tiles -> cells -> groups, and groups -> cells
// =====================================================================================================
// one thread per (cell channel, group): sum the tile partials of the group's cells in ascending order
__global__ void __launch_bounds__(kBlock) k_cell_groups(gj_world_desc w, gj_step_params p, Plan pl,
                                                        const float* __restrict__ beta,
                                                        const float* __restrict__ tile_part,
                                                        float* __restrict__ out_scaled, float* __restrict__ out_plain,
                                                        Batch bt) {
  pdl_launch();
  pdl_wait();
  if (bt.nb > 1) {   // batched ensemble: sample blockIdx.z
    const int s = blockIdx.z;
    beta += (int64_t)s * bt.sBeta;
    tile_part = scr_shift(tile_part, bt, s);
    out_scaled += (int64_t)s * bt.sG;
    out_plain += (int64_t)s * bt.sG;
  }
  const int j = blockIdx.y;
  const int k = pl.t2_net[j];
  const gj_net net = p.nets[k];
  const int t = net.type;
  const int64_t G = w.type_group_off[t + 1] - w.type_group_off[t];
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G) return;
  float sum = 0.0f;
  for (uint32_t ci = w.grp_cell_ptr[t][g]; ci < w.grp_cell_ptr[t][g + 1]; ++ci) {
    const uint32_t c = w.grp_cell[t][ci];
    for (uint32_t tl = w.cell_tile_ptr[t][c]; tl < w.cell_tile_ptr[t][c + 1]; ++tl)
      sum += tile_part[(int64_t)tl * GJ_MAX_CHANNELS + j];
  }
  const float cg = beta[k] * w.pc[w.type_group_off[t] + g];
  out_plain[(int64_t)net.s_off + g] = sum;
  out_scaled[(int64_t)net.s_off + g] = cg * sum;
}

// one thread per (cell channel, cell): sum over the cell's groups (agent edge order)
__global__ void __launch_bounds__(kBlock) k_cell_gather(gj_world_desc w, gj_step_params p, Plan pl,
                                                        const float* __restrict__ in_scaled,
                                                        float* __restrict__ cell_buf, Batch bt) {
  pdl_launch();
  pdl_wait();
  if (bt.nb > 1) {
    const int s = blockIdx.z;
    in_scaled += (int64_t)s * bt.sG;
    cell_buf = scr_shift(cell_buf, bt, s);
  }
  const int j = blockIdx.y;
  const gj_net net = p.nets[pl.t2_net[j]];
  const int t = net.type;
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= w.n_cells[t]) return;
  float sum = 0.0f;
  for (uint32_t gi = w.cell_grp_ptr[t][c]; gi < w.cell_grp_ptr[t][c + 1]; ++gi)
    sum += in_scaled[(int64_t)net.s_off + w.cell_grp[t][gi]];
  cell_buf[(w.cell_off[t] + c) * GJ_MAX_CHANNELS + j] = sum;
}

// =====================================================================================================
// shared per-agent tail of the forward step: sample -> infect -> symptoms -> outputs -> reductions
// =====================================================================================================
struct AgentState {
  float s, inf, tinf, cur, nxt, ttn;
};

// kLabel: also add the agent's cases and death indicator to its label's column of the integer accumulator lacc
// kSeed: seeding by label, the agent's fraction is seed_fraction[seed_label[a]]
template <bool kLabel = false, bool kSeed = false>
__device__ __forceinline__ void forward_tail(const gj_step_params& p, const gj_fwd_io& io, int64_t N, int64_t a,
                                             int64_t ga, int age, float q, AgentState st, float* red,
                                             uint32_t* lacc = nullptr) {
  const int dead = p.n_stages - 1;
  if (p.mode == GJ_MODE_SEED) q = 1.0f - io.seed_fraction[kSeed ? io.seed_label[a] : 0] * 1.0f;  // infection.py:36-40
  float n = 0.0f;
  StepNoise nz;
  nz.E0 = nz.E1 = 1.0f;
  nz.u = 0.0f;
  if (p.phases & (GJ_PHASE_SAMPLE | GJ_PHASE_SYMPTOMS)) {
    if (io.inj_E == nullptr || io.inj_u == nullptr) nz = draw_step_noise(p.seed, p.call_index, ga);
    if (io.inj_E) {
      nz.E0 = io.inj_E[a];
      nz.E1 = io.inj_E[N + a];
    }
    if (io.inj_u) nz.u = io.inj_u[a];
  }
  if (p.phases & GJ_PHASE_SAMPLE) {
    const Draw d = gumbel_draw(q, nz.E0, nz.E1, p.tau);
    n = d.n;
    if (io.tape_y0) io.tape_y0[a] = d.ty;
  } else if (io.n_in) {
    n = io.n_in[a];
  }
  if (io.n) io.n[a] = n;
  if (p.phases & GJ_PHASE_INFECT) {
    st.s = fmaxf(0.0f, st.s - n);  // maximum(0, s - n) and clamp(s - n, min=0) agree in value
    st.inf = st.inf + n;
    st.tinf = st.tinf + n * (p.now - st.tinf);
    if (io.s_o) io.s_o[a] = st.s;
    if (io.inf_o) io.inf_o[a] = st.inf;
    if (io.tinf_o) io.tinf_o[a] = st.tinf;
  }
  if (p.phases & GJ_PHASE_SYMPTOMS) {
    const float* inj_z = io.inj_z;
    const uint64_t seed = p.seed;
    const uint32_t call = p.call_index;
    const float uu = nz.u;
    const SympOut so = symptoms_forward(p, io.stage_prob, st.cur, st.nxt, st.ttn, n, age, [&]() { return uu; },
                                        [&](int row) {
      return inj_z ? inj_z[(int64_t)row * N + a] : draw_step_normal(seed, call, ga);
    });
    st.cur = so.cur;
    st.nxt = so.nxt;
    st.ttn = so.ttn;
    if (io.cur_o) io.cur_o[a] = st.cur;
    if (io.nxt_o) io.nxt_o[a] = st.nxt;
    if (io.ttn_o) io.ttn_o[a] = st.ttn;
  }
  if (io.red) {  // runner.py:167-171,198-224 ; per-thread partial sums of small integers: exact in fp32
    red[0] += st.inf;
    red[1] += (st.cur == (float)dead) ? (st.cur / (float)dead) : 0.0f;
#pragma unroll
    for (int b = 0; b < GJ_MAX_AGE_BINS; ++b)
      if (b < p.n_age_bins && age > p.age_bins[b] && age < p.age_bins[b + 1]) red[2 + b] += st.inf;
  }
  if (kLabel) label_add(lacc, io.label, a, (uint32_t)st.inf, st.cur == (float)dead ? 1u : 0u);
}

struct NetMask {
  float mS;     // mask on the susceptible side (without s)
  float mT;     // mask on the transmitting side
  float age_f;  // care-visit (age > 75) factor on the susceptible side
};

__device__ __forceinline__ NetMask tile_net_mask(const TileTables& tb, const Plan& pl, int k, int kind, float mq,
                                                 int cls) {
  NetMask m;
  m.age_f = 1.0f;
  if (kind == GJ_KIND_HOUSEHOLD) {
    m.mS = m.mT = 1.0f;
  } else if (kind == GJ_KIND_PLAIN) {
    m.mS = m.mT = mq;
  } else {
    m.mS = m.mT = mq * tb.prob[pl.net_lei[k]][cls];
    if (kind == GJ_KIND_CARE_VISIT) m.age_f = ((cls % 100) > 75) ? 1.0f : 0.0f;
  }
  return m;
}

// =====================================================================================================
// F3'  forward: pressure from the three tiers -> q -> draw -> update -> symptoms -> reductions
// =====================================================================================================
// pressure of all active networks on agent `a` in the reference's accumulation order; the network loop is
// fully unrolled so that every per-network parameter is a compile-time slot of the constant bank
struct Pressure {
  float lam, X;
};

__device__ __forceinline__ Pressure agent_pressure(const gj_world_desc& w, const gj_step_params& p, const Plan& pl,
                                                   const TileTables& tb, const float* __restrict__ S_scaled,
                                                   const float* __restrict__ Tsrc, const float* __restrict__ Tq,
                                                   uint32_t a, int cls, float s, float mq) {
  uint32_t e0 = 0, deg = 0, ent0 = 0, ent1 = 0;
  if (pl.n_generic > 0) {
    e0 = w.am_ptr[a];
    deg = w.am_ptr[a + 1] - e0;
    if (deg > 0) ent0 = w.am_ent[e0];
    if (deg > 1) ent1 = w.am_ent[e0 + 1];
  }
  const float age_f = ((cls % 100) > 75) ? 1.0f : 0.0f;
  Pressure out;
  out.lam = 0.0f;
  out.X = 0.0f;
#pragma unroll
  for (int k = 0; k < GJ_MAX_NETS; ++k) {
    if (k < p.n_nets) {
      const int kind = p.nets[k].kind;
      const int type = p.nets[k].type;
      const int tier = pl.tier[k];
      float mS = (kind == GJ_KIND_HOUSEHOLD) ? 1.0f : mq;
      if (kind >= GJ_KIND_LEISURE) mS = mq * tb.prob[pl.net_lei[k]][cls];
      float sp = mS * s, sx = mS;  // susceptibilities = mask * [leisure_mask *] susceptibility
      if (kind == GJ_KIND_CARE_VISIT) {
        sp = sp * age_f;
        sx = sx * age_f;
      }
      float Pk = 0.0f, PXk = 0.0f;
      if (tier == GJ_TIER_RANGE) {
        const uint32_t slot = pl.slot[k][a];
        if (slot != kNoSlot) {
          const uint32_t b0 = a - (slot >> 16), nb = slot & 0xFFFFu;
          const float cg = tb.beta[k] * pl.rpc[k][a];
          float Sg = 0.0f;
          for (uint32_t b = b0; b < b0 + nb; ++b) {  // members in id order = the reference's edge order
            const float v = member_value(tb, pl, k, kind, Tsrc[b], Tq[b], kind >= GJ_KIND_LEISURE ? w.cls[b] : 0);
            Sg += v * cg;
          }
          Pk = Sg * sp;
          PXk = Sg * sx;
        }
      } else if (tier == GJ_TIER_CELL) {
        const float B = tb.cellv[pl.net_t2[k]];
        Pk = B * sp;
        PXk = B * sx;
      } else {
        const int64_t so = p.nets[k].s_off;
        if (deg > 0 && (int)(ent0 >> 28) == type) {
          const float Sg = S_scaled[so + (ent0 & 0x0FFFFFFFu)];
          Pk += Sg * sp;  // message = cumulative_trans * susceptibility   base.py:80-87
          PXk += Sg * sx;
        }
        if (deg > 1 && (int)(ent1 >> 28) == type) {
          const float Sg = S_scaled[so + (ent1 & 0x0FFFFFFFu)];
          Pk += Sg * sp;
          PXk += Sg * sx;
        }
        for (uint32_t j = 2; j < deg; ++j) {
          const uint32_t ent = w.am_ent[e0 + j];
          if ((int)(ent >> 28) == type) {
            const float Sg = S_scaled[so + (ent & 0x0FFFFFFFu)];
            Pk += Sg * sp;
            PXk += Sg * sx;
          }
        }
      }
      out.lam += Pk;  // trans_susc += network(...)   base.py:133-135
      out.X += PXk;
    }
  }
  return out;
}

template <bool kLabel>
__global__ void __launch_bounds__(kBlock, 4) k_tile_forward(gj_world_desc w, gj_step_params p, Plan pl, gj_fwd_io io,
                                                            const float* __restrict__ cell_buf,
                                                            double* __restrict__ red_part,
                                                            unsigned int* __restrict__ ticket) {
  __shared__ TileTables tb;
  const int64_t N = w.n_agents;
  const int64_t tile = blockIdx.x;
  const uint32_t a0 = w.tile_begin[tile], a1 = w.tile_begin[tile + 1];
  load_tables(tb, p, pl, io.leisure_prob, io.beta);
  load_cell_values(tb, w, p, pl, cell_buf, tile);
  __syncthreads();
  float red[kMaxRed];
#pragma unroll
  for (int r = 0; r < kMaxRed; ++r) red[r] = 0.0f;
  const float* __restrict__ Tsrc = io.T_in ? io.T_in : io.T;
  const float* __restrict__ Tq = (p.n_quar > 0) ? io.Tq : Tsrc;

  for (uint32_t a = a0 + threadIdx.x; a < a1; a += kBlock) {
    const int cls = w.cls[a];
    AgentState st;
    st.s = io.s[a];
    st.inf = io.inf ? io.inf[a] : 0.0f;
    st.tinf = io.tinf ? io.tinf[a] : 0.0f;
    st.cur = io.cur ? io.cur[a] : 1.0f;
    st.nxt = io.nxt ? io.nxt[a] : 1.0f;
    st.ttn = io.ttn ? io.ttn[a] : 0.0f;
    const float mq = (p.n_quar > 0) ? quarantine_mask(p, st.cur) : 1.0f;
    const Pressure pr = agent_pressure(w, p, pl, tb, io.S_scaled, Tsrc, Tq, a, cls, st.s, mq);
    const float q = not_infected_prob(pr.lam, p.dt);
    io.tape_v[a] = (st.s == 0.0f) ? pr.X : pr.lam;
    if (io.q) io.q[a] = q;
    if (io.lam) io.lam[a] = pr.lam;
    forward_tail<kLabel>(p, io, N, a, noise_agent(w, p, a), cls % 100, q, st, red, io.label_acc);
  }
  if (io.red) {
    double redd[kMaxRed];
#pragma unroll
    for (int r = 0; r < kMaxRed; ++r) redd[r] = (double)red[r];
    block_sums<double, kMaxRed>(redd, 2 + p.n_age_bins, red_part + tile * kMaxRed);
    finish_partials<kMaxRed>(2 + p.n_age_bins, red_part, gridDim.x, ticket, io.red);
  }
}

// =====================================================================================================
// B1'  backward part 1 (per agent), plus tile partial sums of the cell channels
// =====================================================================================================
struct BackAgent {
  float gs, ginf, gtinf, gcur, gnxt, gttn;  // cotangents of the pre-step state (pressure part of gs included)
  float glam;                               // cotangent of the unclamped pressure
  float gq, gn;
};

// symptoms^T, infect^T, sampler^T and the clamp/exp chain: shared by the generic and the tiled kernels
// kLabel: fold in the cotangent of the forward's label table (gj_bwd_io.g_red_label) at the agent's label
// kSeed: seeding by label, the agent's fraction is seed_fraction[seed_label[a]]
template <bool kLabel = false, bool kSeed = false>
__device__ __forceinline__ BackAgent backward_agent(const gj_step_params& p, const gj_bwd_io& io, int64_t N, int64_t a,
                                                    int64_t ga, int age, const AgentState& st, bool with_networks) {
  const int dead = p.n_stages - 1;
  const bool seed_mode = p.mode == GJ_MODE_SEED;
  float n = 0.0f;
  if (io.inf_o) n = io.inf_o[a] - st.inf;  // exact: both are small integers
  else if (io.n_in) n = io.n_in[a];
  const float gs_o = io.g_s_o ? io.g_s_o[a] : 0.0f;
  float ginf_o = io.g_inf_o ? io.g_inf_o[a] : 0.0f;
  const float gtinf_o = io.g_tinf_o ? io.g_tinf_o[a] : 0.0f;
  float gcur_o = io.g_cur_o ? io.g_cur_o[a] : 0.0f;
  const float gnxt_o = io.g_nxt_o ? io.g_nxt_o[a] : 0.0f;
  const float gttn_o = io.g_ttn_o ? io.g_ttn_o[a] : 0.0f;
  float glab_i = 0.0f, glab_d = 0.0f;   // label table: cases and deaths cotangents of the agent's column
  if (kLabel) {
    const int64_t l = io.label[a];
    glab_i = io.g_red_label[2 * l];
    glab_d = io.g_red_label[2 * l + 1] / (float)dead;
  }
  BackAgent r;
  r.gn = io.g_n ? io.g_n[a] : 0.0f;
  r.gcur = gcur_o;
  r.gnxt = gnxt_o;
  r.gttn = gttn_o;
  if (p.phases & GJ_PHASE_SYMPTOMS) {
    const float* inj_u = io.inj_u;
    const float* inj_z = io.inj_z;
    const uint64_t seed = p.seed;
    const uint32_t call = p.call_index;
    // the uniform / normal draws are regenerated only for the few agents whose stage actually updates
    const SympOut so = symptoms_forward(p, io.stage_prob, st.cur, st.nxt, st.ttn, n, age,
                                        [&]() { return inj_u ? inj_u[a] : draw_step_uniform(seed, call, ga); },
                                        [&](int row) {
      return inj_z ? inj_z[(int64_t)row * N + a] : draw_step_normal(seed, call, ga);
    });
    // reductions fold in here: deaths = sum (cur' == dead) * cur' / dead   runner.py:204-209
    if (io.g_red && so.cur == (float)dead) gcur_o += io.g_red[1] / (float)dead;
    if (kLabel && so.cur == (float)dead) gcur_o += glab_d;
    float gcur1 = gcur_o;
    float gnxt1 = gnxt_o;
    const float gttn1 = gttn_o;
    if (so.branch == 1) {         // next += m ; ttn += dwell * m ; m = (cur==i)*cur/i * transition * symp
      gcur1 += (gnxt_o + gttn_o * so.dwell) / (float)so.stage;
    } else if (so.branch == 2) {  // next -= next * m ; ttn += dwell * m
      gcur1 += (gttn_o * so.dwell - gnxt_o * so.nxt1) / (float)so.stage;
      gnxt1 = 0.0f;               // d(next - next*m)/dnext = 1 - m = 0
    }
    r.gcur = gcur1 * (1.0f - so.tr);  // cur' = cur - (cur - next1) * transition
    gnxt1 += gcur1 * so.tr;
    r.gnxt = gnxt1 * (1.0f - n);      // next1 = next + n * (2 - next)
    r.gn += gnxt1 * (2.0f - st.nxt);
    r.gttn = gttn1 * (1.0f - n);      // ttn1 = ttn + n * (now - ttn)
    r.gn += gttn1 * (p.now - st.ttn);
  } else if (io.g_red && st.cur == (float)dead) {
    r.gcur += io.g_red[1] / (float)dead;
  }
  if (kLabel && !(p.phases & GJ_PHASE_SYMPTOMS) && st.cur == (float)dead) r.gcur += glab_d;
  r.gs = gs_o;
  r.ginf = ginf_o;
  r.gtinf = gtinf_o;
  if (io.g_red) {
    ginf_o += io.g_red[0];
    for (int b = 0; b < p.n_age_bins; ++b)
      if (age > p.age_bins[b] && age < p.age_bins[b + 1]) ginf_o += io.g_red[2 + b];
    r.ginf = ginf_o;
  }
  if (kLabel) {
    ginf_o += glab_i;
    r.ginf = ginf_o;
  }
  if (p.phases & GJ_PHASE_INFECT) {
    const float d = st.s - n;
    float wgt;
    if (seed_mode) wgt = (d >= 0.0f) ? 1.0f : 0.0f;              // clamp(min=0): gradient where x >= min
    else wgt = (d > 0.0f) ? 1.0f : ((d == 0.0f) ? 0.5f : 0.0f);  // maximum(0, x): ties split 1/2
    r.gs = gs_o * wgt;
    r.gn += -(gs_o * wgt) + ginf_o + gtinf_o * (p.now - st.tinf);
    r.ginf = ginf_o;
    r.gtinf = gtinf_o * (1.0f - n);
  }
  r.gq = io.g_q ? io.g_q[a] : 0.0f;
  float lam = 0.0f, q = 1.0f, v = 0.0f;
  if (with_networks) {
    v = io.tape_v[a];
    lam = (st.s == 0.0f) ? 0.0f : v;
    q = not_infected_prob(lam, p.dt);
  }
  if (seed_mode) q = 1.0f - io.seed_fraction[kSeed ? io.seed_label[a] : 0] * 1.0f;
  if (p.phases & GJ_PHASE_SAMPLE) {
    if (!with_networks && !seed_mode && io.q_in) q = io.q_in[a];  // stand-alone sampler
    float y0, y1;
    decode_soft(io.tape_y0[a], y0, y1);
    const float gret0 = -r.gn;                      // new_infected = 1 - ret[0]
    const float dot = gret0 * y0;                   // softmax^T: (g - sum(g*y)) * y with g = (gret0, 0)
    const float gx0 = (gret0 - dot) * y0;
    const float gx1 = (0.0f - dot) * y1;
    const float gl0 = gx0 / p.tau, gl1 = gx1 / p.tau;
    r.gq += gl0 / q - gl1 / (1.0f - q);             // logits = log([q, 1-q])
  }
  r.glam = 0.0f;
  if (with_networks) {
    // q = clamp(exp(-clamp(lam)*dt), 0, 1): clamp passes the gradient on its closed interval
    if (q >= 0.0f && q <= 1.0f) {
      const float glc = r.gq * q * (-p.dt);
      if (lam >= 1e-6f && lam <= 100.0f) r.glam = glc;
    }
    if (io.g_lam) r.glam += io.g_lam[a];
    const float X = (st.s == 0.0f) ? v : v / st.s;
    r.gs += r.glam * X;
  }
  return r;
}

template <bool kLabel>
__global__ void __launch_bounds__(kBlock, 3) k_tile_backward(gj_world_desc w, gj_step_params p, Plan pl, gj_bwd_io io,
                                                          float* __restrict__ tile_part) {
  __shared__ TileTables tb;
  const int64_t N = w.n_agents;
  const int64_t tile = blockIdx.x;
  const uint32_t a0 = w.tile_begin[tile], a1 = w.tile_begin[tile + 1];
  if (pl.n_t2 > 0) load_tables(tb, p, pl, io.leisure_prob, nullptr);
  __syncthreads();
  float acc[GJ_MAX_CHANNELS];
#pragma unroll
  for (int j = 0; j < GJ_MAX_CHANNELS; ++j) acc[j] = 0.0f;
  for (uint32_t a = a0 + threadIdx.x; a < a1; a += kBlock) {
    const int cls = w.cls[a];
    AgentState st;
    st.s = io.s[a];
    st.inf = io.inf ? io.inf[a] : 0.0f;
    st.tinf = io.tinf ? io.tinf[a] : 0.0f;
    st.cur = io.cur ? io.cur[a] : 1.0f;
    st.nxt = io.nxt ? io.nxt[a] : 1.0f;
    st.ttn = io.ttn ? io.ttn[a] : 0.0f;
    const BackAgent r = backward_agent<kLabel>(p, io, N, a, noise_agent(w, p, a), cls % 100, st, true);
    const float mq = (p.n_quar > 0) ? quarantine_mask(p, st.cur) : 1.0f;
    const float wv = r.glam * st.s;
    const float wqv = r.glam * (mq * st.s);
    io.w[a] = wv;
    if (io.wq != io.w) io.wq[a] = wqv;
    if (pl.n_t2 > 0 && r.glam != 0.0f) {
#pragma unroll
      for (int j = 0; j < GJ_MAX_CHANNELS; ++j) {
        if (j < pl.n_t2) {
          const int k = pl.t2_net[j];
          const int kind = p.nets[k].kind;
          float v = member_value(tb, pl, k, kind, wv, wqv, cls);
          if (kind == GJ_KIND_CARE_VISIT) v = v * (((cls % 100) > 75) ? 1.0f : 0.0f);
          acc[j] += v;
        }
      }
    }
    if (io.g_s) io.g_s[a] = r.gs;
    if (io.g_inf) io.g_inf[a] = r.ginf;
    if (io.g_tinf) io.g_tinf[a] = r.gtinf;
    if (io.g_cur) io.g_cur[a] = r.gcur;
    if (io.g_nxt) io.g_nxt[a] = r.gnxt;
    if (io.g_ttn) io.g_ttn[a] = r.gttn;
  }
  if (pl.n_t2 > 0) block_sums<float, GJ_MAX_CHANNELS>(acc, pl.n_t2, tile_part + tile * GJ_MAX_CHANNELS);
}

// =====================================================================================================
// B3'  backward part 2: dL/dT from the three tiers -> (is_infected, infection_time); d/dbeta of RANGE nets
// =====================================================================================================
__global__ void __launch_bounds__(kBlock, 4) k_tile_backward_gather(gj_world_desc w, gj_step_params p, Plan pl,
                                                                    gj_bwd_io io, const float* __restrict__ cell_buf,
                                                                    double* __restrict__ dbeta_tile) {
  __shared__ TileTables tb;
  const int64_t tile = blockIdx.x;
  const uint32_t a0 = w.tile_begin[tile], a1 = w.tile_begin[tile + 1];
  load_tables(tb, p, pl, io.leisure_prob, io.beta);
  load_cell_values(tb, w, p, pl, cell_buf, tile);
  __syncthreads();
  double db[GJ_MAX_RANGE_NETS];
#pragma unroll
  for (int i = 0; i < GJ_MAX_RANGE_NETS; ++i) db[i] = 0.0;
  const bool quar = p.n_quar > 0;
  const float* __restrict__ T = io.T_in;  // the forward's transmissions

  for (uint32_t a = a0 + threadIdx.x; a < a1; a += kBlock) {
    const int cls = w.cls[a];
    const float mq = quar ? quarantine_mask(p, io.cur[a]) : 1.0f;
    uint32_t e0 = 0, deg = 0, ent0 = 0, ent1 = 0;
    if (pl.n_generic > 0) {
      e0 = w.am_ptr[a];
      deg = w.am_ptr[a + 1] - e0;
      if (deg > 0) ent0 = w.am_ent[e0];
      if (deg > 1) ent1 = w.am_ent[e0 + 1];
    }
    float gT = 0.0f;
#pragma unroll
    for (int k = 0; k < GJ_MAX_NETS; ++k) {
      if (k < p.n_nets) {
        const int kind = p.nets[k].kind;
        const int type = p.nets[k].type;
        const int tier = pl.tier[k];
        float mT = (kind == GJ_KIND_HOUSEHOLD) ? 1.0f : mq;
        if (kind >= GJ_KIND_LEISURE) mT = mq * tb.prob[pl.net_lei[k]][cls];
        float acc = 0.0f;
        if (tier == GJ_TIER_RANGE) {
          const uint32_t slot = pl.slot[k][a];
          if (slot != kNoSlot) {
            const uint32_t b0 = a - (slot >> 16), nb = slot & 0xFFFFu;
            const float pcg = pl.rpc[k][a];
            float R = 0.0f;
            for (uint32_t b = b0; b < b0 + nb; ++b) {
              const int cb = (kind >= GJ_KIND_LEISURE) ? w.cls[b] : 0;
              float v = member_value(tb, pl, k, kind, io.w[b], io.wq[b], cb);
              if (kind == GJ_KIND_CARE_VISIT) v = v * (((cb % 100) > 75) ? 1.0f : 0.0f);
              R += v;
            }
            acc = (tb.beta[k] * pcg) * R;
            if (b0 == a && R != 0.0f) {  // first member: d/dbeta += pc_g * (sum of the group's transmissions) * R_g
              float S = 0.0f;
              for (uint32_t b = b0; b < b0 + nb; ++b) {
                const float Tb = T[b];
                const float Tqb = quar ? quarantine_mask(p, io.cur[b]) * Tb : Tb;
                S += member_value(tb, pl, k, kind, Tb, Tqb, kind >= GJ_KIND_LEISURE ? w.cls[b] : 0);
              }
              db[pl.net_t1[k]] += (double)(pcg * S) * (double)R;
            }
          }
        } else if (tier == GJ_TIER_CELL) {
          acc = tb.cellv[pl.net_t2[k]];
        } else {
          const int64_t so = p.nets[k].s_off;
          if (deg > 0 && (int)(ent0 >> 28) == type) acc += io.cR[so + (ent0 & 0x0FFFFFFFu)];
          if (deg > 1 && (int)(ent1 >> 28) == type) acc += io.cR[so + (ent1 & 0x0FFFFFFFu)];
          for (uint32_t j = 2; j < deg; ++j) {
            const uint32_t ent = w.am_ent[e0 + j];
            if ((int)(ent >> 28) == type) acc += io.cR[so + (ent & 0x0FFFFFFFu)];
          }
        }
        gT += mT * acc;
      }
    }
    if (io.g_T) {
      io.g_T[a] = gT;
    } else if (gT != 0.0f) {
      const TransTerms tt =
          transmission_terms<true>(p.now, io.tinf[a], io.maxinf[a], io.shape[a], io.rate[a], io.shift[a], io.k0[a]);
      io.g_inf[a] += gT * tt.coef;
      io.g_tinf[a] += gT * (tt.dcoef * io.inf[a]);
    }
  }
  if (pl.n_t1 > 0) block_sums<double, GJ_MAX_RANGE_NETS>(db, pl.n_t1, dbeta_tile + tile * GJ_MAX_RANGE_NETS);
}

}  // namespace gj
