// Device-side building blocks of the infection step (sm_100a).
//
// Compiled with --fmad=false and without fast-math: every a*b+c below rounds twice, exactly like the
// reference's separate torch ops, and expf/logf/powf/lgammaf are the IEEE-accurate libdevice routines
// (the same ones torch's CUDA kernels call).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "gradjune_b200.h"

namespace gj {

// Programmatic dependent launch (sm_90+): a kernel launched with the programmatic-stream-serialization attribute may
// become resident while its predecessor in the stream is still running its last CTAs; it runs its own prologue
// (shared-memory tables, barrier init, static index loads) and then waits for the predecessor's completion and memory
// flush in pdl_wait().  pdl_launch() at a kernel's top lets ITS successor do the same.  Launched without the attribute
// both are no-ops.  Rule: nothing written by an earlier kernel (state, beta, sums, scratch) is read, and no global
// memory is written, before pdl_wait().
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

constexpr int kBlock = 256;
constexpr int kRedBlocks = 148 * 8;  // persistent grid of the agent passes: 8 CTAs per SM
constexpr int kMaxRed = 2 + GJ_MAX_AGE_BINS;

// ------------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11), counter-based: the draw for (agent, call, stream) does not
// depend on launch geometry, so forward, backward and gj_philox_fill regenerate identical noise.
// ------------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ void philox_round(uint32_t& c0, uint32_t& c1, uint32_t& c2, uint32_t& c3,
                                                      uint32_t k0, uint32_t k1) {
  const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
  const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
  const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
  const uint32_t n1 = (uint32_t)p1;
  const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
  const uint32_t n3 = (uint32_t)p0;
  c0 = n0; c1 = n1; c2 = n2; c3 = n3;
}

__host__ __device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                       uint32_t k0, uint32_t k1, uint32_t out[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    philox_round(c0, c1, c2, c3, k0, k1);
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// Philox2x32-10 (same family, Random123): one 32x32->64 multiply per round instead of two.  The hot draw of a step
// needs exactly two words per agent (the two exponentials of the Gumbel-softmax), so it comes from this generator:
// about half the integer work of a 4x32 block per agent in the forward kernel (Philox was ~18 % of its
// instructions, profiles/r1_final_56M_stalls_k_pipe_forward.txt).  Known answers: tests/test_host_logic.py.
__host__ __device__ __forceinline__ void philox2x32_10(uint32_t c0, uint32_t c1, uint32_t k, uint32_t out[2]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r > 0) k += 0x9E3779B9u;
    const uint64_t p = (uint64_t)0xD256D193u * c0;
    const uint32_t n0 = (uint32_t)(p >> 32) ^ k ^ c1;
    c1 = (uint32_t)p;
    c0 = n0;
  }
  out[0] = c0;
  out[1] = c1;
}

// uniforms: (0,1) for logs, [0,1) for the Bernoulli comparison
// (23 bits + 1/2) * 2^-23: exactly representable, so 0 < u < 1 strictly.  (24 bits + 1/2 rounds its largest value to
// 1.0f: then E = -ln u = 0, its Gumbel is +inf and the reference-order softmax returns NaN — once per 2^24 draws.)
__device__ __forceinline__ float u01_open(uint32_t r) { return ((float)(r >> 9) + 0.5f) * 1.1920928955078125e-07f; }
__device__ __forceinline__ float u01_half(uint32_t r) { return (float)(r >> 8) * 5.9604644775390625e-08f; }

struct StepNoise {
  float E0, E1, u;
};

// The noise of one (agent, call) — THE definition of the stream; forward, backward and gj_philox_fill all come through
// these functions.  The two exponentials of the Gumbel draw (by inversion with the hardware log2): Philox2x32-10,
// counter = (agent, call + seed_hi), key = seed_lo (philox_step_pair).  The uniform of the symptomatic / recovery
// branch (needed only by the few agents whose stage changes in the step): word 2 of the Philox4x32-10 block of
// stream 0, counter = (agent, call).  Stream 1 of Philox4x32-10: the standard normal of the dwell time.
// Agent ids are < 2^32 (checked where worlds are built).
// (One block per PAIR of neighbouring agents, with a thread of the pipelined forward taking both, was built and
// measured: fewer instructions but slower — the pair's 32-bit stores touch every sector twice, and 64-bit stores of
// both agents' results spill at the 64-register budget.)
__device__ __forceinline__ void philox_step_block(uint64_t seed, uint32_t call, uint64_t agent, uint32_t r[4]) {
  philox4x32_10((uint32_t)agent, (uint32_t)(agent >> 32), call, 0u, (uint32_t)seed, (uint32_t)(seed >> 32), r);
}
__device__ __forceinline__ void philox_step_pair(uint64_t seed, uint32_t call, uint64_t agent, uint32_t r[2]) {
  philox2x32_10((uint32_t)agent, call + (uint32_t)(seed >> 32), (uint32_t)seed, r);
}
__device__ __forceinline__ float draw_step_uniform(uint64_t seed, uint32_t call, int64_t agent) {
  uint32_t r[4];
  philox_step_block(seed, call, (uint64_t)agent, r);
  return u01_half(r[2]);
}
// E = -ln u by inversion.  The largest u is 1 - 2^-24, whose E = 5.96e-8 is below the absolute error of the
// hardware log2 near 1: without the floor the approximation may return E = 0, a Gumbel value of +inf and a forced
// draw (ADVICE r1).  The floor is the exact E of that largest u.
constexpr float kMinE = 5.9604645e-08f;         // -ln(1 - 2^-24)
constexpr float kMinE2 = 8.5991327e-08f;        // -log2(1 - 2^-24)
__device__ __forceinline__ StepNoise draw_step_noise(uint64_t seed, uint32_t call, int64_t agent) {
  uint32_t r[4], e[2];
  philox_step_pair(seed, call, (uint64_t)agent, e);
  philox_step_block(seed, call, (uint64_t)agent, r);
  StepNoise n;
  n.E0 = fmaxf(-__logf(u01_open(e[0])), kMinE);
  n.E1 = fmaxf(-__logf(u01_open(e[1])), kMinE);
  n.u = u01_half(r[2]);
  return n;
}
// counter of agent a's noise: its id in the numbering the world was loaded in (renumbered worlds), else its global
// index (agent_offset = first agent of this rank's partition)
__device__ __forceinline__ int64_t noise_agent(const gj_world_desc& w, const gj_step_params& p, int64_t a) {
  return w.orig_id ? (int64_t)w.orig_id[a] : (int64_t)p.agent_offset + a;
}

// results by label (gj_fwd_io.label): add one agent's post-step cases (0..3) and death indicator (0/1), exact small
// integers, to column label[a] of the integer accumulator acc[n_labels][2].  The warp's values are counted with ballots;
// a warp without cases or deaths (most warps early in an epidemic) returns before it loads a label.  Lanes that share a
// label are combined first — without __match_any_sync when the whole warp holds one label, as after renumbering by
// area — so a warp issues one atomic per distinct label and value; any labels stay correct.  Integer sums are exact
// and independent of the order of the atomics.
__device__ __forceinline__ void label_add(uint32_t* __restrict__ acc, const int32_t* __restrict__ label, uint32_t a,
                                          uint32_t cases, uint32_t deaths) {
  const unsigned act = __activemask();
  const unsigned c0 = __ballot_sync(act, cases & 1u), c1 = __ballot_sync(act, cases & 2u);
  const unsigned dd = __ballot_sync(act, deaths != 0u);
  if ((c0 | c1 | dd) == 0u) return;
  const int32_t lab = label[a];
  const int32_t l0 = __shfl_sync(act, lab, __ffs(act) - 1);
  const unsigned grp = __all_sync(act, lab == l0) ? act : __match_any_sync(act, lab);
  if ((int)(threadIdx.x & 31u) == __ffs(grp) - 1) {
    const uint32_t c = __popc(c0 & grp) + 2u * __popc(c1 & grp), d = __popc(dd & grp);
    if (c) atomicAdd(acc + 2 * (int64_t)lab, c);
    if (d) atomicAdd(acc + 2 * (int64_t)lab + 1, d);
  }
}

// one standard normal per (agent, call): Box-Muller on stream 1
__device__ __forceinline__ float draw_step_normal(uint64_t seed, uint32_t call, int64_t agent) {
  uint32_t r[4];
  philox4x32_10((uint32_t)agent, (uint32_t)((uint64_t)agent >> 32), call, 1u, (uint32_t)seed,
                (uint32_t)(seed >> 32), r);
  const float u1 = u01_open(r[0]);
  const float u2 = u01_half(r[1]);
  return sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
}

// ------------------------------------------------------------------------------------------------
// a1  TransmissionUpdater.forward — transmission.py:38-51
//     T = ((((maxinf * sign) * aux) * aux2) * is_infected), aux = exp(-lgamma(shape)) * pow(b, shape-1),
//     aux2 = exp((shift - t) * rate) * rate, b = (t - shift) * rate, t = now - infection_time
// ------------------------------------------------------------------------------------------------
struct TransTerms {
  float coef;   // T / is_infected
  float dcoef;  // d coef / d infection_time
};

template <bool kGrad>
__device__ __forceinline__ TransTerms transmission_terms(float now, float tinf, float maxinf, float shape,
                                                         float rate, float shift, float k0) {
  const float t = now - tinf;
  const float d = t - shift;
  const float sg = d + 1e-10f;
  const float sign = (float)((0.0f < sg) - (sg < 0.0f));
  const float sign01 = (sign + 1.0f) / 2.0f;
  const float b = d * rate;
  const float e = shape - 1.0f;
  const float pw = powf(b, e);
  const float aux = k0 * pw;
  const float ex = expf((shift - t) * rate);
  const float aux2 = ex * rate;
  const float head = maxinf * sign01;
  TransTerms r;
  r.coef = (head * aux) * aux2;
  r.dcoef = 0.0f;
  if (kGrad) {
    // d/dt [k0 * b^e * exp((shift-t)*rate) * rate] = k0*rate*( e*b^(e-1)*rate*ex - b^e*rate*ex ), dt/dtinf = -1
    const float dpw = (e == 0.0f) ? 0.0f : e * (pw / b) * rate;  // e*b^(e-1)*rate ; torch: 0 where exponent == 0
    const float daux = k0 * dpw;
    const float daux2 = -(ex * rate) * rate;
    const float dcoef_dt = head * (daux * aux2 + aux * daux2);
    r.dcoef = -dcoef_dt;
  }
  return r;
}

// ------------------------------------------------------------------------------------------------
// a2  quarantine mask — policies/quarantine_policies.py:13-33
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float quarantine_mask(const gj_step_params& p, float cur) {
  float m = 1.0f;
  for (int i = 0; i < p.n_quar; ++i) m = m * ((cur < p.quar_thr[i]) ? 1.0f : 0.0f);
  return m;
}

__device__ __forceinline__ float leisure_prob(const float* __restrict__ table, int row, int day_type, int cls) {
  return __ldg(table + ((size_t)(row * 2 + day_type) * 200 + cls));
}

// ------------------------------------------------------------------------------------------------
// a3 tail + a8  q = clamp(exp(-clamp(L,1e-6,100)*dt),0,1); Gumbel-softmax hard draw
//     base.py:136-140 ; infection.py:13-17 + torch functional.py:2218-2232
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float not_infected_prob(float lam, float dt) {
  const float lc = fminf(fmaxf(lam, 1e-6f), 100.0f);
  const float q = expf(-lc * dt);
  return fminf(fmaxf(q, 0.0f), 1.0f);
}

struct Draw {
  float n;   // new_infected, exactly 0 or 1
  float ty;  // tape: the smaller of the two soft probabilities, +y1 (infected) or -y0 (not infected)
};

// The backward needs BOTH softmax outputs as the forward rounded them (torch's softmax backward uses
// y1 itself, not 1 - y0: for y1 ~ 1e-9 and q -> 1 the product y0*y1/(1-q) is far from negligible).
// Storing the smaller one with a sign bit keeps it exact; the larger one is 1 - small to 1 ulp.
__device__ __forceinline__ void decode_soft(float ty, float& y0, float& y1) {
  if (signbit(ty)) {
    y0 = -ty;
    y1 = 1.0f - y0;
  } else {
    y1 = ty;
    y0 = 1.0f - y1;
  }
}

__device__ __forceinline__ Draw gumbel_draw(float q, float E0, float E1, float tau) {
  const float l0 = logf(q);
  const float l1 = logf(1.0f - q);
  const float g0 = -logf(E0);
  const float g1 = -logf(E1);
  const float x0 = (l0 + g0) / tau;  // torch CPU divides (CUDA torch multiplies by 1/tau); see DESIGN.md
  const float x1 = (l1 + g1) / tau;
  const float m = fmaxf(x0, x1);
  const float e0 = expf(x0 - m);
  const float e1 = expf(x1 - m);
  const float sum = e0 + e1;
  const float y0 = e0 / sum;
  const float y1 = e1 / sum;
  Draw d;
  d.n = (y1 > y0) ? 1.0f : 0.0f;  // max() returns the first index on ties -> not infected
  d.ty = (y1 <= y0) ? y1 : -y0;
  return d;
}

// ------------------------------------------------------------------------------------------------
// a10  SymptomsUpdater.forward + SymptomsSampler.sample_next_stage — symptoms.py:204-247, 82-128
// ------------------------------------------------------------------------------------------------
struct SympOut {
  float cur, nxt, ttn;
  // for the backward pass
  float tr;       // mask_transition
  int stage;      // int(cur) after the transition
  int branch;     // 0 none, 1 progressed, 2 recovered
  float dwell;    // sampled dwell time of the taken branch
  float nxt1;     // next_stage before the stage loop
};

__device__ __forceinline__ float dwell_time(const gj_dist& d, float z) {
  const float x = d.loc + z * d.scale;
  return d.kind == 0 ? expf(x) : x;
}

template <typename UF, typename ZF>
__device__ __forceinline__ SympOut symptoms_forward(const gj_step_params& p, const float* __restrict__ stage_prob,
                                                    float cur, float nxt, float ttn, float n, int age, UF uf, ZF zf) {
  SympOut o;
  const float nxt1 = nxt + n * (2.0f - nxt);
  const float ttn1 = ttn + n * (p.now - ttn);
  const float tr = ((p.now >= ttn1) && (cur < (float)(p.n_stages - 1))) ? 1.0f : 0.0f;
  const float cur1 = cur - (cur - nxt1) * tr;
  const int st = (int)cur1;  // .long(): truncation
  o.cur = cur1;
  o.nxt = nxt1;
  o.ttn = ttn1;
  o.tr = tr;
  o.stage = st;
  o.branch = 0;
  o.dwell = 0.0f;
  o.nxt1 = nxt1;
  if (tr != 0.0f && st >= 2 && st <= p.n_stages - 2 && cur1 == (float)st) {
    const float pr = __ldg(stage_prob + st * 100 + age);
    const bool symp = uf() < pr;
    const gj_dist& d = symp ? p.trans_time[st] : p.rec_time[st];
    if (d.kind >= 0) {
      const float z = zf((st - 2) * 2 + (symp ? 0 : 1));
      const float dw = dwell_time(d, z);
      o.dwell = dw;
      if (symp) {
        o.branch = 1;
        o.nxt = nxt1 + 1.0f;
        o.ttn = ttn1 + dw * 1.0f;
      } else {
        o.branch = 2;
        o.nxt = nxt1 - nxt1 * 1.0f;
        o.ttn = ttn1 + dw * 1.0f;
      }
    }
  }
  return o;
}

// ------------------------------------------------------------------------------------------------
// reductions
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ int type_of_group(const gj_world_desc& w, uint32_t g) {
  int t = 0;
#pragma unroll
  for (int i = 1; i < GJ_MAX_TYPES; ++i) t += (i < w.n_types && (int64_t)g >= w.type_group_off[i]) ? 1 : 0;
  return t;
}

}  // namespace gj
