/*
 * gradjune_b200.h — C ABI of the B200-native per-timestep infection path of GradABM-JUNE.
 *
 * One shared library (libgradjune_b200.so, sm_100a), plain pointers and sizes only, no torch types.
 * The reference has no FFI: its boundary for this path is the Python nn.Module API
 * (/root/reference/grad_june/model.py:112-144 and the modules it calls).  Each entry point below
 * names the reference interface it replaces; INTEGRATION.md shows the ctypes stubs that bind them.
 *
 * Conventions
 *   - every array pointer is DEVICE memory owned by the caller and borrowed for the call;
 *   - every call is stream-ordered on `stream` (a cudaStream_t passed as void*), performs no
 *     allocation and no host synchronisation;
 *   - return value 0 = ok, negative = error (text via gj_last_error());
 *   - floating point is fp32, compiled without FMA contraction (--fmad=false) and without --use_fast_math.
 *     The reference-order kernels (injected noise, exact_order) use the IEEE libdevice expf/logf/powf and true
 *     divisions, so their elementwise arithmetic rounds like the reference's op-by-op torch graph.  The
 *     throughput-mode kernels (in-kernel Philox noise) keep q = expf(-lam*dt) IEEE but evaluate the Gumbel draw
 *     and the infectiousness profile with the hardware lg2.approx / ex2.approx / rcp.approx (explicit fmaf where
 *     written): masks then differ from the reference only at certified near-ties (DESIGN.md 2).
 */
#ifndef GRADJUNE_B200_H
#define GRADJUNE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GJ_ABI_VERSION 12

#define GJ_MAX_TYPES 8      /* edge types (household, company, school, university, care_home, leisure, ...) */
#define GJ_MAX_NETS 16      /* infection networks active in one step */
#define GJ_MAX_STAGES 16    /* symptom stages */
#define GJ_MAX_QUAR 4       /* simultaneously active quarantine policies */
#define GJ_MAX_AGE_BINS 8   /* cases-by-age result bins */
#define GJ_MAX_CHANNELS 8   /* networks sharing one edge type (the six leisure networks) */

/* group-size split of the group-major passes (the world builder must use the same values,
 * read them through gj_config) */
#define GJ_SMALL_GROUP 16   /* <= this many members: one lane sums the group sequentially */
#define GJ_CHUNK 1024       /* larger groups are cut into chunks of this many members, one warp each */

/* throughput-mode forward: members of a generic-tier group of at most this many agents ADD their transmission into
 * the group's 64-bit fixed-point accumulator (exact, order-independent: deterministic); larger ("giant") groups are
 * summed group-major by the chunk kernel.  Fixed point: GJ_SCATTER_FRAC fractional bits, member values below
 * 2^GJ_SCATTER_CAP_LOG2 (a larger / non-finite value marks its group for an exact re-sum): the sum of
 * GJ_SCATTER_MAX_GROUP such members stays below 2^62 */
#define GJ_SCATTER_MAX_GROUP 32768
#define GJ_SCATTER_CAP_LOG2 10
#define GJ_SCATTER_FRAC 37

enum { GJ_TIER_GENERIC = 0, GJ_TIER_RANGE = 1, GJ_TIER_CELL = 2 };
#define GJ_TILE_AGENTS 1024
#define GJ_MAX_RANGE_NETS 4 /* networks running on RANGE-tier types in one step */

/* how a network masks transmissions / susceptibilities
 * (grad_june/infection_networks/base.py:47-59,144-149; leisure_network.py:61-85,107-120) */
enum { GJ_KIND_PLAIN = 0, GJ_KIND_HOUSEHOLD = 1, GJ_KIND_LEISURE = 2, GJ_KIND_CARE_VISIT = 3 };

/* phases of one timestep (grad_june/model.py:112-144); the fused step runs all of them, the
 * stand-alone module entry points run one */
enum {
  GJ_PHASE_NETWORKS = 1, /* InfectionNetworks.forward            base.py:118-141            */
  GJ_PHASE_SAMPLE = 2,   /* IsInfectedSampler.forward            infection.py:3-18          */
  GJ_PHASE_INFECT = 4,   /* GradJune.infect_people               model.py:90-110            */
  GJ_PHASE_SYMPTOMS = 8, /* SymptomsUpdater.forward              symptoms.py:204-247        */
  GJ_PHASE_ALL = 15
};

enum { GJ_STAGE_ALL = 0, GJ_STAGE_SUMS = 1, GJ_STAGE_REST = 2 };

/* mode flags */
enum {
  GJ_MODE_STEP = 0,
  GJ_MODE_SEED = 1 /* infect_fraction_of_people: uniform q = 1 - fraction and the clamp variant of the
                      susceptibility update (infection.py:21-42, runner.py:138-149) */
};

/* ------------------------------------------------------------------------------------------
 * World: CSR-sorted agent<->group edges for every edge type (replaces the int64 [2,E]
 * edge_index pairs of HeteroData, june_world_loader/graph_loader.py:16-39).
 * ------------------------------------------------------------------------------------------ */
typedef struct gj_world_desc {
  int64_t n_agents;
  int64_t n_groups; /* all types */
  int64_t n_edges;  /* all types */
  int32_t n_types;
  int32_t _pad0;
  int64_t type_group_off[GJ_MAX_TYPES + 1]; /* global group id range of each type */

  /* agent-major CSR, all types merged; an agent's entries are sorted by (type, reference edge order) */
  const uint32_t* am_ptr; /* [n_agents+1] */
  const uint32_t* am_ent; /* [n_edges]  (type << 28) | group id local to the type */

  /* group-major CSR in global group order; members keep the reference's edge order */
  const uint32_t* gm_ptr;   /* [n_groups+1] */
  const uint32_t* gm_agent; /* [n_edges] */
  const float* pc;          /* [n_groups] clamp(1/(people-1), 0, 1)  (base.py:64-69) */

  const uint8_t* cls; /* [n_agents] sex*100 + age */

  /* work lists of the group-major passes */
  const uint32_t* small_groups; /* [n_small] global ids of groups with <= GJ_SMALL_GROUP members */
  int64_t n_small;
  const uint32_t* chunk_group; /* [n_chunks] global group id */
  const uint32_t* chunk_begin; /* [n_chunks] first entry in gm_agent */
  const uint32_t* chunk_end;   /* [n_chunks] one past the last entry */
  const int32_t* chunk_part;   /* [n_chunks] -1: the group's only chunk (write the sum directly);
                                  else index into the partial-sum buffer */
  int64_t n_chunks;
  const uint32_t* big_groups;   /* [n_big] groups with >= 2 chunks */
  const uint32_t* big_part_ptr; /* [n_big+1] their partial-sum ranges */
  int64_t n_big;
  int64_t n_parts; /* total partial sums (= big_part_ptr[n_big]) */

  /* ---- layout tiers: each edge type is stored in the cheapest layout its structure allows; the CSR
   *      arrays above hold the GENERIC types only ---- */
  int32_t type_tier[GJ_MAX_TYPES]; /* GJ_TIER_* */
  /* RANGE tier: [n_agents] (a - first_member) << 16 | group_size, 0xFFFFFFFF = not a member; and the
   * contact probability of the agent's group */
  const uint32_t* range_slot[GJ_MAX_TYPES];
  const float* range_pc[GJ_MAX_TYPES];
  /* 1: range_pc of this type equals clamp(1 / (group_size - 1), 0, 1) for every member, i.e. `people` is the member
   * count (true of every JUNE world): the pipelined kernels then take the contact probability from a 65-entry table
   * indexed by the size in the slot word instead of streaming 4 more bytes per agent and pass */
  int32_t range_pc_from_size[GJ_MAX_TYPES];
  /* CTA tiles of the agent-major kernels: tile i = agents [tile_begin[i], tile_begin[i+1]), at most
   * GJ_TILE_AGENTS, never straddling a cell boundary of a CELL-tier type */
  int64_t n_tiles;
  const uint32_t* tile_begin;
  /* [n_tiles] bit 0: the tile lies in another cell (of any CELL-tier type) than the tile before it; tile 0 has it set.
   * What the pipelined kernels' tile walk prefetches instead of comparing the tile -> cell maps per tile */
  const uint32_t* tile_flags;
  /* CELL tier: runs of consecutive agents with the same ordered group list */
  int64_t n_cells[GJ_MAX_TYPES];
  int64_t cell_off[GJ_MAX_TYPES]; /* offset of the type's cells in per-cell buffers */
  int64_t n_cells_total;
  const uint32_t* tile_cell[GJ_MAX_TYPES];     /* [n_tiles] cell of each tile */
  const uint32_t* cell_tile_ptr[GJ_MAX_TYPES]; /* [n_cells+1] consecutive tiles of each cell */
  const uint32_t* cell_grp_ptr[GJ_MAX_TYPES];  /* [n_cells+1] */
  const uint32_t* cell_grp[GJ_MAX_TYPES];      /* groups (ids local to the type) of each cell, agent edge order */
  const uint32_t* grp_cell_ptr[GJ_MAX_TYPES];  /* [G_type+1] */
  const uint32_t* grp_cell[GJ_MAX_TYPES];      /* cells of each group, ascending */
  /* one-entry-per-agent view of the GENERIC types (throughput-mode kernels): the GLOBAL id of the agent's only
   * generic group (bit 31 set: a giant group, > GJ_SCATTER_MAX_GROUP members), 0xFFFFFFFF = none,
   * 0xFFFFFFFE = several (walk am_ptr / am_ent); NULL = not built */
  const uint32_t* ent1;
  /* the chunk list starts with the n_giant_chunks chunks of the giant groups and the list of multi-chunk groups
   * with the n_giant_big giant ones: the throughput-mode forward sums only those group-major */
  int64_t n_giant_chunks;
  int64_t n_giant_big;
  /* geographic partition (one process per GPU, each owning an agent range and the groups its agents attend):
   * [n_groups] weight of each group in d/dbeta, 1 for groups this rank owns and 0 for groups owned by another
   * rank (their sums are exchanged between the two stages of a step); NULL = all ones */
  const float* dbeta_w;
  /* agent renumbering (grad_june.world.renumber_world / gj_world_build): [n_agents] id of every agent in the
   * numbering the world was LOADED in.  The Philox counter of agent a is orig_id[a] (then agent_offset is not
   * added), so a renumbered world draws exactly the noise of the world as loaded; NULL = the identity */
  const uint32_t* orig_id;
} gj_world_desc;

/* ---- building the world behind the C ABI (replaces the repo-side Python builder for callers that bind the .so
 * directly): the reference's own arrays in, the layout above out.  All pointers are DEVICE memory
 * (gj_world_build) — the reference keeps its HeteroData on `system.device` (runner.py:65-91) — or HOST memory
 * (gj_world_build_host, the same code on the CPU: test infrastructure for boxes without a GPU). */
typedef struct gj_world_src {
  int64_t n_agents;
  int32_t n_types;
  int32_t renumber;                            /* 1: renumber the agents household-contiguous inside their leisure
                                                  cell (grad_june.world.layout_order) before building */
  const char* type_name[GJ_MAX_TYPES];         /* "household", "company", ..., "leisure": data["attends_<name>"] */
  const int64_t* edge_agent[GJ_MAX_TYPES];     /* edge_index[0]  [n_edges[t]]  unsorted */
  const int64_t* edge_group[GJ_MAX_TYPES];     /* edge_index[1] */
  int64_t n_edges[GJ_MAX_TYPES];
  int64_t n_groups[GJ_MAX_TYPES];              /* len(data[name]["id"]) */
  const int64_t* people_i64[GJ_MAX_TYPES];     /* data[name]["people"] as int64 (pickles) ... */
  const float* people_f32[GJ_MAX_TYPES];       /* ... or as float32 (test fixtures); exactly one is non-NULL */
  const int64_t* age;                          /* [n_agents] in [0, 99] */
  const int64_t* sex;                          /* [n_agents] in {0, 1} */
  const int64_t* original_index;               /* optional [n_agents]: ids in an earlier numbering (composed) */
  const int32_t* want_tier;                    /* optional [n_types]: the tier to try per type (partitioned worlds
                                                  pass the tiers their ranks agreed on); NULL = the default policy */
} gj_world_src;
typedef struct gj_world gj_world;
int gj_world_build(const gj_world_src* src, gj_world** out);
int gj_world_build_host(const gj_world_src* src, gj_world** out);
/* the descriptor to pass to gj_step_forward / gj_step_backward (owned by the handle; pointers into its arrays) */
const struct gj_world_desc* gj_world_descriptor(const gj_world* world);
/* [n_agents] perm[new] = old of the renumbering (same memory space as the build), NULL = identity: per-agent
 * inputs (state, profile parameters) are gathered through it, outputs scattered back */
const int64_t* gj_world_permutation(const gj_world* world);
/* synchronous copy between any two of host / device memory (cudaMemcpyDefault): reading a handle's arrays */
int gj_memcpy(void* dst, const void* src, int64_t bytes);
const char* gj_world_last_error(void);
int gj_world_destroy(gj_world* world);

typedef struct gj_net {
  int32_t type;     /* edge type index */
  int32_t kind;     /* GJ_KIND_* */
  int32_t prob_row; /* leisure table index for LEISURE / CARE_VISIT, else -1 */
  int32_t s_off;    /* offset of this network's per-group sums in the S buffers */
} gj_net;

typedef struct gj_dist {
  int32_t kind; /* -1 none, 0 LogNormal, 1 Normal (utils.py:75-83 distributions used by default.yaml / tests) */
  float loc, scale;
} gj_dist;

/* scalars of one timestep, all host values (timer.py, policies/*.py stay on the host) */
typedef struct gj_step_params {
  int32_t mode;   /* GJ_MODE_* */
  int32_t phases; /* GJ_PHASE_* mask */
  float now;      /* timer.now   (days) */
  float dt;       /* timer.duration (days) */
  int32_t day_type; /* 0 weekday, 1 weekend */
  int32_t n_nets;
  gj_net nets[GJ_MAX_NETS]; /* in accumulation order = timer.get_activity_order() minus closed venues */
  int32_t n_quar;           /* -1: no quarantine collection (mask is the scalar 1.0) */
  float quar_thr[GJ_MAX_QUAR];
  int32_t n_stages;
  gj_dist trans_time[GJ_MAX_STAGES];
  gj_dist rec_time[GJ_MAX_STAGES];
  int32_t n_age_bins;
  int32_t age_bins[GJ_MAX_AGE_BINS + 1];
  float tau; /* gumbel-softmax temperature (0.1, infection.py:15) */
  /* noise: counter-based Philox keyed by seed, counter (agent, call_index[, stream]) — Philox2x32-10 for the two
   * exponentials of the draw, Philox4x32-10 for the symptoms' uniform and normal; ignored where an injected array
   * is given */
  uint64_t seed;
  uint32_t call_index;
  /* 0: with in-kernel Philox noise run the throughput-mode kernels where the step allows it (same arithmetic,
   * re-associated sums, hardware log2/exp2 in the draw and the infectiousness profile); 1: always run the
   * reference-order kernels (they also run whenever noise is injected) */
  uint32_t exact_order;
  /* two-stage execution for partitioned worlds: GJ_STAGE_ALL runs the whole step; GJ_STAGE_SUMS stops after the
   * per-group sums (forward: S_scaled / S_unscaled, backward: cR / R) are written, so that the caller can
   * all-reduce the sums of groups that straddle partitions; GJ_STAGE_REST continues from the (summed) buffers */
  uint32_t stage;
  /* 1: io->T (and io->Tq) and the scratch tile sums of the cell channels were already produced for this step by the
   * previous step's gj_step_forward_next (same state tensors, same schedule): skip the transmission pass */
  uint32_t t_ready;
  /* 1: a look-ahead (gj_step_forward_next) whose result was then NOT used left transmissions in the scratch
   * accumulators of the generic groups: clear them before this step's transmission pass */
  uint32_t reset_scatter;
  uint32_t _pad1;
  /* global id of this rank's first agent: the Philox counter is (agent_offset + local agent index), so a
   * partitioned world draws exactly the noise of the unpartitioned one */
  uint64_t agent_offset;
} gj_step_params;

/* device arrays of one forward call; unused ones may be NULL */
typedef struct gj_fwd_io {
  const float* beta;         /* [n_nets] beta_eff per network (base.py:36-42 evaluated on the host) */
  const float* leisure_prob; /* [n_tables][2][2][100] */
  const float* stage_prob;   /* [n_stages][100] */
  const float* seed_fraction; /* [1] (GJ_MODE_SEED), or [n_seed_labels] with seed_label */
  /* injected noise (NULL -> Philox) */
  const float* inj_E; /* [2][N] */
  const float* inj_u; /* [N] */
  const float* inj_z; /* [2*(n_stages-3)][N] */
  /* state in */
  const float *s, *inf, *tinf, *cur, *nxt, *ttn;
  /* per-agent infectiousness profile (transmission.py:8-35); k0 = exp(-lgamma(shape)) */
  const float *maxinf, *shape, *rate, *shift, *k0;
  /* the same profile packed by gj_profile_pack: [N][4] = {maxinf*k0*rate, rate, shape-1, shift}; optional,
   * enables the throughput-mode kernels */
  const float* prof4;
  /* phase inputs when the producing phase is not run */
  const float* T_in; /* transmissions (NETWORKS phase without gj_transmission) */
  const float* q_in; /* not-infected probabilities (SAMPLE without NETWORKS) */
  const float* n_in; /* new_infected (INFECT/SYMPTOMS without SAMPLE) */
  /* state out */
  float *s_o, *inf_o, *tinf_o, *cur_o, *nxt_o, *ttn_o;
  float* T;  /* [N] transmissions (written by the fused step, read by the group pass) */
  float* Tq; /* [N] quarantine-masked transmissions; may alias T when n_quar <= 0 */
  float* q;  /* [N] optional: not_infected_probs */
  float* lam; /* [N] optional: summed pressure before the clamp (InfectionNetwork.forward, base.py:61-84) */
  float* n;  /* [N] optional: new_infected */
  /* saved for backward */
  float* tape_v;  /* [N] pressure (s != 0) or pressure per unit susceptibility (s == 0) */
  float* tape_y0; /* [N] the smaller soft probability of the draw: +y1 (infected) or -y0 (not infected) */
  /* group-sum buffers, [sum_k G(type_k) + n_groups] floats each: network k's sums at nets[k].s_off (reference-order
   * kernels, cell tier), then one value per GLOBAL group id (throughput-mode kernels, generic tier) */
  float* S_scaled;   /* beta*pc-weighted group sums (forward operand) */
  float* S_unscaled; /* plain group sums (saved: d/dbeta) */
  float* red;        /* [2 + n_age_bins] cases, deaths, cases by age bin */
  void* scratch;     /* gj_scratch_bytes() bytes, zero-initialised once by the caller */
  /* gj_step_forward_next: transmissions of the NEXT step (from this step's output state), [N] each; Tq_next only
   * when the next step has an active quarantine */
  float* T_next;
  float* Tq_next;
  /* results by label (cases and deaths per region, area, ...; NULL = off): label[a] is agent a's column in
   * [0, n_labels).  Every kernel that writes `red` also adds the agent's post-step is_infected and its death indicator
   * (current_stage == dead) to red_label[label[a]][0] / [1].  The sums are exact: they are accumulated as integers in
   * label_acc and converted to fp32 once per step, so they are independent of the summation order and sum over the
   * columns to red[0] / red[1].  Label codes must lie in [0, n_labels): they are not checked on the device.  A call with
   * a label table does not produce the look-ahead of gj_step_forward_next. */
  const int32_t* label;  /* [N] */
  int32_t n_labels;      /* 1 .. 2^30 */
  int32_t _pad_label;
  float* red_label;      /* [n_labels][2] cases, deaths */
  uint32_t* label_acc;   /* [n_labels][2] integer workspace, zero-initialised once by the caller; the library leaves it
                            zeroed (gj_scratch_bytes depends on the world only, so it cannot cover it) */
  /* seeding by label (GJ_MODE_SEED only; NULL = one national fraction): seed_label[a] is agent a's region in
   * [0, n_seed_labels), and the seeding step draws agent a with q = 1 - seed_fraction[seed_label[a]] instead of
   * 1 - seed_fraction[0].  The Philox counter is unchanged, so an agent whose region holds the national value draws
   * exactly what it draws without a label table.  Codes are not checked on the device. */
  const int32_t* seed_label;  /* [N] */
  int32_t n_seed_labels;      /* 1 .. 2^30 */
  int32_t _pad_seed;
} gj_fwd_io;

typedef struct gj_bwd_io {
  const float* beta;
  const float* leisure_prob;
  const float* stage_prob;
  const float* seed_fraction;
  const float* inj_E;
  const float* inj_u;
  const float* inj_z;
  /* forward inputs and saved tensors */
  const float *s, *inf, *tinf, *cur, *nxt, *ttn;
  const float *maxinf, *shape, *rate, *shift, *k0;
  const float* prof4;
  const float* inf_o; /* post-step is_infected (new_infected = inf_o - inf) or NULL with n_in */
  const float* n_in;
  const float* T_in; /* transmissions: the stand-alone input, or the T written by the fused forward */
  const float* q_in; /* stand-alone SAMPLE: the q it was given */
  const float* tape_v;
  const float* tape_y0;
  const float* S_unscaled;
  /* cotangents of the outputs (NULL = zero) */
  const float *g_s_o, *g_inf_o, *g_tinf_o, *g_cur_o, *g_nxt_o, *g_ttn_o;
  const float* g_red; /* [2 + n_age_bins] */
  const float* g_q;   /* cotangent of q (NETWORKS without SAMPLE) */
  const float* g_lam; /* cotangent of lam */
  const float* g_n;   /* extra cotangent of new_infected */
  /* cotangents of the inputs (NULL = not wanted) */
  float *g_s, *g_inf, *g_tinf, *g_cur, *g_nxt, *g_ttn;
  float* g_T;       /* cotangent of T_in (stand-alone NETWORKS) */
  float* g_q_out;   /* cotangent of q_in (stand-alone SAMPLE) */
  float* g_n_out;   /* cotangent of n_in (stand-alone INFECT / SYMPTOMS) */
  float* g_beta;    /* [n_nets] */
  float* g_seed_fraction; /* [1], or [n_seed_labels] with seed_label */
  /* workspaces */
  float* w;   /* [N] */
  float* wq;  /* [N], may alias w when n_quar <= 0 */
  float* R;   /* [sum_k G(type_k) + n_groups], laid out like S_unscaled */
  float* cR;  /* [sum_k G(type_k) + n_groups] */
  void* scratch;
  /* results by label: the forward's label codes and the cotangent of its red_label ([n_labels][2]); both non-NULL
   * adds g_red_label[label[a]][0] to the cotangent of agent a's post-step is_infected and g_red_label[label[a]][1] / dead
   * to that of its post-step current_stage where it equals dead; NULL = no label table */
  const int32_t* label;
  const float* g_red_label;
  /* seeding by label (GJ_MODE_SEED only; NULL = one national fraction): the forward's seed_label / n_seed_labels.  The
   * per-agent pass writes each agent's d/dseed_fraction (-dL/dq) to seed_work instead of folding it into one sum, and a
   * reduction then writes g_seed_fraction[l] = sum over the agents of label l.  The library never allocates, so the
   * caller passes the agents in label order: seed_order holds the agent ids stably sorted by label and seed_offsets
   * the start of every label in it (seed_offsets[0] = 0, seed_offsets[n_seed_labels] = N; empty labels allowed).  The
   * sum runs in fp64 over fixed chunks of seed_order whose partials are combined in chunk order: it is bit-reproducible
   * and independent of the launch grid.  Each agent's fraction is q = 1 - seed_fraction[l]; a fraction below ~2^-24
   * rounds q to 1 in fp32, and the sampler's d/dq then divides 0 by 0 for that agent, as the reference's torch code
   * does (DESIGN.md, "Seeding by label"). */
  const int32_t* seed_label;    /* [N] */
  int32_t n_seed_labels;
  int32_t _pad_seed;
  const int32_t* seed_order;    /* [N] */
  const int32_t* seed_offsets;  /* [n_seed_labels + 1] */
  float* seed_work;             /* [N] workspace */
} gj_bwd_io;

/* ---- library ---------------------------------------------------------------------------- */
int gj_abi_version(void);
const char* gj_last_error(void);
/* out[0]=GJ_SMALL_GROUP, out[1]=GJ_CHUNK, out[2]=sizeof(gj_world_desc), out[3]=sizeof(gj_step_params),
 * out[4]=sizeof(gj_fwd_io), out[5]=sizeof(gj_bwd_io), out[6]=reduction grid size, out[7]=GJ_TILE_AGENTS,
 * out[8]=GJ_SCATTER_MAX_GROUP, out[9]=sizeof(gj_batch) */
int gj_config(int64_t* out, int n);
/* bytes of the caller-provided scratch buffer (zero it once; the library leaves it zeroed) */
int64_t gj_scratch_bytes(const gj_world_desc* w);

/* ---- TransmissionUpdater.forward (grad_june/transmission.py:38-51) ------------------------ */
/* k0[i] = exp(-lgamma(shape[i])), the time-independent factor of the gamma profile */
int gj_profile_prepare(int64_t n, const float* shape, float* k0, void* stream);
/* prof4[i] = {maxinf*k0*rate, rate, shape-1, shift}: one 16-byte load per agent in the throughput-mode kernels */
int gj_profile_pack(int64_t n, const float* maxinf, const float* shape, const float* rate, const float* shift,
                    const float* k0, float* prof4, void* stream);
int gj_transmission_forward(int64_t n, float now, const float* tinf, const float* inf, const float* maxinf,
                            const float* shape, const float* rate, const float* shift, const float* k0,
                            float* T, void* stream);
int gj_transmission_backward(int64_t n, float now, const float* tinf, const float* inf, const float* maxinf,
                             const float* shape, const float* rate, const float* shift, const float* k0,
                             const float* g_T, float* g_tinf, float* g_inf, void* stream);

/* ---- GradJune.forward (grad_june/model.py:112-144) and, through `phases`, its parts:
 *      InfectionNetworks.forward (infection_networks/base.py:118-141, 61-87; leisure_network.py),
 *      IsInfectedSampler.forward (infection.py:3-18), infect_people (model.py:90-110,
 *      infection.py:21-28), SymptomsUpdater.forward (symptoms.py:204-247), plus the per-step result
 *      reductions of Runner.forward (runner.py:167-171,198-224) ------------------------------- */
int gj_step_forward(const gj_world_desc* w, const gj_step_params* p, const gj_fwd_io* io, void* stream);
/* gj_step_forward that ALSO runs the transmission pass of the following step (params `next`) inside its agent kernel,
 * from the state it has just written: the next call then sets next->t_ready = 1, passes T_next / Tq_next as its T / Tq,
 * and skips a whole pass over the agents (TransmissionUpdater.forward of step t+1 fused into GradJune.forward of step
 * t).  Returns 1 when the look-ahead was produced, 0 when this (world, params, next) combination cannot (then it
 * behaved exactly like gj_step_forward), < 0 on error. */
int gj_step_forward_next(const gj_world_desc* w, const gj_step_params* p, const gj_step_params* next,
                         const gj_fwd_io* io, void* stream);
/* reverse-mode derivative of gj_step_forward (replaces autograd's replay of the op tape) */
int gj_step_backward(const gj_world_desc* w, const gj_step_params* p, const gj_bwd_io* io, void* stream);

/* ---- batched ensemble [N, b] (SURVEY.md 8e-2, BASELINE config 5; the reference evaluates one parameter sample per
 * Python-driven run, example_scripts/run_model.py:6-11): ONE call steps `n_samples` independent epidemics on the same
 * world.  `io` describes sample 0; sample s reads and writes every per-sample array at a fixed stride behind it:
 *   per-agent arrays  (state in/out, T, Tq, tapes, q/lam/n, cotangents, w, wq)        + s * agent_stride  elements
 *   group-sum buffers (S_scaled, S_unscaled, R, cR)                                   + s * group_stride  elements
 *   beta, g_beta                                                                      + s * beta_stride   elements
 *   red, g_red                                                                        + s * red_stride    elements
 *   red_label, g_red_label, label_acc                                                 + s * label_stride  elements
 *   scratch                                                                           + s * scratch_stride bytes
 * while the world (index words, classes, tiles), the label codes, the packed infectiousness profile and the lookup
 * tables are shared.
 * The CTAs of the b samples that walk the same run of agent tiles are launched next to each other (block index =
 * run * b + sample) and advance in step, so the tile's index words, class bytes and profile are fetched from HBM once
 * and served to the other b-1 samples out of L2: one index read per b samples.  All samples draw the SAME Philox
 * stream (seed, call_index): common random numbers across the parameter samples of an ensemble.  Sample s of a batched
 * call is bit-identical to a gj_step_forward / gj_step_backward call on its slices.
 * Requirements (else an error is returned, nothing runs): the whole fused step in throughput mode (gj_step_plan = 1,
 * prof4 given, no injected noise, GJ_MODE_STEP, GJ_STAGE_ALL), the pipelined kernels enabled, agent_stride a multiple
 * of 4 with every per-agent array 16-byte aligned, n_samples * agent_stride < 2^32, scratch_stride a multiple of 256
 * and >= gj_scratch_bytes(). */
typedef struct gj_batch {
  int32_t n_samples;
  int32_t _pad0;
  int64_t agent_stride;
  int64_t group_stride;
  int64_t beta_stride;
  int64_t red_stride;
  int64_t scratch_stride;
  /* optional workspace of agent_stride floats.  All samples of a batch draw the same Philox stream, so the Gumbel
   * noise of the infection draw (two Philox words and four log2 per agent) is the same for every sample: given this
   * buffer, gj_step_forward_batch evaluates it ONCE per agent (one small kernel) and the b samples read it, instead
   * of every sample regenerating it.  Same arithmetic: results are bit-identical.  NULL = every sample computes it. */
  float* noise;
  /* stride of red_label / g_red_label / label_acc (elements, >= 2 * n_labels when a label table is given) */
  int64_t label_stride;
} gj_batch;
int gj_step_forward_batch(const gj_world_desc* w, const gj_step_params* p, const gj_fwd_io* io, const gj_batch* batch,
                          void* stream);
int gj_step_backward_batch(const gj_world_desc* w, const gj_step_params* p, const gj_bwd_io* io, const gj_batch* batch,
                           void* stream);

/* ---- geographic partition: boundary groups (SURVEY.md 8e; no counterpart in the reference, which is single-device)
 * Between GJ_STAGE_SUMS and GJ_STAGE_REST the caller all-reduces (NCCL, owned by the caller) the sums of the groups
 * that straddle partitions.  pack[2][n_pack]: position q = boundary group q of the step's edge types; inv[q] = index
 * of that group in this rank's two group-sum buffers a / b (S_scaled / S_unscaled forward, cR / R backward), or -1
 * when this rank does not attend it (packs 0, unpacks nothing). */
int gj_boundary_pack(int64_t n_pack, const int32_t* inv, const float* a, const float* b, float* pack, void* stream);
int gj_boundary_unpack(int64_t n_pack, const int32_t* inv, const float* pack, float* a, float* b, void* stream);

/* ---- the same exchange over NVLink peer memory, ONE kernel instead of pack -> ncclAllReduce -> unpack.
 * Every rank owns a receive buffer (cudaMalloc'ed by the library, exported as a CUDA IPC handle, opened by its
 * peers).  gj_peer_exchange: each rank STORES the partial sums of the boundary groups it attends straight into the
 * receive buffers of the other ranks attending them (attend[q] = bit mask of ranks), raises a flag in every peer's
 * memory, waits for the peers' flags in its own, and adds the contributions in ascending rank order — the same
 * order on every rank, so the totals are bit-identical everywhere and run to run.  Two buffer sets alternate
 * (a rank can be at most one exchange ahead of a peer); the exchange counter lives on the device, so the call can
 * be captured in a CUDA graph and replayed.  A peer that does not arrive within ~10 s sets an error flag (read by
 * gj_peer_status) instead of hanging the GPU.  One process per GPU; every rank must issue the same sequence of
 * exchanges. */
typedef struct gj_peer gj_peer;
#define GJ_IPC_HANDLE_BYTES 64
/* capacity: the largest n_pack that will be exchanged; allocates and zeroes this rank's buffers */
int gj_peer_create(int rank, int world_size, int64_t capacity, gj_peer** out);
int gj_peer_handle(gj_peer* peer, void* handle /* GJ_IPC_HANDLE_BYTES */);
/* handles: world_size x GJ_IPC_HANDLE_BYTES, rank-major (an all-gather of gj_peer_handle) */
int gj_peer_connect(gj_peer* peer, const void* handles);
/* mine[n_mine]: the packed positions q this rank attends (inv[q] >= 0), ascending — the kernel then walks only
 * those; NULL walks all n_pack positions */
int gj_peer_exchange(gj_peer* peer, int64_t n_pack, const int32_t* inv, const uint32_t* attend, float* a, float* b,
                     int64_t n_mine, const int32_t* mine, void* stream);
/* 0 = ok, 1 = a wait timed out since the last call (synchronises on nothing: read it after a stream sync) */
int gj_peer_status(gj_peer* peer);
int gj_peer_destroy(gj_peer* peer);

/* ---- kernel family of the throughput mode -------------------------------------------------------
 * 1 (default; GJ_PIPE=0 in the environment turns it off): the agent kernels stage every per-agent array of a tile
 * in shared memory with TMA bulk copies (two-stage mbarrier pipeline) — needs every per-agent array 16-byte aligned
 * and readable up to the next multiple of 16 bytes past its end (true of any allocator with >= 16-byte granules);
 * 0: register-batched loads.  Results are bit-identical.  on < 0 only queries.  Returns the previous setting.
 * Bit 1 of `on` (value 2, default clear: measured neutral on B200, see DESIGN.md) allows gj_step_forward_next to
 * produce the look-ahead.  Bit 2 (value 4, default clear) selects the uncompacted transmission pass
 * (k_lean_transmission) instead of the per-warp compacted one (k_lean_transmission_c): same T bit for bit, the
 * partial sums of the cell channels associated differently. */
int gj_pipeline_enable(int on);

/* ---- measurement (bench.py): CUDA events recorded on the launching stream around every kernel ---- */
int gj_profile_enable(int on); /* also resets the counters */
/* per kernel id: summed event time (ms), number of timed launches, number of launches since enable;
 * synchronises on the recorded events; returns the number of kernel ids */
int gj_profile_read(double* ms, int64_t* timed, int64_t* launches, int n);
const char* gj_profile_kernel_name(int id);

/* which kernel family gj_step_forward / gj_step_backward run for this (world, params) when no noise is injected and
 * the packed profile is given: returns 1 = throughput mode, 0 = reference order, < 0 = error; out[0] = offset of
 * the per-global-group region inside the group-sum buffers (throughput mode).  Host-only; used by partitioned
 * callers to locate the sums they exchange. */
int gj_step_plan(const gj_world_desc* w, const gj_step_params* p, int64_t* out, int n);

/* ---- noise ------------------------------------------------------------------------------- */
/* the exact draws gj_step_forward makes for (seed, call_index) and agents first_agent .. first_agent+n-1:
 * E[2][N], u[N], z[N] */
int gj_philox_fill(uint64_t seed, uint32_t call_index, int64_t n, float* E, float* u, float* z, void* stream);
int gj_philox_fill_at(uint64_t seed, uint32_t call_index, uint64_t first_agent, int64_t n, float* E, float* u, float* z,
                      void* stream);
/* raw Philox4x32-10 block for known-answer tests: out[4] = philox(ctr[4], key[2]) (host function) */
void gj_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);
/* raw Philox2x32-10 block (the generator of the step's two exponentials): out[2] = philox(ctr[2], key) */
void gj_philox2x32_10(const uint32_t ctr[2], uint32_t key, uint32_t out[2]);

#ifdef __cplusplus
}
#endif
#endif /* GRADJUNE_B200_H */
