"""Autograd operators over the C ABI (``include/gradjune_b200.h``).

``infection_step`` is the fused timestep (GradJune.forward, model.py:112-144); the stand-alone module
classes call the same entry point with a sub-set of phases.  All tensors must live on a CUDA device;
there is no CPU fallback.
"""
import ctypes as C
import os
from dataclasses import dataclass, field, replace
from typing import Dict, List, Optional, Sequence

import torch

from . import _lib
from ._lib import (KIND_CARE_VISIT, KIND_HOUSEHOLD, KIND_LEISURE, KIND_PLAIN, MODE_SEED, MODE_STEP, PHASE_ALL,
                   PHASE_INFECT, PHASE_NETWORKS, PHASE_SAMPLE, PHASE_SYMPTOMS)
from .world import DeviceWorld

TAU = 0.1
EXACT_ORDER = False   # module-wide switch: run the reference-order kernels even in Philox mode
# batched ensembles: evaluate the draw's noise once for all samples (gj_batch.noise); GJ_BATCH_OWN_NOISE=1 in the
# environment makes every sample regenerate it (measurement switch; bit-identical results)
BATCH_SHARED_NOISE = os.environ.get("GJ_BATCH_OWN_NOISE", "0") != "1"


def require_cuda(t: torch.Tensor, what: str):
    if not t.is_cuda:
        raise _lib.GradJuneLibraryError(
            f"{what} lives on {t.device}: the infection step runs only as CUDA kernels on a B200 "
            "(there is no CPU fallback); move the world to a cuda device (system.device: cuda:0)."
        )


def _f32(t: Optional[torch.Tensor], device=None):
    if t is None:
        return None
    if t.dtype != torch.float32 or not t.is_contiguous() or (device is not None and t.device != device):
        t = t.to(device=device or t.device, dtype=torch.float32).contiguous()
    return t


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _stream(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _on(device):
    """Context that makes ``device`` the current CUDA device for a library call: kernels are launched on the
    current device, so a world on cuda:1 in a process whose current device is cuda:0 would otherwise launch with a
    foreign stream and foreign pointers (ADVICE r1)."""
    return torch.cuda.device(device)


def _noise_order(world: DeviceWorld, t: Optional[torch.Tensor]):
    """Injected noise arrives indexed by the agents' ORIGINAL ids (the order the world was loaded in, which is the
    order the reference / the oracle draws it in); a renumbered world reads it through its permutation."""
    if t is None or world.__dict__.get("orig_id") is None:
        return t
    oi = world.__dict__.get("_orig_index")
    if oi is None:
        oi = world.__dict__["_orig_index"] = world.orig_id.long() & 0xFFFFFFFF
    return t.index_select(-1, oi).contiguous()


# --------------------------------------------------------------------------------------
# noise control
# --------------------------------------------------------------------------------------
class NoiseSource:
    """Where the step's random draws come from.

    Default: counter-based Philox inside the kernels; each call takes a fresh 62-bit key from
    torch's CPU generator, so ``torch.manual_seed`` makes runs reproducible like the reference.
    ``inject`` replaces it by explicit arrays (parity tests): a callable ``call_index -> (E, u, z)``.
    """

    def __init__(self):
        self.injected = None
        self.fixed_seed = None
        self.calls = 0

    def next(self, n_agents, device):
        """-> (seed, call_index, E, u, z)"""
        c = self.calls
        self.calls += 1
        if self.injected is not None:
            E, u, z = self.injected(c)
            return 0, c, _f32(torch.as_tensor(E), device), _f32(torch.as_tensor(u), device), _f32(torch.as_tensor(z), device)
        if self.fixed_seed is not None:
            return int(self.fixed_seed), c, None, None, None
        seed = int(torch.randint(0, 2**62, (1,)).item())
        return seed, 0, None, None, None


NOISE = NoiseSource()


class inject_noise:
    """``with inject_noise(lambda c: (E, u, z)):`` — feed explicit noise arrays to every sampler /
    symptoms call inside the block; call c = 0, 1, 2, ... in call order."""

    def __init__(self, provider):
        self.provider = provider

    def __enter__(self):
        self._saved = (NOISE.injected, NOISE.calls)
        NOISE.injected, NOISE.calls = self.provider, 0
        return NOISE

    def __exit__(self, *exc):
        NOISE.injected, NOISE.calls = self._saved


class philox_seed:
    """``with philox_seed(1234):`` — fixed Philox key, call_index counts calls inside the block."""

    def __init__(self, seed):
        self.seed = seed

    def __enter__(self):
        self._saved = (NOISE.fixed_seed, NOISE.calls)
        NOISE.fixed_seed, NOISE.calls = self.seed, 0
        return NOISE

    def __exit__(self, *exc):
        NOISE.fixed_seed, NOISE.calls = self._saved


def philox_fill(seed: int, call_index: int, n: int, device, first_agent: int = 0):
    """The exact (E[2,N], u[N], z[N]) draws the kernels make for (seed, call_index) and the agents
    first_agent .. first_agent + n - 1 (global ids)."""
    E = torch.empty(2, n, device=device)
    u = torch.empty(n, device=device)
    z = torch.empty(n, device=device)
    with _on(E.device):
        _lib.check(_lib.lib().gj_philox_fill_at(seed, call_index, first_agent, n, E.data_ptr(), u.data_ptr(),
                                                z.data_ptr(), _stream(E.device)), "gj_philox_fill_at")
    return E, u, z


# --------------------------------------------------------------------------------------
# step description
# --------------------------------------------------------------------------------------
@dataclass
class NetSpec:
    name: str
    edge_type: str
    kind: int
    prob_row: int = -1


@dataclass
class SymptomsTables:
    n_stages: int
    stage_prob: torch.Tensor                  # [S, 100] device
    trans: Dict[int, Optional[tuple]]         # i -> (kind, loc, scale) | None
    rec: Dict[int, Optional[tuple]]


@dataclass
class StepSpec:
    now: float
    dt: float
    day_type: int
    nets: List[NetSpec]
    quarantine: Optional[Sequence[float]]     # None / thresholds of the active policies
    phases: int = PHASE_ALL
    mode: int = MODE_STEP
    age_bins: Sequence[int] = ()
    want_reductions: bool = True
    want_lam: bool = False
    want_probs: bool = True     # fused step: also return q (not_infected_probs) and n (new_infected)
    exact_order: bool = False   # force the reference-order kernels even with in-kernel Philox noise


@dataclass(frozen=True)
class Labels:
    """Per-agent label codes of a results-by-label table (cases and deaths per region, area, ...): ``codes[a]`` is
    agent a's column in ``[0, n)``.  Build it with :func:`make_labels`, which checks the range once."""
    codes: torch.Tensor     # [N] int32
    n: int


def make_labels(codes, n: int, device=None) -> Labels:
    """Validated :class:`Labels` (the kernels index the table with the codes unchecked)."""
    codes = torch.as_tensor(codes)
    if codes.dim() != 1 or codes.dtype.is_floating_point or codes.dtype == torch.bool:
        raise ValueError("label codes must be a 1-D integer array")
    n = int(n)
    if not 1 <= n <= 1 << 30:
        raise ValueError(f"the number of label columns must lie in [1, 2^30], got {n}")
    if codes.numel() and (int(codes.min()) < 0 or int(codes.max()) >= n):
        raise ValueError(f"label codes must lie in [0, {n}), got [{int(codes.min())}, {int(codes.max())}]")
    return Labels(codes.to(device=device or codes.device, dtype=torch.int32).contiguous(), n)


@dataclass(frozen=True)
class SeedLabels:
    """Per-agent region codes of seeding by label: ``codes[a]`` in ``[0, n)`` picks agent a's initial-case fraction.
    ``order`` lists the agents stably sorted by code and ``offsets[l]`` is where region l starts in it ([n + 1]):
    the backward's deterministic per-region reduction walks them.  Build it with :func:`make_seed_labels`."""
    codes: torch.Tensor     # [N] int32
    n: int
    order: torch.Tensor     # [N] int32
    offsets: torch.Tensor   # [n + 1] int32


def make_seed_labels(codes, n: int, device=None) -> SeedLabels:
    """Validated :class:`SeedLabels` (range-checked like :func:`make_labels`); ``codes`` may be the codes of a
    :class:`Labels` already on the device, which are then shared."""
    lab = make_labels(codes, n, device)
    if lab.codes.numel() >= 1 << 31:
        raise ValueError("seeding by label supports fewer than 2^31 agents per world")
    order = torch.sort(lab.codes, stable=True).indices.to(torch.int32)
    counts = torch.bincount(lab.codes.long(), minlength=lab.n)
    offsets = torch.zeros(lab.n + 1, dtype=torch.int64, device=lab.codes.device)
    offsets[1:] = torch.cumsum(counts, 0)
    return SeedLabels(lab.codes, lab.n, order.contiguous(), offsets.to(torch.int32).contiguous())


def _set_seed_labels(io, world: DeviceWorld, seed_label: SeedLabels, seed_fraction, nb: int = 1):
    """Point the io struct at the region codes; checks the fraction tensor holds ``n`` values per sample (or ``n``
    shared by the samples)."""
    if seed_label.codes.numel() != world.n_agents or seed_label.codes.device != world.device:
        raise ValueError(f"seed label codes must hold one entry per agent ({world.n_agents}) on {world.device}")
    if seed_fraction.numel() not in (seed_label.n, nb * seed_label.n):
        raise ValueError(f"seed_fraction must hold {seed_label.n} values (one per region)"
                         + (f" or {nb} x {seed_label.n}" if nb > 1 else "") + f", got {seed_fraction.numel()}")
    io.seed_label, io.n_seed_labels = seed_label.codes.data_ptr(), seed_label.n
    if hasattr(io, "seed_order"):
        io.seed_order, io.seed_offsets = seed_label.order.data_ptr(), seed_label.offsets.data_ptr()
        io.seed_work = _buffer(world, "seed_work", world.n_agents).data_ptr()


@dataclass(frozen=True)
class Region:
    """Regional transmission factor of one step: every agent's summed pressure is multiplied by
    ``factor[labels.codes[a]]`` before the clamp.  ``labels`` (:class:`SeedLabels`) holds the per-agent region codes
    and the order / offsets of the backward's deterministic per-region reduction; ``factor`` is [n] ([n] or [b, n]
    batched), differentiable."""
    labels: SeedLabels
    factor: torch.Tensor


def _set_region(io, world: DeviceWorld, labels: SeedLabels, factor):
    """Point the io struct at the region codes and the factors (and, on the backward's struct, at the reduction's order,
    offsets and the per-agent workspace of ``nb`` rows)."""
    if labels.codes.numel() != world.n_agents or labels.codes.device != world.device:
        raise ValueError(f"region codes must hold one entry per agent ({world.n_agents}) on {world.device}")
    io.region, io.n_regions, io.region_factor = labels.codes.data_ptr(), labels.n, factor.data_ptr()
    if hasattr(io, "region_order"):
        io.region_order, io.region_offsets = labels.order.data_ptr(), labels.offsets.data_ptr()


def _region_factor(region: Region, dev, nb: int = 0):
    """The factors as a contiguous fp32 tensor on ``dev``: [n], or [nb, n] for a batch of ``nb`` samples."""
    f = _f32(region.factor, dev)
    n = region.labels.n
    if nb:
        if tuple(f.shape) not in ((n,), (nb, n)):
            raise ValueError(f"a regional factor must hold {n} values (one per region) or {nb} x {n}, got "
                             f"{tuple(f.shape)}")
        return f.expand(nb, n).contiguous()
    if tuple(f.shape) != (n,):
        raise ValueError(f"a regional factor must hold {n} values (one per region), got {tuple(f.shape)}")
    return f.contiguous()


@dataclass(frozen=True)
class VenueLabels:
    """Region codes of the GROUPS (venues) of a world: ``codes[g]`` in ``[0, n)`` is the region of global group g (the
    group's location).  For the backward's deterministic per-region reduction, ``order`` holds every edge type's groups
    (indices within the type) stably sorted by region at the type's positions ``[type_group_off[t],
    type_group_off[t + 1])``, and ``offsets[t * (n + 1) + r]`` is where region r starts in that part.  Build it with
    :func:`make_venue_labels`."""
    codes: torch.Tensor     # [n_groups] int32
    n: int
    order: torch.Tensor     # [n_groups] int32
    offsets: torch.Tensor   # [n_types * (n + 1)] int32


def make_venue_labels(codes, n: int, type_group_off: Sequence[int], device=None) -> VenueLabels:
    """Validated :class:`VenueLabels` from the per-group codes (global group ids, types concatenated as in
    ``type_group_off``): :func:`make_seed_labels` over the groups of each type."""
    lab = make_labels(codes, n, device)
    if lab.codes.numel() != type_group_off[-1]:
        raise ValueError(f"venue region codes must hold one entry per group ({type_group_off[-1]}), "
                         f"got {lab.codes.numel()}")
    orders, offsets = [], []
    for t in range(len(type_group_off) - 1):
        sl = make_seed_labels(lab.codes[type_group_off[t]:type_group_off[t + 1]], lab.n)
        orders.append(sl.order)
        offsets.append(sl.offsets)
    order = torch.cat(orders) if orders else torch.zeros(0, dtype=torch.int32, device=lab.codes.device)
    return VenueLabels(lab.codes, lab.n, order.contiguous(), torch.cat(offsets).contiguous())


@dataclass(frozen=True)
class Venue:
    """Regional venue factor of one step: network k's beta is multiplied by ``factor[k, labels.codes[g]]`` wherever
    group g's ``beta * pc`` is formed (the group passes, the cell tier and d/dbeta), so a factor of 0 closes network k's
    venues in that region.  Row k belongs to the step's k-th network (``StepSpec.nets``); ``factor`` is [K, n]
    ([K, n] or [b, K, n] batched), differentiable."""
    labels: VenueLabels
    factor: torch.Tensor

    def row(self, k: int) -> "Venue":
        """The venue factor of the step's k-th network alone (a one-network call of the same step)."""
        return Venue(self.labels, self.factor[..., k:k + 1, :])


def _venue_factor(labels: VenueLabels, factor, K: int, dev, nb: int = 0):
    """The factor table as a contiguous fp32 tensor on ``dev``: [K, n], or [nb, K, n] for a batch of ``nb``."""
    f = _f32(factor, dev)
    n = labels.n
    if nb:
        if tuple(f.shape) not in ((K, n), (nb, K, n)):
            raise ValueError(f"a venue factor table must hold {K} x {n} values (network x region) or {nb} x {K} x {n}, "
                             f"got {tuple(f.shape)}")
        return f.expand(nb, K, n).contiguous()
    if tuple(f.shape) != (K, n):
        raise ValueError(f"a venue factor table must hold {K} x {n} values (network x region), got {tuple(f.shape)}")
    return f.contiguous()


def _set_venue(io, world: DeviceWorld, labels: VenueLabels, factor):
    """Point the io struct at the group region codes and the factor table (and, on the backward's struct, at the
    reduction's order and offsets)."""
    if labels.codes.numel() != world.n_groups or labels.codes.device != world.device:
        raise ValueError(f"venue region codes must hold one entry per group ({world.n_groups}) on {world.device}")
    io.venue_region, io.n_venue_regions, io.venue_factor = labels.codes.data_ptr(), labels.n, factor.data_ptr()
    if hasattr(io, "venue_order"):
        io.venue_order, io.venue_offsets = labels.order.data_ptr(), labels.offsets.data_ptr()


def _label_acc(world: DeviceWorld, n: int):
    """The integer accumulator of the label table ([n] uint32, zero; every call leaves it zero)."""
    t = world.__dict__.get("_label_acc")
    if t is None or t.numel() < n:
        t = world.__dict__["_label_acc"] = torch.zeros(n, dtype=torch.int32, device=world.device)
    return t


def _set_labels(io, world: DeviceWorld, label: Labels, nb: int = 1):
    """Point the io struct at the label codes, a new [nb, n, 2] table and the accumulator; returns the table."""
    if label.codes.numel() != world.n_agents or label.codes.device != world.device:
        raise ValueError(f"label codes must hold one entry per agent ({world.n_agents}) on {world.device}")
    table = torch.empty(nb, label.n, 2, dtype=torch.float32, device=world.device)
    io.label, io.n_labels, io.red_label = label.codes.data_ptr(), label.n, table.data_ptr()
    io.label_acc = _label_acc(world, nb * 2 * label.n).data_ptr()
    return table


def _scratch(world: DeviceWorld):
    sc = getattr(world, "_scratch", None)
    if sc is None:
        nbytes = _lib.lib().gj_scratch_bytes(C.byref(world.desc()))
        sc = torch.zeros(nbytes, dtype=torch.uint8, device=world.device)
        world._scratch = sc
    return sc


def _buffer(world: DeviceWorld, name: str, n: int):
    """Reusable per-world workspace (transient between the launches of one call)."""
    cache = world.__dict__.setdefault("_buffers", {})
    t = cache.get(name)
    if t is None or t.numel() < n:
        t = torch.empty(max(n, 1), dtype=torch.float32, device=world.device)
        cache[name] = t
    return t


_PARAMS_CACHE: dict = {}


def _fill_params(world: DeviceWorld, spec: StepSpec, sym: Optional[SymptomsTables], seed: int, call_index: int):
    """gj_step_params of this call.  Everything but (now, dt, seed, call_index) depends only on the step's
    structure, so the filled struct is cached per structure and copied."""
    key = (id(world), tuple((n.edge_type, n.kind, n.prob_row) for n in spec.nets),
           None if spec.quarantine is None else tuple(float(t) for t in spec.quarantine), id(sym),
           tuple(spec.age_bins), spec.mode, spec.phases, int(spec.day_type), bool(spec.exact_order))
    hit = _PARAMS_CACHE.get(key)
    if hit is None or hit[2] is not world or hit[3] is not sym:
        if len(_PARAMS_CACHE) > 256:
            _PARAMS_CACHE.clear()
        p0, off = _build_params(world, spec, sym)
        _PARAMS_CACHE[key] = hit = (bytes(p0), off, world, sym)
    p = _lib.StepParams.from_buffer_copy(hit[0])
    p.now, p.dt = float(spec.now), float(spec.dt)
    p.seed, p.call_index = int(seed), int(call_index)
    return p, hit[1]


def _build_params(world: DeviceWorld, spec: StepSpec, sym: Optional[SymptomsTables]):
    p = _lib.StepParams()
    p.mode, p.phases = spec.mode, spec.phases
    p.day_type = int(spec.day_type)
    if len(spec.nets) > _lib.GJ_MAX_NETS:
        raise ValueError(f"at most {_lib.GJ_MAX_NETS} networks per step")
    p.n_nets = len(spec.nets)
    off = 0
    for k, net in enumerate(spec.nets):
        ti = world.types.index(net.edge_type)
        p.nets[k].type, p.nets[k].kind, p.nets[k].prob_row, p.nets[k].s_off = ti, net.kind, net.prob_row, off
        off += world.type_group_off[ti + 1] - world.type_group_off[ti]
    if off >= (1 << 31):
        raise ValueError("group-sum buffer too large")
    if spec.quarantine is None:
        p.n_quar = -1
    else:
        if len(spec.quarantine) > _lib.GJ_MAX_QUAR:
            raise ValueError(f"at most {_lib.GJ_MAX_QUAR} simultaneous quarantine policies")
        p.n_quar = len(spec.quarantine)
        for i, thr in enumerate(spec.quarantine):
            p.quar_thr[i] = float(thr)
    if sym is not None:
        if sym.n_stages > _lib.GJ_MAX_STAGES:
            raise ValueError("too many symptom stages")
        p.n_stages = sym.n_stages
        for i in range(_lib.GJ_MAX_STAGES):
            for arr, table in ((p.trans_time, sym.trans), (p.rec_time, sym.rec)):
                e = table.get(i)
                if e is None:
                    arr[i].kind = -1
                else:
                    arr[i].kind, arr[i].loc, arr[i].scale = int(e[0]), float(e[1]), float(e[2])
    else:
        p.n_stages = 8
        for i in range(_lib.GJ_MAX_STAGES):
            p.trans_time[i].kind = p.rec_time[i].kind = -1
    bins = list(spec.age_bins)
    if len(bins) - 1 > _lib.GJ_MAX_AGE_BINS:
        raise ValueError("too many age bins")
    p.n_age_bins = max(len(bins) - 1, 0)
    for i, b in enumerate(bins):
        p.age_bins[i] = int(b)
    p.tau = TAU
    p.exact_order = 1 if spec.exact_order else 0
    return p, off


@dataclass
class StepStatic:
    """Per-world constants of the step: profile parameters and lookup tables (device tensors)."""
    world: DeviceWorld
    maxinf: Optional[torch.Tensor] = None
    shape: Optional[torch.Tensor] = None
    rate: Optional[torch.Tensor] = None
    shift: Optional[torch.Tensor] = None
    k0: Optional[torch.Tensor] = None
    prof4: Optional[torch.Tensor] = None          # [N, 4] packed profile (gj_profile_pack)
    leisure_prob: Optional[torch.Tensor] = None   # [n_tables, 2, 2, 100]
    symptoms: Optional[SymptomsTables] = None
    exchange: object = None                       # partition.BoundaryExchange of a partitioned world


def profile_k0(shape: torch.Tensor) -> torch.Tensor:
    require_cuda(shape, "infection_parameters['shape']")
    shape = _f32(shape)
    k0 = torch.empty_like(shape)
    with _on(shape.device):
        _lib.check(_lib.lib().gj_profile_prepare(shape.numel(), shape.data_ptr(), k0.data_ptr(), _stream(shape.device)),
                   "gj_profile_prepare")
    return k0


def profile_pack(maxinf, shape, rate, shift, k0) -> torch.Tensor:
    """[N, 4] = {maxinf*k0*rate, rate, shape-1, shift}: the profile as one 16-byte word per agent."""
    out = torch.empty(shape.numel(), 4, dtype=torch.float32, device=shape.device)
    with _on(shape.device):
        _lib.check(_lib.lib().gj_profile_pack(shape.numel(), maxinf.data_ptr(), shape.data_ptr(), rate.data_ptr(),
                                              shift.data_ptr(), k0.data_ptr(), out.data_ptr(), _stream(shape.device)),
                   "gj_profile_pack")
    return out


class _Transmission(torch.autograd.Function):
    """TransmissionUpdater.forward (transmission.py:38-51) and its derivative."""

    @staticmethod
    def forward(ctx, now, tinf, inf, maxinf, shape, rate, shift, k0):
        dev = tinf.device
        tinf, inf = _f32(tinf), _f32(inf)
        T = torch.empty_like(tinf)
        with _on(dev):
            _lib.check(_lib.lib().gj_transmission_forward(
                tinf.numel(), float(now), tinf.data_ptr(), inf.data_ptr(), maxinf.data_ptr(), shape.data_ptr(),
                rate.data_ptr(), shift.data_ptr(), k0.data_ptr(), T.data_ptr(), _stream(dev)), "gj_transmission_forward")
        ctx.save_for_backward(tinf, inf, maxinf, shape, rate, shift, k0)
        ctx.now = float(now)
        return T

    @staticmethod
    def backward(ctx, gT):
        tinf, inf, maxinf, shape, rate, shift, k0 = ctx.saved_tensors
        gT = _f32(gT)
        g_tinf = torch.empty_like(tinf)
        g_inf = torch.empty_like(tinf)
        with _on(tinf.device):
            _lib.check(_lib.lib().gj_transmission_backward(
                tinf.numel(), ctx.now, tinf.data_ptr(), inf.data_ptr(), maxinf.data_ptr(), shape.data_ptr(),
                rate.data_ptr(), shift.data_ptr(), k0.data_ptr(), gT.data_ptr(), g_tinf.data_ptr(), g_inf.data_ptr(),
                _stream(tinf.device)), "gj_transmission_backward")
        return None, g_tinf, g_inf, None, None, None, None, None


def transmission(now, tinf, inf, maxinf, shape, rate, shift, k0=None):
    for t, name in ((tinf, "infection_time"), (inf, "is_infected"), (shape, "infection_parameters")):
        require_cuda(t, name)
    maxinf, shape, rate, shift = _f32(maxinf), _f32(shape), _f32(rate), _f32(shift)
    if k0 is None:
        k0 = profile_k0(shape)
    return _Transmission.apply(now, tinf, inf, maxinf, shape, rate, shift, k0)


_STATE = ("s", "inf", "tinf", "cur", "nxt", "ttn")


def step_plan(static: "StepStatic", spec: "StepSpec") -> str:
    """Which kernel family ``gj_step_forward`` runs for this step when the noise is the in-kernel Philox stream:
    "throughput" (gj_lean.cuh / gj_pipe.cuh) or "reference-order" (gj_tiled.cuh) — ``gj_step_plan``."""
    if EXACT_ORDER and not spec.exact_order:
        spec = replace(spec, exact_order=True)
    p, _ = _fill_params(static.world, spec, static.symptoms, 0, 0)
    out = (C.c_int64 * 1)()
    rc = _lib.lib().gj_step_plan(C.byref(static.world.desc()), C.byref(p), out, 1)
    if rc < 0:
        _lib.check(rc, "gj_step_plan")
    return "throughput" if (rc == 1 and static.prof4 is not None) else "reference-order"


def _staged_call(fn, what, static: "StepStatic", desc, p, io, stream, sum_buffers, lean_inputs: bool, p_next=None):
    """One library call, or — for a partitioned world — the two stages of it with the all-reduce of the boundary
    groups' sums (``sum_buffers``: the two group-sum tensors of this call) in between.  ``p_next``: parameters of
    the following step for gj_step_forward_next.  Returns the library's (non-negative) return code."""
    world = static.world
    world.__dict__["_calls"] = world.__dict__.get("_calls", 0) + 1   # the per-world scratch changes hands

    def call():
        with _on(world.device):
            if p_next is not None:
                rc = _lib.lib().gj_step_forward_next(C.byref(desc), C.byref(p), C.byref(p_next), C.byref(io), stream)
            else:
                rc = fn(C.byref(desc), C.byref(p), C.byref(io), stream)
        if rc < 0:
            _lib.check(rc, what)
        return rc

    ex = static.exchange
    if ex is None or sum_buffers is None:
        return call()
    out = (C.c_int64 * 1)()
    lean = _lib.lib().gj_step_plan(C.byref(desc), C.byref(p), out, 1)
    if lean < 0:
        _lib.check(lean, "gj_step_plan")
    lean = bool(lean) and lean_inputs
    region = ex.regions(lean, int(out[0]), [(p.nets[k].type, p.nets[k].s_off) for k in range(p.n_nets)])
    p.stage = _lib.STAGE_SUMS
    call()
    ex.exchange(sum_buffers, region)
    p.stage = _lib.STAGE_REST
    rc = call()
    p.stage = _lib.STAGE_ALL
    return rc


def _spec_key(spec: "StepSpec"):
    """What the transmission pass of a step depends on besides the state (look-ahead bookkeeping)."""
    return (float(spec.now), int(spec.day_type), tuple((n.edge_type, n.kind, n.prob_row) for n in spec.nets),
            None if spec.quarantine is None else tuple(float(t) for t in spec.quarantine), spec.mode, spec.phases,
            bool(spec.exact_order))


def _same(t, ref):
    return t is not None and ref is not None and t.data_ptr() == ref.data_ptr() and t._version == ref._version \
        and t.shape == ref.shape


class _Step(torch.autograd.Function):
    """gj_step_forward / gj_step_backward.

    Differentiable inputs: beta[K], the six state tensors, T_in / q_in / n_in (stand-alone phases)
    and the seeding fraction.  Outputs: six new state tensors, T, q, n, reductions.
    """

    @staticmethod
    def forward(ctx, static: StepStatic, spec: StepSpec, noise, beta, s, inf, tinf, cur, nxt, ttn, T_in, q_in, n_in,
                seed_fraction, next_spec=None, label: Optional[Labels] = None, seed_label: Optional[SeedLabels] = None,
                region_labels: Optional[SeedLabels] = None, region_factor=None,
                venue_labels: Optional[VenueLabels] = None, venue_factor=None):
        world = static.world
        dev = world.device
        N = world.n_agents
        L = _lib.lib()
        seed, call_index, E, u, z = noise
        E, u, z = _noise_order(world, E), _noise_order(world, u), _noise_order(world, z)
        if EXACT_ORDER and not spec.exact_order:   # pin the choice: the backward must run the same kernel family
            spec = replace(spec, exact_order=True)
        p, s_total = _fill_params(world, spec, static.symptoms, seed, call_index)
        io = _lib.FwdIO()
        keep = []

        def put(name, t):
            t = _f32(t, dev)
            if t is not None:
                keep.append(t)
                setattr(io, name, t.data_ptr())
            return t

        phases, seed_mode = spec.phases, spec.mode == MODE_SEED
        nets_on = bool(phases & PHASE_NETWORKS) and not seed_mode
        beta = put("beta", beta) if nets_on else None
        region_labels = region_labels if nets_on else None
        if region_labels is not None:
            region_factor = _region_factor(Region(region_labels, region_factor), dev)
            keep.append(region_factor)
            _set_region(io, world, region_labels, region_factor)
        else:
            region_factor = None
        venue_labels = venue_labels if nets_on else None
        if venue_labels is not None:
            venue_factor = _venue_factor(venue_labels, venue_factor, p.n_nets, dev)
            keep.append(venue_factor)
            _set_venue(io, world, venue_labels, venue_factor)
        else:
            venue_factor = None
        put("leisure_prob", static.leisure_prob)
        if static.symptoms is not None:
            put("stage_prob", static.symptoms.stage_prob)
        seed_fraction = put("seed_fraction", seed_fraction) if seed_mode else None
        seed_label = seed_label if seed_mode else None
        if seed_label is not None:
            _set_seed_labels(io, world, seed_label, seed_fraction)
        put("inj_E", E), put("inj_u", u), put("inj_z", z)
        st = {}
        for name, t in zip(_STATE, (s, inf, tinf, cur, nxt, ttn)):
            st[name] = put(name, t)
        fused_T = nets_on and T_in is None
        if fused_T:
            for name in ("maxinf", "shape", "rate", "shift", "k0", "prof4"):
                put(name, getattr(static, name))
        T_in, q_in, n_in = put("T_in", T_in), put("q_in", q_in), put("n_in", n_in)

        def new(name):
            t = torch.empty(N, dtype=torch.float32, device=dev)
            setattr(io, name, t.data_ptr())
            return t

        out = {}
        if phases & PHASE_INFECT:
            for name in ("s_o", "inf_o", "tinf_o"):
                out[name] = new(name)
        if phases & PHASE_SYMPTOMS:
            for name in ("cur_o", "nxt_o", "ttn_o"):
                out[name] = new(name)
        T = None
        fused_all = fused_T and phases == PHASE_ALL
        # look-ahead: the previous step's forward may already have run this step's transmission pass
        pf = world.__dict__.pop("_prefetch", None)
        tq_name = "Tq0"
        if (pf is not None and fused_all and E is None and u is None and z is None and pf["key"] == _spec_key(spec)
                and pf["calls"] == world.__dict__.get("_calls", 0) and _same(st["inf"], pf["inf"])
                and _same(st["tinf"], pf["tinf"]) and _same(st["cur"], pf["cur"])):
            T = pf["T"]
            io.T = T.data_ptr()
            io.Tq = pf["Tq"].data_ptr() if p.n_quar > 0 else T.data_ptr()
            tq_name = pf["tq_name"]
            p.t_ready = 1
            keep.append(pf)
            world.__dict__["_scatter_pending"] = False
        elif fused_T:
            T = new("T")
            io.Tq = _buffer(world, tq_name, N).data_ptr() if p.n_quar > 0 else T.data_ptr()
        elif nets_on and p.n_quar > 0:
            io.Tq = _buffer(world, tq_name, N).data_ptr()
        probs = spec.want_probs or not fused_all   # the fused step needs neither q nor n for its own backward
        q = new("q") if (nets_on and probs) else None
        lam = new("lam") if (nets_on and spec.want_lam) else None
        n = new("n") if ((phases & PHASE_SAMPLE) and probs) else None
        tape_v = new("tape_v") if nets_on else None
        tape_y0 = new("tape_y0") if (phases & PHASE_SAMPLE) else None
        S_un = S_sc = None
        if nets_on:
            s_total += world.n_groups   # per-network sums, then one value per global group (throughput mode)
            S_sc = _buffer(world, "S_scaled", s_total)
            io.S_scaled = S_sc.data_ptr()
            S_un = torch.empty(max(s_total, 1), dtype=torch.float32, device=dev)
            io.S_unscaled = S_un.data_ptr()
        red = None
        if spec.want_reductions:
            red = torch.empty(2 + p.n_age_bins, dtype=torch.float32, device=dev)
            io.red = red.data_ptr()
        red_label = _set_labels(io, world, label)[0] if label is not None else None
        io.scratch = _scratch(world).data_ptr()
        desc = world.desc()
        if world.__dict__.get("_scatter_pending"):
            # a look-ahead scattered the next step's transmissions into the group accumulators, but this call is not
            # that step: have the library clear them first
            p.reset_scatter = 1
            world.__dict__["_scatter_pending"] = False
        if static.exchange is not None:
            p.agent_offset = static.exchange.part.agent_lo
        lean_inputs = E is None and u is None and z is None and T_in is None and lam is None and static.prof4 is not None
        p_next = T_next = Tq_next = None
        if (next_spec is not None and fused_all and lean_inputs and not seed_mode and label is None
                and region_labels is None):
            # also run the NEXT step's transmission pass inside this step's agent kernel (gj_step_forward_next)
            p_next, _ = _fill_params(world, next_spec, static.symptoms, 0, 0)
            T_next = torch.empty(N, dtype=torch.float32, device=dev)
            io.T_next = T_next.data_ptr()
            if p_next.n_quar > 0:
                next_tq_name = "Tq1" if tq_name == "Tq0" else "Tq0"   # this step's kernels still read the other one
                Tq_next = _buffer(world, next_tq_name, N)
                io.Tq_next = Tq_next.data_ptr()
        rc = _staged_call(L.gj_step_forward, "gj_step_forward", static, desc, p, io, _stream(dev),
                          (S_sc, S_un) if nets_on else None, lean_inputs, p_next=p_next)
        if p_next is not None and rc == 1:
            world.__dict__["_scatter_pending"] = True
            world.__dict__["_prefetch"] = dict(
                key=_spec_key(next_spec), calls=world.__dict__.get("_calls", 0), T=T_next, Tq=Tq_next,
                tq_name=next_tq_name if Tq_next is not None else "Tq0", inf=out.get("inf_o"), tinf=out.get("tinf_o"),
                cur=out.get("cur_o"))

        ctx.static, ctx.spec, ctx.noise_key, ctx.label = static, spec, (seed, call_index), label
        ctx.seed_label, ctx.region_labels, ctx.venue_labels = seed_label, region_labels, venue_labels
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(beta, st["s"], st["inf"], st["tinf"], st["cur"], st["nxt"], st["ttn"],
                              T_in if T_in is not None else T, q_in, n_in,
                              seed_fraction, out.get("inf_o"), tape_v, tape_y0, S_un, E, u, z, q, n, region_factor,
                              venue_factor)
        ctx.fused_T = fused_T
        outs = (out.get("s_o"), out.get("inf_o"), out.get("tinf_o"), out.get("cur_o"), out.get("nxt_o"),
                out.get("ttn_o"), T, q, n, red, lam, red_label)
        nd = [t for t in (T,) if t is not None]
        if (phases & PHASE_SAMPLE) and q is not None:
            nd.append(q)   # fused: q is a by-product; its cotangent path runs through the sampler
        if (phases & PHASE_INFECT) and n is not None:
            nd.append(n)
        ctx.mark_non_differentiable(*nd)
        return outs

    @staticmethod
    def backward(ctx, g_s_o, g_inf_o, g_tinf_o, g_cur_o, g_nxt_o, g_ttn_o, g_T, g_q, g_n, g_red, g_lam, g_red_label):
        static, spec = ctx.static, ctx.spec
        world = static.world
        dev, N = world.device, world.n_agents
        (beta, s, inf, tinf, cur, nxt, ttn, T_in, q_in, n_in, seed_fraction, inf_o, tape_v, tape_y0, S_un, E, u, z,
         q_saved, n_saved, region_factor, venue_factor) = ctx.saved_tensors
        seed, call_index = ctx.noise_key
        p, s_total = _fill_params(world, spec, static.symptoms, seed, call_index)
        phases, seed_mode = spec.phases, spec.mode == MODE_SEED
        nets_on = bool(phases & PHASE_NETWORKS) and not seed_mode
        io = _lib.BwdIO()
        keep = []

        def put(name, t):
            t = _f32(t, dev)
            if t is not None:
                keep.append(t)
                setattr(io, name, t.data_ptr())
            return t

        put("beta", beta), put("leisure_prob", static.leisure_prob)
        if static.symptoms is not None:
            put("stage_prob", static.symptoms.stage_prob)
        put("seed_fraction", seed_fraction)
        put("inj_E", E), put("inj_u", u), put("inj_z", z)
        for name, t in zip(_STATE, (s, inf, tinf, cur, nxt, ttn)):
            put(name, t)
        fused_T = ctx.fused_T
        if fused_T:
            for name in ("maxinf", "shape", "rate", "shift", "k0", "prof4"):
                put(name, getattr(static, name))
        put("inf_o", inf_o)
        if inf_o is None:
            put("n_in", n_in if n_in is not None else n_saved)
        put("T_in", T_in), put("q_in", q_in if q_in is not None else None)
        put("tape_v", tape_v), put("tape_y0", tape_y0), put("S_unscaled", S_un)
        for name, g in (("g_s_o", g_s_o), ("g_inf_o", g_inf_o), ("g_tinf_o", g_tinf_o), ("g_cur_o", g_cur_o),
                        ("g_nxt_o", g_nxt_o), ("g_ttn_o", g_ttn_o), ("g_red", g_red)):
            put(name, g)
        if nets_on and not (phases & PHASE_SAMPLE):
            put("g_q", g_q)
        if nets_on:
            put("g_lam", g_lam)
        if (phases & PHASE_SAMPLE) and not (phases & PHASE_INFECT):
            put("g_n", g_n)
        if g_red_label is not None:
            put("g_red_label", g_red_label)
            io.label = ctx.label.codes.data_ptr()

        need = ctx.needs_input_grad  # (static, spec, noise, beta, s, inf, tinf, cur, nxt, ttn, T_in, q_in, n_in, frac,
        #                                next_spec, label, seed_label, region_labels, region_factor, venue_labels,
        #                                venue_factor)
        g_region = None
        if ctx.region_labels is not None:   # the per-agent terms always; their per-region sums when wanted
            _set_region(io, world, ctx.region_labels, region_factor)
            io.region_work = _buffer(world, "region_work", N).data_ptr()
            if need[18]:
                g_region = torch.empty(ctx.region_labels.n, dtype=torch.float32, device=dev)
                io.g_region_factor = g_region.data_ptr()

        def new(name, n=N, zero=False):
            t = (torch.zeros if zero else torch.empty)(n, dtype=torch.float32, device=dev)
            setattr(io, name, t.data_ptr())
            return t

        grads = {}
        for i, name in enumerate(_STATE):
            src = (s, inf, tinf, cur, nxt, ttn)[i]
            if src is not None and need[4 + i]:
                grads[name] = new("g_" + name)
        # the gather pass accumulates into g_inf / g_tinf, so they must exist when the fused networks ran
        if fused_T:
            for name in ("inf", "tinf"):
                if name not in grads:
                    grads[name] = new("g_" + name)
        g_T_in = new("g_T") if (nets_on and not fused_T) else None
        g_q_in = new("g_q_out") if (q_in is not None and need[11]) else None
        g_n_in = new("g_n_out") if (n_in is not None and need[12]) else None
        g_beta = new("g_beta", max(p.n_nets, 1), zero=True) if nets_on else None
        g_frac = None
        if seed_mode and ctx.seed_label is not None:   # one gradient per region
            _set_seed_labels(io, world, ctx.seed_label, seed_fraction)
            g_frac = new("g_seed_fraction", ctx.seed_label.n).reshape(seed_fraction.shape)
        elif seed_mode:
            g_frac = new("g_seed_fraction", 1, zero=True)
        R_buf = cR_buf = None
        if nets_on:
            s_total += world.n_groups
            io.w = _buffer(world, "w", N).data_ptr()
            io.wq = _buffer(world, "wq", N).data_ptr() if p.n_quar > 0 else io.w
            R_buf, cR_buf = _buffer(world, "R", s_total), _buffer(world, "cR", s_total)
            io.R, io.cR = R_buf.data_ptr(), cR_buf.data_ptr()
        g_venue = None
        if ctx.venue_labels is not None:   # the group passes always; the per-region gradient when wanted
            _set_venue(io, world, ctx.venue_labels, venue_factor)
            if need[20]:
                g_venue = torch.empty(p.n_nets, ctx.venue_labels.n, dtype=torch.float32, device=dev)
                io.g_venue_factor = g_venue.data_ptr()
                io.venue_work = _buffer(world, "venue_work", s_total).data_ptr()
        io.scratch = _scratch(world).data_ptr()
        desc = world.desc()
        if static.exchange is not None:
            p.agent_offset = static.exchange.part.agent_lo
        lean_inputs = (E is None and u is None and z is None and g_T_in is None and g_lam is None
                       and static.prof4 is not None and io.g_q is None and io.g_n is None)
        _staged_call(_lib.lib().gj_step_backward, "gj_step_backward", static, desc, p, io, _stream(dev),
                     (cR_buf, R_buf) if nets_on else None, lean_inputs)
        if g_beta is not None:
            g_beta = g_beta[: p.n_nets]
        return (None, None, None, g_beta if need[3] else None,
                grads.get("s") if need[4] else None, grads.get("inf") if need[5] else None,
                grads.get("tinf") if need[6] else None, grads.get("cur") if need[7] else None,
                grads.get("nxt") if need[8] else None, grads.get("ttn") if need[9] else None,
                g_T_in if need[10] else None, g_q_in, g_n_in, g_frac if need[13] else None, None, None, None, None,
                g_region, None, g_venue)


# --------------------------------------------------------------------------------------
# batched ensemble: b samples per call (gj_step_forward_batch / gj_step_backward_batch)
# --------------------------------------------------------------------------------------
# which stride every pointer field of the io structs moves by from one sample to the next (fields not listed are
# shared by the samples: the lookup tables and the infectiousness profile)
_AGENT_FIELDS = {"s", "inf", "tinf", "cur", "nxt", "ttn", "T_in", "q_in", "n_in", "s_o", "inf_o", "tinf_o", "cur_o",
                 "nxt_o", "ttn_o", "T", "Tq", "q", "lam", "n", "tape_v", "tape_y0", "g_s_o", "g_inf_o", "g_tinf_o",
                 "g_cur_o", "g_nxt_o", "g_ttn_o", "g_s", "g_inf", "g_tinf", "g_cur", "g_nxt", "g_ttn", "w", "wq"}
_GROUP_FIELDS = {"S_scaled", "S_unscaled", "R", "cR"}


def _scratch_batch(world: DeviceWorld, nb: int):
    """Per-sample scratch buffers of a batched call: (tensor, stride in bytes)."""
    stride = int(_lib.lib().gj_scratch_bytes(C.byref(world.desc())))
    stride = (stride + 255) // 256 * 256
    hit = world.__dict__.get("_scratch_b")
    if hit is None or hit[0].numel() < nb * stride:
        hit = world.__dict__["_scratch_b"] = (torch.zeros(nb * stride, dtype=torch.uint8, device=world.device), stride)
    return hit


def _row_calls(fn, what, world, desc, p, io, nb, strides, stream):
    """A call the library does not batch (the seeding step): one ordinary call per sample on its slices."""
    for r in range(nb):
        row = type(io)()
        for name, _ in io._fields_:
            v = getattr(io, name)
            if v:
                v += r * strides.get(name, 0)
            setattr(row, name, v)
        with _on(world.device):
            _lib.check(fn(C.byref(desc), C.byref(p), C.byref(row), stream), what)


class _BatchStep(torch.autograd.Function):
    """The fused step (and the seeding step) for a batch of b independent samples on one world: state tensors
    [b, Np] (Np = n_agents rounded up to a multiple of 4; sample rows 16-byte aligned), beta [b, K], reductions
    [b, 2 + bins].  The fused step is ONE library call (``gj_step_forward_batch``): the b samples share every read of
    the world's index data and of the infectiousness profile; the seeding step (once per window) runs per sample.
    All samples draw the same Philox stream (common random numbers), so sample r is bit-identical to an unbatched
    run with the same seed and beta[r]."""

    @staticmethod
    def forward(ctx, static: StepStatic, spec: StepSpec, noise, beta, s, inf, tinf, cur, nxt, ttn, seed_fraction,
                label: Optional[Labels] = None, seed_label: Optional[SeedLabels] = None,
                region_labels: Optional[SeedLabels] = None, region_factor=None,
                venue_labels: Optional[VenueLabels] = None, venue_factor=None):
        world = static.world
        dev, N = world.device, world.n_agents
        L = _lib.lib()
        seed, call_index, E, u, z = noise
        if E is not None or u is not None or z is not None:
            raise _lib.GradJuneLibraryError("batched ensembles draw the in-kernel Philox noise (no injected arrays)")
        nb, Np = s.shape
        if Np % 4 or Np < N:
            raise ValueError(f"batched state must be [b, Np] with Np >= n_agents and Np % 4 == 0, got {tuple(s.shape)}")
        seed_mode = spec.mode == MODE_SEED
        if EXACT_ORDER or spec.exact_order:
            raise _lib.GradJuneLibraryError("batched ensembles run the throughput-mode kernels only")
        if not seed_mode and (spec.phases != PHASE_ALL or step_plan(static, spec) != "throughput"):
            raise _lib.GradJuneLibraryError(
                "batched ensembles need the whole fused step on the throughput-mode kernels (gj_step_plan = 1): "
                "renumber the world (Runner.get_data does) and use the built-in network kinds")
        p, s_total = _fill_params(world, spec, static.symptoms, seed, call_index)
        io = _lib.FwdIO()
        keep = []

        def put(name, t):
            t = _f32(t, dev)
            if t is not None:
                keep.append(t)
                setattr(io, name, t.data_ptr())
            return t

        def new(name):
            t = torch.empty(nb, Np, dtype=torch.float32, device=dev)
            if Np > N:
                t[:, N:] = 0.0          # the kernels never touch the padding
            setattr(io, name, t.data_ptr())
            return t

        put("leisure_prob", static.leisure_prob)
        put("stage_prob", static.symptoms.stage_prob)
        st = {}
        for name, t in zip(_STATE, (s, inf, tinf, cur, nxt, ttn)):
            st[name] = put(name, t)
            if tuple(st[name].shape) != (nb, Np):
                raise ValueError(f"batched state '{name}' has shape {tuple(st[name].shape)}, expected {(nb, Np)}")
        out = {name: new(name) for name in ("s_o", "inf_o", "tinf_o", "cur_o", "nxt_o", "ttn_o")}
        tape_y0 = new("tape_y0")
        nr = 2 + p.n_age_bins
        red = None
        if spec.want_reductions:
            red = torch.empty(nb, nr, dtype=torch.float32, device=dev)
            io.red = red.data_ptr()
        red_label = _set_labels(io, world, label, nb) if label is not None else None
        n_lab = 2 * label.n if label is not None else 0
        scratch, scr_stride = _scratch_batch(world, nb)
        io.scratch = scratch.data_ptr()
        desc = world.desc()
        strides = {name: 4 * Np for name in _AGENT_FIELDS}
        strides.update(red=4 * nr, scratch=scr_stride, red_label=4 * n_lab, label_acc=4 * n_lab)
        T = tape_v = S_un = None
        sG = K = 0
        if not seed_mode:
            seed_label = None
        if seed_mode:
            region_labels = venue_labels = None
        rf, n_reg = None, 0
        if region_labels is not None:   # [b, R]: every sample its own row of factors
            rf = _region_factor(Region(region_labels, region_factor), dev, nb)
            keep.append(rf)
            _set_region(io, world, region_labels, rf)
            n_reg = region_labels.n
        vf, n_ven = None, 0
        if venue_labels is not None:    # [b, K, R]: every sample its own table of factors
            vf = _venue_factor(venue_labels, venue_factor, p.n_nets, dev, nb)
            keep.append(vf)
            _set_venue(io, world, venue_labels, vf)
            n_ven = p.n_nets * venue_labels.n
        if seed_mode:
            seed_fraction = put("seed_fraction", seed_fraction)
            R = 1
            if seed_label is not None:   # seeding by label: [R] shared by the samples or [b, R]
                _set_seed_labels(io, world, seed_label, seed_fraction, nb)
                R = seed_label.n
            elif seed_fraction.numel() not in (1, nb):
                raise ValueError("seed_fraction must hold 1 or b values")
            strides["seed_fraction"] = 4 * R if seed_fraction.numel() == nb * R else 0
            beta = None
            _row_calls(L.gj_step_forward, "gj_step_forward", world, desc, p, io, nb, strides, _stream(dev))
        else:
            seed_fraction = None
            beta = put("beta", beta)
            K = p.n_nets
            if tuple(beta.shape) != (nb, K):
                raise ValueError(f"batched beta has shape {tuple(beta.shape)}, expected {(nb, K)}")
            for name in ("maxinf", "shape", "rate", "shift", "k0", "prof4"):
                put(name, getattr(static, name))
            T = new("T")
            io.Tq = _buffer(world, "Tq_b", nb * Np).data_ptr() if p.n_quar > 0 else T.data_ptr()
            tape_v = new("tape_v")
            sG = s_total + world.n_groups
            io.S_scaled = _buffer(world, "S_scaled_b", nb * sG).data_ptr()
            S_un = torch.empty(nb, max(sG, 1), dtype=torch.float32, device=dev)
            io.S_unscaled = S_un.data_ptr()
            # the samples share the Philox stream: the draw's Gumbel noise is evaluated once per agent
            noise_buf = _buffer(world, "noise_b", Np) if BATCH_SHARED_NOISE else None
            bt = _lib.Batch(n_samples=nb, agent_stride=Np, group_stride=max(sG, 1), beta_stride=K, red_stride=nr,
                            scratch_stride=scr_stride, noise=_ptr(noise_buf), label_stride=n_lab, region_stride=n_reg,
                            venue_stride=n_ven)
            with _on(dev):
                _lib.check(L.gj_step_forward_batch(C.byref(desc), C.byref(p), C.byref(io), C.byref(bt), _stream(dev)),
                           "gj_step_forward_batch")
        ctx.static, ctx.spec, ctx.noise_key, ctx.label = static, spec, (seed, call_index), label
        ctx.seed_label, ctx.region_labels = seed_label, region_labels
        ctx.region_shape = tuple(region_factor.shape) if region_labels is not None else None
        ctx.venue_labels = venue_labels
        ctx.venue_shape = tuple(venue_factor.shape) if venue_labels is not None else None
        ctx.shape = (nb, Np, sG, K, nr)
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(beta, st["s"], st["inf"], st["tinf"], st["cur"], st["nxt"], st["ttn"], T, seed_fraction,
                              out["inf_o"], tape_v, tape_y0, S_un, rf, vf)
        if T is not None:
            ctx.mark_non_differentiable(T)
        return (out["s_o"], out["inf_o"], out["tinf_o"], out["cur_o"], out["nxt_o"], out["ttn_o"], T, red, red_label)

    @staticmethod
    def backward(ctx, g_s_o, g_inf_o, g_tinf_o, g_cur_o, g_nxt_o, g_ttn_o, g_T, g_red, g_red_label):
        static, spec = ctx.static, ctx.spec
        world = static.world
        dev = world.device
        nb, Np, sG, K, nr = ctx.shape
        beta, s, inf, tinf, cur, nxt, ttn, T, seed_fraction, inf_o, tape_v, tape_y0, S_un, rf, vf = ctx.saved_tensors
        seed, call_index = ctx.noise_key
        p, _ = _fill_params(world, spec, static.symptoms, seed, call_index)
        seed_mode = spec.mode == MODE_SEED
        L = _lib.lib()
        io = _lib.BwdIO()
        keep = []

        def put(name, t):
            t = _f32(t, dev)
            if t is not None:
                keep.append(t)
                setattr(io, name, t.data_ptr())
            return t

        put("beta", beta), put("leisure_prob", static.leisure_prob), put("stage_prob", static.symptoms.stage_prob)
        put("seed_fraction", seed_fraction)
        for name, t in zip(_STATE, (s, inf, tinf, cur, nxt, ttn)):
            put(name, t)
        put("inf_o", inf_o), put("tape_y0", tape_y0)
        for name, g in (("g_s_o", g_s_o), ("g_inf_o", g_inf_o), ("g_tinf_o", g_tinf_o), ("g_cur_o", g_cur_o),
                        ("g_nxt_o", g_nxt_o), ("g_ttn_o", g_ttn_o), ("g_red", g_red)):
            g = put(name, g)
            if g is not None and name != "g_red" and tuple(g.shape) != (nb, Np):
                raise ValueError(f"cotangent {name} has shape {tuple(g.shape)}, expected {(nb, Np)}")
        n_lab = 0
        if g_red_label is not None:
            put("g_red_label", g_red_label)
            io.label = ctx.label.codes.data_ptr()
            n_lab = 2 * ctx.label.n
        need = ctx.needs_input_grad   # (static, spec, noise, beta, s, inf, tinf, cur, nxt, ttn, seed_fraction, label,
        #                                 seed_label, region_labels, region_factor, venue_labels, venue_factor)
        g_region, n_reg = None, 0
        if ctx.region_labels is not None:
            n_reg = ctx.region_labels.n
            _set_region(io, world, ctx.region_labels, rf)
            io.region_work = _buffer(world, "region_work_b", nb * Np).data_ptr()
            if need[14]:
                g_region = torch.empty(nb, n_reg, dtype=torch.float32, device=dev)
                io.g_region_factor = g_region.data_ptr()
        g_venue, n_ven = None, 0
        if ctx.venue_labels is not None:
            n_ven = K * ctx.venue_labels.n
            _set_venue(io, world, ctx.venue_labels, vf)
            if need[16]:
                g_venue = torch.empty(nb, K, ctx.venue_labels.n, dtype=torch.float32, device=dev)
                io.g_venue_factor = g_venue.data_ptr()
                io.venue_work = _buffer(world, "venue_work_b", nb * sG).data_ptr()

        def new(name):
            t = torch.empty(nb, Np, dtype=torch.float32, device=dev)
            if Np > world.n_agents:
                t[:, world.n_agents:] = 0.0
            setattr(io, name, t.data_ptr())
            return t

        grads = {}
        for i, name in enumerate(_STATE):
            if need[4 + i] or (not seed_mode and name in ("inf", "tinf")):   # the gather pass accumulates into these two
                grads[name] = new("g_" + name)
        scratch, scr_stride = _scratch_batch(world, nb)
        io.scratch = scratch.data_ptr()
        desc = world.desc()
        g_beta = g_frac = None
        if seed_mode:
            R = 1
            if ctx.seed_label is not None:
                _set_seed_labels(io, world, ctx.seed_label, seed_fraction, nb)
                R = ctx.seed_label.n
            g_frac = torch.zeros(nb, R, dtype=torch.float32, device=dev)
            io.g_seed_fraction = g_frac.data_ptr()
            strides = {name: 4 * Np for name in _AGENT_FIELDS}
            strides.update(g_red=4 * nr, scratch=scr_stride, g_seed_fraction=4 * R, g_red_label=4 * n_lab,
                           seed_fraction=4 * R if seed_fraction.numel() == nb * R else 0)
            _row_calls(L.gj_step_backward, "gj_step_backward", world, desc, p, io, nb, strides, _stream(dev))
            if seed_fraction.numel() != nb * R:
                g_frac = g_frac.sum(0).reshape(seed_fraction.shape)    # one fraction (per region) shared by the samples
            else:
                g_frac = g_frac.reshape(seed_fraction.shape)
        else:
            for name in ("maxinf", "shape", "rate", "shift", "k0", "prof4"):
                put(name, getattr(static, name))
            put("T_in", T), put("tape_v", tape_v), put("S_unscaled", S_un)
            g_beta = torch.zeros(nb, max(K, 1), dtype=torch.float32, device=dev)
            io.g_beta = g_beta.data_ptr()
            io.w = _buffer(world, "w_b", nb * Np).data_ptr()
            io.wq = _buffer(world, "wq_b", nb * Np).data_ptr() if p.n_quar > 0 else io.w
            io.R, io.cR = _buffer(world, "R_b", nb * sG).data_ptr(), _buffer(world, "cR_b", nb * sG).data_ptr()
            bt = _lib.Batch(n_samples=nb, agent_stride=Np, group_stride=max(sG, 1), beta_stride=K, red_stride=nr,
                            scratch_stride=scr_stride, label_stride=n_lab, region_stride=n_reg, venue_stride=n_ven)
            with _on(dev):
                _lib.check(L.gj_step_backward_batch(C.byref(desc), C.byref(p), C.byref(io), C.byref(bt), _stream(dev)),
                           "gj_step_backward_batch")
            g_beta = g_beta[:, :K]
            if g_region is not None and ctx.region_shape != (nb, n_reg):
                g_region = g_region.sum(0)   # one row of factors shared by the samples
            if g_venue is not None and len(ctx.venue_shape) == 2:
                g_venue = g_venue.sum(0)     # one table shared by the samples
        return (None, None, None, g_beta if need[3] else None,
                grads.get("s") if need[4] else None, grads.get("inf") if need[5] else None,
                grads.get("tinf") if need[6] else None, grads.get("cur") if need[7] else None,
                grads.get("nxt") if need[8] else None, grads.get("ttn") if need[9] else None,
                g_frac if (seed_mode and need[10]) else None, None, None, None, g_region, None, g_venue)


def infection_step(static: StepStatic, spec: StepSpec, beta, state: dict, T_in=None, q_in=None, n_in=None,
                   seed_fraction=None, noise=None, next_spec=None, label: Optional[Labels] = None,
                   seed_label: Optional[SeedLabels] = None, region: Optional[Region] = None,
                   venue: Optional[Venue] = None):
    """Run one (fused or partial) step.  ``state``: s, inf, tinf, cur, nxt, ttn (any may be None when
    the phases do not need it).  Returns a dict with s, inf, tinf, cur, nxt, ttn, T, q, n, red and red_label:
    with ``label`` the post-step cases and deaths per label column, [n, 2] ([b, n, 2] batched), else None.
    ``seed_label`` (seeding step only): ``seed_fraction`` then holds one fraction per region ([n], or [b, n]
    batched) and agent a is seeded with ``seed_fraction[seed_label.codes[a]]``.
    ``region`` (:class:`Region`, steps with the networks phase): every agent's pressure is multiplied by its region's
    factor before the clamp; the factor is differentiable.  The seeding step ignores it.
    ``venue`` (:class:`Venue`, steps with the networks phase): network k's beta is multiplied by the factor of each
    group's region, ``venue.factor[k, venue.labels.codes[g]]``, in the group passes; differentiable."""
    world = static.world
    if world.device.type != "cuda":
        raise _lib.GradJuneLibraryError(
            "the infection step runs only as CUDA kernels on a B200 (no CPU fallback): world is on "
            f"{world.device}; use system.device: cuda:0")
    if noise is None:
        if spec.phases & (PHASE_SAMPLE | PHASE_SYMPTOMS):
            noise = NOISE.next(world.n_agents, world.device)
        else:
            noise = (0, 0, None, None, None)
    if state.get("s") is not None and state["s"].dim() == 2:      # [b, Np]: a batched ensemble
        if T_in is not None or q_in is not None or n_in is not None or static.exchange is not None:
            raise _lib.GradJuneLibraryError("batched ensembles run the whole fused step on an unpartitioned world")
        outs = _BatchStep.apply(static, spec, noise, beta, state["s"], state["inf"], state["tinf"], state["cur"],
                                state["nxt"], state["ttn"], seed_fraction, label, seed_label,
                                None if region is None else region.labels, None if region is None else region.factor,
                                None if venue is None else venue.labels, None if venue is None else venue.factor)
        names = ("s", "inf", "tinf", "cur", "nxt", "ttn", "T", "red", "red_label")
        ret = dict(zip(names, outs))
        ret.update(q=None, n=None, lam=None)
        return ret
    outs = _Step.apply(static, spec, noise, beta, state.get("s"), state.get("inf"), state.get("tinf"),
                       state.get("cur"), state.get("nxt"), state.get("ttn"), T_in, q_in, n_in, seed_fraction, next_spec,
                       label, seed_label, None if region is None else region.labels,
                       None if region is None else region.factor, None if venue is None else venue.labels,
                       None if venue is None else venue.factor)
    names = ("s", "inf", "tinf", "cur", "nxt", "ttn", "T", "q", "n", "red", "lam", "red_label")
    return dict(zip(names, outs))
