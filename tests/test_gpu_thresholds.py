"""The throughput kernels at every size threshold of the world layout, against the fp32 / fp64 oracle.

``make_threshold_world`` builds a ~124 k-agent world, already in layout order, whose groups sit exactly on the
thresholds the layout and the kernels branch on: generic groups of 16 / 17 members (one lane vs the chunk lists),
1023 / 1024 / 1025 / 2049 (chunks of GJ_CHUNK and the multi-chunk fix-up), 32768 / 32769 (the largest scatter-tier
group and the smallest giant one), an empty group with ``people`` > 0; households of up to 64 members straddling
agent tiles and the ends of the world; leisure cells of 1 / 63 / 1024 / 1025 / 3000 agents (a 1-agent tile),
agents with 16 leisure edges and with none; a 40 000-member university whose members partly also work, and a few
duplicated edges.  A few hundred designated "hot" agents get ``max_infectiousness`` x 1e4, so that their
transmission passes 2^GJ_SCATTER_CAP_LOG2 = 1024 and the fixed-point scatter hands their groups to the exact re-sum.

The world asserts its own coverage (``_coverage``) before anything is compared, so that a change of the generator or
of the builders cannot quietly turn a case off.  The CPU test compares the native builder with the torch one on every
variant; the GPU tests compare one teacher-forced step (three pressure regimes x three kernel configurations), a
BPTT window, the look-ahead pass, the batched ensemble and the native world with the oracle or with each other."""
import numpy as np
import pytest
import torch

import helpers as H
from grad_june import world as W
from oracle import gj_oracle as O

DEV = "cuda:0"
VARIANTS = ("size", "people", "hh65")     # people = member count / people != count for some households / a 65-member one
N_BASE = 124_000
SPECIAL_AGES = (0, 17, 18, 64, 65, 75, 76, 99)
# company groups on the thresholds, and how many of each group's members are "hot" (max_infectiousness x 1e4)
COMPANY_SIZES = (0, 1, 2, 16, 17, 1023, 1024, 1025, 2049, 32768, 32769)
HOT = {2: 1, 17: 2, 1025: 8, 32768: 80, 32769: 80}
N_HOT_MULTI = 40                          # university members who also work: hot, university + a small company
N_UNIVERSITY = 40_000
N_UNI_WORKERS, N_UNI_PUPILS = 3000, 1000


def make_threshold_world(variant):
    """Deterministic world of N_BASE + {1, 2, 3} agents (N mod 4 = 1, 2, 3 for the three variants), numbered in layout
    order (run it with ``system: {renumber_agents: false}``).  ``data["threshold"]`` records what the tests need to
    find again: the hot agents, the company group of every threshold size, the households placed on tile edges."""
    assert variant in VARIANTS
    n = N_BASE + 1 + VARIANTS.index(variant)
    g = torch.Generator().manual_seed(20261020)

    # ---- leisure cells (CELL tier): consecutive agents with the same ordered list of leisure groups ----------------
    cells = [("three", 1), ("three", 63), ("three", 1024), ("three", 1025), ("three", 3000), ("sixteen", 2000),
             ("none", 1500)]
    used = sum(s for _, s in cells)
    while n - used - 1 > 3000:
        cells.append(("three", 3000))
        used += 3000
    cells += [("three", n - used - 1), ("three", 1)]
    n_lg = len(cells) + 16
    starts = np.cumsum([0] + [s for _, s in cells])
    la, lg = [], []
    for c, (kind, size) in enumerate(cells):
        ids = torch.arange(int(starts[c]), int(starts[c + 1]))
        k = {"three": 3, "sixteen": W.CELL_MAX_GROUPS, "none": 0}[kind]
        for j in range(k):
            la.append(ids)
            lg.append(torch.full_like(ids, (c + j) % n_lg))
    la, lg = torch.cat(la), torch.cat(lg)
    # the agent-major order of the edge list is the attendance order; keep it per agent
    order = torch.argsort(la, stable=True)
    la, lg = la[order], lg[order]
    big_cell = int(starts[4])                      # the 3000-agent cell: tiles start at +0, +1024, +2048
    none_lo, none_hi = int(starts[6]), int(starts[7])

    # ---- households (RANGE tier): contiguous runs; 64-member ones on tile edges and at both ends of the world ------
    tile = W.TILE_AGENTS
    fixed = [(0, 64), (big_cell + tile - 1, big_cell + tile + 63), (big_cell + 2 * tile - 63, big_cell + 2 * tile + 1),
             (n - 64, n)]
    fixed += [(a, a + 1) for a in range(none_lo, none_hi)]           # the none cell: everybody lives alone
    if variant == "hh65":
        fixed.append((big_cell + 2500, big_cell + 2565))
    fixed.sort()
    sizes = torch.tensor([1, 2, 3, 4, 8, 9, 63, 64])
    probs = torch.tensor([0.30, 0.30, 0.12, 0.10, 0.08, 0.06, 0.02, 0.02])
    runs, pos = [], 0
    for a, b in fixed + [(n, n)]:
        while pos < a:
            s = int(sizes[torch.multinomial(probs, 1, generator=g)])
            runs.append((pos, min(pos + s, a)))
            pos = runs[-1][1]
        if a < b:
            runs.append((a, b))
        pos = b
    hh = torch.empty(n, dtype=torch.long)
    for h, (a, b) in enumerate(runs):
        hh[a:b] = h
    n_hh = len(runs)
    hh_size = torch.bincount(hh, minlength=n_hh)
    hh_people = hh_size.clone()
    if variant == "people":
        hh_people[::7] += 3                                          # r_pc_lut = 0: the staged per-agent array

    # ---- ages: every bin edge of cases_by_age and both sides of care_visit's age > 75 -----------------------------
    age = torch.randint(0, 100, (n,), generator=g)
    for j, a in enumerate(SPECIAL_AGES):
        age[j * 997 + 5] = a
        age[n - 1 - j * 1009] = a
    sex = torch.randint(0, 2, (n,), generator=g)

    # ---- generic types ------------------------------------------------------------------------------------------
    hot_pool = torch.arange(none_lo, none_hi)                         # alone, no leisure: their T reaches only groups
    n_hot = sum(HOT.values()) + N_HOT_MULTI
    hot = hot_pool[:n_hot]
    ordinary = torch.cat((torch.arange(0, none_lo), hot_pool[n_hot:], torch.arange(none_hi, n)))
    ordinary = ordinary[torch.randperm(ordinary.numel(), generator=g)]
    hot_multi = hot[sum(HOT.values()):]
    uni = torch.cat((hot_multi, ordinary[:N_UNIVERSITY - N_HOT_MULTI]))
    rest = ordinary[N_UNIVERSITY - N_HOT_MULTI:]
    uni_workers = uni[N_HOT_MULTI:N_HOT_MULTI + N_UNI_WORKERS]
    uni_pupils = uni[N_HOT_MULTI + N_UNI_WORKERS:N_HOT_MULTI + N_UNI_WORKERS + N_UNI_PUPILS]

    # companies: the threshold sizes, then small filler groups; hot agents first in their group's member list
    n_fill_members = 6000
    workers = torch.cat((uni_workers, rest[:sum(COMPANY_SIZES) + n_fill_members - N_UNI_WORKERS]))
    workers = workers[torch.randperm(workers.numel(), generator=g)]
    rest = rest[sum(COMPANY_SIZES) + n_fill_members - N_UNI_WORKERS:]
    ca, cg, comp_of_size, p = [], [], {}, 0
    hot_at = 0
    for gid, s in enumerate(COMPANY_SIZES):
        k = HOT.get(s, 0)
        members = torch.cat((hot[hot_at:hot_at + k], workers[p:p + s - k]))
        hot_at += k
        p += s - k
        ca.append(members)
        cg.append(torch.full_like(members, gid))
        comp_of_size[s] = gid
    gid = len(COMPANY_SIZES)
    while p < workers.numel():
        s = min(int(torch.randint(3, 13, (1,), generator=g)), workers.numel() - p)
        ca.append(workers[p:p + s])
        cg.append(torch.full((s,), gid))
        p, gid = p + s, gid + 1
    n_comp = gid
    # the hot university members work in small filler companies (one each): their CSR is university (giant) + company
    ca.append(hot_multi)
    cg.append(len(COMPANY_SIZES) + torch.arange(N_HOT_MULTI) * 7)
    # the 32768-member company's hot agents all work in a small company too: only the agent-major walk of lean_scatter
    # (its size check against GJ_SCATTER_MAX_GROUP) carries their T >= 1024 into that group and marks it dirty
    first_32768 = HOT[2] + HOT[17] + HOT[1025]
    ca.append(hot[first_32768:first_32768 + HOT[32768]])
    cg.append(len(COMPANY_SIZES) + 3 + torch.arange(HOT[32768]) * 7)
    # duplicated edges: an agent listed twice in the same group counts twice, in the kernels and in the oracle
    ca.append(ca[-3][:2])
    cg.append(cg[-3][:2])
    ca, cg = torch.cat(ca), torch.cat(cg)

    ua = torch.cat((uni, uni[100:105]))
    ug = torch.zeros(ua.numel(), dtype=torch.long)

    pupils = torch.cat((uni_pupils, rest[:7000]))
    rest = rest[7000:]
    sa_ = pupils[torch.randperm(pupils.numel(), generator=g)]
    sg = torch.arange(sa_.numel()) // 250
    care = rest[:1200]
    care_g = torch.arange(care.numel()) // 30
    age[care[:600]] = 75 + torch.randint(0, 25, (600,), generator=g)   # residents: both sides of the age > 75 mask

    data = W.HeteroData()
    data["agent"].id = torch.arange(n)
    data["agent"].age = age
    data["agent"].sex = sex
    data["agent"].ethnicity = np.array(["A"])

    def add(name, a, grp, n_groups, people=None):
        data[name].id = torch.arange(n_groups)
        data[name].people = torch.bincount(grp, minlength=n_groups) if people is None else people
        data["agent", "attends_" + name, name].edge_index = torch.stack((a, grp))

    add("household", torch.arange(n), hh, n_hh, hh_people)
    comp_people = torch.bincount(cg, minlength=n_comp)
    comp_people[comp_of_size[0]] = 5                                  # an empty group that says it has people
    add("company", ca, cg, n_comp, comp_people)
    add("school", sa_, sg, int(sg.max()) + 1)
    add("university", ua, ug, 1)
    add("care_home", care, care_g, int(care_g.max()) + 1)
    add("leisure", la, lg, n_lg)
    tb = big_cell + tile
    data["threshold"] = {"hot": hot.clone(), "company_of_size": comp_of_size, "hot_multi": hot_multi.clone(),
                         "tile_edges": (tb, tb + tile)}
    return data


def _types(data):
    return data.venue_types()


def _python_build(data, device="cpu"):
    from grad_june import _lib
    cfg = _lib.config()
    types = _types(data)
    return W.build_csr(len(data["agent"].id), types, {t: data["attends_" + t].edge_index for t in types},
                       {t: torch.as_tensor(data[t]["people"]) for t in types}, {t: len(data[t]["id"]) for t in types},
                       data["agent"].age, data["agent"].sex, cfg["small_group"], cfg["chunk"], device)


def _coverage(data, world, variant):
    """What the world must contain; thresholds read from the library and the layout module, never restated."""
    from grad_june import _lib
    cfg = _lib.config()
    small, chunk, smax, tile = cfg["small_group"], cfg["chunk"], cfg["scatter_max"], cfg["tile_agents"]
    assert tile == W.TILE_AGENTS and smax == W.SCATTER_MAX_GROUP
    types = _types(data)
    tier = dict(zip(types, world.type_tier))
    hh_tier = W.TIER_GENERIC if variant == "hh65" else W.TIER_RANGE
    assert tier["household"] == hh_tier and tier["leisure"] == W.TIER_CELL, tier
    assert tier["company"] == tier["university"] == W.TIER_GENERIC
    n = world.n_agents
    assert n % 4 == 1 + VARIANTS.index(variant)
    size = world.group_size.cpu()
    off = world.type_group_off
    comp = {s: off[types.index("company")] + gid for s, gid in data["threshold"]["company_of_size"].items()}
    for s, gid in comp.items():
        assert int(size[gid]) == s, (s, int(size[gid]))
    assert int(torch.as_tensor(data["company"]["people"])[data["threshold"]["company_of_size"][0]]) > 0
    # exact boundaries around every threshold
    for s in (small, small + 1, chunk - 1, chunk, chunk + 1, 2 * chunk + 1, smax, smax + 1):
        assert s in comp, s
    assert world.n_giant_big >= 1 and world.n_parts > 0
    small_groups = set(world.small_groups.cpu().long().tolist())
    chunk_groups = set(world.chunk_group.cpu().long().tolist())
    assert comp[small] in small_groups and comp[small + 1] in chunk_groups and comp[small + 1] not in small_groups
    assert comp[smax + 1] in world.big_groups.cpu().long().tolist()[:world.n_giant_big]
    assert comp[smax] in chunk_groups
    uni_g = off[types.index("university")]
    assert int(size[uni_g]) > smax
    # giant = more than scatter_max members, nothing else: the listed giant groups and the giant bit of ent1
    generic = torch.zeros(world.n_groups, dtype=torch.bool)
    for ti, t in enumerate(types):
        generic[off[ti]:off[ti + 1]] = world.type_tier[ti] == W.TIER_GENERIC
    giant = set(torch.nonzero(generic & (size > smax)).flatten().tolist())
    assert set(world.big_groups.cpu().long().tolist()[:world.n_giant_big]) == giant and comp[smax] not in giant
    ent1_all = world.ent1.cpu().long()[:n] & 0xFFFFFFFF
    one = ent1_all < 0xFFFFFFFE
    assert torch.equal((ent1_all[one] >> 31) == 1, size[ent1_all[one] & 0x7FFFFFFF] > smax)
    # multi-edge agents whose agent-major run holds a giant group (and a scatter-tier one)
    ent1 = world.ent1.cpu().long() & 0xFFFFFFFF
    multi = torch.nonzero(ent1 == 0xFFFFFFFE).flatten()
    am_ptr, am_ent = world.am_ptr.cpu().long(), world.am_ent.cpu().long() & 0xFFFFFFFF
    giant_multi = 0
    for a in multi.tolist():
        gs = [off[e >> 28] + (e & 0x0FFFFFFF) for e in am_ent[am_ptr[a]:am_ptr[a + 1]].tolist()]
        sz = [int(size[x]) for x in gs]
        giant_multi += any(s > smax for s in sz) and any(s <= smax for s in sz)
    assert giant_multi >= N_HOT_MULTI, giant_multi
    ei = data["attends_company"].edge_index.cpu()
    hot = data["threshold"]["hot"].cpu()
    hot_32768 = hot[torch.isin(hot, ei[0][ei[1] == data["threshold"]["company_of_size"][smax]])]
    assert hot_32768.numel() > 0 and bool((ent1[hot_32768] == 0xFFFFFFFE).all())
    tb = world.tile_begin.cpu().long()
    assert int(tb[-1]) == n
    assert int((tb[1:] - tb[:-1]).min()) == 1                         # a 1-agent tile
    if hh_tier == W.TIER_RANGE:
        hi = types.index("household")
        slot = world.range_slot[hi].cpu().long() & 0xFFFFFFFF
        gsize, goff = slot & 0xFFFF, slot >> 16
        assert int(gsize.max()) == W.RANGE_MAX_GROUP
        first = torch.arange(n) - goff                                # first member of every agent's household
        crossing = [int(t) for t in tb[1:-1].tolist() if int(gsize[t]) == W.RANGE_MAX_GROUP and int(first[t]) < t]
        assert crossing, "no 64-member household crosses a tile boundary"
        e0, e1 = data["threshold"]["tile_edges"]
        assert int(first[e0]) == e0 - 1 and int(first[e1]) == e1 - 63 and int(goff[e1 + 1]) == 0
        assert int(gsize[0]) == int(gsize[n - 1]) == W.RANGE_MAX_GROUP and int(goff[n - 1]) == W.RANGE_MAX_GROUP - 1
    else:
        assert int(torch.bincount(data["attends_household"].edge_index[1]).max()) == W.RANGE_MAX_GROUP + 1
    ldeg = torch.bincount(data["attends_leisure"].edge_index[0], minlength=n)
    assert int(ldeg.max()) == W.CELL_MAX_GROUPS and int((ldeg == 0).sum()) > 0
    age = data["agent"].age
    assert all(bool((age == a).any()) for a in SPECIAL_AGES)


@pytest.mark.parametrize("variant", VARIANTS)
def test_native_builder_matches_python_on_the_threshold_world(variant):
    from test_world_build import _compare
    data = make_threshold_world(variant)
    ref = _python_build(data)
    _coverage(data, ref, variant)
    native = W.NativeWorld(data, host=True, renumber=False)
    assert native.permutation() is None
    _compare(native, ref, _types(data))
    if variant != "hh65":
        hi = _types(data).index("household")
        assert bool(ref.range_pc_from_size[hi]) == (variant == "size")
    native.close()


# ------------------------------------------------------------------------------------------------------------------
# GPU: the kernels on the threshold world
# ------------------------------------------------------------------------------------------------------------------
# log-beta shifts.  floor: -6 rather than -3, because a hot agent (T >= 1024) in each of the two 32 k-member companies
# alone lifts their members - over half of the world - above the 1e-6 floor down to a shift of about -5.5
REGIMES = {"default": {}, "saturated": {"company": 2.5, "university": 2.5}, "floor": "all-6"}
CONFIGS = ("pipelined", "register", "reference-order")
THRESHOLD_SIZES = (2, 17, 1025, 32768, 32769)     # the company groups whose members must feel mostly that group


def _params(days):
    from grad_june.default_config import default_parameters
    p = default_parameters()
    p["system"]["device"] = DEV
    p["system"]["renumber_agents"] = False
    p["policies"] = {}
    p["timer"]["total_days"] = days
    p["infection_seed"]["log_fraction_initial_cases"] = -1.0
    return p


def _threshold_data(params, variant):
    """The world on DEV with sampled profiles; the hot agents' max_infectiousness x 1e4."""
    from grad_june.runner import Runner
    torch.manual_seed(7)
    data = Runner.get_data(params, data=make_threshold_world(variant))
    hot = data["threshold"]["hot"]
    data["agent"].infection_parameters["max_infectiousness"][hot] *= 1e4
    return data


def _log_betas(params, regime):
    base = {k: float(v["log_beta"]) for k, v in params["networks"].items()}
    shift = REGIMES[regime]
    if shift == "all-6":
        return {k: v - 6.0 for k, v in base.items()}
    return {k: v + shift.get(k, 0.0) for k, v in base.items()}


def _pressure_by_type(w, spec, T, s):
    """Per edge type, the pressure every agent receives (oracle arithmetic, no quarantine in these runs)."""
    assert not spec.quarantine
    out = {}
    for net in spec.nets:
        p = O.network_pressure(w, net, T, s, 1.0, spec.day_type)
        out[net.edge_type] = out.get(net.edge_type, 0) + p
    return out


def _check_pressure_design(data, w, spec, T, s, regime):
    """The hot agents reach every threshold group with T >= 1024, and a member of a threshold group receives most of
    its pressure from that group (so that a wrong sum of it cannot hide under the household's or leisure's)."""
    from grad_june import _lib
    cap = 2.0 ** 10
    assert _lib.config()["scatter_max"] == W.SCATTER_MAX_GROUP
    ei = data["attends_company"].edge_index.to(T.device)
    comp = data["threshold"]["company_of_size"]
    hotT = torch.zeros_like(T, dtype=torch.bool)
    hotT[data["threshold"]["hot"].to(T.device)] = True
    big = (T >= cap) & hotT
    assert int(big[data["threshold"]["hot_multi"].to(T.device)].sum()) >= 5
    press = _pressure_by_type(w, spec, T, s)
    total = sum(press.values())
    shares = {}
    for size in THRESHOLD_SIZES:
        members = ei[0][ei[1] == comp[size]]
        if size < 32769:
            assert int(big[members].sum()) >= 1, f"no member with T >= 1024 in the {size}-member group"
        m = members[(s[members] > 0) & (total[members] > 0)]
        share = press["company"][m] / total[m]
        shares[size] = float(share.detach().min())
        assert float(share.min()) > 0.5, (size, float(share.min()))
    return shares


def _teacher_forced(variant, regime, config):
    """One step from a mid-epidemic state with the kernels' own Philox draws against the oracle (on the CPU)."""
    from grad_june import GradJune, Timer, _lib, ops
    params = _params(10)
    data = _threshold_data(params, variant)
    n = len(data["agent"].id)
    model = GradJune.from_parameters(params)
    lbs = _log_betas(params, regime)
    for k, net in model.infection_networks.networks.items():
        net.log_beta = torch.nn.Parameter(torch.tensor(lbs[k], device=DEV))
    timer = Timer.from_parameters(params)
    for _ in range(8):
        next(timer)
    state = H.mid_epidemic_state(n, timer.now, 11, DEV)
    hot = data["threshold"]["hot"]
    for key, v in (("is_infected", 1.0), ("susceptibility", 0.0), ("infection_time", timer.now - 0.25),
                   ("current_stage", 2.0), ("next_stage", 3.0), ("time_to_next_stage", timer.now + 2.0)):
        state[key][hot] = v
    for k in ("susceptibility", "is_infected", "infection_time"):
        data["agent"][k] = state[k]
    data["agent"].symptoms = {k: state[k] for k in ("current_stage", "next_stage", "time_to_next_stage")}
    world = W.get_device_world(data, DEV)
    _coverage(data, world, variant)
    assert model.kernel_family(data, timer) == "throughput"
    seed = 4099
    prev = _lib.pipeline_enable(None)
    _lib.pipeline_enable(config == "pipelined", lookahead=False)
    ops.EXACT_ORDER = config == "reference-order"
    try:
        with ops.philox_seed(seed):
            res = model(data=data, timer=timer)
    finally:
        ops.EXACT_ORDER = False
        _lib.pipeline_enable(*prev)
    agent = res["agent"]
    E, u, z = (t.cpu() for t in ops.philox_fill(seed, 0, n, DEV))
    noise = O.StepNoise(E=E, u=u, z=z.expand(10, n))
    # the oracle on the CPU: its fp32 group sums then run in edge order, the same sums on every run
    w, nets, spec, sym, prof, st = H.oracle_step_inputs(params, data, model, timer, state, "cpu")
    aux = {}
    O.step(w, st, prof, spec, sym, noise, aux)
    what = f"threshold world {variant}/{regime}/{config}"

    shares = _check_pressure_design(data, w, spec, aux["transmission"], state["susceptibility"].cpu(), regime)
    lam = aux["lam"].detach()
    sat, low = float((lam > 100).float().mean()), float((lam < 1e-6).float().mean())
    if regime == "saturated":
        assert sat >= 0.05, sat
    if regime == "floor":
        assert low >= 0.5, low

    def cpu(t):
        return t.detach().cpu().numpy()

    T, To = cpu(agent.transmission), cpu(aux["transmission"])
    assert np.allclose(T, To, rtol=1e-5, atol=1e-30), np.max(np.abs(T - To) / np.maximum(np.abs(To), 1e-30))
    q, qo = cpu(agent["not_infected_probs"]), cpu(aux["q"])
    q_rel = np.abs(q - qo) / qo
    # q = exp(-lam dt) carries lam's absolute rounding error: its relative error is dt x |d lam|.  Up to the cap of 100,
    # a few fp32 ulps of lam (re-associated sums) move q by up to ~3e-5, and a q below 2^-126 is a denormal with fewer
    # significant bits; both allowances are added to the 1e-5 (they vanish for the small lam of the other tests).  The
    # fp32 oracle's own one-by-one sum over a 32 k-member group can be further off than that (the kernels' fixed-point
    # sums are exact), so an agent also passes at 1e-5 from the fp64 witness or no further from it than 4 x the fp32
    # oracle is (as assert_grad_parity's criterion b).
    w64, _, spec64, sym64, prof64, st64 = H.oracle_step_inputs(params, data, model, timer, state, "cpu")
    for sp in spec64.nets:
        sp.beta = sp.beta.detach().double()
    aux64 = {}
    with torch.no_grad():
        O.step(w64, {k: v.double() for k, v in st64.items()}, {k: v.double() for k, v in prof64.items()}, spec64,
               sym64, O.StepNoise(E=E.double(), u=u.double(), z=z.double().expand(10, n)), aux64)
    q64 = cpu(aux64["q"])
    lam32 = np.clip(cpu(aux["lam"]), 1e-6, 100.0).astype(np.float32)
    tol = 1e-5 + 4.0 * spec.dt * np.spacing(lam32).astype(np.float64) + 2.0 ** -149 / np.maximum(qo, 2.0 ** -149)
    q_ok = (q_rel <= tol) | (np.abs(q - q64) <= np.maximum(1e-5 * q64, 4.0 * np.abs(qo - q64)))
    bad = np.nonzero(~q_ok)[0]
    assert len(bad) == 0, (f"{len(bad)} agents: q {q[bad[:5]]} fp32 oracle {qo[bad[:5]]} fp64 {q64[bad[:5]]} "
                           f"lam {cpu(aux['lam'])[bad[:5]]}")
    q_fallback = int((q_rel > 1e-5).sum())
    q_rel = float(q_rel.max())
    nn, no = cpu(agent["new_infected"]), cpu(aux["new_infected"])
    mism = np.nonzero(nn != no)[0]
    # a draw where the kernels agree with the fp64 witness is the fp32 oracle's rounding (its q can be ~1e-4 off
    # in a 32 k-member group); every other mismatch must be a certified near-tie
    by64 = nn[mism] == cpu(aux64["new_infected"])[mism]
    worst = H.certify_near_ties(qo, E.numpy(), mism[~by64], what=what)
    assert len(mism) <= max(2, int(1e-6 * n)), len(mism)
    ok = np.ones(n, dtype=bool)
    ok[mism] = False
    assert nn.sum() > 0 or regime == "floor"
    for mine, theirs, exact in ((agent.susceptibility, st["susceptibility"], True),
                                (agent.is_infected, st["is_infected"], True),
                                (agent.symptoms["current_stage"], st["current_stage"], True),
                                (agent.symptoms["next_stage"], st["next_stage"], True),
                                (agent.infection_time, st["infection_time"], False),
                                (agent.symptoms["time_to_next_stage"], st["time_to_next_stage"], False)):
        a, b = cpu(mine)[ok], cpu(theirs)[ok]
        if exact:
            assert np.array_equal(a, b)
        else:
            assert np.allclose(a, b, rtol=2e-6, atol=1e-6)

    # gradients: flipped agents (certified near-ties) left out of the loss on both sides
    gw = torch.Generator(device="cpu").manual_seed(5)
    keep = torch.from_numpy(ok.astype(np.float32))
    wts = [torch.rand(n, generator=gw) * keep for _ in range(4)]
    keys = list(model.infection_networks.networks.keys())

    def loss_of(inf, cur, s, tinf, dtype=torch.float32):
        w0, w1, w2, w3 = (t.to(device=inf.device, dtype=dtype) for t in wts)
        return (inf * w0).sum() + (cur * w1).sum() + 0.5 * (s * w2).sum() + 0.05 * (tinf * w3).sum()

    def oracle_grads(dtype, perturb=None):
        wo, netso, speco, symo, profo, sto = H.oracle_step_inputs(params, data, model, timer, state, "cpu")
        for sp in speco.nets:
            sp.beta = sp.beta.to(dtype)
        sto = {k: v.to(dtype) for k, v in sto.items()}
        profo = {k: v.to(dtype) for k, v in profo.items()}
        nz = O.StepNoise(E=noise.E.to(dtype), u=noise.u.to(dtype), z=noise.z.to(dtype))
        if perturb is None:
            O.step(wo, sto, profo, speco, symo, nz)
        else:
            with H.perturb_q(perturb):
                O.step(wo, sto, profo, speco, symo, nz)
        loss_of(sto["is_infected"], sto["current_stage"], sto["susceptibility"], sto["infection_time"], dtype).backward()
        gr = np.array([netso.networks[k].log_beta.grad.item() if netso.networks[k].log_beta.grad is not None
                       else 0.0 for k in keys])
        return gr, torch.equal(sto["is_infected"].float() * keep, st["is_infected"] * keep)

    loss_of(agent.is_infected, agent.symptoms["current_stage"], agent.susceptibility, agent.infection_time).backward()
    mine = np.array([model.infection_networks.networks[k].log_beta.grad.item() for k in keys])
    ref, _ = oracle_grads(torch.float32)
    g64, same = oracle_grads(torch.float64)
    assert same, "fp64 witness drew different masks"
    sens = np.zeros_like(ref)
    for sd in (1, 2, 3):
        gp, _ = oracle_grads(torch.float32, perturb=sd)
        sens = np.maximum(sens, np.abs(gp - ref))
    used = H.assert_grad_parity(mine, ref, g64, sens, rtol=1e-5, what=f"{what}: d/dlog_beta")
    H.report(f"{what}: teacher-forced step", {"mismatches": int(len(mism)), "fp64_agrees": int(by64.sum()), "worst_near_tie": worst, "q_max_rel": q_rel,
                                             "q_via_fp64": q_fallback, "saturated_frac": sat, "floor_frac": low, "criteria": used,
                                             "min_group_share": shares})


# every regime meets every variant and every kernel configuration once (a Latin square)
CASES = [(VARIANTS[(i + j) % 3], regime, config) for i, regime in enumerate(REGIMES) for j, config in enumerate(CONFIGS)]


@pytest.mark.gpu
@pytest.mark.parametrize("variant,regime,config", CASES)
def test_teacher_forced_step_on_the_threshold_world(variant, regime, config):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    _teacher_forced(variant, regime, config)


def _runner(variant, days, native=False):
    from grad_june import GradJune, Timer
    from grad_june.runner import Runner
    params = _params(days)
    data = _threshold_data(params, variant)
    model = GradJune.from_parameters(params)
    keys = list(model.infection_networks.networks.keys())
    for k in keys:
        model.infection_networks.networks[k].log_beta = torch.tensor(float(params["networks"][k]["log_beta"]),
                                                                     device=DEV, requires_grad=True)
    runner = Runner(model=model, data=data, timer=Timer.from_parameters(params),
                    log_fraction_initial_cases=torch.tensor(-1.0, requires_grad=True),
                    save_path="/tmp/gj_test", parameters=params)
    world = W.get_device_world(data, DEV, native=native)
    if not native:
        _coverage(data, world, variant)
    return runner, params, keys


def _hot_in_scatter_groups(data):
    """Hot agents that are members of a non-giant company group."""
    ei = data["attends_company"].edge_index
    size = torch.bincount(ei[1])
    members = ei[0][size[ei[1]] <= W.SCATTER_MAX_GROUP]
    hot = data["threshold"]["hot"]
    return hot[torch.isin(hot, members)]


def _assert_hot_transmission(runner):
    """The last step of the window still scattered T >= 2^GJ_SCATTER_CAP_LOG2 into scatter-tier groups."""
    T = runner.data["agent"].transmission.detach()
    assert int((T[_hot_in_scatter_groups(runner.data)] >= 1024).sum()) >= 1


@pytest.mark.gpu
def test_bptt_window_on_the_threshold_world_vs_oracle():
    """Five steps of Runner() + backward in throughput mode against oracle.run in fp32 and fp64 (test_gpu_layout's
    criterion): the fixed-point accumulators and dirty flags have to be clean again at every step."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from test_gpu_layout import _window_vs_oracle
    runner, params, keys = _runner("people", 5)
    _window_vs_oracle(runner, params, keys, seed=4242, what="threshold world window (5 steps)")
    _assert_hot_transmission(runner)


def _run_window(runner, keys, lb, seed):
    from grad_june import ops
    nets = runner.model.infection_networks.networks
    leaves = []
    for i, k in enumerate(keys):
        leaf = (lb[:, i] if runner.batch else lb[i]).detach().clone().requires_grad_(True)
        nets[k].log_beta = leaf
        leaves.append(leaf)
    frac = torch.tensor(-1.0, device=DEV, requires_grad=True)
    runner.log_fraction_initial_cases = frac
    with ops.philox_seed(seed):
        results, is_inf = runner()
    loss = results["cases_per_timestep"].sum(0) + 3.0 * results["deaths_per_timestep"].sum(0) \
        + 0.5 * results["cases_by_age_65"].sum(0)
    loss.sum().backward()
    agent = runner.data["agent"]
    n = runner.n_agents
    state = [agent.susceptibility, agent.infection_time, agent.symptoms["current_stage"], agent.symptoms["next_stage"],
             agent.symptoms["time_to_next_stage"]]
    return dict(loss=loss.detach().clone(), grads=torch.stack([l.grad for l in leaves], dim=-1),
                frac=frac.grad.clone(), inf=is_inf.detach().clone(),
                series={k: v.detach().clone() for k, v in results.items() if k != "dates"},
                state=[t.detach()[..., :n].clone() for t in state],
                T=None if runner.batch else agent.transmission.detach().clone())


def _base_lb(params, keys):
    return torch.tensor([float(params["networks"][k]["log_beta"]) for k in keys], device=DEV)


@pytest.mark.gpu
def test_lookahead_pass_on_the_threshold_world():
    """The look-ahead transmission pass scatters step t+1's values (dirty flags included) while step t runs: the same
    trajectory, transmissions and state as without it, gradients to 5e-5."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from grad_june import _lib
    runner, params, keys = _runner("size", 4)
    lb = _base_lb(params, keys)
    outs = {}
    prev = _lib.pipeline_enable(None)
    try:
        for look in (False, True):
            _lib.pipeline_enable(True, lookahead=look)
            outs[look] = _run_window(runner, keys, lb, 61)
            _assert_hot_transmission(runner)
    finally:
        _lib.pipeline_enable(*prev)
    a, b = outs[False], outs[True]
    assert a["series"]["cases_per_timestep"][-1] > a["series"]["cases_per_timestep"][0] > 0
    for k, v in a["series"].items():
        assert torch.equal(v, b["series"][k]), k
    assert torch.equal(a["inf"], b["inf"])
    for x, y in zip(a["state"] + [a["T"]], b["state"] + [b["T"]]):
        assert torch.equal(x, y)
    ga, gb = a["grads"], b["grads"]
    assert torch.allclose(ga, gb, rtol=5e-5, atol=1e-6 * float(ga.abs().max())), (ga, gb)


@pytest.mark.gpu
def test_batched_ensemble_on_the_threshold_world():
    """runner.batch = 3 with distinct log-beta rows against three unbatched runs: series, infections and state
    bit-identical, gradients to 2e-6 (the per-sample scratch shift of the accumulators and dirty flags, the giant-group
    pass with several samples).  N = 3 mod 4: padded rows."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    runner, params, keys = _runner("hh65", 3)
    b = 3
    base = _base_lb(params, keys)
    lbs = torch.stack([base + (r - 1) * torch.linspace(-0.25, 0.25, len(keys), device=DEV) for r in range(b)])
    singles = [_run_window(runner, keys, lbs[r], 71) for r in range(b)]
    runner.batch = b
    try:
        bat = _run_window(runner, keys, lbs, 71)
    finally:
        runner.batch = None
    for r, one in enumerate(singles):
        for k, v in one["series"].items():
            assert torch.equal(bat["series"][k][:, r], v), (k, r)
        assert torch.equal(bat["inf"][r], one["inf"])
        for tb, ts in zip(bat["state"], one["state"]):
            assert torch.equal(tb[r], ts), r
        assert torch.equal(bat["loss"][r], one["loss"])
        g1 = one["grads"]
        assert torch.allclose(bat["grads"][r], g1, rtol=2e-6, atol=2e-8 * float(g1.abs().max())), (r, bat["grads"][r], g1)
    gsum = sum(one["frac"] for one in singles)
    assert torch.allclose(bat["frac"], gsum, rtol=2e-6, atol=2e-8 * float(gsum.abs()))
    assert not torch.equal(bat["series"]["cases_per_timestep"][:, 0], bat["series"]["cases_per_timestep"][:, 2])


@pytest.mark.gpu
def test_native_builder_on_the_threshold_world_is_bit_identical(monkeypatch):
    """Runner on the world built by gj_world_build against the torch builder: identical results and gradients."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    outs = []
    for native in ("0", "1"):
        monkeypatch.setenv("GJ_NATIVE_BUILD", native)
        runner, params, keys = _runner("people", 3, native=native == "1")
        assert isinstance(W.get_device_world(runner.data, DEV), W.NativeWorld) == (native == "1")
        outs.append(_run_window(runner, keys, _base_lb(params, keys), 81))
    a, b = outs
    for k, v in a["series"].items():
        assert torch.equal(v, b["series"][k]), k
    assert torch.equal(a["inf"], b["inf"]) and torch.equal(a["grads"], b["grads"]) and torch.equal(a["frac"], b["frac"])
    assert a["series"]["cases_per_timestep"][-1] > a["series"]["cases_per_timestep"][0]
