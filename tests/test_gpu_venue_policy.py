"""Regional venue restrictions on the GPU: network k's beta at a group times the factor of the group's region.

1. identity: factors of 1 over the whole window reproduce the run without the policy bit for bit (pipelined
   throughput kernels, register-batched throughput kernels, reference-order kernels);
2. the renumbered sample world with three group regions, two overlapping windows and factors 0 to 3 against the
   oracle with the per-group beta vector f[code] (``venue_oracle.venue_factor``): exact masks, stages and series;
   d/dlog_beta and d/dfactor through ``assert_grad_parity``;
3. factor 0 in every region for one network equals national CloseVenue of that network;
4. batched b = 4 against the unbatched runs; graph replay against the eager window; Calibrator(fit_venue=True);
5. the modular path (a user network subclass);
6. two generic networks on one edge type: each gets its own factor gradient;
7. a 1 M-agent world with super-area, 300-agent area and 100 000 random group labels: sum_r dL/dlog10 f[k, r] =
   dL/dlog_beta_k for every network, and bit-identical reruns;
8. 2 GPUs against 1: a partitioned world, graphed with fit_venue=True (skips on one GPU)."""
import datetime

import numpy as np
import pytest
import torch

import helpers as H
from oracle import gj_oracle as O
from venue_oracle import venue_factor

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
RTOL = 1e-5
FA = [0.0, 1.5, 3.0]      # pub: closed in region 0
FB = [2.0, 0.5, 1.2]      # company, window A
FC = [0.2, 1.0, 2.5]      # company, window B (overlaps A)
FU = [1.4, 0.6, 0.3]      # university, window B
ALL = 0.8                 # every other non-household network, window A


@pytest.fixture(autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")


def _day(params, d):
    return datetime.datetime.strptime(str(params["timer"]["initial_day"]), "%Y-%m-%d") + datetime.timedelta(days=d)


def _windows(params):
    return [(_day(params, 2), _day(params, 9)), (_day(params, 6), _day(params, 13))]


def _group_region(arrays, t):
    return np.arange(int(arrays[f"{t}_ngroups"]), dtype=np.int64) % 3


def _sample_runner(tag, entries=None, windows=None, close=None):
    """The renumbered sample world; every non-household group type carries ``region`` = group id % 3.  ``entries``:
    the beta_factors of one venue policy per window.  Log-betas are leaves."""
    from grad_june import GradJune, Runner, Timer
    from grad_june.policies import CloseVenue, CloseVenuePolicies, RegionalVenueDistancing, VenuePolicies
    from grad_june.world import layout_order_of, world_from_arrays
    g = np.load(H.GOLDEN / f"run_{tag}.npz")
    params, _ = H.load_params(tag)
    params["system"]["device"] = DEV
    params["system"]["renumber_agents"] = True
    arrays = np.load(H.GOLDEN / "sample_world.npz")
    world = world_from_arrays(arrays, H.SAMPLE_TYPES)
    for t in H.SAMPLE_TYPES[1:]:
        world[t].region = torch.from_numpy(_group_region(arrays, t))
    data = Runner.get_data(params, data=world)
    data["agent"].infection_parameters = {k: layout_order_of(data, v.to(DEV)).contiguous()
                                          for k, v in H.profile_params(g).items()}
    model = GradJune.from_parameters(params)
    if entries is not None:
        windows = windows or _windows(params)
        model.policies.venue_policies = VenuePolicies(
            [RegionalVenueDistancing(w[0], w[1], "region", e, device=DEV) for w, e in zip(windows, entries)])
    if close is not None:
        model.policies.close_venue_policies = CloseVenuePolicies(
            [CloseVenue(w[0], w[1], names=close, device=DEV) for w in (windows or _windows(params))[:1]])
    nets = model.infection_networks.networks
    for key in nets.keys():
        nets[key].log_beta = torch.nn.Parameter(nets[key].log_beta)
    runner = Runner(model=model, data=data, timer=Timer.from_parameters(params),
                    log_fraction_initial_cases=float(params["infection_seed"]["log_fraction_initial_cases"]),
                    save_path=params["save_path"], parameters=params,
                    age_bins=params.get("age_bins_to_save", (0, 18, 65, 100)))
    return runner, g, params, arrays


def _loss(results):
    return results["cases_per_timestep"].sum() + 0.7 * results["deaths_per_timestep"].sum() \
        + 0.3 * results["cases_by_age_65"].sum()


def _run(runner, family, tag, n_steps, leaves=()):
    from grad_june import ops
    from gpu_helpers import noise_provider
    nets = runner.model.infection_networks.networks
    for net in nets.values():
        net.log_beta.grad = None
    pipe = None
    if family == "register-batched":
        pipe = ops._lib.pipeline_enable(False)
    try:
        if family in ("throughput", "register-batched"):
            with ops.philox_seed(4242 + H.RUNS[tag]):
                results, is_inf = runner()
        else:
            with ops.inject_noise(noise_provider(H.RUNS[tag], n_steps + 1, runner.n_agents)):
                results, is_inf = runner()
        _loss(results).backward()
    finally:
        if pipe is not None:
            ops._lib.pipeline_enable(*pipe)
    grads = torch.stack([nets[k].log_beta.grad.detach().clone() if nets[k].log_beta.grad is not None
                         else torch.zeros((), device=DEV) for k in nets.keys()])
    res = {k: v.detach().clone() for k, v in results.items() if k != "dates"}
    return res, is_inf.detach().clone(), grads, [l.grad.detach().clone() for l in leaves]


def _stages(runner):
    from grad_june.world import original_order
    return original_order(runner.data, runner.data["agent"].symptoms["current_stage"]).detach().cpu()


@pytest.mark.parametrize("family", ["throughput", "register-batched", "reference-order"])
def test_identity_with_unit_factors(family):
    tag = "sample_default"
    plain, g, params, _ = _sample_runner(tag)
    n_steps = int(g["n_steps"])
    whole = [(_day(params, -1), _day(params, 100))]
    leaf = torch.ones(3, device=DEV, requires_grad=True)
    pub = torch.ones(3, device=DEV, requires_grad=True)
    ones, _, _, _ = _sample_runner(tag, entries=[{"all": leaf, "pub": pub}], windows=whole)
    assert ones.venue_labels.tolist() == [0, 1, 2]
    a = _run(plain, family, tag, n_steps)
    b = _run(ones, family, tag, n_steps, [leaf, pub])
    for k, v in a[0].items():
        assert torch.equal(b[0][k], v), k
    assert torch.equal(a[1], b[1]), "infection masks"
    assert torch.equal(a[2], b[2]), (a[2], b[2])
    assert torch.equal(_stages(plain), _stages(ones))
    for gl in b[3]:
        assert gl.shape == (3,) and bool(torch.isfinite(gl).all()) and float(gl.abs().max()) > 0.0


def _oracle(tag, arrays, windows, noises, dtype=torch.float32, perturb=None):
    """The oracle with the venue factors as per-group beta vectors: (result, d/dlog_beta, {entry: d/dfactor})."""
    import contextlib
    from grad_june import Timer
    from grad_june.policies import Policies
    from grad_june.symptoms import SymptomsSampler
    g = np.load(H.GOLDEN / f"run_{tag}.npz")
    params, _ = H.load_params(tag)
    w = H.oracle_world(arrays, H.SAMPLE_TYPES)
    nets = H.make_leaf_networks(params)
    steps = H.oracle_schedule(params, nets, Policies.from_parameters(params))
    if dtype != torch.float32:
        for s in steps:
            for n in s.nets:
                n.beta = n.beta.to(dtype)
    sym = H.oracle_symptoms(SymptomsSampler.from_parameters(params))
    noises = [O.StepNoise(E=n.E.to(dtype), u=n.u.to(dtype), z=n.z.to(dtype)) for n in noises]
    leaves = {k: torch.tensor(v, dtype=dtype, requires_grad=True) for k, v in (("pub", FA), ("companyA", FB),
                                                                                  ("companyB", FC), ("university", FU))}
    codes = {t: torch.from_numpy(_group_region(arrays, t)) for t in H.SAMPLE_TYPES[1:]}
    on = {}
    timer = Timer.from_parameters(params)
    while timer.date < timer.final_date:
        next(timer)
        on[float(timer.now)] = [i for i, (a, b) in enumerate(windows) if a <= timer.date < b]

    def factor_of(spec, net):
        act = on[float(spec.now)]
        f = None
        if 0 in act:   # window A: pub, company, all (not household) 0.8
            if net.name == "pub":
                f = leaves["pub"]
            elif net.name == "company":
                f = leaves["companyA"]
            elif net.name != "household":
                f = torch.full((3,), ALL, dtype=dtype)
        if 1 in act:   # window B: company, university
            x = {"company": leaves.get("companyB"), "university": leaves.get("university")}.get(net.name)
            if x is not None:
                f = x if f is None else f * x
        return None if f is None else f[codes[net.edge_type]]

    prof = {k: v.to(dtype) for k, v in H.profile_params(g).items()}
    lf = torch.tensor(float(params["infection_seed"]["log_fraction_initial_cases"]), dtype=dtype)
    with venue_factor(factor_of), (H.perturb_q(perturb) if perturb is not None else contextlib.nullcontext()):
        res = O.run(w, prof, sym, lf, steps, noises, dtype=dtype)
    (res["cases_per_timestep"].sum() + 0.7 * res["deaths_per_timestep"].sum()
     + 0.3 * res["cases_by_age"][:, 1].sum()).backward()
    names = [str(n) for n in g["net_names"]]
    grads = np.array([nets.networks[n].log_beta.grad.item() if nets.networks[n].log_beta.grad is not None else 0.0
                      for n in names])
    return res, grads, {k: v.grad.numpy().copy() for k, v in leaves.items()}


@pytest.mark.parametrize("family,tag", [("throughput", "sample_default"), ("reference-order", "sample_default")])
def test_sample_world_venue_factor_vs_oracle(family, tag):
    leaves = {k: torch.tensor(v, device=DEV, requires_grad=True) for k, v in (("pub", FA), ("companyA", FB),
                                                                                 ("companyB", FC), ("university", FU))}
    entries = [{"pub": leaves["pub"], "company": leaves["companyA"], "all": ALL},
               {"company": leaves["companyB"], "university": leaves["university"]}]
    runner, g, params, arrays = _sample_runner(tag, entries=entries)
    n, n_steps = runner.n_agents, int(g["n_steps"])
    order = list(leaves)
    res, is_inf, grads, gf = _run(runner, family, tag, n_steps, [leaves[k] for k in order])
    if family == "throughput":
        noises = H.philox_noises(4242 + H.RUNS[tag], n_steps + 1, n)
    else:
        noises = H.torch_noise(H.RUNS[tag], n_steps + 1, n)
    windows = _windows(params)
    ref, og, ogf = _oracle(tag, arrays, windows, noises)
    assert torch.equal(is_inf.cpu(), ref["state"]["is_infected"]), "infection masks"
    assert torch.equal(res["cases_per_timestep"].cpu(), ref["cases_per_timestep"])
    assert torch.equal(res["deaths_per_timestep"].cpu(), ref["deaths_per_timestep"])
    assert torch.equal(res["cases_by_age_65"].cpu(), ref["cases_by_age"][:, 1])
    assert torch.equal(_stages(runner).to(ref["state"]["current_stage"].dtype), ref["state"]["current_stage"])
    _, g64, gf64 = _oracle(tag, arrays, windows, noises, torch.float64)
    sens = np.zeros_like(og)
    sensf = {k: np.zeros(3) for k in order}
    for sd in (1, 2, 3):
        _, gp, gpf = _oracle(tag, arrays, windows, noises, perturb=sd)
        sens = np.maximum(sens, np.abs(gp - og))
        sensf = {k: np.maximum(sensf[k], np.abs(gpf[k] - ogf[k])) for k in order}
    names = [str(x) for x in g["net_names"]]
    keys = list(runner.model.infection_networks.networks.keys())
    mine = np.array([float(grads[keys.index(k)]) for k in names])
    H.assert_grad_parity(mine, og, g64, sens, rtol=RTOL, what=f"{family}/{tag}: venue d/dlog_beta")
    for i, k in enumerate(order):
        assert float(np.abs(ogf[k]).max()) > 0.0, k
        for r in range(3):
            H.assert_grad_parity(float(gf[i][r]), float(ogf[k][r]), float(gf64[k][r]), float(sensf[k][r]), rtol=RTOL,
                                 what=f"{family}/{tag}: d/dfactor[{k}][{r}]")


def test_factor_zero_everywhere_equals_close_venue():
    tag = "sample_default"
    zero, g, params, _ = _sample_runner(tag, entries=[{"company": 0.0}])
    closed, _, _, _ = _sample_runner(tag, close=["company"])
    n_steps = int(g["n_steps"])
    a = _run(zero, "throughput", tag, n_steps)
    b = _run(closed, "throughput", tag, n_steps)
    for k, v in a[0].items():
        assert torch.equal(b[0][k], v), k
    assert torch.equal(a[1], b[1])
    assert torch.equal(_stages(zero), _stages(closed))
    keys = list(zero.model.infection_networks.networks.keys())
    other = [i for i, k in enumerate(keys) if k != "company"]
    assert torch.allclose(a[2][other], b[2][other], rtol=1e-5, atol=0.0), (a[2], b[2])


def _batched(tag, rows):
    """One batched window of b = len(rows) samples, the pub factor row r for sample r."""
    from grad_june import ops
    runner, g, _, _ = _sample_runner(tag, entries=[{"pub": rows}] if rows is not None else None,
                                     windows=None)
    b = 4
    nets = runner.model.infection_networks.networks
    lbs = {}
    for k, net in nets.items():
        v = torch.as_tensor(net.log_beta).detach().to(DEV).reshape(()).expand(b).clone().requires_grad_(True)
        net._parameters.pop("log_beta", None)
        net.log_beta = lbs[k] = v
    runner.batch = b
    with ops.philox_seed(4242 + H.RUNS[tag]):
        results, is_inf = runner()
    _loss(results).sum().backward()
    gb = torch.stack([lbs[k].grad for k in nets.keys()], dim=1)
    return ({k: v.detach() for k, v in results.items() if k != "dates"}, is_inf.detach(), gb,
            rows.grad if rows is not None and rows.requires_grad else None)


def test_batched_rows_equal_unbatched_runs():
    tag = "sample_default"
    rows = torch.tensor([FA, [1.0, 1.0, 1.0], [0.5, 2.5, 0.7], [3.0, 0.2, 1.1]], device=DEV, requires_grad=True)
    results, is_inf, gb, gf = _batched(tag, rows)
    for r in range(4):
        leaf = rows[r].detach().clone().requires_grad_(True)
        runner, g, _, _ = _sample_runner(tag, entries=[{"pub": leaf}])
        single = _run(runner, "throughput", tag, int(g["n_steps"]), [leaf])
        for k, v in single[0].items():
            assert torch.equal(results[k][:, r], v), (r, k)
        assert torch.equal(is_inf[r].to(single[1].device), single[1]), r
        assert torch.equal(gb[r].cpu(), single[2].cpu()), r
        assert torch.equal(gf[r], single[3][0]), (r, gf[r], single[3][0])


def test_graphed_replay_and_calibrator_fit_the_venue_factors():
    from grad_june import ops
    from grad_june.calibration import Calibrator
    from grad_june.graphed import GraphedRunner
    tag = "sample_default"
    caller = torch.tensor(FB, device=DEV)
    runner, g, _, _ = _sample_runner(tag, entries=[{"pub": [0.5, 1.5, 3.0], "company": caller}])
    K = len(runner.model.infection_networks.networks)
    graphed = GraphedRunner(runner, loss_fn=_loss, seed=77, fit_venue=True)
    assert graphed.venue_names == ["0_pub_0", "0_pub_1", "0_pub_2", "0_company_0", "0_company_1", "0_company_2"]
    x = graphed.log_beta.detach().clone()
    x[K:] = torch.log10(torch.tensor([0.3, 2.0, 1.0, 1.5, 0.6, 0.9], device=DEV))
    loss, grads, _ = graphed(x)
    loss, grads = loss.clone(), grads.clone()
    pol = runner.model.policies.venue_policies.policies[0]
    assert pol.beta_factors["pub"] == [0.5, 1.5, 3.0] and pol.beta_factors["company"] is caller
    assert torch.equal(caller, torch.tensor(FB, device=DEV))
    fp = (10.0 ** x[K:K + 3]).detach().clone().requires_grad_(True)
    fc = (10.0 ** x[K + 3:]).detach().clone().requires_grad_(True)
    runner2, _, _, _ = _sample_runner(tag, entries=[{"pub": fp, "company": fc}])
    nets2 = runner2.model.infection_networks.networks
    leaves = []
    for i, k in enumerate(nets2.keys()):
        nets2[k]._parameters.pop("log_beta", None)
        nets2[k].log_beta = x[i].clone().requires_grad_(True)
        leaves.append(nets2[k].log_beta)
    with ops.philox_seed(77):
        results, _ = runner2()
    eager = _loss(results)
    eager.backward()
    assert torch.equal(loss, eager.detach())
    assert torch.equal(grads[:K], torch.stack([l.grad for l in leaves]))
    ln10 = float(np.log(10.0))
    expect = torch.cat([fp.grad * fp.detach() * ln10, fc.grad * fc.detach() * ln10])
    assert torch.allclose(grads[K:], expect, rtol=1e-5, atol=1e-6 * float(expect.abs().max())), (grads[K:], expect)

    # a target made with the company factors changed: the fit lowers its loss
    target_runner, _, _, _ = _sample_runner(tag, entries=[{"pub": [0.5, 1.5, 3.0], "company": [0.5, 0.1, 3.0]}])
    with ops.philox_seed(77):
        target = target_runner()[0]["cases_per_timestep"].detach()
    runner4, _, _, _ = _sample_runner(tag, entries=[{"pub": [0.5, 1.5, 3.0], "company": FB}])
    cal = Calibrator(runner4, loss_fn=lambda r: ((r["cases_per_timestep"] - target) ** 2).mean(), lr=0.05, seed=77,
                     fit_venue=True)
    hist = cal.fit(8)
    assert "log_venue_factor_0_pub_2" in hist.columns and "grad_log_venue_factor_0_company_0" in hist.columns
    assert float(hist["loss"].iloc[-1]) < float(hist["loss"].iloc[0]), hist["loss"].tolist()


def test_modular_path_unit_factors_and_parity():
    """A user network subclass sends the step through the modular path: unit factors change nothing, and with
    factors its probabilities and gradients at one step match the fused networks phase."""
    from grad_june import ops
    from grad_june.infection_networks import CompanyNetwork

    class MyCompany(CompanyNetwork):
        @classmethod
        def _get_name(cls):
            return "company"

        def _get_transmissions(self, data, policies, timer):
            return super()._get_transmissions(data, policies, timer) * 1.0

    tag = "sample_default"
    whole = None
    plain, g, params, _ = _sample_runner(tag)
    whole = [(_day(params, -1), _day(params, 100))]
    ones, _, _, _ = _sample_runner(tag, entries=[{"all": 1.0}], windows=whole)
    for r in (plain, ones):
        old = r.model.infection_networks.networks["company"]
        new = MyCompany(log_beta=old.log_beta, device=DEV)
        r.model.infection_networks.networks["company"] = new
    n_steps = int(g["n_steps"])
    a = _run(plain, "throughput", tag, n_steps)
    b = _run(ones, "throughput", tag, n_steps)
    for k, v in a[0].items():
        assert torch.equal(b[0][k], v), k
    assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])

    # one step: modular (user subclass) against the fused networks phase, same factors
    f = torch.tensor([0.3, 1.7, 2.2], device=DEV, requires_grad=True)
    fused, _, _, _ = _sample_runner(tag, entries=[{"company": f, "pub": 0.5}], windows=whole)
    mod, _, _, _ = _sample_runner(tag, entries=[{"company": f, "pub": 0.5}], windows=whole)
    mod.model.infection_networks.networks["company"] = MyCompany(
        log_beta=mod.model.infection_networks.networks["company"].log_beta, device=DEV)
    outs = []
    for r in (fused, mod):
        r.timer.reset()
        with ops.philox_seed(5):
            r.set_initial_cases()
        next(r.timer)
        data = r.data
        data["agent"].transmission = ops.transmission(
            r.timer.now, data["agent"].infection_time, data["agent"].is_infected,
            *[data["agent"].infection_parameters[k] for k in ("max_infectiousness", "shape", "rate", "shift")])
        venue = r._venue(r.timer)
        f.grad = None
        q = r.model.infection_networks(data=data, timer=r.timer, policies=r.model.policies, venue=venue)
        q.sum().backward()
        outs.append((q.detach().clone(), f.grad.detach().clone()))
    assert torch.allclose(outs[0][0], outs[1][0], rtol=1e-6, atol=1e-7)
    assert torch.allclose(outs[0][1], outs[1][1], rtol=1e-4, atol=1e-6), (outs[0][1], outs[1][1])


def test_networks_sharing_an_edge_type_get_their_own_factor_gradient():
    """Two PLAIN networks on the company type share the group sums of the throughput path, but each has its own beta
    and its own row of factors: d/df[k, r] = beta_k * sum over the region's groups of own * pc * S * R, so the two rows
    differ exactly by beta_1 / beta_0."""
    from grad_june import ops
    tag = "sample_default"
    runner, _, _, _ = _sample_runner(tag)
    runner.timer.reset()
    with ops.philox_seed(11):
        runner._restore_for_window()
        runner.set_initial_cases()
    for _ in range(3):
        next(runner.timer)
    timer = runner.timer
    static, _ = runner.model._static(runner.data, torch.device(DEV))
    world = static.world
    nets = [ops.NetSpec("a", "company", ops.KIND_PLAIN), ops.NetSpec("b", "company", ops.KIND_PLAIN),
            ops.NetSpec("household", "household", ops.KIND_HOUSEHOLD)]
    spec = ops.StepSpec(now=timer.now, dt=timer.duration, day_type=0, nets=nets, quarantine=None, want_probs=False)
    assert ops.step_plan(static, spec) == "throughput"
    codes = torch.arange(world.n_groups) % 3
    venue_labels = ops.make_venue_labels(codes, 3, world.type_group_off, DEV)
    beta = torch.tensor([0.3, 0.7, 0.5], device=DEV, requires_grad=True)
    f = torch.tensor([[0.5, 1.5, 2.5], [2.0, 0.4, 1.1], [1.0, 1.0, 1.0]], device=DEV, requires_grad=True)
    agent = runner.data["agent"]
    sym = agent.symptoms
    state = {"s": agent.susceptibility, "inf": agent.is_infected, "tinf": agent.infection_time,
             "cur": sym["current_stage"], "nxt": sym["next_stage"], "ttn": sym["time_to_next_stage"]}
    with ops.philox_seed(12):
        out = ops.infection_step(static, spec, beta, state, venue=ops.Venue(venue_labels, f))
    (out["inf"].sum() + 0.3 * out["s"].sum() + out["red"][1]).backward()
    g = f.grad
    assert float(g[0].abs().max()) > 0.0
    if world.type_tier[world.types.index("household")] == 1:   # a RANGE-tier network's row is 0
        assert torch.equal(g[2], torch.zeros(3, device=DEV))
    assert torch.allclose(g[1], g[0] * (0.7 / 0.3), rtol=1e-5, atol=0.0), g


_SYN = {}
N_SYN = 1_000_000
_SYN_BY = {"super_area": "venue_super_area", "area": "venue_area", "random": "venue_random"}


def _syn_world():
    if "data" not in _SYN:
        from grad_june.default_config import default_parameters
        from grad_june.runner import Runner
        from grad_june.world import group_labels, make_synthetic_world
        params = default_parameters()
        params["system"]["device"] = DEV
        params["timer"]["total_days"] = 6
        params["infection_seed"]["log_fraction_initial_cases"] = -2.0
        world = make_synthetic_world(N_SYN, seed=4, device=DEV, agents_per_super_area=7500)
        ids = torch.arange(N_SYN, device=DEV)
        world["agent"].super_area = ids // 7500
        world["agent"].area = ids // 300
        rng = np.random.default_rng(9)
        for t in world.venue_types():
            if t == "household":
                continue
            world[t].venue_super_area = torch.as_tensor(group_labels(world, t, "super_area"))
            world[t].venue_area = torch.as_tensor(group_labels(world, t, "area"))
            world[t].venue_random = torch.as_tensor(rng.integers(0, 100_000, len(world[t]["id"])))
        torch.manual_seed(5)
        data = Runner.get_data(params, data=world)
        agent = data["agent"]
        _SYN["start"] = ({k: agent[k].clone() for k in ("susceptibility", "is_infected", "infection_time", "transmission")},
                         {k: v.clone() for k, v in agent.symptoms.items()})
        _SYN["data"], _SYN["params"] = data, params
    agent = _SYN["data"]["agent"]
    for k, v in _SYN["start"][0].items():
        agent[k] = v.clone()
    agent.symptoms = {k: v.clone() for k, v in _SYN["start"][1].items()}
    return _SYN["data"], _SYN["params"]


def _syn_window(by):
    """One 1 M-agent window with a venue policy active on every step that gives every non-household network its own
    differentiable [R] factor: (results, d/dlog_beta {name}, {name: (factor, d/dfactor)})."""
    from grad_june import GradJune, Timer, ops
    from grad_june.policies import RegionalVenueDistancing, VenuePolicies
    from grad_june.runner import Runner
    data, params = _syn_world()
    model = GradJune.from_parameters(params)
    nets = model.infection_networks.networks
    for key in nets.keys():
        nets[key].log_beta = torch.nn.Parameter(torch.as_tensor(nets[key].log_beta, dtype=torch.float32).to(DEV))
    types = [t for t in data.venue_types() if t != "household"]
    R = len(np.unique(np.concatenate([data[t][_SYN_BY[by]].cpu().numpy() for t in types])))
    leaves = {}
    for i, name in enumerate(k for k in nets.keys() if k != "household"):
        leaves[name] = (0.2 + 2.8 * torch.rand(R, generator=torch.Generator().manual_seed(i))).to(DEV).requires_grad_(True)
    model.policies.venue_policies = VenuePolicies([RegionalVenueDistancing(
        _day(params, -1), _day(params, 100), _SYN_BY[by], dict(leaves), device=DEV)])
    runner = Runner(model=model, data=data, timer=Timer.from_parameters(params), log_fraction_initial_cases=-2.0,
                    save_path="/tmp/gj_test_venue", parameters=params)
    assert len(runner.venue_labels) == R
    with ops.philox_seed(321):
        results, _ = runner()
    (results["cases_per_timestep"].sum() + 3.0 * results["deaths_per_timestep"].sum()).backward()
    gb = {k: (nets[k].log_beta.grad.detach().clone() if nets[k].log_beta.grad is not None
              else torch.zeros((), device=DEV)) for k in nets.keys()}
    res = {k: v.detach().clone() for k, v in results.items() if k != "dates"}
    return res, gb, {k: (v.detach(), v.grad.detach().clone()) for k, v in leaves.items()}


@pytest.mark.parametrize("by", ["super_area", "area", "random"])
def test_synthetic_world_factor_gradients_sum_to_the_log_beta_gradient(by):
    """sum_r dL/dlog10 f[k, r] = dL/dlog_beta_k for every network (both are sums of beta_k * f * own * pc * S * R over
    the groups), with a factor per network over thousands to 100 000 group regions, and bit-identical reruns."""
    res, gb, gf = _syn_window(by)
    ln10 = float(np.log(10.0))
    scale = max(float(gb[k].abs()) for k in gf)
    assert scale > 0.0
    for k, (f, g) in gf.items():
        lhs = ln10 * float((f.double() * g.double()).sum())
        rhs = float(gb[k])
        assert abs(lhs - rhs) <= 1e-4 * abs(rhs) + 1e-6 * scale, (by, k, lhs, rhs)
    res2, gb2, gf2 = _syn_window(by)
    for k, v in res.items():
        assert torch.equal(res2[k], v), k
    for k in gb:
        assert torch.equal(gb[k], gb2[k]), k
    for k in gf:
        assert torch.equal(gf[k][1], gf2[k][1]), k


def _free_port():
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _partition_worker(rank, world_size, port, out):
    import os

    import torch.distributed as dist
    from grad_june import GradJune, Timer
    from grad_june.default_config import default_parameters
    from grad_june.graphed import GraphedRunner
    from grad_june.partition import partition_world
    from grad_june.policies import RegionalVenueDistancing, VenuePolicies
    from grad_june.runner import Runner
    from grad_june.world import group_labels, make_synthetic_world
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = f"cuda:{rank}"
    dist.init_process_group("nccl", rank=rank, world_size=world_size, device_id=torch.device(dev))
    try:
        params = default_parameters()
        params["system"]["device"] = dev
        params["timer"]["total_days"] = 4
        params["infection_seed"]["log_fraction_initial_cases"] = -1.5
        torch.manual_seed(5)
        world = make_synthetic_world(200_000, seed=5, device=dev, agents_per_super_area=5000)
        world["agent"].area = torch.arange(200_000, device=dev) // 300
        types = [t for t in world.venue_types() if t != "household"]
        for t in types:     # labels set on the complete world, before partitioning
            world[t].region = torch.as_tensor(group_labels(world, t, "area"))
        R = len(np.unique(np.concatenate([world[t].region.cpu().numpy() for t in types])))
        full = Runner.get_data(params, data=world)

        def run(data):
            """The window as one CUDA graph (exchanges and the gradient all-reduce included) with the venue factors
            fitted: (venue labels, cases, is_infected of this rank's agents, [log-betas..., log10 factors...] grad)."""
            model = GradJune.from_parameters(params)
            model.policies.venue_policies = VenuePolicies([RegionalVenueDistancing(
                _day(params, 1), _day(params, 3), "region", {"all": torch.linspace(0.3, 2.5, R, device=dev)},
                device=dev)])
            runner = Runner(model=model, data=data, timer=Timer.from_parameters(params), log_fraction_initial_cases=-1.5,
                            save_path="/tmp/gj_test_venue", parameters=params)
            loss_fn = lambda r: r["cases_per_timestep"].sum() + 2.0 * r["deaths_per_timestep"].sum()  # noqa: E731
            g = GraphedRunner(runner, loss_fn, seed=4242, fit_venue=True)
            for _ in range(2):
                _, grads, results = g()
            torch.cuda.synchronize()
            ret = (np.asarray(runner.venue_labels), results["cases_per_timestep"].detach().cpu().numpy(),
                   g.is_infected.detach().cpu().numpy(), grads.detach().cpu().numpy().copy(), g.n_beta)
            g.graph.reset()
            return ret

        local = partition_world(full, rank, world_size)
        part = local._gj_partition
        labels, cases, inf, grads, K = run(local)
        out[f"inf{rank}"] = (part.agent_lo, part.agent_hi, inf)
        if rank == 0:
            out["part"] = (labels, cases, grads, K)
            labels1, cases1, inf1, grads1, _ = run(full)
            out["full"] = (labels1, cases1, inf1, grads1, R)
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_two_gpus_venue_factor_gradients_match_one():
    """A partitioned world with a venue policy, graphed with fit_venue=True: boundary groups carry their global label
    on every rank, the owner alone adds their d/df terms (dbeta_w) and the ranks' gradients are summed in the captured
    all-reduce.  The trajectory equals the single-GPU one exactly, the gradients to rounding."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 CUDA devices")
    import torch.multiprocessing as mp
    out = mp.Manager().dict()
    mp.spawn(_partition_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    labels, cases, grads, K = out["part"]
    labels1, cases1, inf1, grads1, R = out["full"]
    inf = np.empty_like(inf1)
    for r in range(2):
        lo, hi, x = out[f"inf{r}"]
        inf[lo:hi] = x
    assert np.array_equal(labels, labels1) and len(labels1) == R > 100
    assert cases1[-1] > cases1[0] > 0
    assert np.array_equal(inf, inf1), int((inf != inf1).sum())
    assert np.array_equal(cases, cases1)
    assert grads.shape == grads1.shape == (K + R,)
    for part, ref in ((grads[:K], grads1[:K]), (grads[K:], grads1[K:])):
        assert np.abs(ref).max() > 0
        assert np.allclose(part, ref, rtol=1e-4, atol=1e-6 * np.abs(ref).max()), (part, ref)
