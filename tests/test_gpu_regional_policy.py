"""Regional social distancing on the GPU: a per-region factor on every agent's force of infection, before the clamp.

1. identity: factors of 1 over the whole window reproduce the run without the policy bit for bit (throughput,
   reference-order and batched kernels, and a 1 M-agent world);
2. the renumbered sample world with the agents' leisure group as region (3 regions, factors 0.2 to 3, two overlapping
   windows) against the oracle with the factor gathered per agent (``region_oracle.regional_factor``): exact masks,
   stages and series; d/dlog_beta and d/dfactor per region and policy through ``assert_grad_parity``;
3. a 1 M-agent world with super-area, 300-agent area and 100 000 random labels: the homogeneity invariant
   sum_r m_r dL/dm_r = sum_k dL/dlog10(beta_k) / ln 10, run-to-run bit identity of the factor gradient, and the steps
   outside the window equal to the policy-free run;
4. batched b = 4 against the unbatched runs, graph replay against the eager window, Calibrator(fit_regional=True);
5. a user network subclass (the modular path): unit factors change nothing, the homogeneity invariant holds, and at one
   step its probabilities and gradients match the library's networks phase with the factor applied in the kernels;
6. 2 GPUs against 1: a partitioned world, graphed with fit_regional=True (skips on one GPU)."""
import contextlib
import datetime
import os
import socket

import numpy as np
import pytest
import torch

import helpers as H
from oracle import gj_oracle as O
from region_oracle import regional_factor

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
RTOL = 1e-5
N_SYN = 1_000_000
FA = [0.2, 1.5, 3.0]
FB = [2.0, 0.5, 1.2]


@pytest.fixture(autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")


def _leisure_label(arrays):
    label = np.zeros(len(arrays["age"]), dtype=np.int64)
    label[arrays["leisure_src"]] = arrays["leisure_dst"]
    return label


def _day(params, d):
    return datetime.datetime.strptime(str(params["timer"]["initial_day"]), "%Y-%m-%d") + datetime.timedelta(days=d)


def _windows(params):
    """Two overlapping windows: A on days [2, 9), B on [6, 13)."""
    return [(_day(params, 2), _day(params, 9)), (_day(params, 6), _day(params, 13))]


def _policies(params, factors, by="leisure_group", windows=None):
    from grad_june.policies import RegionalPolicies, RegionalSocialDistancing
    windows = windows or _windows(params)
    return RegionalPolicies([RegionalSocialDistancing(w[0], w[1], by, f, device=DEV) for w, f in zip(windows, factors)])


def _sample_runner(tag, factors=None, windows=None):
    """The renumbered sample world with ``data["agent"].leisure_group`` as the region; ``factors``: one entry per
    regional policy (None: no regional policy).  Log-betas are leaves."""
    from grad_june import GradJune, Runner, Timer
    from grad_june.world import layout_order_of, world_from_arrays
    g = np.load(H.GOLDEN / f"run_{tag}.npz")
    params, _ = H.load_params(tag)
    params["system"]["device"] = DEV
    params["system"]["renumber_agents"] = True
    arrays = np.load(H.GOLDEN / "sample_world.npz")
    world = world_from_arrays(arrays, H.SAMPLE_TYPES)
    world["agent"].leisure_group = torch.from_numpy(_leisure_label(arrays))
    data = Runner.get_data(params, data=world)
    data["agent"].infection_parameters = {k: layout_order_of(data, v.to(DEV)).contiguous()
                                          for k, v in H.profile_params(g).items()}
    model = GradJune.from_parameters(params)
    if factors is not None:
        model.policies.regional_policies = _policies(params, factors, windows=windows)
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
    """One eager window and backward: (results, is_infected, d/dlog_beta, [d/dfactor per leaf])."""
    from grad_june import ops
    from gpu_helpers import noise_provider
    nets = runner.model.infection_networks.networks
    for net in nets.values():
        net.log_beta.grad = None
    if family == "throughput":
        with ops.philox_seed(4242 + H.RUNS[tag]):
            results, is_inf = runner()
    else:
        with ops.inject_noise(noise_provider(H.RUNS[tag], n_steps + 1, runner.n_agents)):
            results, is_inf = runner()
    _loss(results).backward()
    grads = torch.stack([nets[k].log_beta.grad.detach().clone() if nets[k].log_beta.grad is not None
                         else torch.zeros((), device=DEV) for k in nets.keys()])
    res = {k: v.detach().clone() for k, v in results.items() if k != "dates"}
    return res, is_inf.detach().clone(), grads, [l.grad.detach().clone() for l in leaves]


def _state(runner):
    agent = runner.data["agent"]
    out = {k: agent[k].detach().clone() for k in ("susceptibility", "is_infected", "infection_time")}
    out.update({k: v.detach().clone() for k, v in agent.symptoms.items()})
    return out


@pytest.mark.parametrize("family", ["throughput", "reference-order"])
def test_identity_with_unit_factors(family):
    tag = "sample_default"
    plain, g, params, _ = _sample_runner(tag)
    n_steps = int(g["n_steps"])
    whole = [(_day(params, -1), _day(params, 100))]
    leaf = torch.ones(3, device=DEV, requires_grad=True)
    ones, _, _, _ = _sample_runner(tag, factors=[leaf], windows=whole)
    a = _run(plain, family, tag, n_steps)
    b = _run(ones, family, tag, n_steps, [leaf])
    for k, v in a[0].items():
        assert torch.equal(b[0][k], v), k
    assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])
    sa, sb = _state(plain), _state(ones)
    for k, v in sa.items():
        assert torch.equal(v, sb[k]), k
    assert b[3][0].shape == (3,) and bool(torch.isfinite(b[3][0]).all())


def _oracle(tag, label, factors, windows, noises, dtype=torch.float32, perturb=None):
    """The oracle with the regional factors gathered per agent: (result, d/dlog_beta, [d/dfactor per policy]).
    ``perturb``: a ``helpers.perturb_q`` seed; its hook wraps the regional one, so the perturbed q include the factor."""
    from grad_june import Timer
    from grad_june.policies import Policies
    from grad_june.symptoms import SymptomsSampler
    g = np.load(H.GOLDEN / f"run_{tag}.npz")
    params, _ = H.load_params(tag)    # the oracle runs on the host
    w = H.oracle_world(np.load(H.GOLDEN / "sample_world.npz"), H.SAMPLE_TYPES)
    nets = H.make_leaf_networks(params)
    steps = H.oracle_schedule(params, nets, Policies.from_parameters(params))
    if dtype != torch.float32:
        for s in steps:
            for n in s.nets:
                n.beta = n.beta.to(dtype)
    sym = H.oracle_symptoms(SymptomsSampler.from_parameters(params))
    noises = [O.StepNoise(E=n.E.to(dtype), u=n.u.to(dtype), z=n.z.to(dtype)) for n in noises]
    leaves = [torch.tensor(f, dtype=dtype, requires_grad=True) for f in factors]
    idx = torch.as_tensor(label, dtype=torch.long)
    active = {}
    timer = Timer.from_parameters(params)
    while timer.date < timer.final_date:
        next(timer)
        active[float(timer.now)] = [i for i, (a, b) in enumerate(windows) if a <= timer.date < b]

    def factor_of(spec):
        on = active[float(spec.now)]
        if not on:
            return None
        f = leaves[on[0]]
        for i in on[1:]:
            f = f * leaves[i]
        return f[idx]

    prof = {k: v.to(dtype) for k, v in H.profile_params(g).items()}
    lf = torch.tensor(float(params["infection_seed"]["log_fraction_initial_cases"]), dtype=dtype)
    with regional_factor(factor_of), (H.perturb_q(perturb) if perturb is not None else contextlib.nullcontext()):
        res = O.run(w, prof, sym, lf, steps, noises, dtype=dtype)
    (res["cases_per_timestep"].sum() + 0.7 * res["deaths_per_timestep"].sum()
     + 0.3 * res["cases_by_age"][:, 1].sum()).backward()
    names = [str(n) for n in g["net_names"]]
    grads = np.array([nets.networks[n].log_beta.grad.item() if nets.networks[n].log_beta.grad is not None else 0.0
                      for n in names])
    return res, grads, [l.grad.numpy().copy() for l in leaves]


@pytest.mark.parametrize("family,tag", [("throughput", "sample_default"), ("throughput", "sample_deadly"),
                                        ("reference-order", "sample_default"), ("reference-order", "sample_policies")])
def test_sample_world_regional_factor_vs_oracle(family, tag):
    leaves = [torch.tensor(FA, device=DEV, requires_grad=True), torch.tensor(FB, device=DEV, requires_grad=True)]
    runner, g, params, arrays = _sample_runner(tag, factors=leaves)
    assert runner.region_labels.tolist() == [0, 1, 2]
    n, n_steps = runner.n_agents, int(g["n_steps"])
    res, is_inf, grads, gf = _run(runner, family, tag, n_steps, leaves)
    if family == "throughput":
        noises = H.philox_noises(4242 + H.RUNS[tag], n_steps + 1, n)
    else:
        noises = H.torch_noise(H.RUNS[tag], n_steps + 1, n)
    label = _leisure_label(arrays)
    windows = _windows(params)
    ref, og, ogf = _oracle(tag, label, [FA, FB], windows, noises)
    assert torch.equal(is_inf.cpu(), ref["state"]["is_infected"]), "infection masks"
    assert torch.equal(res["cases_per_timestep"].cpu(), ref["cases_per_timestep"])
    assert torch.equal(res["deaths_per_timestep"].cpu(), ref["deaths_per_timestep"])
    assert torch.equal(res["cases_by_age_65"].cpu(), ref["cases_by_age"][:, 1])
    from grad_june.world import original_order
    stages = original_order(runner.data, runner.data["agent"].symptoms["current_stage"]).cpu()
    assert torch.equal(stages.to(ref["state"]["current_stage"].dtype), ref["state"]["current_stage"]), "stages"
    _, g64, gf64 = _oracle(tag, label, [FA, FB], windows, noises, torch.float64)
    sens = np.zeros_like(og)
    sensf = [np.zeros(3), np.zeros(3)]
    for sd in (1, 2, 3):
        _, gp, gpf = _oracle(tag, label, [FA, FB], windows, noises, perturb=sd)
        sens = np.maximum(sens, np.abs(gp - og))
        sensf = [np.maximum(s, np.abs(a - b)) for s, a, b in zip(sensf, gpf, ogf)]
    names = [str(x) for x in g["net_names"]]
    keys = list(runner.model.infection_networks.networks.keys())
    mine = np.array([float(grads[keys.index(k)]) for k in names])
    H.assert_grad_parity(mine, og, g64, sens, rtol=RTOL, what=f"{family}/{tag}: regional d/dlog_beta")
    for p in range(2):
        assert float(np.abs(ogf[p]).max()) > 0.0
        for r in range(3):
            H.assert_grad_parity(float(gf[p][r]), float(ogf[p][r]), float(gf64[p][r]), float(sensf[p][r]), rtol=RTOL,
                                 what=f"{family}/{tag}: d/dfactor[{p}][{r}]")


def _homogeneity_tolerance():
    """The fp32 oracle's relative residual of the homogeneity invariant on the sample world (one policy over the whole
    window), with the fp64 oracle's as the reference: the tolerance of the large-world check."""
    tag = "sample_default"
    params, _ = H.load_params(tag)
    g = np.load(H.GOLDEN / f"run_{tag}.npz")
    arrays = np.load(H.GOLDEN / "sample_world.npz")
    label = _leisure_label(arrays)
    whole = [(_day(params, -1), _day(params, 100))]
    noises = H.torch_noise(H.RUNS[tag], int(g["n_steps"]) + 1, len(arrays["age"]))
    out = []
    for dt in (torch.float32, torch.float64):
        _, gb, gf = _oracle(tag, label, [FA], whole, noises, dt)
        lhs = float(np.dot(np.asarray(FA, dtype=np.float64), gf[0]))
        rhs = float(gb.sum()) / np.log(10.0)
        out.append(abs(lhs - rhs) / max(abs(rhs), 1e-30))
    return max(10.0 * out[0], 1e-4), out


_SYN = {}


def _syn_world():
    if "data" not in _SYN:
        from grad_june.default_config import default_parameters
        from grad_june.runner import Runner
        from grad_june.world import make_synthetic_world
        params = default_parameters()
        params["system"]["device"] = DEV
        params["timer"]["total_days"] = 6
        params["infection_seed"]["log_fraction_initial_cases"] = -2.0
        world = make_synthetic_world(N_SYN, seed=4, device=DEV, agents_per_super_area=7500)
        ids = torch.arange(N_SYN, device=DEV)
        world["agent"].super_area = ids // 7500
        world["agent"].area = ids // 300
        world["agent"].random_label = torch.randint(0, 100_000, (N_SYN,), device=DEV,
                                                    generator=torch.Generator(DEV).manual_seed(9))
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


def _syn_window(by, factor, window):
    """(runner, results, d/dlog_beta [K], d/dfactor or None) of one 1 M-agent window; ``factor(R)`` builds the
    factors, ``window`` = (first day, end day) or None for no policy."""
    from grad_june import GradJune, Timer, ops
    from grad_june.runner import Runner
    data, params = _syn_world()
    model = GradJune.from_parameters(params)
    nets = model.infection_networks.networks
    for key in nets.keys():
        nets[key].log_beta = torch.nn.Parameter(torch.as_tensor(nets[key].log_beta, dtype=torch.float32).to(DEV))
    leaf = None
    if window is not None:
        n_reg = len(np.unique(data["agent"][by].cpu().numpy()))
        leaf = factor(n_reg).to(DEV).requires_grad_(True)
        w = (_day(params, window[0]), _day(params, window[1]))
        model.policies.regional_policies = _policies(params, [leaf], by=by, windows=[w])
    runner = Runner(model=model, data=data, timer=Timer.from_parameters(params), log_fraction_initial_cases=-2.0,
                    save_path="/tmp/gj_test_regional", parameters=params)
    with ops.philox_seed(321):
        results, _ = runner()
    (results["cases_per_timestep"].sum() + 3.0 * results["deaths_per_timestep"].sum()).backward()
    gb = torch.stack([nets[k].log_beta.grad.detach().clone() if nets[k].log_beta.grad is not None
                      else torch.zeros((), device=DEV) for k in nets.keys()])
    res = {k: v.detach().clone() for k, v in results.items() if k != "dates"}
    return runner, res, gb, (leaf.grad.detach().clone() if leaf is not None else None)


@pytest.mark.parametrize("by", ["super_area", "area", "random_label"])
def test_synthetic_world_homogeneity_and_reproducibility(by):
    tol, measured = _homogeneity_tolerance()

    def factors(R):
        return 0.2 + 2.8 * torch.rand(R, generator=torch.Generator().manual_seed(3))
    whole = (-1, 100)
    _, res, gb, gf = _syn_window(by, factors, whole)
    lhs = float((factors(len(gf)).double().to(DEV) * gf.double()).sum())
    rhs = float(gb.double().sum()) / np.log(10.0)
    assert abs(lhs - rhs) <= tol * abs(rhs), (by, lhs, rhs, tol, measured)
    _, res2, gb2, gf2 = _syn_window(by, factors, whole)
    assert torch.equal(gf, gf2) and torch.equal(gb, gb2)
    for k, v in res.items():
        assert torch.equal(res2[k], v), k


def test_synthetic_world_identity_and_off_steps():
    _, plain, gb0, _ = _syn_window("super_area", None, None)
    _, ones, gb1, gf1 = _syn_window("super_area", lambda R: torch.ones(R), (-1, 100))
    for k, v in plain.items():
        assert torch.equal(ones[k], v), k
    assert torch.equal(gb0, gb1) and bool(torch.isfinite(gf1).all())
    # a window on days [3, 5): every series equals the policy-free run before day 3
    _, late, _, _ = _syn_window("super_area", lambda R: torch.full((R,), 0.3), (3, 5))
    for k, v in plain.items():
        assert torch.equal(late[k][:3], v[:3]), k
    assert not torch.equal(late["cases_per_timestep"], plain["cases_per_timestep"])


def _batched(tag, factors):
    """One batched b = 4 window of the sample world (equal log-betas in every row): (results, is_infected,
    d/dlog_beta [4, K], d/dfactor [4, 3] or None).  ``factors``: [4, 3] rows of the policy's factors, or None."""
    from grad_june import ops
    leaf = None if factors is None else factors.clone().requires_grad_(True)
    runner, g, _, _ = _sample_runner(tag, factors=None if leaf is None else [leaf])
    runner.batch = 4
    nets = runner.model.infection_networks.networks
    for k in nets.keys():
        value = nets[k].log_beta.detach().reshape(()).to(DEV)
        nets[k]._parameters.pop("log_beta", None)
        nets[k].log_beta = value.repeat(4).requires_grad_(True)
    with ops.philox_seed(4242 + H.RUNS[tag]):
        results, is_inf = runner()
    _loss(results).sum().backward()
    gb = torch.stack([nets[k].log_beta.grad for k in nets.keys()], dim=1)
    return results, is_inf, gb, (None if leaf is None else leaf.grad)


def test_batched_rows_equal_unbatched_runs():
    tag = "sample_default"
    rows = torch.tensor([FA, [1.0, 1.0, 1.0], [0.5, 2.5, 0.7], [3.0, 0.2, 1.1]], device=DEV)
    singles = []
    for r in range(4):
        leaf = rows[r].clone().requires_grad_(True)
        runner, g, _, _ = _sample_runner(tag, factors=[leaf])
        singles.append(_run(runner, "throughput", tag, int(g["n_steps"]), [leaf]))
    results, is_inf, gb, gf = _batched(tag, rows)
    for r in range(4):
        for k, v in singles[r][0].items():
            assert torch.equal(results[k][:, r] if results[k].dim() > 1 else results[k], v), (r, k)
        assert torch.equal(is_inf[r].to(singles[r][1].device), singles[r][1]), r
        assert torch.equal(gf[r], singles[r][3][0]), (r, gf[r], singles[r][3][0])
        assert torch.equal(gb[r].cpu(), singles[r][2].cpu()), r
    # identity: row 1 holds factors of 1, so it equals the rows of a batched window without the policy
    plain, plain_inf, plain_gb, _ = _batched(tag, None)
    for k, v in plain.items():
        if k == "dates":
            continue
        for r in range(4):
            assert torch.equal(results[k][:, 1], v[:, r]), (k, r)
    for r in range(4):
        assert torch.equal(is_inf[1], plain_inf[r]) and torch.equal(gb[1], plain_gb[r]), r
    assert not torch.equal(results["cases_per_timestep"][:, 0], plain["cases_per_timestep"][:, 0])


def test_graphed_replay_and_calibrator_fit_the_regional_factors():
    from grad_june import ops
    from grad_june.calibration import Calibrator
    from grad_june.graphed import GraphedRunner
    tag = "sample_default"
    runner, g, _, _ = _sample_runner(tag, factors=[list(FA), 0.8])
    K = len(runner.model.infection_networks.networks)
    graphed = GraphedRunner(runner, loss_fn=_loss, seed=77, fit_regional=True)
    assert graphed.regional_names == ["0_0", "0_1", "0_2", "1_0", "1_1", "1_2"]
    assert tuple(graphed.log_beta.shape) == (K + 6,)
    x = graphed.log_beta.detach().clone()
    x[K:] = torch.log10(torch.tensor([0.3, 2.0, 1.0, 1.5, 0.6, 0.9], device=DEV))
    loss, grads, _ = graphed(x)
    loss, grads = loss.clone(), grads.clone()
    # the eager window at the same parameters and Philox key
    fa = (10.0 ** x[K:K + 3]).detach().clone().requires_grad_(True)
    fb = (10.0 ** x[K + 3:]).detach().clone().requires_grad_(True)
    runner2, _, _, _ = _sample_runner(tag, factors=[fa, fb])
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
    expect = torch.cat([fa.grad * fa.detach() * ln10, fb.grad * fb.detach() * ln10])
    assert torch.allclose(grads[K:], expect, rtol=1e-5, atol=1e-6 * float(expect.abs().max())), (grads[K:], expect)

    # a target made with region 2's first factor changed: the fit lowers its loss
    runner3, _, _, _ = _sample_runner(tag, factors=[[FA[0], FA[1], 0.5], 0.8])
    with ops.philox_seed(77):
        target = runner3()[0]["cases_per_timestep"].detach()
    runner4, _, _, _ = _sample_runner(tag, factors=[list(FA), 0.8])
    cal = Calibrator(runner4, loss_fn=lambda r: ((r["cases_per_timestep"] - target) ** 2).mean(), lr=0.05, seed=77,
                     fit_regional=True)
    hist = cal.fit(15)
    for col in ("log_factor_0_2", "grad_log_factor_1_0"):
        assert col in hist.columns, col
    assert hist["loss"].iloc[-1] < hist["loss"].iloc[0], hist["loss"].tolist()
    assert runner4.model.policies.regional_policies.policies[0].beta_factors == list(FA)   # the policy is left as built

    # factors that are not fitted stay the caller's: an nn.Parameter keeps its registration and its identity
    param = torch.nn.Parameter(torch.tensor(FA, device=DEV))
    runner5, _, _, _ = _sample_runner(tag, factors=[param])
    g5 = GraphedRunner(runner5, loss_fn=_loss, seed=77)
    g5()
    pol = runner5.model.policies.regional_policies.policies[0]
    assert pol.beta_factors is param and pol._parameters.get("beta_factors") is param
    # a factor of 0 has no log10: fitting it is refused with a clear error
    runner6, _, _, _ = _sample_runner(tag, factors=[[0.0, 1.0, 2.0]])
    with pytest.raises(ValueError, match="factor > 0"):
        GraphedRunner(runner6, loss_fn=_loss, seed=77, fit_regional=True)


def test_modular_path_applies_the_factor():
    """A user network subclass runs the modular path, which applies the same factor in torch before the clamp: unit
    factors reproduce the run without the policy bit for bit, and the gradient satisfies the homogeneity invariant
    sum_r m_r dL/dm_r = sum_k dL/dlog10(beta_k) / ln 10 (the pressure is linear in the betas)."""
    from grad_june import ops
    from grad_june.infection_networks.base import InfectionNetwork
    tag = "sample_default"

    def modular(factors, windows=None):
        runner, g, params, _ = _sample_runner(tag, factors=factors, windows=windows)
        nets = runner.model.infection_networks.networks
        name = next(k for k, net in nets.items() if net.kind == ops.KIND_PLAIN)   # a plain venue

        class Custom(type(nets[name])):
            def _get_susceptibilities(self, data, policies, timer):
                return 1.0 * InfectionNetwork._get_susceptibilities(self, data, policies, timer)

        nets[name].__class__ = Custom
        assert runner.model.kernel_family(runner.data, runner.timer).startswith("modular")
        return runner, g, params

    plain, g, params = modular(None)
    n_steps = int(g["n_steps"])
    whole = [(_day(params, -1), _day(params, 100))]
    one = torch.ones(3, device=DEV, requires_grad=True)
    ones, _, _ = modular([one], whole)
    a = _run(plain, "throughput", tag, n_steps)
    b = _run(ones, "throughput", tag, n_steps, [one])
    for k, v in a[0].items():
        assert torch.equal(b[0][k], v), k
    assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])
    leaf = torch.tensor(FA, device=DEV, requires_grad=True)
    runner, _, _ = modular([leaf], whole)
    res, _, gb, gf = _run(runner, "throughput", tag, n_steps, [leaf])
    assert not torch.equal(res["cases_per_timestep"], a[0]["cases_per_timestep"])
    lhs = float((leaf.detach().double() * gf[0].double()).sum())
    rhs = float(gb.double().sum()) / np.log(10.0)
    tol, measured = _homogeneity_tolerance()
    assert abs(lhs - rhs) <= tol * abs(rhs), (lhs, rhs, tol, measured)


def test_modular_path_matches_the_kernels_at_one_step():
    """At one mid-epidemic step with factors 0.2 / 1.5 / 3 per region: the modular path (a user network subclass, the
    factor gathered in torch) gives the probabilities and the gradients of the library's networks phase (the factor
    applied inside the kernels) — with respect to every region's factor and every log-beta."""
    from grad_june import ops
    from grad_june.infection_networks.base import InfectionNetwork
    tag = "sample_default"
    leaf = torch.tensor(FA, device=DEV, requires_grad=True)
    _, _, params, _ = _sample_runner(tag)
    runner, _, _, _ = _sample_runner(tag, factors=[leaf], windows=[(_day(params, -1), _day(params, 100))])
    with ops.philox_seed(4242):
        runner()                                  # an epidemic state to evaluate the step on
    model, data, timer = runner.model, runner.data, runner.timer
    agent = data["agent"]
    for k in ("susceptibility", "is_infected", "infection_time"):
        agent[k] = agent[k].detach().clone()
    agent.symptoms = {k: v.detach().clone() for k, v in agent.symptoms.items()}
    # the timer stays at the window's end, the time of this state (an earlier time would precede infection times)
    agent.transmission = model.transmission_updater(data=data, timer=timer).detach()
    nets = model.infection_networks.networks
    w = torch.rand(runner.n_agents, generator=torch.Generator(DEV).manual_seed(8), device=DEV)

    def evaluate():
        leaf.grad = None
        for net in nets.values():
            net.log_beta.grad = None
        q = model.infection_networks(data=data, timer=timer, policies=model.policies, region=runner._region(timer))
        (q * w).sum().backward()
        gb = torch.stack([net.log_beta.grad if net.log_beta.grad is not None else torch.zeros((), device=DEV)
                          for net in nets.values()])
        return q.detach().clone(), gb.detach().clone(), leaf.grad.detach().clone()

    q_k, gb_k, gf_k = evaluate()
    assert bool(torch.isfinite(q_k).all()) and float(q_k.min()) < 0.999
    q_plain = model.infection_networks(data=data, timer=timer, policies=model.policies).detach()
    assert not torch.allclose(q_k, q_plain, rtol=1e-4)
    name = next(k for k, net in nets.items() if net.kind == ops.KIND_PLAIN)   # a plain venue

    class Custom(type(nets[name])):
        def _get_susceptibilities(self, data, policies, timer):
            return 1.0 * InfectionNetwork._get_susceptibilities(self, data, policies, timer)

    nets[name].__class__ = Custom
    assert model.infection_networks.has_custom()
    q_m, gb_m, gf_m = evaluate()
    assert torch.allclose(q_m, q_k, rtol=2e-6, atol=0), float(((q_m - q_k).abs() / q_k).max())
    assert bool((gf_k != 0).all())
    assert torch.allclose(gf_m, gf_k, rtol=1e-4, atol=1e-6 * float(gf_k.abs().max())), (gf_m, gf_k)
    assert torch.allclose(gb_m, gb_k, rtol=1e-4, atol=1e-6 * float(gb_k.abs().max())), (gb_m, gb_k)


# ---------------------------------------------------------------------------------------------------------------
# 2 GPUs against 1
# ---------------------------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _partition_worker(rank, world_size, port, out):
    import torch.distributed as dist
    from grad_june import GradJune, Timer
    from grad_june.default_config import default_parameters
    from grad_june.graphed import GraphedRunner
    from grad_june.partition import partition_world
    from grad_june.policies import RegionalPolicies, RegionalSocialDistancing
    from grad_june.runner import Runner
    from grad_june.world import make_synthetic_world
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
        full = Runner.get_data(params, data=world)
        R = len(torch.unique(full["agent"].area))

        def run(data):
            """The window as one CUDA graph (exchanges and the gradient all-reduce included) with the regional factors
            fitted: (region labels, cases, is_infected of this rank's agents, [log-betas..., log10 factors...] grad)."""
            model = GradJune.from_parameters(params)
            model.policies.regional_policies = RegionalPolicies([RegionalSocialDistancing(
                _day(params, 1), _day(params, 3), "area", torch.linspace(0.3, 2.5, R, device=dev), device=dev)])
            runner = Runner(model=model, data=data, timer=Timer.from_parameters(params), log_fraction_initial_cases=-1.5,
                            save_path="/tmp/gj_test_regional", parameters=params)
            loss_fn = lambda r: r["cases_per_timestep"].sum() + 2.0 * r["deaths_per_timestep"].sum()  # noqa: E731
            g = GraphedRunner(runner, loss_fn, seed=4242, fit_regional=True)
            for _ in range(2):
                _, grads, results = g()
            torch.cuda.synchronize()
            ret = (np.asarray(runner.region_labels), results["cases_per_timestep"].detach().cpu().numpy(),
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
            out["full"] = (labels1, cases1, inf1, grads1)
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_two_gpus_regional_factor_gradients_match_one():
    """A partitioned world with a regional policy, graphed with fit_regional=True: every rank holds part of each region,
    its factor gradients cover its own agents and are summed in the captured all-reduce.  The trajectory equals the
    single-GPU one exactly; the gradients (sums re-associated across ranks) to rounding — a partial or twice-counted
    factor gradient is off by a whole share, far outside it."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 CUDA devices")
    import torch.multiprocessing as mp
    out = mp.Manager().dict()
    mp.spawn(_partition_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    labels, cases, grads, K = out["part"]
    labels1, cases1, inf1, grads1 = out["full"]
    inf = np.empty_like(inf1)
    for r in range(2):
        lo, hi, x = out[f"inf{r}"]
        inf[lo:hi] = x
    assert np.array_equal(labels, labels1) and len(labels1) > 600
    assert cases1[-1] > cases1[0] > 0
    assert np.array_equal(inf, inf1), int((inf != inf1).sum())
    assert np.array_equal(cases, cases1)
    assert grads.shape == grads1.shape == (K + len(labels1),)
    for part, ref in ((grads[:K], grads1[:K]), (grads[K:], grads1[K:])):
        assert np.abs(ref).max() > 0
        assert np.allclose(part, ref, rtol=1e-4, atol=1e-6 * np.abs(ref).max()), (part, ref)
