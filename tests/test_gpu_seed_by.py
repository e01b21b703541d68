"""Seeding by label on the GPU: one initial-case fraction per region, differentiable per region.

1. identity: every region at the national value reproduces the national seed bit for bit (throughput, reference-order
   and batched kernels), and the per-region gradients sum to the national d/dlog_fraction;
2. the renumbered sample world, seeded by each agent's leisure group (3 regions, fractions from 1e-3 to 0.3), against
   the oracle with a per-agent log-fraction: exact masks, stages and series, d/dlog_fraction per region and
   d/dlog_beta through ``assert_grad_parity`` (throughput kernels on their Philox draws, reference-order kernels on
   injected noise);
3. a 1 M-agent synthetic world with super-area, 300-agent area and uniformly random (100 000-region) labels: the
   per-region gradient equals an fp64 index_add of the per-agent terms, and repeats bit for bit;
4. batched b = 4 with a different row of fractions per sample against the unbatched runs;
5. GraphedRunner(fit_seed=True) against the eager window, and Calibrator(fit_seed=True);
6. 2 GPUs against 1 (skips on one GPU);
7. a region seeded at log-fraction -30: no agent of it is infected, and the other regions are unaffected."""
import os
import socket

import numpy as np
import pytest
import torch

import helpers as H
from seed_oracle import seed_log_fraction
from oracle import gj_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
RTOL = 1e-5
N_SYN = 1_000_000
LF3 = [-3.0, float(np.log10(0.03)), float(np.log10(0.3))]     # fractions 1e-3, 0.03, 0.3


@pytest.fixture(autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")


# ---------------------------------------------------------------------------------------------------------------
# sample world
# ---------------------------------------------------------------------------------------------------------------
def _leisure_label(arrays):
    label = np.zeros(len(arrays["age"]), dtype=np.int64)
    label[arrays["leisure_src"]] = arrays["leisure_dst"]
    return label


def _sample_runner(tag, seed_by="leisure_group", log_fraction=None):
    """The renumbered sample world with ``data["agent"].leisure_group`` attached before renumbering; log-betas are
    leaves.  Returns (runner, golden arrays, params, world arrays)."""
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
    nets = model.infection_networks.networks
    for key in nets.keys():
        nets[key].log_beta = torch.nn.Parameter(nets[key].log_beta)
    if log_fraction is None:
        log_fraction = float(params["infection_seed"]["log_fraction_initial_cases"])
    runner = Runner(model=model, data=data, timer=Timer.from_parameters(params), log_fraction_initial_cases=log_fraction,
                    save_path=params["save_path"], parameters=params,
                    age_bins=params.get("age_bins_to_save", (0, 18, 65, 100)), seed_by=seed_by)
    return runner, g, params, arrays


def _loss(results):
    return results["cases_per_timestep"].sum() + 0.7 * results["deaths_per_timestep"].sum() \
        + 0.3 * results["cases_by_age_65"].sum()


def _run(runner, family, tag, n_steps, lf):
    """One eager window and backward with log-fraction leaf ``lf``: (results, is_infected, d/dlog_beta, d/dlf)."""
    from grad_june import ops
    from gpu_helpers import noise_provider
    runner.log_fraction_initial_cases = lf
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
    return res, is_inf.detach().clone(), grads, lf.grad.detach().clone()


@pytest.mark.parametrize("family", ["throughput", "reference-order"])
def test_identity_with_the_national_seed(family):
    tag = "sample_default"
    national, g, params, _ = _sample_runner(tag, seed_by=None)
    by, _, _, _ = _sample_runner(tag)
    n_steps = int(g["n_steps"])
    lf0 = float(params["infection_seed"]["log_fraction_initial_cases"])
    a = _run(national, family, tag, n_steps, torch.tensor(lf0, device=DEV, requires_grad=True))
    b = _run(by, family, tag, n_steps, torch.full((3,), lf0, device=DEV, requires_grad=True))
    for k, v in a[0].items():
        assert torch.equal(b[0][k], v), k
    assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])
    for k in ("susceptibility", "is_infected", "infection_time"):
        assert torch.equal(national.data["agent"][k], by.data["agent"][k]), k
    for k, v in national.data["agent"].symptoms.items():
        assert torch.equal(v, by.data["agent"].symptoms[k]), k
    assert b[3].shape == (3,)
    total, ref = float(b[3].double().sum()), float(a[3])
    assert abs(total - ref) <= 1e-6 * abs(ref), (b[3], ref)


def _oracle(tag, label, lf, noises, dtype=torch.float32):
    """The oracle on the world as loaded with per-agent log-fractions lf[label]: (result, d/dlog_beta, d/dlf[R])."""
    from grad_june.policies import Policies
    from grad_june.symptoms import SymptomsSampler
    g = np.load(H.GOLDEN / f"run_{tag}.npz")
    params, _ = H.load_params(tag)
    w = H.oracle_world(np.load(H.GOLDEN / "sample_world.npz"), H.SAMPLE_TYPES)
    nets = H.make_leaf_networks(params)
    steps = H.oracle_schedule(params, nets, Policies.from_parameters(params))
    if dtype != torch.float32:
        for s in steps:
            for n in s.nets:
                n.beta = n.beta.to(dtype)
    sym = H.oracle_symptoms(SymptomsSampler.from_parameters(params))
    noises = [O.StepNoise(E=n.E.to(dtype), u=n.u.to(dtype), z=n.z.to(dtype)) for n in noises]
    leaf = torch.tensor(lf, dtype=dtype, requires_grad=True)
    prof = {k: v.to(dtype) for k, v in H.profile_params(g).items()}
    res = O.run(w, prof, sym, seed_log_fraction(leaf, label), steps, noises, dtype=dtype)
    (res["cases_per_timestep"].sum() + 0.7 * res["deaths_per_timestep"].sum()
     + 0.3 * res["cases_by_age"][:, 1].sum()).backward()
    names = [str(n) for n in g["net_names"]]
    grads = np.array([nets.networks[n].log_beta.grad.item() if nets.networks[n].log_beta.grad is not None else 0.0
                      for n in names])
    return res, grads, leaf.grad.numpy().copy()


@pytest.mark.parametrize("family,tag", [("throughput", "sample_default"), ("throughput", "sample_deadly"),
                                        ("reference-order", "sample_default"), ("reference-order", "sample_policies")])
def test_sample_world_per_region_seed_vs_oracle(family, tag):
    runner, g, params, arrays = _sample_runner(tag)
    assert runner.seed_labels.tolist() == [0, 1, 2]
    assert tuple(runner.age_bins.tolist())[1:3] == (18, 65)
    n, n_steps = runner.n_agents, int(g["n_steps"])
    lf = torch.tensor(LF3, device=DEV, requires_grad=True)
    res, is_inf, grads, gfrac = _run(runner, family, tag, n_steps, lf)
    if family == "throughput":
        noises = H.philox_noises(4242 + H.RUNS[tag], n_steps + 1, n)
    else:
        noises = H.torch_noise(H.RUNS[tag], n_steps + 1, n)
    label = _leisure_label(arrays)
    ref, og, ogf = _oracle(tag, label, LF3, noises)
    assert torch.equal(is_inf.cpu(), ref["state"]["is_infected"]), "infection masks"
    assert torch.equal(res["cases_per_timestep"].cpu(), ref["cases_per_timestep"])
    assert torch.equal(res["deaths_per_timestep"].cpu(), ref["deaths_per_timestep"])
    assert torch.equal(res["cases_by_age_65"].cpu(), ref["cases_by_age"][:, 1])
    from grad_june.world import original_order
    stages = original_order(runner.data, runner.data["agent"].symptoms["current_stage"]).cpu()
    assert torch.equal(stages.to(ref["state"]["current_stage"].dtype), ref["state"]["current_stage"]), "stages"
    # the three regions started differently: more seeds where the fraction is larger
    seeds0 = [int(((torch.as_tensor(label) == r) & (ref["state"]["infection_time"] == 0)
                   & (ref["state"]["is_infected"] > 0)).sum()) for r in range(3)]
    assert seeds0[2] > seeds0[0], seeds0
    _, g64, gf64 = _oracle(tag, label, LF3, noises, torch.float64)
    sens, sensf = np.zeros_like(og), np.zeros_like(ogf)
    for sd in (1, 2, 3):
        with H.perturb_q(sd):
            _, gp, gpf = _oracle(tag, label, LF3, noises)
        sens, sensf = np.maximum(sens, np.abs(gp - og)), np.maximum(sensf, np.abs(gpf - ogf))
    names = [str(x) for x in g["net_names"]]
    keys = list(runner.model.infection_networks.networks.keys())
    mine = np.array([float(grads[keys.index(k)]) for k in names])
    H.assert_grad_parity(mine, og, g64, sens, rtol=RTOL, what=f"{family}/{tag}: seed by label d/dlog_beta")
    for r in range(3):
        H.assert_grad_parity(float(gfrac[r]), float(ogf[r]), float(gf64[r]), float(sensf[r]), rtol=RTOL,
                             what=f"{family}/{tag}: d/dlog_fraction[{r}]")


def test_batched_rows_equal_unbatched_runs():
    from grad_june import ops
    tag = "sample_default"
    rows = torch.tensor([LF3, [-1.0, -1.0, -1.0], [-1.0, -2.5, -0.7], [-0.52, -3.0, -1.52]], device=DEV)
    singles = []
    for r in range(4):
        runner, g, _, _ = _sample_runner(tag)
        singles.append(_run(runner, "throughput", tag, int(g["n_steps"]), rows[r].clone().requires_grad_(True)))
    # row 1 holds the national value (-1) in every region: the same window as the national seed
    national, _, _, _ = _sample_runner(tag, seed_by=None)
    nat = _run(national, "throughput", tag, int(g["n_steps"]), torch.tensor(-1.0, device=DEV, requires_grad=True))
    for k, v in nat[0].items():
        assert torch.equal(singles[1][0][k], v), k
    assert torch.equal(nat[1], singles[1][1]) and torch.equal(nat[2], singles[1][2])
    runner, g, _, _ = _sample_runner(tag)
    runner.batch = 4
    nets = runner.model.infection_networks.networks
    for k in nets.keys():
        value = nets[k].log_beta.detach().reshape(()).to(DEV)
        nets[k]._parameters.pop("log_beta", None)
        nets[k].log_beta = value.repeat(4).requires_grad_(True)
    lf = rows.clone().requires_grad_(True)
    runner._parameters.pop("log_fraction_initial_cases", None)
    runner.log_fraction_initial_cases = lf
    with ops.philox_seed(4242 + H.RUNS[tag]):
        results, is_inf = runner()
    _loss(results).sum().backward()
    for r in range(4):
        for k, v in singles[r][0].items():
            assert torch.equal(results[k][:, r] if results[k].dim() > 1 else results[k], v), (r, k)
        assert torch.equal(is_inf[r].to(singles[r][1].device), singles[r][1]), r
        assert torch.equal(lf.grad[r], singles[r][3]), (r, lf.grad[r], singles[r][3])
        assert torch.equal(torch.stack([nets[k].log_beta.grad[r] for k in nets.keys()]).cpu(), singles[r][2].cpu()), r


def test_graphed_replay_and_calibrator_fit_the_seed():
    from grad_june.calibration import Calibrator
    from grad_june.graphed import GraphedRunner
    tag = "sample_default"
    runner, g, _, _ = _sample_runner(tag, log_fraction=list(LF3))
    nets = runner.model.infection_networks.networks
    K = len(nets)
    graphed = GraphedRunner(runner, loss_fn=_loss, seed=77, fit_seed=True)
    assert graphed.seed_names == ["0", "1", "2"] and tuple(graphed.log_beta.shape) == (K + 3,)
    x = graphed.log_beta.detach().clone()
    x[K:] = torch.tensor([-2.0, -1.0, -2.5], device=DEV)
    loss, grads, _ = graphed(x)
    loss, grads = loss.clone(), grads.clone()
    # eager window at the same parameters and Philox key
    from grad_june import ops
    runner2, _, _, _ = _sample_runner(tag)
    nets2 = runner2.model.infection_networks.networks
    leaves = []
    for i, k in enumerate(nets2.keys()):
        nets2[k]._parameters.pop("log_beta", None)
        nets2[k].log_beta = x[i].clone().requires_grad_(True)
        leaves.append(nets2[k].log_beta)
    lf = x[K:].clone().requires_grad_(True)
    runner2.log_fraction_initial_cases = lf
    with ops.philox_seed(77):
        results, _ = runner2()
    eager = _loss(results)
    eager.backward()
    assert torch.equal(loss, eager.detach())
    assert torch.equal(grads[K:], lf.grad), (grads[K:], lf.grad)
    assert torch.equal(grads[:K], torch.stack([l.grad for l in leaves]))

    # a fixed-seed loss on the sample world: fit the regional seeds to a target series
    runner3, _, _, _ = _sample_runner(tag, log_fraction=-2.0)
    target = results["cases_per_timestep"].detach()
    cal = Calibrator(runner3, loss_fn=lambda r: ((r["cases_per_timestep"] - target) ** 2).mean(), lr=0.1, seed=77,
                     fit_seed=True)
    hist = cal.fit(20)
    for col in ("log_fraction_0", "log_fraction_2", "grad_log_fraction_1"):
        assert col in hist.columns, col
    assert hist["loss"].iloc[-1] < hist["loss"].iloc[0], hist["loss"].tolist()
    # a national seed fits one value
    runner4, _, _, _ = _sample_runner(tag, seed_by=None)
    g4 = GraphedRunner(runner4, loss_fn=_loss, seed=77, fit_seed=True)
    assert g4.seed_names == ["national"] and tuple(g4.log_beta.shape) == (K + 1,)
    _, gr, _ = g4()
    assert bool(torch.isfinite(gr).all()) and float(gr[K]) != 0.0


def test_unfitted_seed_keeps_graphed_shapes():
    from grad_june.graphed import GraphedRunner
    runner, _, _, _ = _sample_runner("sample_default", log_fraction=list(LF3))
    graphed = GraphedRunner(runner, loss_fn=_loss, seed=77)
    assert tuple(graphed.log_beta.shape) == (len(runner.model.infection_networks.networks),)
    _, grads, _ = graphed()
    assert grads.shape == graphed.log_beta.shape


def test_barely_seeded_region_is_never_infected():
    """log-fraction -30 rounds q to exactly 1 in fp32: no agent of that region is seeded; its gradient is NaN (0/0
    in the sampler's d/dq, as in the reference's torch code) and the other regions' gradients are unchanged."""
    tag = "sample_default"
    runner, g, _, arrays = _sample_runner(tag)
    n_steps = int(g["n_steps"])
    lf = torch.tensor([-30.0, LF3[1], LF3[2]], device=DEV, requires_grad=True)
    from grad_june import ops
    from grad_june.world import original_order
    label = torch.from_numpy(_leisure_label(arrays))
    res, _, _, gf = _run(runner, "throughput", tag, n_steps, lf)
    runner2, _, _, _ = _sample_runner(tag)
    with ops.philox_seed(4242):
        runner2.log_fraction_initial_cases = lf
        runner2.set_initial_cases()
    inf0 = original_order(runner2.data, runner2.data["agent"].is_infected).cpu()
    assert float(inf0[label == 0].sum()) == 0.0 and float(inf0[label != 0].sum()) > 0
    assert bool(torch.isnan(gf[0])) and bool(torch.isfinite(gf[1:]).all())
    runner3, _, _, _ = _sample_runner(tag)
    ref = _run(runner3, "throughput", tag, n_steps, torch.tensor([-20.0, LF3[1], LF3[2]], device=DEV,
                                                                  requires_grad=True))
    assert torch.equal(ref[3][1:], gf[1:]), (ref[3], gf)
    for k, v in ref[0].items():
        assert torch.equal(res[k], v), k


# ---------------------------------------------------------------------------------------------------------------
# synthetic 1 M-agent world
# ---------------------------------------------------------------------------------------------------------------
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


def _syn_window(seed_by, lf):
    from grad_june import GradJune, Timer, ops
    from grad_june.runner import Runner
    data, params = _syn_world()
    model = GradJune.from_parameters(params)
    runner = Runner(model=model, data=data, timer=Timer.from_parameters(params), log_fraction_initial_cases=-2.0,
                    save_path="/tmp/gj_test_seed_by", parameters=params, seed_by=seed_by)
    lf = lf(runner).detach().clone().requires_grad_(True)
    runner.log_fraction_initial_cases = lf
    with ops.philox_seed(321):
        results, is_inf = runner()
    (results["cases_per_timestep"].sum() + 3.0 * results["deaths_per_timestep"].sum()).backward()
    work = None
    if seed_by is not None:
        static, _ = model._static(data, torch.device(DEV))
        work = static.world.__dict__["_buffers"]["seed_work"][: runner.n_agents].clone()
    return runner, {k: v.detach().clone() for k, v in results.items() if k != "dates"}, is_inf.clone(), \
        lf.grad.clone(), work


@pytest.mark.parametrize("name,min_cols", [("super_area", 130), ("area", 3000), ("random_label", 65_536)])
def test_synthetic_world_per_region_gradient(name, min_cols):
    gen = torch.Generator().manual_seed(11)

    def spread(runner):
        R = len(runner.seed_labels)
        return (-3.0 + 2.5 * torch.rand(R, generator=gen)).to(DEV)

    runner, res, inf, gf, work = _syn_window(name, spread)
    R = len(runner.seed_labels)
    assert R > min_cols and gf.shape == (R,)
    assert runner.model.kernel_family(runner.data, runner.timer) == "throughput"
    assert bool(torch.isfinite(gf).all()) and float(res["cases_per_timestep"][0]) > 0
    codes = runner._seed_label_codes().codes.long()
    # d loss / d log_fraction[r] = fraction[r] * ln 10 * sum over region r of d loss / d fraction
    # d/dlog_fraction[r] = ln 10 * fraction[r] * (sum over region r of the per-agent d/dfraction), to fp32 rounding
    frac = 10.0 ** runner.log_fraction_initial_cases.detach().double()
    g_frac = torch.zeros(R, dtype=torch.float64, device=DEV).index_add(0, codes, work.double())
    expect = g_frac * frac * np.log(10.0)
    err = (gf.double() - expect).abs()
    assert bool((err <= 1e-6 * expect.abs() + 1e-30).all()), float((err / expect.abs().clamp_min(1e-30)).max())
    assert float((g_frac != 0).double().mean()) > 0.9
    gen.manual_seed(11)
    _, res2, inf2, gf2, _ = _syn_window(name, spread)
    assert torch.equal(gf, gf2) and torch.equal(inf, inf2)
    for k, v in res.items():
        assert torch.equal(res2[k], v), k


def test_synthetic_world_identity_one_region_per_super_area():
    """Throughput kernels at 1 M agents: every region at the national value equals the national seed bit for bit, and
    a single region covering every agent (a one-element label) sums its gradient over the whole world."""
    _, res0, inf0, gf0, _ = _syn_window(None, lambda r: torch.tensor(-2.0, device=DEV))
    runner, res1, inf1, gf1, _ = _syn_window("super_area", lambda r: torch.full((len(r.seed_labels),), -2.0,
                                                                                device=DEV))
    for k, v in res0.items():
        assert torch.equal(res1[k], v), k
    assert torch.equal(inf0, inf1)
    assert abs(float(gf1.double().sum()) - float(gf0)) <= 1e-6 * abs(float(gf0))
    data, _ = _syn_world()
    data["agent"].one_region = np.array(["all"])
    runner, res2, inf2, gf2, _ = _syn_window("one_region", lambda r: torch.tensor([-2.0], device=DEV))
    assert runner.seed_labels.tolist() == ["all"] and gf2.shape == (1,)
    assert torch.equal(inf0, inf2)
    assert abs(float(gf2[0]) - float(gf0)) <= 1e-6 * abs(float(gf0))


# ---------------------------------------------------------------------------------------------------------------
# 2 GPUs against 1
# ---------------------------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _partition_worker(rank, world_size, port, out):
    import torch.distributed as dist
    from grad_june import GradJune, Timer, ops
    from grad_june.default_config import default_parameters
    from grad_june.partition import partition_world
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
        torch.manual_seed(5)
        world = make_synthetic_world(200_000, seed=5, device=dev, agents_per_super_area=5000)
        world["agent"].area = torch.arange(200_000, device=dev) // 300
        full = Runner.get_data(params, data=world)

        def run(data):
            model = GradJune.from_parameters(params)
            runner = Runner(model=model, data=data, timer=Timer.from_parameters(params), log_fraction_initial_cases=-1.5,
                            save_path="/tmp/gj_test", parameters=params, seed_by="area")
            R = len(runner.seed_labels)
            lf = torch.linspace(-3.0, -1.0, R, device=dev).requires_grad_(True)
            runner.log_fraction_initial_cases = lf
            with ops.philox_seed(4242):
                results, is_inf = runner()
            (results["cases_per_timestep"].sum() + 2.0 * results["deaths_per_timestep"].sum()).backward()
            return runner.seed_labels, results["cases_per_timestep"].detach().cpu(), is_inf.detach().cpu(), lf.grad

        labels, cases, _, grads = run(partition_world(full, rank, world_size))
        dist.all_reduce(grads)
        if rank == 0:
            out["part"] = (labels, cases, grads.cpu())
            labels1, cases1, _, grads1 = run(full)
            out["full"] = (labels1, cases1, grads1.cpu())
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_two_gpus_seed_gradients_match_one():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 CUDA devices")
    import torch.multiprocessing as mp
    out = mp.Manager().dict()
    mp.spawn(_partition_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    labels, cases, grads = out["part"]
    labels1, cases1, grads1 = out["full"]
    assert np.array_equal(labels, labels1)
    assert torch.equal(cases, cases1)
    assert torch.allclose(grads, grads1, rtol=1e-5, atol=1e-6 * float(grads1.abs().max())), (grads, grads1)
