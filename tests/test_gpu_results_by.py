"""Results by label on the GPU: cases and deaths per label column and timestep, reduced inside the step kernels.

- the renumbered 769-agent sample world, labelled by each agent's leisure super-area group (3 columns), against the
  oracle: per-step tables equal, d loss / d log_beta and d / d log_fraction through ``assert_grad_parity`` for a loss
  that weights the new series with fixed random weights per (t, column) — throughput kernels on the kernels' Philox
  draws, and reference-order kernels on injected noise;
- a synthetic 1 M-agent world with super-area, 300-agent area (> 3 000 columns) and uniformly random (> 65 536 columns)
  labels: columns sum to the national series bit for bit, tables equal a torch index_add of the per-step state, the
  feature leaves every other output and the gradient of a loss without the new series bit-identical, runs repeat;
- every execution mode: batched b = 4, GraphedRunner replay, EnsembleEvaluator with a padded replay, the look-ahead
  step, a user-defined network subclass (modular path), and 2 GPUs against 1 (skips on one GPU)."""
import os
import socket

import numpy as np
import pytest
import torch

import helpers as H
from label_oracle import run_with_labels
from oracle import gj_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
RTOL = 1e-5
N_SYN = 1_000_000


@pytest.fixture(autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")


# ---------------------------------------------------------------------------------------------------------------
# sample world against the oracle
# ---------------------------------------------------------------------------------------------------------------
def _leisure_label(arrays):
    label = np.zeros(len(arrays["age"]), dtype=np.int64)
    label[arrays["leisure_src"]] = arrays["leisure_dst"]
    return label


def _sample_runner(tag):
    """gpu_helpers.make_runner with the leisure group attached as ``data["agent"].leisure_group`` before the world is
    renumbered (the label follows the agents)."""
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
    assert "original_index" in data["agent"]
    data["agent"].infection_parameters = {k: layout_order_of(data, v.to(DEV)).contiguous()
                                          for k, v in H.profile_params(g).items()}
    model = GradJune.from_parameters(params)
    nets = model.infection_networks.networks
    for key in nets.keys():
        nets[key].log_beta = torch.nn.Parameter(nets[key].log_beta)
    log_frac = torch.nn.Parameter(torch.tensor(float(params["infection_seed"]["log_fraction_initial_cases"])))
    runner = Runner(model=model, data=data, timer=Timer.from_parameters(params), log_fraction_initial_cases=log_frac,
                    save_path=params["save_path"], parameters=params,
                    age_bins=params.get("age_bins_to_save", (0, 18, 65, 100)), results_by="leisure_group")
    return runner, g, params, arrays


def _weights(n_rows, n_cols, seed):
    gen = torch.Generator().manual_seed(seed)
    return torch.rand(n_rows, n_cols, generator=gen), torch.rand(n_rows, n_cols, generator=gen)


def _loss(cases, deaths, cases_by, deaths_by, wc, wd):
    return cases.sum() + 0.7 * deaths.sum() + (wc * cases_by).sum() + 3.0 * (wd * deaths_by).sum()


def _oracle(tag, label, wc, wd, noises, dtype=torch.float32):
    """The oracle on the world AS LOADED with the label table; returns (result, d/dlog_beta[K], d/dlog_fraction)."""
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
    log_frac = torch.tensor(float(params["infection_seed"]["log_fraction_initial_cases"]), requires_grad=True,
                            dtype=dtype)
    prof = {k: v.to(dtype) for k, v in H.profile_params(g).items()}
    res = run_with_labels(w, prof, sym, log_frac, steps, noises, label, dtype=dtype)
    _loss(res["cases_per_timestep"], res["deaths_per_timestep"], res["cases_by_label"], res["deaths_by_label"],
          wc.to(dtype), wd.to(dtype)).backward()
    names = [str(n) for n in g["net_names"]]
    grads = np.array([nets.networks[n].log_beta.grad.item() if nets.networks[n].log_beta.grad is not None else 0.0
                      for n in names])
    return res, grads, log_frac.grad.item()


def _sensitivity(tag, label, wc, wd, noises, seeds=(1, 2, 3)):
    _, base, basef = _oracle(tag, label, wc, wd, noises)
    sens, sensf = np.zeros_like(base), 0.0
    for sd in seeds:
        with H.perturb_q(sd):
            _, gp, gpf = _oracle(tag, label, wc, wd, noises)
        sens = np.maximum(sens, np.abs(gp - base))
        sensf = max(sensf, abs(gpf - basef))
    return sens, sensf


def _sample_vs_oracle(tag, family):
    from grad_june import ops
    from gpu_helpers import noise_provider
    runner, g, params, arrays = _sample_runner(tag)
    n, n_steps = runner.n_agents, int(g["n_steps"])
    assert runner.result_labels.tolist() == [0, 1, 2]
    wc, wd = _weights(n_steps + 1, 3, 17 + H.RUNS[tag])
    if family == "throughput":
        seed = 4242 + H.RUNS[tag]
        with ops.philox_seed(seed):
            results, _ = runner()
        noises = H.philox_noises(seed, n_steps + 1, n)
    else:
        with ops.inject_noise(noise_provider(H.RUNS[tag], n_steps + 1, n)):
            results, _ = runner()
        noises = H.torch_noise(H.RUNS[tag], n_steps + 1, n)
    by_c, by_d = results["cases_by_leisure_group"], results["deaths_by_leisure_group"]
    assert tuple(by_c.shape) == (n_steps + 1, 3) == tuple(by_d.shape)
    _loss(results["cases_per_timestep"], results["deaths_per_timestep"], by_c, by_d, wc.to(DEV), wd.to(DEV)).backward()
    nets = runner.model.infection_networks.networks
    names = [str(x) for x in g["net_names"]]
    grads = np.array([nets[k].log_beta.grad.item() if nets[k].log_beta.grad is not None else 0.0 for k in names])
    gfrac = runner.log_fraction_initial_cases.grad.item()

    label = _leisure_label(arrays)
    res, og, ogf = _oracle(tag, label, wc, wd, noises)
    assert float(res["cases_by_label"][-1].detach().min()) > 0
    if tag == "sample_deadly":
        assert float(res["deaths_by_label"][-1].detach().sum()) > 0
    assert torch.equal(by_c.detach().cpu(), res["cases_by_label"]), "cases by label"
    assert torch.equal(by_d.detach().cpu(), res["deaths_by_label"]), "deaths by label"
    assert torch.equal(by_c.sum(1), results["cases_per_timestep"])
    assert torch.equal(by_d.sum(1), results["deaths_per_timestep"])
    _, g64, gf64 = _oracle(tag, label, wc, wd, noises, torch.float64)
    sens, sensf = _sensitivity(tag, label, wc, wd, noises)
    H.assert_grad_parity(grads, og, g64, sens, rtol=RTOL, what=f"{family}/{tag}: by label d/dlog_beta")
    H.assert_grad_parity(gfrac, ogf, gf64, sensf, rtol=RTOL, what=f"{family}/{tag}: by label d/dlog_fraction")


@pytest.mark.parametrize("tag", ["sample_default", "sample_policies", "sample_deadly"])
def test_sample_world_philox_label_tables_vs_oracle(tag):
    _sample_vs_oracle(tag, "throughput")


@pytest.mark.parametrize("tag", ["sample_default", "sample_policies"])
def test_sample_world_injected_noise_label_tables_vs_oracle(tag):
    _sample_vs_oracle(tag, "reference-order")


# ---------------------------------------------------------------------------------------------------------------
# synthetic world
# ---------------------------------------------------------------------------------------------------------------
_SYN = {}


def _syn_world():
    """A 1 M-agent synthetic world (renumbered) with three label attributes, built once per session."""
    if "data" not in _SYN:
        from grad_june.default_config import default_parameters
        from grad_june.runner import Runner
        from grad_june.world import make_synthetic_world
        params = default_parameters()
        params["system"]["device"] = DEV
        params["timer"]["total_days"] = 10
        params["infection_seed"]["log_fraction_initial_cases"] = -2.0
        params["policies"] = {"quarantine": {"quarantine": {1: {"start_date": "2022-02-03", "end_date": "2023-01-01",
                                                                 "stage_threshold": 4}}}}
        for k in params["networks"]:
            params["networks"][k]["log_beta"] = float(params["networks"][k]["log_beta"]) + 0.5
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
        _SYN["data"] = data
        _SYN["params"] = params
    # the runners share the world: every new one starts from the initial state, not from where the last one stopped
    agent = _SYN["data"]["agent"]
    for k, v in _SYN["start"][0].items():
        agent[k] = v.clone()
    agent.symptoms = {k: v.clone() for k, v in _SYN["start"][1].items()}
    return _SYN["data"], _SYN["params"]


def _syn_runner(results_by, batch=None):
    from grad_june import GradJune, Timer
    from grad_june.runner import Runner
    data, params = _syn_world()
    model = GradJune.from_parameters(params)
    return Runner(model=model, data=data, timer=Timer.from_parameters(params), log_fraction_initial_cases=-2.0,
                  save_path="/tmp/gj_test_results_by", parameters=params, results_by=results_by)


def _leaves(runner, batch=None, lbs=None):
    nets = runner.model.infection_networks.networks
    leaves = []
    for i, k in enumerate(nets.keys()):
        v = lbs[:, i] if batch else torch.tensor(float(runner.input_parameters["networks"][k]["log_beta"]), device=DEV)
        leaf = v.detach().clone().requires_grad_(True)
        nets[k].log_beta = leaf
        leaves.append(leaf)
    frac = torch.tensor(-2.0, device=DEV, requires_grad=True)
    runner.log_fraction_initial_cases = frac
    return leaves, frac


def _window(runner, name, seed=321, label_loss=True, wseed=3):
    """One eager window + backward: (results, is_infected, d/dlog_beta, d/dlog_fraction)."""
    from grad_june import ops
    leaves, frac = _leaves(runner)
    with ops.philox_seed(seed):
        results, is_inf = runner()
    loss = results["cases_per_timestep"].sum() + 3.0 * results["deaths_per_timestep"].sum() \
        + 0.5 * results["cases_by_age_65"].sum()
    if label_loss:
        c, d = results[f"cases_by_{name}"], results[f"deaths_by_{name}"]
        wc, wd = _weights(c.shape[0], c.shape[1], wseed)
        loss = loss + (wc.to(DEV) * c).sum() * 1e-3 + (wd.to(DEV) * d).sum() * 1e-2
    loss.backward()
    res = {k: v.detach().clone() for k, v in results.items() if k != "dates"}
    return res, is_inf.detach().clone(), torch.stack([l.grad for l in leaves]), frac.grad.clone()


@pytest.mark.parametrize("name,min_cols", [("super_area", 130), ("area", 3000), ("random_label", 65_536)])
def test_synthetic_world_invariants(name, min_cols):
    from grad_june import ops
    runner = _syn_runner(name)
    assert len(runner.result_labels) > min_cols
    assert runner.model.kernel_family(runner.data, runner.timer) == "throughput"
    res, inf, g, gf = _window(runner, name)
    c, d = res[f"cases_by_{name}"], res[f"deaths_by_{name}"]
    assert c.shape == d.shape and c.shape[1] == len(runner.result_labels)
    assert float(res["cases_per_timestep"][-1]) > float(res["cases_per_timestep"][0]) > 0
    assert bool(torch.isfinite(g).all()) and bool(torch.isfinite(gf))
    # columns sum to the national series bit for bit
    assert torch.equal(c.sum(1), res["cases_per_timestep"])
    assert torch.equal(d.sum(1), res["deaths_per_timestep"])
    assert torch.equal(res["daily_cases_per_timestep"], torch.diff(c.sum(1), prepend=torch.zeros_like(c[:1, 0])))
    # two runs: identical tables and gradients
    res2, _, g2, gf2 = _window(runner, name)
    assert torch.equal(res2[f"cases_by_{name}"], c) and torch.equal(res2[f"deaths_by_{name}"], d)
    assert torch.equal(g2, g) and torch.equal(gf2, gf)
    # the feature on leaves every other output, and a gradient that does not use the new series, bit-identical
    on, inf_on, g_on, gf_on = _window(runner, name, label_loss=False)
    off, inf_off, g_off, gf_off = _window(_syn_runner(None), name, label_loss=False)
    assert set(on) - set(off) == {f"cases_by_{name}", f"deaths_by_{name}"}
    for k, v in off.items():
        assert torch.equal(on[k], v), k
    assert torch.equal(inf_on, inf_off) and torch.equal(g_on, g_off) and torch.equal(gf_on, gf_off)
    assert not torch.equal(g, g_off)                  # the label loss does reach log_beta
    # per step: the table equals a torch index_add of the step's is_infected / current_stage
    labels = runner._labels()
    idx = labels.codes.long()
    dead = float(len(runner.model.symptoms_updater.stages_ids) - 1)
    timer, model, data = runner.timer, runner.model, runner.data
    timer.reset()
    runner._restore_for_window()
    with ops.philox_seed(99), torch.no_grad():
        _, _, tab = model.step(data, timer, age_bins=(0, 18, 65, 100), mode=ops.MODE_SEED,
                               seed_fraction=runner._fraction_tensor(), label=labels)
        for t in range(4):
            inf_t = data["agent"].is_infected
            cur = data["agent"].symptoms["current_stage"]
            ref_c = torch.zeros(labels.n, dtype=torch.float64, device=DEV).index_add(0, idx, inf_t.double())
            ref_d = torch.zeros(labels.n, dtype=torch.float64, device=DEV).index_add(0, idx, (cur == dead).double())
            assert torch.equal(tab[:, 0].double(), ref_c), t
            assert torch.equal(tab[:, 1].double(), ref_d), t
            next(timer)
            _, _, tab = model.step(data, timer, age_bins=(0, 18, 65, 100), want_probs=False, label=labels)


def test_batched_samples_equal_unbatched_slices():
    """runner.batch = 4 with shared noise: sample r of the table, and its gradients, equal the unbatched run with
    log_beta[r] to the last bit (the gradient of a loss on the label series has no d/dbeta partials of its own)."""
    from grad_june import ops
    name = "area"
    runner = _syn_runner(name)
    keys = list(runner.model.infection_networks.networks.keys())
    base = torch.tensor([float(runner.input_parameters["networks"][k]["log_beta"]) for k in keys], device=DEV)
    lbs = torch.stack([base + (r - 1.5) * 0.1 for r in range(4)])

    def run(batch, lb):
        runner.batch = batch
        nets = runner.model.infection_networks.networks
        leaves = []
        for i, k in enumerate(keys):
            leaf = (lb[:, i] if batch else lb[i]).detach().clone().requires_grad_(True)
            nets[k].log_beta = leaf
            leaves.append(leaf)
        with ops.philox_seed(55):
            results, _ = runner()
        c, d = results[f"cases_by_{name}"], results[f"deaths_by_{name}"]
        gen = torch.Generator().manual_seed(8)
        w = torch.rand(c.shape[0], c.shape[-1], generator=gen).to(DEV)
        w = w[:, None, :] if batch else w
        loss = (w * c).sum(-1).sum(0) + 2.0 * (w * d).sum(-1).sum(0)
        loss.sum().backward()
        return c.detach().clone(), d.detach().clone(), torch.stack([l.grad for l in leaves], dim=-1)

    try:
        singles = [run(None, lbs[r]) for r in range(4)]
        cb, db, gb = run(4, lbs)
    finally:
        runner.batch = None
    assert cb.dim() == 3 and cb.shape[1] == 4
    for r in range(4):
        assert torch.equal(cb[:, r], singles[r][0]) and torch.equal(db[:, r], singles[r][1]), r
        assert torch.allclose(gb[r], singles[r][2], rtol=2e-6, atol=0), (gb[r], singles[r][2])
    assert not torch.equal(cb[:, 0], cb[:, 3])


def test_graphed_runner_and_ensemble_see_the_label_series():
    from grad_june.calibration import EnsembleEvaluator
    from grad_june.graphed import GraphedRunner
    name = "super_area"
    runner = _syn_runner(name)
    keys = list(runner.model.infection_networks.networks.keys())
    base = torch.tensor([float(runner.input_parameters["networks"][k]["log_beta"]) for k in keys], device=DEV)
    lbs = torch.stack([base + (r - 2) * 0.1 for r in range(5)])

    def loss_fn(r):
        c, d = r[f"cases_by_{name}"], r[f"deaths_by_{name}"]
        return (c[-1] * torch.linspace(0.5, 1.5, c.shape[-1], device=DEV)).sum(-1) + 5.0 * d[-1].sum(-1)

    from grad_june import ops
    eager = []
    for r in range(5):
        _leaves(runner)
        nets = runner.model.infection_networks.networks
        leaf = lbs[r].clone().requires_grad_(True)
        for i, k in enumerate(keys):
            nets[k].log_beta = leaf[i]
        with ops.philox_seed(77):
            results, _ = runner()
        loss = loss_fn(results)
        loss.backward()
        eager.append((loss.detach().clone(), leaf.grad.clone(), results[f"cases_by_{name}"].detach().clone()))
    # a leaf made outside the capture stream (as _leaves does) cannot take its gradient inside a captured backward
    runner.log_fraction_initial_cases = -2.0
    g = GraphedRunner(runner, loss_fn, seed=77)
    for r in (0, 3, 1):
        loss, grads, results = g(lbs[r])
        torch.cuda.synchronize()
        assert torch.equal(results[f"cases_by_{name}"], eager[r][2]), r
        assert torch.equal(loss, eager[r][0]), r
        assert torch.allclose(grads, eager[r][1], rtol=2e-6, atol=0), (grads, eager[r][1])
    g.graph.reset()
    del g
    ens = EnsembleEvaluator(runner, loss_fn, seed=77, batch=2)         # 5 samples: the last replay is padded
    losses, grads = ens(lbs)
    runner.batch = None
    for r in range(5):
        assert torch.equal(losses[r], eager[r][0]), r
        assert torch.allclose(grads[r], eager[r][1], rtol=2e-6, atol=0), r


def test_lookahead_step_with_labels():
    """With the look-ahead transmission pass enabled, a step with a label table runs without it (the library falls
    back); the tables and every other output equal the runs without the look-ahead."""
    from grad_june import _lib
    name = "area"
    runner = _syn_runner(name)
    ref = _window(runner, name)
    prev = _lib.pipeline_enable(None)
    _lib.pipeline_enable(True, lookahead=True)
    try:
        got = _window(runner, name)
        off_la = _window(_syn_runner(None), name, label_loss=False)
    finally:
        _lib.pipeline_enable(prev[0], lookahead=prev[1], uncompacted=prev[2])
    off = _window(_syn_runner(None), name, label_loss=False)
    for k, v in ref[0].items():
        assert torch.equal(got[0][k], v), k
    assert torch.equal(got[2], ref[2]) and torch.equal(got[3], ref[3])
    for k, v in off[0].items():
        assert torch.equal(off_la[0][k], v), k


def test_user_defined_network_subclass_label_table():
    """The modular path (a user subclass of a network) builds the same table with index_add: columns sum to the
    national series and a loss on the table reaches the log-betas."""
    from grad_june import infection_networks as IN
    name = "super_area"
    runner = _syn_runner(name)
    nets = runner.model.infection_networks.networks

    class CompanyNetwork(IN.CompanyNetwork):
        def _get_transmissions(self, data, policies, timer):
            qp = policies.quarantine_policies
            return (qp.quarantine_mask if qp else 1.0) * data["agent"].transmission

    nets["company"] = CompanyNetwork(log_beta=torch.tensor(float(runner.input_parameters["networks"]["company"]["log_beta"])))
    assert runner.model.kernel_family(runner.data, runner.timer).startswith("modular")
    res, _, g, _ = _window(runner, name)
    c, d = res[f"cases_by_{name}"], res[f"deaths_by_{name}"]
    assert c.shape[1] == len(runner.result_labels)
    assert torch.equal(c.sum(1), res["cases_per_timestep"]) and torch.equal(d.sum(1), res["deaths_per_timestep"])
    assert float(res["cases_per_timestep"][-1]) > float(res["cases_per_timestep"][0])
    assert bool((g != 0).all()), g


# ---------------------------------------------------------------------------------------------------------------
# 2 GPUs against 1
# ---------------------------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _partition_worker(rank, world_size, port, peer, out):
    import torch.distributed as dist
    from grad_june import GradJune, Timer, ops
    from grad_june.default_config import default_parameters
    from grad_june.partition import partition_world
    from grad_june.runner import Runner
    from grad_june.world import make_synthetic_world
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), GJ_PEER="1" if peer else "0")
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

        def run(data):
            model = GradJune.from_parameters(params)
            keys = list(model.infection_networks.networks.keys())
            leaves = []
            for k in keys:
                leaf = torch.tensor(float(params["networks"][k]["log_beta"]) + 0.4, device=dev, requires_grad=True)
                model.infection_networks.networks[k].log_beta = leaf
                leaves.append(leaf)
            runner = Runner(model=model, data=data, timer=Timer.from_parameters(params), log_fraction_initial_cases=-1.5,
                            save_path="/tmp/gj_test", parameters=params, results_by="area")
            with ops.philox_seed(4242):
                results, _ = runner()
            c = results["cases_by_area"]
            w = torch.linspace(0.5, 1.5, c.shape[1], device=dev)
            ((c * w).sum() + 2.0 * (results["deaths_by_area"] * w).sum()).backward()
            return runner.result_labels, c.detach().cpu(), results["deaths_by_area"].detach().cpu(), \
                torch.stack([l.grad for l in leaves])

        labels, c, d, grads = run(partition_world(full, rank, world_size))
        dist.all_reduce(grads)
        if rank == 0:
            out["part"] = (labels, c, d, grads.cpu())
            out["full"] = tuple(x.cpu() if torch.is_tensor(x) else x for x in run(full))
        dist.barrier()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("peer", [True, False])
def test_two_gpus_label_tables_match_one(peer):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 CUDA devices")
    import torch.multiprocessing as mp
    out = mp.Manager().dict()
    mp.spawn(_partition_worker, args=(2, _free_port(), peer, out), nprocs=2, join=True)
    labels, c, d, grads = out["part"]
    labels1, c1, d1, grads1 = out["full"]
    assert np.array_equal(labels, labels1)
    assert torch.equal(c, c1) and torch.equal(d, d1)
    assert torch.allclose(grads, grads1, rtol=1e-4, atol=1e-6 * float(grads1.abs().max())), (grads, grads1)
