"""Regional social distancing (``RegionalSocialDistancing``) on the host: parsing of the YAML form and of the factor
argument (scalar, mapping with a default, tensor), the errors, the half-open date window and the product of
overlapping policies, the union of the region labels over the ranks of a partitioned world (gloo), the codes shared
with ``results_by``, the sm_100a build, and the register / spill / shared-memory report of every kernel that existed
before the feature (it must not change)."""
import datetime
import os
import socket
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from grad_june import GradJune, Timer, ops
from grad_june.default_config import default_parameters
from grad_june.policies import Policies, RegionalSocialDistancing
from grad_june.runner import Runner
from grad_june.world import make_synthetic_world

ROOT = Path(__file__).resolve().parent.parent


def _world(n=3001, per=500):
    data = make_synthetic_world(n, seed=2, device="cpu", agents_per_super_area=per)
    data["agent"].super_area = torch.arange(len(data["agent"].id)) // per
    return data


def _params(regional=None, device="cpu"):
    params = default_parameters()
    params["system"]["device"] = device
    params["system"]["renumber_agents"] = False
    params["timer"]["total_days"] = 4
    if regional is not None:
        params.setdefault("policies", {})
        params["policies"] = dict(params["policies"] or {})
        params["policies"]["regional"] = {"regional_social_distancing": regional}
    return params


def _runner(params, data=None, results_by=None, seed_by=None):
    data = Runner.get_data(params, data=data if data is not None else _world())
    return Runner(model=GradJune.from_parameters(params), data=data, timer=Timer.from_parameters(params),
                  log_fraction_initial_cases=-1.5, save_path="/tmp/gj_test_regional", parameters=params,
                  results_by=results_by, seed_by=seed_by)


def _start(params, days=0):
    return (datetime.datetime.strptime(str(params["timer"]["initial_day"]), "%Y-%m-%d")
            + datetime.timedelta(days=days)).strftime("%Y-%m-%d")


def test_yaml_form_with_mapping_and_default():
    params = _params()
    cfg = {1: {"start_date": _start(params), "end_date": _start(params, 2), "by": "super_area",
               "beta_factors": {1: 0.4, "3": 2.0, "default": 0.6}}}
    params = _params(cfg)
    runner = _runner(params)
    rp = runner.model.policies.regional_policies
    assert len(list(rp.policies)) == 1 and rp.by() == "super_area"
    assert runner.region_by == "super_area" and runner.region_labels.tolist() == list(range(7))
    f = rp.policies[0].factors(runner.region_labels, "cpu")
    assert f.dtype == torch.float32
    assert torch.equal(f, torch.tensor([0.6, 0.4, 0.6, 2.0, 0.6, 0.6, 0.6], dtype=torch.float32))


def test_scalar_and_tensor_factors():
    labels = np.arange(5)
    pol = RegionalSocialDistancing("2020-03-01", "2020-03-10", "super_area", 0.5, device="cpu")
    assert torch.equal(pol.factors(labels, "cpu"), torch.full((5,), 0.5))
    t = torch.nn.Parameter(torch.linspace(0.2, 3.0, 5))
    pol = RegionalSocialDistancing("2020-03-01", "2020-03-10", "super_area", t, device="cpu")
    f = pol.factors(labels, "cpu")
    assert torch.equal(f, t.detach())
    f.sum().backward()
    assert t.grad is not None and torch.equal(t.grad, torch.ones(5))
    batched = RegionalSocialDistancing("2020-03-01", "2020-03-10", "super_area", torch.ones(3, 5), device="cpu")
    assert tuple(batched.factors(labels, "cpu", batch=3).shape) == (3, 5)
    listed = RegionalSocialDistancing("2020-03-01", "2020-03-10", "super_area", [1, 2, 3, 4, 5], device="cpu")
    assert torch.equal(listed.factors(labels, "cpu"), torch.arange(1.0, 6.0))


def test_errors():
    labels = np.arange(5)
    mk = lambda f, by="super_area": RegionalSocialDistancing("2020-03-01", "2020-03-10", by, f, device="cpu")  # noqa
    with pytest.raises(ValueError, match="not carried"):
        mk({9: 0.5, "default": 1.0}).factors(labels, "cpu")
    with pytest.raises(ValueError, match="default"):
        mk({1: 0.5}).factors(labels, "cpu")
    with pytest.raises(ValueError, match=">= 0"):
        mk(-0.1)
    with pytest.raises(ValueError, match=">= 0"):
        mk({1: 0.5, "default": -1.0})
    with pytest.raises(ValueError, match=">= 0"):
        mk(torch.tensor([1.0, -1.0, 1.0, 1.0, 1.0]))
    with pytest.raises(ValueError, match="one value"):
        mk(torch.ones(4)).factors(labels, "cpu")
    with pytest.raises(ValueError, match="one value"):
        mk(torch.ones(2, 5)).factors(labels, "cpu", batch=3)
    params = _params()
    two = {1: {"start_date": _start(params), "end_date": _start(params, 2), "by": "super_area", "beta_factors": 0.5},
           2: {"start_date": _start(params), "end_date": _start(params, 2), "by": "area", "beta_factors": 0.5}}
    with pytest.raises(ValueError, match="same 'by'"):
        Policies.from_parameters(_params(two))


def test_active_policy_without_region_raises():
    params = _params()
    cfg = {1: {"start_date": _start(params), "end_date": _start(params, 2), "by": "super_area", "beta_factors": 0.5}}
    params = _params(cfg)
    runner = _runner(params)
    runner.timer.reset()
    next(runner.timer)
    with pytest.raises(ValueError, match="regional policy is active"):
        runner.model.step(runner.data, runner.timer)


def test_half_open_window_and_product_of_overlapping_policies():
    params = _params()
    cfg = {1: {"start_date": _start(params, 1), "end_date": _start(params, 3), "by": "super_area",
               "beta_factors": {0: 0.5, "default": 2.0}},
           2: {"start_date": _start(params, 2), "end_date": _start(params, 4), "by": "super_area",
               "beta_factors": 0.25}}
    runner = _runner(_params(cfg))
    timer = runner.timer
    timer.reset()
    seen = {}
    while timer.date < timer.final_date:
        r = runner._region(timer)
        seen[(timer.date - timer.initial_date).days] = None if r is None else r.factor.clone()
        next(timer)
    f1 = torch.tensor([0.5] + [2.0] * 6)
    assert seen[0] is None                        # before the first window
    assert torch.equal(seen[1], f1)               # first policy only
    assert torch.equal(seen[2], f1 * 0.25)        # both: the elementwise product
    assert torch.equal(seen[3], torch.full((7,), 0.25))   # the first window is half-open: its end date is excluded


def test_region_codes_share_the_results_by_and_seed_by_codes():
    params = _params()
    cfg = {1: {"start_date": _start(params), "end_date": _start(params, 2), "by": "super_area", "beta_factors": 0.5}}
    runner = _runner(_params(cfg), results_by="super_area")
    assert runner.region_labels is runner.result_labels
    reg = runner._region_codes()
    assert reg.codes.data_ptr() == runner._labels().codes.data_ptr()
    assert runner._region_codes() is reg
    assert np.array_equal(reg.order.numpy(), np.argsort(reg.codes.numpy(), kind="stable"))
    seeded = _runner(_params(cfg), seed_by="super_area")
    assert seeded._region_codes() is seeded._seed_label_codes()
    other = _runner(_params(cfg), results_by="ethnicity")
    assert other._region_codes().codes.data_ptr() != other._labels().codes.data_ptr()


def test_no_regional_policy_changes_nothing():
    runner = _runner(_params())
    assert runner.region_by is None and runner.region_labels is None
    runner.timer.reset()
    assert runner._region(runner.timer) is None and runner._region_codes() is None


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _union_worker(rank, world_size, port, out):
    from grad_june.partition import partition_world
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world_size)
    try:
        data = make_synthetic_world(20_000, seed=3, device="cpu", agents_per_super_area=2000)
        n = len(data["agent"].id)
        data["agent"].area = np.array([f"A{i // 700:03d}" for i in range(n)])
        local = partition_world(data, rank, world_size)
        params = _params()
        cfg = {1: {"start_date": _start(params), "end_date": _start(params, 2), "by": "area",
                   "beta_factors": {"A003": 0.3, "default": 0.8}}}
        params = _params(cfg)
        local = Runner.get_data(params, data=local)
        runner = Runner(model=GradJune.from_parameters(params), data=local, timer=Timer.from_parameters(params),
                        log_fraction_initial_cases=-1.5, save_path="/tmp/gj_test_regional", parameters=params)
        codes = runner._region_codes().codes.numpy()
        f = runner.model.policies.regional_policies.policies[0].factors(runner.region_labels, "cpu")
        out[rank] = (runner.region_labels.tolist(), np.unique(local["agent"].area).tolist(),
                     bool(np.array_equal(runner.region_labels[codes], local["agent"].area)), f.tolist())
    finally:
        dist.destroy_process_group()


def test_partitioned_world_region_labels_are_the_union_over_ranks():
    out = mp.Manager().dict()
    mp.spawn(_union_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    cols0, mine0, ok0, f0 = out[0]
    cols1, mine1, ok1, f1 = out[1]
    assert cols0 == cols1 == sorted(set(mine0) | set(mine1)) == [f"A{i:03d}" for i in range(29)]
    assert mine0 != cols0 and mine1 != cols1
    assert ok0 and ok1
    assert f0 == f1 and abs(f0[3] - 0.3) < 1e-7 and sum(abs(v - 0.8) < 1e-7 for v in f0) == 28


def test_kernels_build_for_sm_100a(tmp_path):
    """The regional-factor kernels compile for sm_100a (nvcc needs no GPU) and are in the object."""
    obj = tmp_path / "gj_kernels.o"
    cmd = ["/usr/local/cuda/bin/nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "--fmad=false", "-std=c++17",
           "-I", str(ROOT / "include"), "-I", str(ROOT / "gradabm-june_b200/csrc"), "-c", "-o", str(obj),
           str(ROOT / "gradabm-june_b200/csrc/gj_kernels.cu")]
    subprocess.run(cmd, check=True)
    syms = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-symbols", str(obj)], capture_output=True, text=True,
                          check=True).stdout
    for name in ("k_pipe_forward_region", "k_lean_forward_region", "k_tile_forward_region", "k_pipe_backward_region",
                 "k_lean_backward_region", "k_tile_backward_region", "k_seed_label_grad", "k_seed_label_fix"):
        assert name in syms, name


def test_ptxas_report_of_existing_kernels_is_unchanged():
    """tests/golden/ptxas_parent.txt lists kernels that existed before the regional factor: every one keeps its
    registers, spills, stack and shared memory."""
    out = subprocess.run([sys.executable, str(ROOT / "scripts/ptxas_report.py")], capture_output=True, text=True,
                         check=True).stdout
    now = {line.split(" regs ")[0].strip(): line for line in out.splitlines() if " regs " in line}
    before = [line for line in (ROOT / "tests/golden/ptxas_parent.txt").read_text().splitlines() if line.strip()]
    assert len(before) > 50
    for line in before:
        name = line.split(" regs ")[0].strip()
        assert now.get(name) == line, f"{name}: was\n{line}\nnow\n{now.get(name)}"
    assert any(name.startswith("k_pipe_forward_region") for name in now)
