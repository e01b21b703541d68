"""Seeding by label (``Runner(seed_by=...)``) on the host: parsing of the YAML form and of the ``Runner`` argument,
the per-region fraction tensors, the label order the backward's reduction walks, the union of the seed labels over
the ranks of a partitioned world (gloo), the sm_100a build, and the register / spill / shared-memory report of every
kernel that existed before the feature (it must not change)."""
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
from grad_june.runner import Runner, seed_log_fractions
from grad_june.world import make_synthetic_world

ROOT = Path(__file__).resolve().parent.parent


def _world(n=3001, per=500):
    data = make_synthetic_world(n, seed=2, device="cpu", agents_per_super_area=per)
    data["agent"].super_area = torch.arange(len(data["agent"].id)) // per
    return data


def _runner(data, seed_by, log_fraction=-1.5, results_by=None):
    params = default_parameters()
    params["system"]["device"] = "cpu"
    params["system"]["renumber_agents"] = False
    params["timer"]["total_days"] = 2
    params["infection_seed"] = {"log_fraction_initial_cases": log_fraction}
    if seed_by is not None:
        params["infection_seed"]["by"] = seed_by
    params["results_by"] = results_by
    data = Runner.get_data(params, data=data)
    return Runner(model=GradJune.from_parameters(params), data=data, timer=Timer.from_parameters(params),
                  log_fraction_initial_cases=params["infection_seed"]["log_fraction_initial_cases"],
                  save_path="/tmp/gj_test_seed_by", parameters=params, results_by=params["results_by"],
                  seed_by=params["infection_seed"].get("by"))


def test_yaml_form_is_read_by_from_parameters(tmp_path):
    params = default_parameters()
    params["system"]["device"] = "cpu"
    params["infection_seed"] = {"by": "super_area", "log_fraction_initial_cases": {1: -2.0, "3": -3.0, "default": -1.0}}
    params["save_path"] = str(tmp_path)
    data = _world()
    runner = Runner(model=GradJune.from_parameters(params), data=Runner.get_data(params, data=data),
                    timer=Timer.from_parameters(params),
                    log_fraction_initial_cases=params["infection_seed"]["log_fraction_initial_cases"],
                    save_path=tmp_path, parameters=params, seed_by=params["infection_seed"]["by"])
    assert runner.seed_by == "super_area"
    assert runner.seed_labels.tolist() == list(range(7))
    assert runner.log_fraction_initial_cases == [-1.0, -2.0, -1.0, -3.0, -1.0, -1.0, -1.0]
    frac = runner._fraction_tensor()
    expect = torch.tensor([10.0 ** v for v in runner.log_fraction_initial_cases], dtype=torch.float32)
    assert frac.dtype == torch.float32 and torch.equal(frac, expect)


def test_mapping_with_default_and_string_labels():
    labels = np.array(["east", "north", "south"])
    assert seed_log_fractions({"north": -2, "default": -4}, labels) == [-4.0, -2.0, -4.0]
    assert seed_log_fractions({"north": -2, "east": -1, "south": -3}, labels) == [-1.0, -2.0, -3.0]
    with pytest.raises(ValueError, match="not carried"):
        seed_log_fractions({"west": -2, "default": -4}, labels)
    with pytest.raises(ValueError, match="default"):
        seed_log_fractions({"north": -2}, labels)
    with pytest.raises(ValueError, match="not carried"):
        seed_log_fractions({9: -2, "default": -1}, np.arange(3))
    with pytest.raises(ValueError, match="not carried"):
        seed_log_fractions({"x": -2, "default": -1}, np.arange(3))


def test_scalar_broadcasts_to_every_region_like_the_national_seed():
    data = _world()
    national = _runner(data, None)
    by = _runner(_world(), "super_area")
    R = len(by.seed_labels)
    f = by._fraction_tensor()
    assert tuple(f.shape) == (R,) and torch.equal(f, national._fraction_tensor().expand(R))
    lf = torch.nn.Parameter(torch.tensor(-1.5))
    national.log_fraction_initial_cases = by.log_fraction_initial_cases = lf
    f = by._fraction_tensor()
    assert tuple(f.shape) == (R,) and torch.equal(f, national._fraction_tensor().expand(R))
    f.sum().backward()        # the gradient reaches the scalar through the broadcast
    assert lf.grad is not None


def test_per_region_tensor_and_shape_errors():
    by = _runner(_world(), "super_area")
    R = len(by.seed_labels)
    lf = torch.nn.Parameter(torch.linspace(-3.0, -0.5, R))
    by.log_fraction_initial_cases = lf
    assert torch.equal(by._fraction_tensor(), (10.0 ** lf).detach())
    by._parameters.pop("log_fraction_initial_cases")
    by.log_fraction_initial_cases = torch.zeros(R + 1)
    with pytest.raises(ValueError, match="one value"):
        by._fraction_tensor()
    with pytest.raises(ValueError, match="one value"):
        _runner(_world(), "super_area", log_fraction=[-1.0, -2.0])
    with pytest.raises(ValueError, match="needs infection_seed.by"):
        _runner(_world(), None, log_fraction={"default": -1.0})
    with pytest.raises(ValueError, match="not carried"):
        _runner(_world(), "super_area", log_fraction={99: -1.0, "default": -2.0})
    by.batch = 3
    by.log_fraction_initial_cases = torch.zeros(3, R)
    assert tuple(by._fraction_tensor().shape) == (3, R)
    by.log_fraction_initial_cases = torch.zeros(2, R)
    with pytest.raises(ValueError, match="one value"):
        by._fraction_tensor()


def test_seed_codes_share_the_results_by_codes():
    data = _world()
    runner = _runner(data, "super_area", results_by="super_area")
    assert runner.seed_labels is runner.result_labels
    seed = runner._seed_label_codes()
    assert seed.codes.data_ptr() == runner._labels().codes.data_ptr()
    assert runner._seed_label_codes() is seed       # cached per label array
    other = _runner(_world(), "super_area", results_by="ethnicity")
    assert other._seed_label_codes().codes.data_ptr() != other._labels().codes.data_ptr()


def test_unset_seed_by_keeps_the_national_seed():
    runner = _runner(_world(), None)
    assert runner.seed_by is None and runner.seed_labels is None and runner._seed_label_codes() is None
    assert tuple(runner._fraction_tensor().shape) == (1,)


@pytest.mark.parametrize("n_labels,n,seed", [(1, 1000, 0), (7, 5000, 1), (300, 20_000, 2), (100_000, 60_000, 3)])
def test_seed_order_and_offsets_match_a_stable_argsort(n_labels, n, seed):
    rng = np.random.default_rng(seed)
    codes = rng.integers(0, n_labels, n)
    if n_labels > 3:
        codes[codes == 2] = 3                    # an empty label in the middle
    s = ops.make_seed_labels(torch.from_numpy(codes), n_labels)
    assert s.n == n_labels and s.codes.dtype == s.order.dtype == s.offsets.dtype == torch.int32
    assert np.array_equal(s.order.numpy(), np.argsort(codes, kind="stable"))
    expect = np.concatenate([[0], np.cumsum(np.bincount(codes, minlength=n_labels))])
    assert np.array_equal(s.offsets.numpy(), expect)
    if n_labels > 3:
        assert s.offsets[2] == s.offsets[3]
    with pytest.raises(ValueError):
        ops.make_seed_labels(torch.from_numpy(codes), int(codes.max()))


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
        params = default_parameters()
        params["system"]["device"] = "cpu"
        params["timer"]["total_days"] = 2
        local = Runner.get_data(params, data=local)
        runner = Runner(model=GradJune.from_parameters(params), data=local, timer=Timer.from_parameters(params),
                        log_fraction_initial_cases={"A003": -2.0, "default": -1.5}, save_path="/tmp/gj_test_seed_by",
                        parameters=params, seed_by="area")
        codes = runner._seed_label_codes().codes.numpy()
        out[rank] = (runner.seed_labels.tolist(), np.unique(local["agent"].area).tolist(),
                     bool(np.array_equal(runner.seed_labels[codes], local["agent"].area)),
                     list(runner.log_fraction_initial_cases))
    finally:
        dist.destroy_process_group()


def test_partitioned_world_seed_labels_are_the_union_over_ranks():
    out = mp.Manager().dict()
    mp.spawn(_union_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    cols0, mine0, ok0, lf0 = out[0]
    cols1, mine1, ok1, lf1 = out[1]
    assert cols0 == cols1 == sorted(set(mine0) | set(mine1)) == [f"A{i:03d}" for i in range(29)]
    assert mine0 != cols0 and mine1 != cols1
    assert ok0 and ok1
    assert lf0 == lf1 and lf0[3] == -2.0 and lf0.count(-1.5) == 28


def test_kernels_build_for_sm_100a(tmp_path):
    """The seeding-by-label kernels compile for sm_100a (nvcc needs no GPU) and are in the object."""
    obj = tmp_path / "gj_kernels.o"
    cmd = ["/usr/local/cuda/bin/nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "--fmad=false", "-std=c++17",
           "-I", str(ROOT / "include"), "-I", str(ROOT / "gradabm-june_b200/csrc"), "-c", "-o", str(obj),
           str(ROOT / "gradabm-june_b200/csrc/gj_kernels.cu")]
    subprocess.run(cmd, check=True)
    syms = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-symbols", str(obj)], capture_output=True, text=True,
                          check=True).stdout
    for name in ("k_seed_label_grad", "k_seed_label_fix", "k_lean_seed_by", "k_agent_seed_forward",
                 "k_agent_seed_backward"):
        assert name in syms, name


def test_ptxas_report_of_existing_kernels_is_unchanged():
    """tests/golden/ptxas_parent.txt is scripts/ptxas_report.py before seeding by label: every kernel listed there
    keeps its registers, spills, stack and shared memory."""
    out = subprocess.run([sys.executable, str(ROOT / "scripts/ptxas_report.py")], capture_output=True, text=True,
                         check=True).stdout
    now = {line.split(" regs ")[0].strip(): line for line in out.splitlines() if " regs " in line}
    before = [line for line in (ROOT / "tests/golden/ptxas_parent.txt").read_text().splitlines() if line.strip()]
    assert len(before) > 50
    for line in before:
        name = line.split(" regs ")[0].strip()
        assert now.get(name) == line, f"{name}: was\n{line}\nnow\n{now.get(name)}"
