"""Results by label (``Runner(results_by=...)``) on the host: the result columns of integer, string and one-element
label attributes, their union over the ranks of a partitioned world (gloo), the range check of the codes the kernels
index with, the loader's ``super_area``, the long-format CSV, the oracle's label tables, and the sm_100a build."""
import os
import socket
import subprocess
from pathlib import Path

import numpy as np
import pandas as pd
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from grad_june import GradJune, Timer, ops
from grad_june.default_config import default_parameters
from grad_june.runner import Runner, agent_labels, label_codes
from grad_june.world import make_synthetic_world

ROOT = Path(__file__).resolve().parent.parent


def _runner(data, results_by, save_path="/tmp/gj_test_results_by"):
    params = default_parameters()
    params["system"]["device"] = "cpu"
    params["system"]["renumber_agents"] = False
    params["timer"]["total_days"] = 2
    params["results_by"] = results_by
    data = Runner.get_data(params, data=data)
    return Runner(model=GradJune.from_parameters(params), data=data, timer=Timer.from_parameters(params),
                  log_fraction_initial_cases=-1.5, save_path=save_path, parameters=params,
                  results_by=params["results_by"])


def test_integer_and_string_labels_factorise_to_sorted_columns():
    data = make_synthetic_world(3001, seed=2, device="cpu", agents_per_super_area=500)
    n = len(data["agent"].id)
    sa = torch.arange(n) // 500
    data["agent"].super_area = sa.flip(0)            # unsorted in agent order
    names = np.array(["north", "south", "east"])[np.arange(n) % 3]
    data["agent"].region = names
    runner = _runner(data, "super_area")
    assert runner.result_labels.tolist() == list(range(int(sa.max()) + 1))
    labels = runner._labels()
    assert labels.n == len(runner.result_labels) and labels.codes.dtype == torch.int32
    assert torch.equal(labels.codes.long(), sa.flip(0))
    assert runner._labels() is labels                # cached per label array
    runner = _runner(data, "region")
    assert runner.result_labels.tolist() == ["east", "north", "south"]
    codes = runner._labels().codes.numpy()
    assert np.array_equal(runner.result_labels[codes], names)


def test_one_element_label_applies_to_every_agent():
    data = make_synthetic_world(2001, seed=2, device="cpu", agents_per_super_area=500)
    assert len(data["agent"].ethnicity) == 1
    runner = _runner(data, "ethnicity")
    assert runner.result_labels.tolist() == ["A"]
    labels = runner._labels()
    assert labels.n == 1 and labels.codes.numel() == runner.n_agents and int(labels.codes.abs().sum()) == 0


def test_label_helpers_reject_bad_input():
    with pytest.raises(ValueError, match="1-D"):
        agent_labels(np.zeros((4, 2)), 4)
    with pytest.raises(ValueError, match="1 or 5"):
        agent_labels(np.arange(3), 5)
    with pytest.raises(ValueError, match="not one of"):
        label_codes(np.array([1, 7]), np.array([1, 2, 3]))
    with pytest.raises(ValueError, match="not one of"):
        label_codes(np.array(["b", "z"]), np.array(["a", "b"]))
    assert label_codes(np.array([3, 1]), np.array([1, 2, 3])).tolist() == [2, 0]


@pytest.mark.parametrize("codes,n", [([0, 1, 2], 2), ([-1, 0], 3), ([0, 1], 0), ([0, 1], (1 << 30) + 1)])
def test_out_of_range_codes_are_rejected(codes, n):
    with pytest.raises(ValueError):
        ops.make_labels(torch.tensor(codes), n)


def test_make_labels_accepts_in_range_codes():
    lab = ops.make_labels(np.array([0, 2, 1, 2], dtype=np.int64), 3)
    assert lab.n == 3 and lab.codes.dtype == torch.int32 and lab.codes.tolist() == [0, 2, 1, 2]
    with pytest.raises(ValueError, match="integer"):
        ops.make_labels(torch.tensor([0.0, 1.0]), 2)


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
                        log_fraction_initial_cases=-1.5, save_path="/tmp/gj_test_results_by", parameters=params,
                        results_by="area")
        mine = np.unique(local["agent"].area)
        codes = runner._labels().codes.numpy()
        out[rank] = (runner.result_labels.tolist(), mine.tolist(),
                     bool(np.array_equal(runner.result_labels[codes], local["agent"].area)))
    finally:
        dist.destroy_process_group()


def test_partitioned_world_columns_are_the_union_over_ranks():
    out = mp.Manager().dict()
    mp.spawn(_union_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    cols0, mine0, ok0 = out[0]
    cols1, mine1, ok1 = out[1]
    assert cols0 == cols1 == sorted(set(mine0) | set(mine1)) == [f"A{i:03d}" for i in range(29)]
    assert mine0 != cols0 and mine1 != cols1            # each rank sees only part of the labels
    assert ok0 and ok1


def test_june_loader_stores_super_area():
    from grad_june import june_world_loader as JL
    from test_june_loader import _fake_june_file
    f = _fake_june_file()
    agent = JL.world_from_june_arrays(f, k_leisure=3)["agent"]
    assert agent.super_area.dtype == torch.int64
    assert np.array_equal(agent.super_area.numpy(), f["population"]["super_area"])


def test_results_by_csv_long_format_round_trips(tmp_path):
    data = make_synthetic_world(2001, seed=2, device="cpu", agents_per_super_area=500)
    data["agent"].super_area = torch.arange(len(data["agent"].id)) // 500
    runner = _runner(data, "super_area", save_path=tmp_path)
    n_dates, n_labels = 4, len(runner.result_labels)
    dates = list(pd.date_range("2022-02-01", periods=n_dates).date)
    g = torch.Generator().manual_seed(5)
    cases = torch.randint(0, 100, (n_dates, n_labels), generator=g).float()
    deaths = torch.randint(0, 5, (n_dates, n_labels), generator=g).float()
    results = {"dates": dates, "cases_per_timestep": cases.sum(1), "deaths_per_timestep": deaths.sum(1),
               "cases_by_super_area": cases, "deaths_by_super_area": deaths}
    runner.save_results(results, torch.zeros(runner.n_agents))
    national = pd.read_csv(tmp_path / "results.csv")
    assert list(national.columns) == ["date", "cases_per_timestep", "deaths_per_timestep"]
    df = pd.read_csv(tmp_path / "results_by_super_area.csv")
    assert list(df.columns) == ["date", "label", "cases", "deaths"] and len(df) == n_dates * n_labels
    assert df["date"].tolist() == [str(d) for d in dates for _ in range(n_labels)]
    assert df["label"].tolist() == runner.result_labels.tolist() * n_dates
    assert np.array_equal(df["cases"].to_numpy().reshape(n_dates, n_labels), cases.numpy())
    assert np.array_equal(df["deaths"].to_numpy().reshape(n_dates, n_labels), deaths.numpy())
    back = df.pivot(index="date", columns="label", values="cases")
    assert np.array_equal(back.sum(axis=1).to_numpy(), national["cases_per_timestep"].to_numpy())


@pytest.mark.parametrize("tag", ["sample_default", "sample_deadly"])
def test_oracle_label_tables_sum_to_the_national_series(tag):
    import helpers as H
    from label_oracle import run_with_labels
    from oracle import gj_oracle as O
    from grad_june.policies import Policies
    from grad_june.symptoms import SymptomsSampler
    g = np.load(H.GOLDEN / f"run_{tag}.npz")
    params, _ = H.load_params(tag)
    arrays = np.load(H.GOLDEN / "sample_world.npz")
    w = H.oracle_world(arrays, H.SAMPLE_TYPES)
    nets = H.make_leaf_networks(params)
    steps = H.oracle_schedule(params, nets, Policies.from_parameters(params))
    sym = H.oracle_symptoms(SymptomsSampler.from_parameters(params))
    noises = H.torch_noise(H.RUNS[tag], len(steps) + 1, w.n_agents)
    label = np.zeros(w.n_agents, dtype=np.int64)
    label[arrays["leisure_src"]] = arrays["leisure_dst"]
    res = run_with_labels(w, H.profile_params(g), sym,
                          torch.tensor(float(params["infection_seed"]["log_fraction_initial_cases"])), steps, noises, label)
    ref = O.run(w, H.profile_params(g), sym, torch.tensor(float(params["infection_seed"]["log_fraction_initial_cases"])),
                steps, noises)
    for key in ("cases_per_timestep", "deaths_per_timestep", "cases_by_age"):
        assert torch.equal(res[key], ref[key]), key
    assert res["cases_by_label"].shape == (len(steps) + 1, 3) == res["deaths_by_label"].shape
    assert torch.equal(res["cases_by_label"].sum(1), res["cases_per_timestep"])
    assert torch.equal(res["deaths_by_label"].sum(1), res["deaths_per_timestep"])
    assert float(res["cases_by_label"][-1].detach().min()) > 0
    if tag == "sample_deadly":
        assert float(res["deaths_per_timestep"][-1]) > 0


def test_kernels_build_for_sm_100a(tmp_path):
    """The label instantiations compile for sm_100a (nvcc needs no GPU) and are in the object."""
    obj = tmp_path / "gj_kernels.o"
    cmd = ["/usr/local/cuda/bin/nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "--fmad=false", "-std=c++17",
           "-I", str(ROOT / "include"), "-I", str(ROOT / "gradabm-june_b200/csrc"), "-c", "-o", str(obj),
           str(ROOT / "gradabm-june_b200/csrc/gj_kernels.cu")]
    subprocess.run(cmd, check=True)
    syms = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-symbols", str(obj)], capture_output=True, text=True,
                          check=True).stdout
    assert "k_label_finish" in syms
    assert "sm_100a" in subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-lelf", str(obj)], capture_output=True,
                                       text=True).stdout
