"""Regional venue restrictions (``RegionalVenueDistancing``) on the host: the YAML and argument forms, mapping defaults,
the ``all`` fallback and every error, the half-open window and the product of overlapping policies, the majority rule
for the regions of groups (ties included), the JUNE loader's leisure labels, ``partition_world`` carrying the group
attributes (gloo, two ranks, with the label union), the sm_100a build and the unchanged register report of the
kernels that existed before the feature."""
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

from grad_june import GradJune, Timer
from grad_june.default_config import default_parameters
from grad_june.policies import RegionalVenueDistancing, VenuePolicies
from grad_june.runner import Runner
from grad_june.world import HeteroData, group_labels, make_synthetic_world

ROOT = Path(__file__).resolve().parent.parent


def _world(n=3001, per=500):
    data = make_synthetic_world(n, seed=2, device="cpu", agents_per_super_area=per)
    data["agent"].super_area = torch.arange(len(data["agent"].id)) // per
    return data


def _params(venue=None):
    params = default_parameters()
    params["system"]["device"] = "cpu"
    params["system"]["renumber_agents"] = False
    params["timer"]["total_days"] = 4
    if venue is not None:
        params["policies"] = dict(params.get("policies") or {})
        params["policies"]["regional"] = {"regional_venue_distancing": venue}
    return params


def _runner(params, data=None):
    data = Runner.get_data(params, data=data if data is not None else _world())
    return Runner(model=GradJune.from_parameters(params), data=data, timer=Timer.from_parameters(params),
                  log_fraction_initial_cases=-1.5, save_path="/tmp/gj_test_venue", parameters=params)


def _start(params, days=0):
    return (datetime.datetime.strptime(str(params["timer"]["initial_day"]), "%Y-%m-%d")
            + datetime.timedelta(days=days)).strftime("%Y-%m-%d")


def _cfg(params, factors, by="super_area", days=(0, 2)):
    return {1: {"start_date": _start(params, days[0]), "end_date": _start(params, days[1]), "by": by,
                "beta_factors": factors}}


def test_yaml_form_mapping_default_and_all_fallback():
    params = _params()
    params = _params(_cfg(params, {"pub": {1: 0.0, "3": 2.0, "default": 0.6}, "company": 0.5, "all": 0.8}))
    runner = _runner(params)
    vp = runner.model.policies.venue_policies
    assert len(list(vp.policies)) == 1 and vp.by() == "super_area"
    # the group labels: a super-area that hosts no group's majority (the last, one-agent one) is not a column
    assert runner.venue_by == "super_area" and runner.venue_labels.tolist() == list(range(6))
    pol = vp.policies[0]
    assert pol.entry("pub") == "pub" and pol.entry("school") == "all" and pol.entry("household") is None
    names = ["household", "company", "pub", "school"]
    runner.timer.reset()
    table = vp.table(runner.timer, names, runner.venue_labels, "cpu")
    assert table.shape == (4, 6) and table.dtype == torch.float32
    assert torch.equal(table[0], torch.ones(6))
    assert torch.equal(table[1], torch.full((6,), 0.5))
    assert torch.equal(table[2], torch.tensor([0.6, 0.0, 0.6, 2.0, 0.6, 0.6]))
    assert torch.equal(table[3], torch.full((6,), 0.8))


def test_tensor_entries_are_differentiable_and_batched():
    labels = np.arange(5)
    t = torch.nn.Parameter(torch.linspace(0.2, 3.0, 5))
    pol = RegionalVenueDistancing("2020-03-01", "2020-03-10", "super_area", {"gym": t}, device="cpu")
    assert any(p is t for p in pol.parameters())
    f = pol.factors("gym", labels, "cpu")
    f.sum().backward()
    assert torch.equal(t.grad, torch.ones(5))
    b = RegionalVenueDistancing("2020-03-01", "2020-03-10", "super_area", {"gym": torch.ones(3, 5), "pub": 0.5},
                                device="cpu")
    timer = type("T", (), {"date": datetime.datetime(2020, 3, 2)})()
    table = VenuePolicies([b]).table(timer, ["pub", "gym"], labels, "cpu", batch=3)
    assert tuple(table.shape) == (3, 2, 5) and torch.equal(table[:, 0], torch.full((3, 5), 0.5))


def test_errors():
    mk = lambda f, by="super_area": RegionalVenueDistancing("2020-03-01", "2020-03-10", by, f, device="cpu")  # noqa
    with pytest.raises(ValueError, match=">= 0"):
        mk({"pub": -0.1})
    with pytest.raises(ValueError, match=">= 0"):
        mk({"pub": {"a": 1.0, "default": -1.0}})
    with pytest.raises(ValueError, match=">= 0"):
        mk({"pub": torch.tensor([1.0, -2.0])})
    with pytest.raises(ValueError, match="not a number"):
        mk({"pub": "x"})
    with pytest.raises(ValueError, match="households"):
        mk({"household": 0.5})
    with pytest.raises(ValueError, match="'by'"):
        mk({"pub": 0.5}, by="")
    with pytest.raises(ValueError, match="same 'by'"):
        VenuePolicies([mk({"pub": 0.5}), mk({"pub": 0.5}, by="area")]).by()
    params = _params()
    with pytest.raises(ValueError, match="no network 'bar'"):
        _runner(_params(_cfg(params, {"bar": 0.5})))
    with pytest.raises(ValueError, match="not carried by any"):
        r = _runner(_params(_cfg(params, {"pub": {99: 0.5, "default": 1.0}})))
        r.timer.reset()
        r.model.policies.venue_policies.table(r.timer, ["pub"], r.venue_labels, "cpu")
    with pytest.raises(ValueError, match="no factor for label"):
        r = _runner(_params(_cfg(params, {"pub": {0: 0.5}})))
        r.timer.reset()
        r.model.policies.venue_policies.table(r.timer, ["pub"], r.venue_labels, "cpu")


def test_all_covering_a_range_tier_type_raises():
    """Without a household edge type the company edges (one per agent, small groups) take the RANGE tier: an 'all'
    entry covers the company network there and raises; naming only other networks is fine."""
    from grad_june.world import tier_candidates
    data = _world()
    data2 = HeteroData()
    for k, v in data["agent"].items():
        data2["agent"][k] = v
    for t in data.venue_types():
        if t == "household":
            continue
        for k, v in data[t].items():
            data2[t][k] = v
        data2["agent", "attends_" + t, t].edge_index = data["attends_" + t].edge_index
    types = data2.venue_types()
    rt, _ = tier_candidates(len(data2["agent"].id), types, {t: data2["attends_" + t].edge_index for t in types},
                            {t: len(data2[t]["id"]) for t in types})
    assert rt is not None and rt != "household"
    params = _params()
    params["networks"].pop("household")
    with pytest.raises(ValueError, match="RANGE tier"):
        _runner(_params_with(params, _cfg(params, {"all": 0.5})), data=data2)
    other = [n for n in params["networks"] if n != "household" and _net_type(n) != rt][0]
    _runner(_params_with(params, _cfg(params, {other: 0.5})), data=_copy(data2))


def _net_type(name):
    return "leisure" if name in ("pub", "gym", "grocery", "visit", "cinema", "care_visit") else name


def _copy(data):
    out = HeteroData()
    for k, v in data["agent"].items():
        out["agent"][k] = v.clone() if torch.is_tensor(v) else v
    for t in data.venue_types():
        for k, v in data[t].items():
            out[t][k] = v
        out["agent", "attends_" + t, t].edge_index = data["attends_" + t].edge_index.clone()
    return out


def _params_with(params, venue):
    params = dict(params)
    params["policies"] = dict(params.get("policies") or {})
    params["policies"]["regional"] = {"regional_venue_distancing": venue}
    return params


def test_half_open_window_and_product_of_overlapping_policies():
    a = RegionalVenueDistancing("2020-03-02", "2020-03-05", "r", {"pub": [0.5, 2.0], "all": 0.9}, device="cpu")
    b = RegionalVenueDistancing("2020-03-04", "2020-03-08", "r", {"pub": [3.0, 0.25]}, device="cpu")
    vp = VenuePolicies([a, b])
    labels = np.array([0, 1])

    def at(day):
        timer = type("T", (), {"date": datetime.datetime(2020, 3, day)})()
        return vp.table(timer, ["pub", "gym", "household"], labels, "cpu")

    assert at(1) is None
    assert torch.equal(at(2), torch.tensor([[0.5, 2.0], [0.9, 0.9], [1.0, 1.0]]))
    assert torch.equal(at(4)[0], torch.tensor([0.5 * 3.0, 2.0 * 0.25]))
    assert torch.equal(at(5), torch.tensor([[3.0, 0.25], [1.0, 1.0], [1.0, 1.0]]))
    assert at(8) is None


def test_group_labels_majority_rule_and_ties():
    data = HeteroData()
    data["agent"].id = torch.arange(9)
    data["agent"].r = np.array(["b", "a", "a", "c", "c", "b", "b", "a", "c"])
    # group 0: a a b -> a ; group 1: c b (tie) -> b ; group 2: c c a b (c) ; group 3: empty -> smallest ("a")
    src = torch.tensor([0, 1, 2, 3, 5, 4, 8, 7, 6])
    dst = torch.tensor([0, 0, 0, 1, 1, 2, 2, 2, 2])
    data["g"].id = torch.arange(4)
    data["agent", "attends_g", "g"].edge_index = torch.stack((src, dst))
    assert group_labels(data, "g", "r").tolist() == ["a", "b", "c", "a"]
    data["g"].r = np.array(["x", "y", "x", "z"])
    assert group_labels(data, "g", "r").tolist() == ["x", "y", "x", "z"]


def test_loader_stores_the_leisure_super_area():
    from grad_june.june_world_loader import world_from_june_arrays
    from test_june_loader import _fake_june_file
    f = _fake_june_file()
    data = world_from_june_arrays(f, k_leisure=3)
    sa = data["leisure"].super_area
    assert torch.equal(sa, torch.as_tensor(np.asarray(f["geography"]["super_area_id"][:]).astype(np.int64)))
    assert group_labels(data, "leisure", "super_area").tolist() == sa.tolist()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _partition_worker(rank, world_size, port, out):
    from grad_june.partition import partition_world
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world_size)
    try:
        data = make_synthetic_world(20_000, seed=3, device="cpu", agents_per_super_area=2000)
        n = len(data["agent"].id)
        data["agent"].super_area = torch.arange(n) // 2000
        whole = {t: group_labels(data, t, "super_area") for t in ("company", "leisure")}
        for t, v in whole.items():
            data[t].super_area = torch.as_tensor(v)
        data["company"].note = np.arange(len(data["company"]["id"])) * 2
        local = partition_world(data, rank, world_size)
        part = local.__dict__["_gj_partition"]
        ok = all(torch.equal(local[t].super_area, torch.as_tensor(whole[t])[part.local_groups[t]])
                 for t in ("company", "leisure"))
        ok = ok and np.array_equal(local["company"].note, part.local_groups["company"].numpy() * 2)
        params = _params()
        params = _params(_cfg(params, {"company": 0.5, "pub": 0.2}))
        local = Runner.get_data(params, data=local)
        runner = Runner(model=GradJune.from_parameters(params), data=local, timer=Timer.from_parameters(params),
                        log_fraction_initial_cases=-1.5, save_path="/tmp/gj_test_venue", parameters=params)
        mine = sorted(set(local["company"].super_area.tolist()) | set(local["leisure"].super_area.tolist()))
        codes = runner._venue_codes().codes
        off = np.cumsum([0] + [len(local[t]["id"]) for t in local.venue_types()])
        ti = local.venue_types().index("company")
        cc = codes[off[ti]:off[ti + 1]].numpy()
        ok = ok and bool(np.array_equal(runner.venue_labels[cc], local["company"].super_area.numpy()))
        del local["company"]["super_area"]
        try:
            group_labels(local, "company", "super_area")
            raised = False
        except ValueError:
            raised = True
        out[rank] = (runner.venue_labels.tolist(), mine, ok, raised)
    finally:
        dist.destroy_process_group()


def test_partition_world_carries_group_attributes_and_labels_are_the_union():
    out = mp.Manager().dict()
    mp.spawn(_partition_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    cols0, mine0, ok0, r0 = out[0]
    cols1, mine1, ok1, r1 = out[1]
    assert cols0 == cols1 == sorted(set(mine0) | set(mine1))
    assert ok0 and ok1 and r0 and r1


def test_kernels_build_for_sm_100a(tmp_path):
    """The venue-factor kernels compile for sm_100a (nvcc needs no GPU) and are in the object."""
    obj = tmp_path / "gj_kernels.o"
    cmd = ["/usr/local/cuda/bin/nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "--fmad=false", "-std=c++17",
           "-I", str(ROOT / "include"), "-I", str(ROOT / "gradabm-june_b200/csrc"), "-c", "-o", str(obj),
           str(ROOT / "gradabm-june_b200/csrc/gj_kernels.cu")]
    subprocess.run(cmd, check=True)
    syms = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-symbols", str(obj)], capture_output=True, text=True,
                          check=True).stdout
    for name in ("k_lean_group_sums_venue", "k_lean_group_fix_venue", "k_lean_scatter_finalize_venue",
                 "k_group_small_venue", "k_group_chunk_venue", "k_group_fix_venue", "k_cell_groups_venue",
                 "k_dbeta_venue", "k_seed_label_grad", "k_seed_label_fix"):
        assert name in syms, name


def test_ptxas_report_of_existing_kernels_is_unchanged_and_venue_kernels_do_not_spill():
    out = subprocess.run([sys.executable, str(ROOT / "scripts/ptxas_report.py")], capture_output=True, text=True,
                         check=True).stdout
    now = {line.split(" regs ")[0].strip(): line for line in out.splitlines() if " regs " in line}
    before = [line for line in (ROOT / "tests/golden/ptxas_parent.txt").read_text().splitlines() if line.strip()]
    for line in before:
        name = line.split(" regs ")[0].strip()
        assert now.get(name) == line, f"{name}: was\n{line}\nnow\n{now.get(name)}"
    venue = [line for name, line in now.items() if "_venue" in name]
    assert len(venue) == 11
    for line in venue:
        assert "spill st/ld    0/0" in line, line
