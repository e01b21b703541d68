#!/usr/bin/env python
"""Cost of a regional venue factor (``RegionalVenueDistancing``) on the flagship 56 M-agent synthetic world.

Three configurations in one process, alternated round by round: off (no venue policy), group labels from the home
super-area of the groups' members (7 500 agents each; majority rule) and uniformly random group labels.  The venue
policy is active on every step and covers every non-household network (``all``), so every group pass runs its venue
instantiation and every backward step runs the per-region reduction of d/dfactor.  Each timed unit is one window
(``--days`` steps) forward plus backward, timed with CUDA events; the library's per-kernel events then locate the cost.
Prints one JSON line with the GPU name and power limit read in the same run.
usage: python scripts/venue_factor_overhead.py [--agents N] [--days D] [--rounds R]"""
import argparse
import json
import subprocess
import sys
import tempfile
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "gradabm-june_b200"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--agents", type=int, default=56_000_000)
    ap.add_argument("--days", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--random-regions", type=int, default=100_000)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("venue_factor_overhead.py measures on a CUDA device; none is available")
    from grad_june import GradJune, Timer, _lib, ops
    from grad_june.default_config import default_parameters
    from grad_june.policies import RegionalVenueDistancing, VenuePolicies
    from grad_june.runner import Runner
    from grad_june.world import group_labels, make_synthetic_world

    dev = "cuda:0"
    n = args.agents
    params = default_parameters()
    params["system"]["device"] = dev
    params["timer"]["total_days"] = args.days
    params["infection_seed"]["log_fraction_initial_cases"] = -2.0
    params["save_path"] = tempfile.gettempdir() + "/gj_venue_factor_overhead"
    world = make_synthetic_world(n, seed=0, device=dev)
    world["agent"].super_area = torch.arange(n, device=dev) // 7500
    rng = np.random.default_rng(1)
    for t in world.venue_types():
        if t == "household":
            continue
        world[t].home_region = torch.as_tensor(group_labels(world, t, "super_area"))
        world[t].random_region = torch.as_tensor(rng.integers(0, args.random_regions, len(world[t]["id"])))
    torch.manual_seed(0)
    data = Runner.get_data(params, data=world)
    start, end = str(params["timer"]["initial_day"]), "2100-01-01"

    configs = {"off": None, "super_area": "home_region", "random": "random_region"}
    runners = {}
    for key, by in configs.items():
        model = GradJune.from_parameters(params)
        nets = model.infection_networks.networks
        for k in nets.keys():
            nets[k].log_beta = torch.nn.Parameter(torch.as_tensor(nets[k].log_beta, dtype=torch.float32).to(dev))
        if by is not None:
            model.policies.venue_policies = VenuePolicies(
                [RegionalVenueDistancing(start, end, by, {"all": 0.8}, device=dev)])
        runners[key] = Runner(model=model, data=data, timer=Timer.from_parameters(params), log_fraction_initial_cases=-2.0,
                              save_path=params["save_path"], parameters=params)
        if by is not None:   # the factor tables as leaves, so the backward computes d/dfactor
            R = len(runners[key].venue_labels)
            model.policies.venue_policies.policies[0].beta_factors["all"] = torch.nn.Parameter(
                torch.full((R,), 0.8, device=dev))

    def window(key):
        with ops.philox_seed(7):
            results, _ = runners[key]()
        (results["cases_per_timestep"].sum() + results["deaths_per_timestep"].sum()).backward()

    for key in configs:                  # warm-up: module loads, workspaces, group codes and order
        window(key)
    torch.cuda.synchronize()
    times = {k: [] for k in configs}
    for _ in range(args.rounds):
        for key in configs:
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            window(key)
            t1.record()
            torch.cuda.synchronize()
            times[key].append(t0.elapsed_time(t1))

    kernels = {}     # the library's CUDA events around every kernel, per window
    for key in configs:
        torch.cuda.synchronize()
        _lib.profile_enable(True)
        window(key)
        torch.cuda.synchronize()
        kernels[key] = {k: round(v[0], 3) for k, v in _lib.profile_read().items() if v[2] > 0}
        _lib.profile_enable(False)

    def median(v):
        v = sorted(v)
        return v[len(v) // 2]

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    off = median(times["off"])
    out = {"metric": "venue_factor_overhead", "agents": n, "steps": args.days, "rounds": args.rounds,
           "gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi,
           "regions": {k: (len(r.venue_labels) if r.venue_labels is not None else 0) for k, r in runners.items()},
           "window_fwd_bwd_ms_median": {k: round(median(v), 2) for k, v in times.items()},
           "window_fwd_bwd_ms_all": {k: [round(x, 2) for x in v] for k, v in times.items()},
           "kernel_ms_per_window": kernels,
           "overhead_pct": {k: round(100.0 * (median(v) - off) / off, 2) for k, v in times.items() if k != "off"}}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
