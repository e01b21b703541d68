#!/usr/bin/env python
"""Cost of the results-by-label tables (``Runner(results_by=...)``) on the flagship 56 M-agent synthetic world.

Four configurations in one process, alternated round by round so that they see the same machine state: off, super-area
labels (7 500 agents each), 300-agent area labels, and uniformly random labels over as many columns as the areas (the
worst case for the warp aggregation of the reduction).  Each timed unit is one 20-step window, forward plus backward,
with a loss on the label series (so the backward folds their cotangents in), timed with CUDA events.  Prints one JSON
line with the GPU name and power limit, the median window time of every configuration and its overhead over off.
usage: python scripts/results_by_overhead.py [--agents N] [--steps K] [--rounds R]"""
import argparse
import json
import subprocess
import sys
import tempfile
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "gradabm-june_b200"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--agents", type=int, default=56_000_000)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--area", type=int, default=300)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("results_by_overhead.py measures on a CUDA device; none is available")
    from grad_june import GradJune, Timer, ops
    from grad_june.default_config import default_parameters
    from grad_june.runner import Runner
    from grad_june.world import make_synthetic_world

    dev = "cuda:0"
    n = args.agents
    params = default_parameters()
    params["system"]["device"] = dev
    params["timer"]["total_days"] = args.steps
    params["infection_seed"]["log_fraction_initial_cases"] = -2.0
    params["save_path"] = tempfile.gettempdir() + "/gj_results_by_overhead"
    world = make_synthetic_world(n, seed=0, device=dev)
    ids = torch.arange(n, device=dev)
    world["agent"].super_area = ids // 7500
    world["agent"].area = ids // args.area
    n_area = (n + args.area - 1) // args.area
    world["agent"].random_label = torch.randint(0, n_area, (n,), device=dev, generator=torch.Generator(dev).manual_seed(1))
    del ids
    torch.manual_seed(0)
    data = Runner.get_data(params, data=world)

    configs = {"off": None, "super_area": "super_area", "area": "area", "random": "random_label"}
    runners = {}
    for key, by in configs.items():
        model = GradJune.from_parameters(params)
        runners[key] = Runner(model=model, data=data, timer=Timer.from_parameters(params), log_fraction_initial_cases=-2.0,
                              save_path=params["save_path"], parameters=params, results_by=by)

    def window(key):
        runner = runners[key]
        for k, net in runner.model.infection_networks.networks.items():
            net.log_beta = torch.tensor(float(params["networks"][k]["log_beta"]), device=dev, requires_grad=True)
        runner.log_fraction_initial_cases = torch.tensor(-2.0, device=dev, requires_grad=True)
        with ops.philox_seed(7):
            results, _ = runner()
        loss = results["cases_per_timestep"].sum() + results["deaths_per_timestep"].sum()
        if runner.results_by is not None:
            loss = loss + 1e-3 * results[f"cases_by_{runner.results_by}"].sum() \
                + 1e-2 * results[f"deaths_by_{runner.results_by}"].sum()
        loss.backward()
        return results

    for key in configs:                  # warm-up: module loads, workspaces, label codes
        window(key)
    torch.cuda.synchronize()
    times = {k: [] for k in configs}
    for _ in range(args.rounds):
        for key in configs:
            start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            start.record()
            window(key)
            end.record()
            torch.cuda.synchronize()
            times[key].append(start.elapsed_time(end))

    # per-kernel times of one window (the library's CUDA events around every kernel), for off and each label set
    from grad_june import _lib
    kernels = {}
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
    out = {"metric": "results_by_overhead", "agents": n, "steps_per_window": args.steps, "rounds": args.rounds,
           "gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi,
           "columns": {k: (len(r.result_labels) if r.result_labels is not None else 0) for k, r in runners.items()},
           "window_ms_median": {k: round(median(v), 2) for k, v in times.items()},
           "window_ms_all": {k: [round(x, 2) for x in v] for k, v in times.items()},
           "kernel_ms_per_window": kernels,
           "overhead_pct": {k: round(100.0 * (median(v) / off - 1.0), 2) for k, v in times.items() if k != "off"}}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
