#!/usr/bin/env python
"""Cost of seeding by label (``Runner(seed_by=...)``) on the flagship 56 M-agent synthetic world.

The seeding step runs once per window: its forward (``k_lean_seed`` / ``k_lean_seed_by``) and its backward (the
per-agent pass, plus ``k_seed_label_grad`` / ``k_seed_label_fix`` with labels).  Four configurations in one process,
alternated round by round: off (one national fraction), super-area labels (7 500 agents each), 300-agent areas, and
uniformly random labels over as many regions as the areas.  Each timed unit is the seeding forward plus backward with a
loss on the seeded state, timed with CUDA events; the library's per-kernel events then separate the seeding kernel,
the per-agent backward and the per-label reduction.  Prints one JSON line with the GPU name and power limit.
usage: python scripts/seed_by_overhead.py [--agents N] [--rounds R]"""
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
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--area", type=int, default=300)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("seed_by_overhead.py measures on a CUDA device; none is available")
    from grad_june import GradJune, Timer, _lib, ops
    from grad_june.default_config import default_parameters
    from grad_june.runner import Runner
    from grad_june.world import make_synthetic_world

    dev = "cuda:0"
    n = args.agents
    params = default_parameters()
    params["system"]["device"] = dev
    params["timer"]["total_days"] = 2
    params["infection_seed"]["log_fraction_initial_cases"] = -2.0
    params["save_path"] = tempfile.gettempdir() + "/gj_seed_by_overhead"
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
                              save_path=params["save_path"], parameters=params, seed_by=by)

    def seeding(key):
        runner = runners[key]
        runner.timer.reset()
        runner._restore_for_window()
        R = len(runner.seed_labels) if runner.seed_by is not None else 1
        lf = torch.full((R,) if runner.seed_by is not None else (), -2.0, device=dev, requires_grad=True)
        runner.log_fraction_initial_cases = lf
        with ops.philox_seed(7):
            red = runner.set_initial_cases()
        agent = runner.data["agent"]
        (red.sum() + agent.is_infected.sum() + 1e-3 * agent.symptoms["current_stage"].sum()).backward()
        return lf.grad

    for key in configs:                  # warm-up: module loads, workspaces, label codes and order
        seeding(key)
    torch.cuda.synchronize()
    times = {k: [] for k in configs}
    for _ in range(args.rounds):
        for key in configs:
            start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            start.record()
            seeding(key)
            end.record()
            torch.cuda.synchronize()
            times[key].append(start.elapsed_time(end))

    # per-kernel times (the library's CUDA events around every kernel), averaged over the rounds
    kernels = {}
    for key in configs:
        torch.cuda.synchronize()
        _lib.profile_enable(True)
        for _ in range(args.rounds):
            seeding(key)
        torch.cuda.synchronize()
        kernels[key] = {k: round(v[0] / args.rounds, 4) for k, v in _lib.profile_read().items() if v[2] > 0}
        _lib.profile_enable(False)

    def median(v):
        v = sorted(v)
        return v[len(v) // 2]

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    off = median(times["off"])
    out = {"metric": "seed_by_overhead", "agents": n, "rounds": args.rounds,
           "gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi,
           "regions": {k: (len(r.seed_labels) if r.seed_labels is not None else 1) for k, r in runners.items()},
           "seeding_fwd_bwd_ms_median": {k: round(median(v), 3) for k, v in times.items()},
           "seeding_fwd_bwd_ms_all": {k: [round(x, 3) for x in v] for k, v in times.items()},
           "kernel_ms_per_seeding": kernels,
           "overhead_ms": {k: round(median(v) - off, 3) for k, v in times.items() if k != "off"}}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
