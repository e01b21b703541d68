#!/usr/bin/env python
"""Benchmark of the per-timestep infection path (fwd+bwd), BASELINE.json metric
"agent-timesteps/sec fwd+bwd ...; HBM GB/s vs roofline".

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W     # the reference's CPU path (oracle port)
    python bench.py --steps K --dump-outputs DIR              # + the last timed window's outputs as DIR/*.npy

One "step" = one simulation timestep forward AND its backward, over every agent of the synthetic
England-scale world (config.workload).  K steps are run as BPTT windows (forward w steps, backward
through them) exactly as Runner.forward() + loss.backward() does; prints ONE JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
for p in (ROOT / "gradabm-june_b200", ROOT, ROOT / "tests", ROOT / "tests" / "golden"):
    if str(p) not in sys.path:
        sys.path.insert(0, str(p))

import numpy as np
import torch

METRIC = "agent_timesteps_per_sec_fwd_bwd"
UNIT = "agent-timesteps/s"
# algorithmic HBM bytes per agent-timestep, fwd+bwd, symptoms on (SURVEY.md §8d; DESIGN.md "Roofline")
B_ALG_STEP = 279.0


def measured_peak_gbs():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        try:
            return float(json.load(open(f))["hbm_gbs"]), "measured"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback"


def bench_params(device, steps, policies=False):
    from grad_june.default_config import default_parameters
    p = default_parameters()
    p["system"]["device"] = device
    p["policies"] = {}
    if policies:   # BASELINE config 4 (SURVEY.md 8d): everything active from day 15 of the run (start 2022-02-01)
        span = {"start_date": "2022-02-16", "end_date": "2030-01-01"}
        leisure = ("pub", "cinema", "gym", "grocery", "visit", "care_visit")
        p["policies"] = {
            "interaction": {"social_distancing": {1: dict(span, beta_factors=dict(
                {"school": 0.5, "company": 0.5}, **{k: 0.5 for k in leisure}))}},
            "close_venue": {"close_venue": {1: dict(span, names=["school", "pub", "cinema", "gym"])}},
            "quarantine": {"quarantine": {1: dict(span, stage_threshold=4)}},
        }
    p["timer"]["total_days"] = steps
    p["infection_seed"]["log_fraction_initial_cases"] = -2.0
    p["save_path"] = tempfile.gettempdir() + "/gj_bench"
    return p


# ------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock and throttle reasons through NVML from a background thread while the timed region
    runs (polling `nvidia-smi -lms` from a subprocess was measured to slow the timed kernels by 2-3x)."""

    def __init__(self, index, period=0.05):
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz, self.error = [], set(), None, None
        self._stop = None
        self._thread = None

    def __enter__(self):
        import threading
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # noqa: BLE001
            self.error = repr(e)[:200]
            return self
        names = {"hw_slowdown": getattr(pynvml, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(pynvml, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(pynvml, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(pynvml, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        self._stop = threading.Event()

        def loop():
            get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                getattr(pynvml, "nvmlDeviceGetCurrentClocksThrottleReasons")
            while not self._stop.is_set():
                try:
                    self.samples.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                    mask = int(get_reasons(h))
                    for k, bit in names.items():
                        if mask & bit:
                            self.reasons.add(k)
                except Exception as e:  # noqa: BLE001
                    self.error = repr(e)[:200]
                    return
                self._stop.wait(self.period)

        self._thread = threading.Thread(target=loop, daemon=True)
        self._thread.start()
        return self

    def __exit__(self, *a):
        if self._stop is not None:
            self._stop.set()
            self._thread.join(timeout=2)

    def summary(self):
        out = {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}
        if self.samples:
            out.update(sm_mhz=float(np.median(self.samples)), samples=len(self.samples))
        if self.error:
            out["error"] = self.error
        return out


# ------------------------------------------------------------------------------------------
# CPU baseline = the oracle port of the reference's path, on the host cores
# ------------------------------------------------------------------------------------------
def cpu_reference_run(n_agents, steps, repeats=1, policies=False):
    """Oracle (torch CPU restatement of the reference) fwd+bwd on a bounded sample of the workload:
    the same synthetic world generator at n_agents, default 11 networks, `steps` timesteps.
    Returns (agent-timesteps/s, seconds per fwd+bwd pass, cores)."""
    import helpers as H
    from grad_june import Timer
    from grad_june.policies import Policies
    from grad_june.symptoms import SymptomsSampler
    from grad_june.transmission import TransmissionSampler
    from grad_june.world import make_synthetic_world
    from oracle import gj_oracle as O

    params = bench_params("cpu", steps, policies)
    torch.manual_seed(0)
    data = make_synthetic_world(n_agents, seed=0, device="cpu")
    w = O.OracleWorld(n_agents=n_agents, age=data["agent"].age, sex=data["agent"].sex)
    for t in data.venue_types():
        ei = data["attends_" + t].edge_index
        w.edges[t] = O.EdgeType(src=ei[0], dst=ei[1], people=data[t]["people"], n_groups=len(data[t]["id"]))
    vals = TransmissionSampler.from_parameters(params)(n_agents)
    prof = {k: vals[i] for i, k in enumerate(("max_infectiousness", "shape", "rate", "shift"))}
    nets = H.make_leaf_networks(params)
    sym = H.oracle_symptoms(SymptomsSampler.from_parameters(params))
    sched = H.oracle_schedule(params, nets, Policies.from_parameters(params))
    g = torch.Generator().manual_seed(1)
    best = None
    for _ in range(repeats):
        noises = [O.StepNoise(E=torch.empty(2, n_agents).exponential_(generator=g), u=torch.rand(n_agents, generator=g),
                              z=torch.randn(10, n_agents, generator=g)) for _ in range(len(sched) + 1)]
        for net in nets.networks.values():
            net.log_beta.grad = None
        # fresh graph each repeat
        sched = H.oracle_schedule(params, nets, Policies.from_parameters(params))
        t0 = time.perf_counter()
        res = O.run(w, prof, sym, torch.tensor(-2.0), sched, noises)
        (res["cases_per_timestep"].sum() + res["deaths_per_timestep"].sum()).backward()
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return n_agents * steps / best, best, torch.get_num_threads()


def run_reference_arm(args, rank, world_size):
    if rank != 0:
        return
    # every host thread this process may use (torchrun pins OMP_NUM_THREADS=1 per rank: the other ranks do no work here)
    try:
        torch.set_num_threads(max(1, len(os.sched_getaffinity(0))))
    except (AttributeError, OSError):
        torch.set_num_threads(max(1, os.cpu_count() or 1))
    n_sample = args.cpu_agents
    # warm-up
    for _ in range(max(args.warmup, 0) and 1):
        cpu_reference_run(min(n_sample, 100_000), 1)
    t0 = time.perf_counter()
    thr, secs, cores = cpu_reference_run(n_sample, args.steps, policies=args.policies)
    line = {
        "impl": "reference", "metric": METRIC, "value": thr, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": secs * 1e3 / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.agents), "sample_agents": n_sample, "networks": 11,
                   "note": "reference is pure Python/torch (no compiled oracle/_ref): oracle port of its CPU path"},
        "cpu_baseline": {"value": thr, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{n_sample} agents of the same synthetic world x {args.steps} timesteps, fwd+bwd"},
        "e2e": {"value": thr, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_name(n_agents, policies=False):
    return (f"synthetic England-scale world ({n_agents / 1e6:.0f}M agents, ~4.6 edges/agent over household/company/school/"
            "university/care_home/leisure), 11 default networks, symptoms on, fwd+bwd wrt log_beta"
            + (", social distancing + school/pub/cinema/gym closure + quarantine(stage 4) from day 15" if policies else ""))


DUMP_AGENTS = 1 << 20      # agents in the sample of the per-agent state that --dump-outputs writes


def window_outputs(out, window, data, per_agent):
    """What a caller of the timed path receives from its last window, as host arrays: the result series and
    d loss / d log_beta (a leading axis over the samples when a rank evaluates several) and, ``per_agent``, the
    agents' final infection state in the order the world was loaded in, for a fixed seeded sample of agents."""
    from grad_june.world import original_order

    out = out.detach().cpu().numpy().astype(np.float32)
    t = window + 1                   # the seeding step + `window` timesteps
    arrays = {"cases_per_timestep": out[..., :t], "deaths_per_timestep": out[..., t:2 * t],
              "grad_log_beta": out[..., 2 * t:]}
    if per_agent:
        inf = original_order(data, data["agent"].is_infected.detach())
        idx = np.sort(np.random.default_rng(0).choice(inf.numel(), size=min(DUMP_AGENTS, inf.numel()), replace=False))
        arrays["is_infected_sample"] = inf[torch.from_numpy(idx).to(inf.device)].cpu().numpy().astype(np.float32)
        arrays["is_infected_sample_agent"] = idx.astype(np.float64)
    return arrays


def write_outputs(dirname, arrays):
    d = Path(dirname)
    d.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(d / f"{name}.npy", np.ascontiguousarray(a))


# ------------------------------------------------------------------------------------------
# parity inside the benchmark: one teacher-forced step at the benchmark's size against the oracle on the same GPU
# ------------------------------------------------------------------------------------------
def verify_step(model, data, params, dev, policies, seed=2024):
    """One fused step of the throughput-mode kernels from a mid-epidemic state against oracle/gj_oracle.py run on
    the SAME GPU (same CUDA libm) with the kernels' own Philox draws (gj_philox_fill): per-agent q, masks, stages.
    The oracle is the checker here, nothing of it is timed."""
    import helpers as H
    from grad_june import Timer, ops
    from oracle import gj_oracle as O

    n = len(data["agent"].id)
    timer = Timer.from_parameters(params)
    for _ in range(min(16 if policies else 8, int(params["timer"]["total_days"]) - 1)):
        next(timer)
    keep = {k: data["agent"][k] for k in ("susceptibility", "is_infected", "infection_time", "transmission")}
    keep_sym = dict(data["agent"].symptoms)
    state = H.mid_epidemic_state(n, timer.now, 11, dev)
    for k in ("susceptibility", "is_infected", "infection_time"):
        data["agent"][k] = state[k]
    data["agent"].symptoms = {k: state[k] for k in ("current_stage", "next_stage", "time_to_next_stage")}
    out = {"agents": n, "step": f"day {timer.now:.0f}, dt {timer.duration:.2f}", "oracle_device": str(dev)}
    try:
        family = model.kernel_family(data, timer)
        with torch.no_grad(), ops.philox_seed(seed):
            model.step(data, timer, want_probs=True)
        agent = data["agent"]
        E, u, z = ops.philox_fill(seed, 0, n, dev)
        w, nets, spec, sym, prof, st = H.oracle_step_inputs(params, data, model, timer, state, dev)
        aux = {}
        with torch.no_grad():
            O.step(w, st, prof, spec, sym, H.layout_noise(data, E, u, z, dev), aux)
        q, qo = agent["not_infected_probs"], aux["q"]
        T, To = agent.transmission, aux["transmission"]
        nz = To != 0
        mism = torch.nonzero(agent["new_infected"] != aux["new_infected"]).flatten()
        Eo = E if "original_index" not in agent else E[:, agent["original_index"]]
        worst = H.certify_near_ties(qo[mism].cpu().numpy(), Eo[:, mism].cpu().numpy(), np.arange(mism.numel()),
                                    what=f"bench --verify, {n} agents")
        ok = torch.ones(n, dtype=torch.bool, device=dev)
        ok[mism] = False
        sym_out = agent.symptoms
        stage_bad = int(((sym_out["current_stage"] != st["current_stage"]) & ok).sum()) \
            + int(((sym_out["next_stage"] != st["next_stage"]) & ok).sum()) \
            + int(((agent.is_infected != st["is_infected"]) & ok).sum())
        out.update(kernel_family=family,
                   q_max_rel=float(((q - qo).abs() / qo).max()),
                   T_max_rel=float(((T[nz] - To[nz]).abs() / To[nz].abs()).max()) if bool(nz.any()) else 0.0,
                   mask_mismatch=int(mism.numel()), max_gap=worst, near_ties_certified=True,
                   state_mismatch_outside_near_ties=stage_bad,
                   new_infections=int(aux["new_infected"].sum()),
                   stages_moved=int((st["current_stage"] != state["current_stage"]).sum()),
                   passed=bool(stage_bad == 0 and float(((q - qo).abs() / qo).max()) <= 1e-5))
    except Exception as e:  # noqa: BLE001 -- the bench line must still be printed
        out.update(passed=False, error=repr(e)[:300])
    finally:
        for k, v in keep.items():
            data["agent"][k] = v
        data["agent"].symptoms = keep_sym
        data["agent"]._mapping.pop("new_infected", None)
        data["agent"]._mapping.pop("not_infected_probs", None)
        torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------
# one measured configuration
# ------------------------------------------------------------------------------------------
def measure(args, ctx, scaling, graph, full=True):
    """Build the world of this configuration, warm up, time exactly K steps (device events, max over ranks), and —
    ``full`` — the per-kernel pass, the end-to-end pass, the repeats and the verification step.  Returns the dict
    rank 0 turns into the JSON line (None on other ranks)."""
    import torch.distributed as dist
    from grad_june import GradJune, Runner, Timer, _lib, ops
    from grad_june.world import freeze_device_world, make_synthetic_world, renumber_world

    rank, world_size, dev = ctx["rank"], ctx["world_size"], ctx["dev"]
    geo = world_size > 1 and args.parallelism == "geo"
    strong = geo and scaling == "strong"
    N = args.agents // world_size if strong else args.agents      # agents this rank owns (about, for strong)
    free, total = torch.cuda.mem_get_info()
    per_step = 40.0 * N            # bytes retained per agent per step until backward (pre-state 24 + tape 8 + sums ~3)
    resident = 120.0 * N           # world CSR + static arrays + transient workspaces + initial state backup
    max_window = int(max(1, (free * 0.85 - resident) // per_step))
    # the timed region is exactly K = --steps timesteps in windows of one length: the longest that divides K
    cap = min(args.steps, args.window or 60, max_window)
    window = max(w for w in range(1, cap + 1) if args.steps % w == 0)
    if world_size > 1:             # the ranks of a partitioned world step together (a divisor of K on every rank)
        wt = torch.tensor([window], device=dev)
        dist.all_reduce(wt, op=dist.ReduceOp.MIN)
        window = int(wt.item())

    params = bench_params(dev, window, args.policies)
    torch.manual_seed(1234 + rank)
    part = None
    if geo:
        from grad_june.partition import partition_from_blocks, partition_world
        if strong:      # the whole world fits every GPU: build it, keep this rank's part
            whole = make_synthetic_world(args.agents, seed=0, device=dev)
            data = partition_world(whole, rank, world_size)
            del whole
        else:           # no rank ever holds the whole world: each generates its own block
            data = partition_from_blocks(make_synthetic_world(N, seed=0, device=dev, block=(rank, world_size)))
        part = data._gj_partition
        N = part.agent_hi - part.agent_lo
        torch.cuda.empty_cache()
    else:
        data = make_synthetic_world(N, seed=0, device=dev)
    if args.shuffle_agents:
        assert not geo, "--shuffle-agents: single-GPU / ensemble runs"
        data = renumber_world(data, torch.randperm(N, device=dev))
        del data["agent"]["original_index"]        # a world that simply arrived in this order
        torch.cuda.empty_cache()
    data = Runner.get_data(params, data=data)
    torch.cuda.empty_cache()
    model = GradJune.from_parameters(params)
    parity = None
    if full and args.verify and world_size == 1:
        parity = verify_step(model, data, params, dev, args.policies)
    world = freeze_device_world(data, dev)   # the int64 edge lists are not needed once the CSR exists
    torch.cuda.empty_cache()
    keys = list(model.infection_networks.networks.keys())
    gen = torch.Generator().manual_seed(99)
    offsets = 0.05 * torch.randn(max(world_size, 1), len(keys), generator=gen)
    # geo: one parameter vector for the one world; ensemble: every rank evaluates its own beta sample (config 5)
    base_log_beta = torch.tensor([float(model.infection_networks.networks[k].log_beta) for k in keys])
    n_samples = 1          # parameter samples this rank evaluates per window
    if not geo and args.samples > max(world_size, 1):
        n_samples = args.samples // max(world_size, 1)
        draws = 0.25 * torch.randn(args.samples, len(keys), generator=torch.Generator().manual_seed(1))
        host_log_beta = (base_log_beta + draws[rank * n_samples:(rank + 1) * n_samples]).contiguous()   # [B/N, K]
    else:
        host_log_beta = (base_log_beta + offsets[0 if geo else rank]).reshape(1, -1)
    host_log_beta = host_log_beta.pin_memory()
    n_total = N * n_samples      # agent-trajectories advanced per timestep over all GPUs
    if geo:
        n_total = part.n_global_agents
    elif world_size > 1:
        n_total = N * n_samples * world_size

    runner = Runner(model=model, data=data, timer=Timer.from_parameters(params), log_fraction_initial_cases=-2.0,
                    save_path=params["save_path"], parameters=params)

    def one_window(e2e):
        """every sample of this rank: forward `window` timesteps + backward; device-side results and grads"""
        lb_all = host_log_beta.to(dev, non_blocking=True) if e2e else resident_log_beta   # H2D of the inputs
        outs = [one_sample(lb_all[i]) for i in range(n_samples)]
        out = outs[0] if n_samples == 1 else torch.stack(outs)
        return out.to("cpu") if e2e else out                                             # D2H of the results

    def one_sample(lb_dev):
        leaves = []
        for i, k in enumerate(keys):
            leaf = lb_dev[i].detach().clone().requires_grad_(True)
            model.infection_networks.networks[k].log_beta = leaf
            leaves.append(leaf)
        with ops.philox_seed(7):
            results, _ = runner()
        loss = results["cases_per_timestep"].sum() + results["deaths_per_timestep"].sum()
        loss.backward()
        grads = torch.stack([l.grad for l in leaves])
        if geo:      # every rank holds the terms of the groups it owns: the world's gradient is their sum
            dist.all_reduce(grads)
        return torch.cat([results["cases_per_timestep"], results["deaths_per_timestep"], grads])

    resident_log_beta = host_log_beta.to(dev)
    n_windows = args.steps // window
    steps_done = n_windows * window
    eager_window = one_window

    def barrier():
        if world_size > 1:
            dist.barrier()
        torch.cuda.synchronize()

    prof = None
    graphed = None
    B = args.batch if (args.batch > 1 and not geo and graph) else 0      # [N, b] batching of the ensemble's samples
    if B:
        # batched ensemble (SURVEY 8e-2): every replay steps B of this rank's samples through gj_step_*_batch
        from grad_june.graphed import GraphedRunner
        if n_samples % B:
            raise SystemExit(f"--batch {B}: needs --parallelism ensemble with --samples a multiple of gpus x batch "
                             f"(this rank has {n_samples} sample(s))")
        loss_fn_b = lambda r: r["cases_per_timestep"].sum(0) + r["deaths_per_timestep"].sum(0)   # noqa: E731

        def eager_batched(lb):          # the same window through the Python loop (per-kernel events need eager launches)
            runner.batch = B
            leaves = []
            for i, k in enumerate(keys):
                leaf = lb[:, i].detach().clone().requires_grad_(True)
                model.infection_networks.networks[k].log_beta = leaf
                leaves.append(leaf)
            with ops.philox_seed(7):
                results, _ = runner()
            loss_fn_b(results).sum().backward()

        eager_batched(resident_log_beta[:B])
        if full:
            _lib.profile_enable(True)
            barrier()
            eager_batched(resident_log_beta[:B])
            barrier()
            scale = n_windows * (n_samples // B)
            prof = {k: (v[0] * scale, v[1] * scale, v[2] * scale) for k, v in _lib.profile_read().items()}
            _lib.profile_enable(False)
        for k in keys:
            model.infection_networks.networks[k].log_beta = torch.tensor(0.0)
        graphed = GraphedRunner(runner, loss_fn=loss_fn_b, seed=7, batch=B)

        def one_window(e2e):  # noqa: F811
            lb_all = host_log_beta.to(dev, non_blocking=True) if e2e else resident_log_beta
            outs = []
            for j in range(0, n_samples, B):
                _, grads, results = graphed(lb_all[j:j + B])
                outs.append(torch.cat([results["cases_per_timestep"].t(), results["deaths_per_timestep"].t(), grads], dim=1))
            out = torch.cat(outs)
            return out.to("cpu") if e2e else out
    elif graph:
        from grad_june.graphed import GraphedRunner
        # per-kernel pass first, eagerly (a replayed graph carries no events), then capture
        eager_window(False)
        if full:
            _lib.profile_enable(True)
            barrier()
            eager_window(False)
            barrier()
            prof = {k: (v[0] * n_windows, v[1] * n_windows, v[2] * n_windows) for k, v in _lib.profile_read().items()}
            _lib.profile_enable(False)
        for k in keys:
            model.infection_networks.networks[k].log_beta = torch.tensor(0.0)
        loss_fn = lambda r: r["cases_per_timestep"].sum() + r["deaths_per_timestep"].sum()   # noqa: E731
        graphed = GraphedRunner(runner, loss_fn=loss_fn, seed=7)     # partitioned: the gradient all-reduce is captured too

        def one_sample(lb_dev, g=None):  # noqa: F811
            _, grads, results = (g or graphed)(lb_dev)
            return torch.cat([results["cases_per_timestep"], results["deaths_per_timestep"], grads])

        if args.streams > 1 and not geo and n_samples > 1:
            # more lanes: each needs its own world object (per-world scratch = one step in flight per world), runner
            # and captured window; the world arrays are rebuilt from the same seed
            lanes = [graphed]
            for _ in range(args.streams - 1):
                torch.manual_seed(1234 + rank)
                d2 = Runner.get_data(params, data=make_synthetic_world(N, seed=0, device=dev))
                freeze_device_world(d2, dev)
                m2 = GradJune.from_parameters(params)
                r2 = Runner(model=m2, data=d2, timer=Timer.from_parameters(params), log_fraction_initial_cases=-2.0,
                            save_path=params["save_path"], parameters=params)
                lanes.append(GraphedRunner(r2, loss_fn=loss_fn, seed=7))
            lane_streams = [torch.cuda.Stream(device=dev) for _ in lanes]

            def one_window(e2e):  # noqa: F811
                lb_all = host_log_beta.to(dev, non_blocking=True) if e2e else resident_log_beta
                main = torch.cuda.current_stream(dev)
                for st in lane_streams:
                    st.wait_stream(main)
                outs = [None] * n_samples
                for i in range(n_samples):
                    k = i % len(lanes)
                    with torch.cuda.stream(lane_streams[k]):
                        outs[i] = one_sample(lb_all[i], lanes[k])
                for st in lane_streams:
                    main.wait_stream(st)
                out = torch.stack(outs)
                return out.to("cpu") if e2e else out

    # warm-up: W >= 3 timesteps
    wsteps = 0
    while wsteps < max(args.warmup, 3) or (world_size > 1 and wsteps < 2 * window):   # N > 1: NCCL channels settle
        one_window(False)
        wsteps += window
    barrier()

    # ---- timed region 1: EXACTLY K steps, device-resident inputs ------------------------------------------
    # (NVML is polled by rank 0 only: eight processes polling it were measured to disturb the step)
    with ClockSampler(ctx["local_rank"], period=0.02 if rank == 0 else 1e9) as clocks:
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.nvtx.range_push("timed")
        e0.record()
        for _ in range(n_windows):
            out = one_window(False)
        e1.record()
        torch.cuda.nvtx.range_pop()
        barrier()
        ms = e0.elapsed_time(e1)
        outputs = None
        if args.dump_outputs and rank == 0 and full:     # before the windows below overwrite the last one's state
            outputs = window_outputs(out, window, data, per_agent=n_samples == 1 and world_size == 1)
        # ---- repeats: the same window R more times, each timed on its own (spread of the measurement) --------
        rep_ms = []
        for _ in range(args.repeats if full else 0):
            barrier()
            r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            r0.record()
            one_window(False)
            r1.record()
            barrier()
            rep_ms.append(r0.elapsed_time(r1) / window)
    clk = clocks.summary()

    # ---- per-kernel pass: the same K steps again with the library's CUDA events around every kernel (kept out
    #      of the timed region above: two event records per launch cost a few per cent on small worlds) ----------
    if prof is None and full:
        _lib.profile_enable(True)
        barrier()
        for _ in range(n_windows):
            one_window(False)
        barrier()
        prof = _lib.profile_read()
        _lib.profile_enable(False)

    # ---- timed region 2: end to end through Runner with host buffers -------------------------------
    e2e_s, h2d, d2h = None, 0.0, 0.0
    if full:
        barrier()
        t0 = time.perf_counter()
        for _ in range(n_windows):
            host_out = one_window(True)
        torch.cuda.synchronize()
        if world_size > 1:
            dist.barrier()
        e2e_s = time.perf_counter() - t0
        h2d = host_log_beta.numel() * 4 / window
        d2h = host_out.numel() * 4 / window

    rank_ms = [ms]
    if world_size > 1:
        t = torch.tensor([ms, e2e_s or 0.0] + rep_ms, device=dev, dtype=torch.float64)
        every = [torch.zeros_like(t) for _ in range(world_size)]
        dist.all_gather(every, t)
        rank_ms = [round(float(x[0]), 3) for x in every]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_s, rep_ms = float(t[0]), (float(t[1]) if full else None), [float(x) for x in t[2:]]
        if not geo:
            gathered = [torch.zeros_like(out) for _ in range(world_size)]
            dist.all_gather(gathered, out)      # the ensemble's only exchange: losses + gradients

    parallelism = "single GPU"
    if geo:
        from grad_june.partition import exchange_for
        nb = {t: part.n_boundary[t] for t in part.types if part.n_boundary[t]}
        parallelism = (f"geographic partition over {world_size} GPUs ({scaling} scaling), boundary-group sums exchanged "
                       f"once per step forward and once backward ({exchange_for(data, world).mode}); boundary "
                       f"groups {nb} of {world.n_groups} local groups")
    elif world_size > 1 or n_samples > 1:
        how = (f"{B} at a time as one batched [N, b] step (gj_step_forward_batch: one read of the world's index data and "
               "profile per b samples)") if B else "one after the other"
        parallelism = (f"ensemble shard: {n_samples * world_size} beta samples per window, {n_samples} per GPU evaluated "
                       f"{how} on a replica of the world, no data-path collective")
    res = None
    if rank == 0:
        total_units = n_total * steps_done
        res = dict(value=total_units / (ms * 1e-3), ms=ms, steps_done=steps_done, window=window, N=N, n_total=n_total,
                   world=world, prof=prof, clk=clk, rank_ms=rank_ms, e2e_s=e2e_s, h2d=h2d, d2h=d2h, rep_ms=rep_ms,
                   parallelism=parallelism, parity=parity, graph=graph, scaling=scaling, total_units=total_units,
                   batch=B, outputs=outputs)
    if graphed is not None:
        ctx["captured_nccl"] = ctx.get("captured_nccl", False) or geo
        graphed.graph.reset()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=120,
                    help="timesteps K of the timed region, run as K / w BPTT windows of w timesteps: the longest w "
                         "that divides K and that --window and the GPU's memory allow")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--agents", type=int, default=56_000_000,
                    help="agents of the whole world (strong scaling, the default for N > 1: BASELINE config 3 is THE 56M "
                         "world on 1/2/4/8 GPUs) / per GPU (weak scaling)")
    ap.add_argument("--parallelism", default="geo", choices=["geo", "ensemble"],
                    help="N > 1: geographic partition of ONE world with the boundary-group exchange (default), or one "
                         "beta sample per GPU on replicas of the world (no data-path collective)")
    ap.add_argument("--scaling", default=None, choices=["weak", "strong"],
                    help="geo: the --agents world is cut into N parts (strong, default), or every GPU owns --agents agents "
                         "of a world of N x --agents (weak; also measured and reported as `weak_scaling` by default)")
    ap.add_argument("--no-weak-companion", action="store_true",
                    help="N > 1, strong scaling: skip the additional weak-scaling measurement")
    ap.add_argument("--samples", type=int, default=0,
                    help="ensemble: beta samples evaluated per window over all GPUs (BASELINE config 5: 1024 on a 9M "
                         "world, --agents 9000000 --window 30); default one per GPU")
    ap.add_argument("--batch", type=int, default=0,
                    help="ensemble: step this many samples together as one batched [N, b] call (gj_step_forward_batch / "
                         "gj_step_backward_batch); 0 = one sample per replay")
    ap.add_argument("--streams", type=int, default=0,
                    help="ensemble + graph: evaluate this many samples concurrently, each lane with its own replica of "
                         "the world, captured window and CUDA stream (bandwidth-bound and issue-bound kernels of "
                         "different samples overlap)")
    ap.add_argument("--graph", action="store_true",
                    help="capture the window (Runner() + backward) once as a CUDA graph and replay it "
                         "(grad_june.graphed.GraphedRunner): removes the per-step Python cost that bounds small worlds. "
                         "This is the default driver")
    ap.add_argument("--no-graph", action="store_true", help="always drive the window from the Python loop (Runner)")
    ap.add_argument("--policies", action="store_true",
                    help="BASELINE config 4: social distancing, school/leisure closures and quarantine from day 15")
    ap.add_argument("--window", type=int, default=0,
                    help="longest BPTT window (0 = 60 timesteps as in BASELINE.json, fewer if memory does not allow); "
                         "the window also divides --steps")
    ap.add_argument("--repeats", type=int, default=5, help="further windows timed one by one (median / spread)")
    ap.add_argument("--no-verify", dest="verify", action="store_false",
                    help="skip the teacher-forced parity step against the oracle (N = 1)")
    ap.add_argument("--shuffle-agents", action="store_true",
                    help="load the synthetic world with its agents in a RANDOM order (as a world that was not numbered "
                         "for this layout): Runner.get_data then renumbers it (world.layout_order) and the kernels key "
                         "their noise by the loaded ids")
    ap.add_argument("--cpu-agents", type=int, default=1_000_000, help="agents of the CPU-baseline sample")
    ap.add_argument("--cpu-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what their last window computed as DIR/<name>.npy: the result "
                         "series, d loss / d log_beta and (one sample, one GPU) the final infection state of a fixed "
                         f"seeded sample of {DUMP_AGENTS} agents; the inputs are the same for the same arguments")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")

    rank = int(os.environ.get("RANK", 0))
    world_size = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference_arm(args, rank, world_size)
        return

    import torch.distributed as dist
    from grad_june import _lib

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = f"cuda:{local_rank}"
    if world_size > 1:
        dist.init_process_group("nccl", device_id=torch.device(dev))
    ctx = {"rank": rank, "world_size": world_size, "local_rank": local_rank, "dev": dev}

    geo = world_size > 1 and args.parallelism == "geo"
    if args.batch > 1:         # a batched replay already fills the GPU: one lane
        args.streams = 1
    if args.streams <= 0:      # ensembles: three concurrent lanes per GPU by default (+17 % over one, profiles/README.md)
        args.streams = 3 if (not geo and args.samples > max(world_size, 1)) else 1
    scaling = args.scaling or ("strong" if geo else "weak")
    per_gpu = args.agents // world_size if (geo and scaling == "strong") else args.agents
    # the captured window (GraphedRunner: Runner() + backward() as one CUDA graph) is the default driver: it removes the
    # per-launch gaps of the Python loop (56 M agents: 2.84 -> 2.75 ms per step; 9 M: host-bound without it)
    graph = not args.no_graph
    _ = per_gpu
    m = measure(args, ctx, scaling, graph, full=True)
    weak = None
    if geo and scaling == "strong" and not args.no_weak_companion:
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        weak = measure(args, ctx, "weak", graph, full=False)

    if rank == 0:
        if args.dump_outputs:
            write_outputs(args.dump_outputs, m["outputs"])
        peak, peak_kind = measured_peak_gbs()
        world, prof, N, value = m["world"], m["prof"], m["N"], m["value"]
        steps_done = m["steps_done"]
        # dominant kernel + its algorithmic bytes per launch (DESIGN.md "Roofline")
        e_bar = world.n_edges / N
        g_bar = world.n_groups / N
        small = (world.group_size <= _lib.config()["small_group"]) & (world.group_size > 0)
        e_small = float(world.group_size[small].sum()) / N
        g_small = float(small.sum()) / N
        e_gen = world.n_generic_edges / N
        g_gen = float((world.group_size > 0).sum()) / N
        alg = kernel_alg_bytes(e_gen, g_gen, e_small, g_small)
        per_launch = N          # agents (agent-samples) one launch processes
        if m.get("batch"):
            # a batched launch steps b samples: the world's index words, class bytes and the packed profile are read
            # once per b samples, everything else per sample
            b = m["batch"]
            shared = {"agent_forward": 1 + 4 + 8, "agent_backward": 1, "backward_gather": 1 + 4 + 8 + 16,
                      "group_small<bwd>": 4 * e_small + 8 * g_small,
                      "group_chunk<bwd>": 4 * (e_gen - e_small) + 8 * (g_gen - g_small)}
            alg = {k: v - shared.get(k, 0.0) * (b - 1) / b for k, v in alg.items()}
            per_launch = N * b
        timed = {k: v for k, v in prof.items() if v[1] > 0}
        dom = max(timed, key=lambda k: timed[k][0]) if timed else None
        roof = None
        if dom is not None:
            avg_ms = timed[dom][0] / timed[dom][1]
            achieved = alg.get(dom, 0.0) * per_launch / (avg_ms * 1e-3) / 1e9
            traffic = ncu_traffic(N)
            step_frac = B_ALG_STEP * value / world_size / 1e9 / peak
            roof = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "traffic": traffic["kernels"].get(dom) if traffic else None,
                    "traffic_source": traffic["source"] if traffic else None, "peak_kind": peak_kind,
                    "alg_bytes_per_agent": alg.get(dom), "avg_launch_ms": avg_ms,
                    "step_alg_bytes_per_agent_timestep": B_ALG_STEP,
                    "step_achieved": B_ALG_STEP * value / world_size / 1e9,
                    "step_frac": step_frac, "step_frac_contract_279B": step_frac,
                    "kernel_frac": {k: round(alg[k] * per_launch / (v[0] / v[1] * 1e-3) / 1e9 / peak, 4)
                                    for k, v in timed.items() if alg.get(k)},
                    "kernel_ms_share": {k: round(v[0] / sum(x[0] for x in timed.values()), 4) for k, v in timed.items()},
                    "kernel_avg_ms": {k: round(v[0] / v[1], 4) for k, v in timed.items()},
                    "kernel_ms_per_step": round(sum(x[0] for x in timed.values()) / steps_done, 4),
                    "note": "per-kernel CUDA events from a second, identical pass over the K steps"}
            if traffic and traffic.get("step_bytes_per_agent"):
                # the same throughput against the bytes ncu counted for one whole step (every kernel, fwd + bwd)
                roof["step_ncu_bytes_per_agent_timestep"] = traffic["step_bytes_per_agent"]
                roof["step_frac_ncu_bytes"] = traffic["step_bytes_per_agent"] * value / world_size / 1e9 / peak
        launches = int(sum(v[2] for v in prof.values()))
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world_size, "steps": steps_done,
            "warmup": max(args.warmup, 3), "ms_per_step": m["ms"] / steps_done, "higher_is_better": True,
            "scaling": m["scaling"] if geo else "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(m["n_total"] if geo else N, args.policies), "agents_per_gpu": N,
                       "agents_total": m["n_total"], "edges_per_agent": round(e_bar, 3),
                       "groups_per_agent": round(g_bar, 3), "bptt_window": m["window"], "networks": 11,
                       "ensemble_batch": m.get("batch") or None,
                       "driver": (f"CUDA graph replay (GraphedRunner), {args.streams} concurrent lane(s)" if m["graph"]
                                  else "Python loop (Runner)"),
                       "layout_tiers": dict(zip(world.types, world.type_tier)),
                       "agents_shuffled_then_renumbered": bool(args.shuffle_agents),
                       "noise_keyed_by_loaded_id": world.__dict__.get("orig_id") is not None,
                       "parallelism": m["parallelism"],
                       "l2": "inputs (>= 2 GB per pass) far larger than the 126 MB L2; no flush needed"},
            "clocks": m["clk"], "rank_ms": m["rank_ms"],
            "e2e": {"value": m["total_units"] / m["e2e_s"], "unit": UNIT, "h2d_bytes_per_step": m["h2d"],
                    "d2h_bytes_per_step": m["d2h"]},
            "gpu_launches": launches,
            "roofline": roof,
        }
        if m["rep_ms"]:
            r = sorted(m["rep_ms"])
            line["repeats"] = {"n": len(r), "ms_per_step_median": r[len(r) // 2], "ms_per_step_min": r[0],
                               "ms_per_step_max": r[-1], "spread_pct": round(100 * (r[-1] - r[0]) / r[len(r) // 2], 2),
                               "value_median": m["n_total"] / (r[len(r) // 2] * 1e-3),
                               "note": "further single windows after the timed K steps, each between its own events"}
        if m["parity"] is not None:
            line["parity"] = m["parity"]
        if weak is not None:
            line["weak_scaling"] = {"value": weak["value"], "unit": UNIT, "ms_per_step": weak["ms"] / weak["steps_done"],
                                    "agents_per_gpu": weak["N"], "agents_total": weak["n_total"],
                                    "driver": "CUDA graph replay (GraphedRunner)" if weak["graph"] else "Python loop (Runner)",
                                    "parallelism": weak["parallelism"],
                                    "rank_ms": weak["rank_ms"]}
        if not args.no_cpu_baseline and world_size == 1:
            thr, secs, cores = cpu_reference_run(args.cpu_agents, args.cpu_steps, policies=args.policies)
            line["cpu_baseline"] = {"value": thr, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": f"{args.cpu_agents} agents of the same synthetic world x {args.cpu_steps} "
                                              f"timesteps fwd+bwd ({secs:.1f} s)"}
        print(json.dumps(line), flush=True)
    if world_size > 1:
        if ctx.get("captured_nccl"):
            # a captured graph that contained NCCL kernels: destroy_process_group was seen to hang after it
            torch.cuda.synchronize()
            dist.barrier()
            sys.stdout.flush()
            os._exit(0)
        dist.destroy_process_group()


def ncu_traffic(n_agents):
    """DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum, per launch) of the throughput-mode kernels from the
    NEWEST committed `ncu --set full` capture of this workload size: profiles/r*_traffic.json, written by
    scripts/ncu_summarise.py together with the git revision it was taken at.  None when no capture matches the
    size (traffic cannot be measured inside an un-profiled run)."""
    best = None
    for f in sorted((ROOT / "profiles").glob("r*_traffic.json")):
        try:
            t = json.load(open(f))
        except Exception:  # noqa: BLE001
            continue
        if int(t.get("agents", -1)) == int(n_agents):
            best = (f, t)            # sorted by name: the round tag orders them
    if best is None:
        return None
    f, t = best
    return {"kernels": t["kernels"], "step_bytes_per_agent": t.get("step_bytes_per_agent"),
            "source": {"file": f"profiles/{f.name}", "git": t.get("git"), "captured": t.get("when")}}


def kernel_alg_bytes(e_gen, g_gen, e_small, g_small):
    """Algorithmic bytes per agent and launch of each throughput-mode kernel: every operand array touched once,
    int32 indices, fp32 values (DESIGN.md "Kernels" lists the terms).  e_gen / g_gen: edges and groups per agent
    of the GENERIC-tier types; e_small / g_small: the part of them in groups <= GJ_SMALL_GROUP."""
    def grp(e, g):   # member index + member value per edge; per group: row pointer, pc, two outputs
        return 8 * e + 16 * g
    return {
        # is_infected in, T out; the profile (tinf 4 + packed 16) is read for infected agents only: not counted
        "transmission": 4 + 4,
        # forward: the scatter tier's finalize pass (accumulator 8 + dirty 1 + row pointers 8 + pc 4 + two outputs 8 per
        # group; the adds themselves come from the infectious few inside the transmission pass) / giant groups only
        "group_small<fwd>": 29 * g_gen, "group_chunk<fwd>": 0.0,
        "group_small<bwd>": grp(e_small, g_small), "group_chunk<bwd>": grp(e_gen - e_small, g_gen - g_small),
        # state in 24 + class 1 + generic entry 4 + household slot+pc 8 + T 4 + group value + state out 24 + tape 8
        "agent_forward": 24 + 1 + 4 + 8 + 4 + 4 * e_gen + 24 + 8,
        # state in 20 + tape 8 + class 1 + cotangents in 24 + cotangents out 24 + w 4
        "agent_backward": 20 + 8 + 1 + 24 + 24 + 4,
        # class 1 + generic entry 4 + household slot+pc 8 + w 4 + group value + is_infected/infection_time 8 +
        # packed profile 16 + read-modify-write of two cotangents 16
        "backward_gather": 1 + 4 + 8 + 4 + 4 * e_gen + 8 + 16 + 16,
    }


if __name__ == "__main__":
    main()
