"""A whole calibration iteration — ``Runner()`` (seeding + T fused timesteps) and ``loss.backward()`` — captured
once as a CUDA graph and replayed per parameter sample (SURVEY.md §8f rank 1: the caller of the hot path).

The reference drives the path from Python: per timestep ~430 torch ops; here it is ~12 kernels per step whose launch
cost (≈ 0.55 ms of Python per step fwd+bwd) dominates worlds below ≈ 10 M agents and strongly-scaled partitions.  The
library's entry points are stream-ordered, never allocate and never synchronise, so the whole window — including
the NCCL all-reduces of a partitioned world — is capturable with ``torch.cuda.graph``.

    graphed = GraphedRunner(runner, loss_fn=lambda r: r["cases_per_timestep"].sum())
    loss, grads, results = graphed(log_beta_vector)       # replay: one graph launch

``fit_seed=True`` calibrates the seeding too: the initial-case log-fractions go next to the log-betas in the parameter
vector — one value for a national seed, one per region of ``runner.seed_labels`` with ``seed_by`` — so a replay takes
[K + R] values ([b, K + R] batched) and returns their gradient.

Noise: the Philox key and call indices are kernel arguments, so every replay draws the SAME noise (common random
numbers across parameter samples — the usual variance reduction for calibration gradients); ``recapture(seed)``
re-records the graph with another key.

``batch=b`` captures a BATCHED window (SURVEY.md §8e-2): b parameter samples advance together through
``gj_step_forward_batch`` / ``gj_step_backward_batch`` — one read of the world's index data and of the infectiousness
profile serves all b samples, and every kernel launch does b samples' work.  ``log_beta`` is then [b, K], ``loss_fn``
receives result series of shape [T+1, b] and must return one loss per sample ([b]); the gradients come back as [b, K]
(the samples are independent, so the gradient of the summed loss IS the per-sample gradient).  Sample r of a batched
replay is bit-identical to an unbatched replay with ``log_beta[r]`` (same Philox key).
"""
import warnings
from typing import Callable, Optional, Sequence

import numpy as np
import torch

from . import ops


class GraphedRunner:
    def __init__(self, runner, loss_fn: Callable[[dict], torch.Tensor], networks: Optional[Sequence[str]] = None,
                 seed: int = 0, warmup: int = 1, batch: Optional[int] = None, fit_seed: bool = False):
        self.runner = runner
        self.fit_seed = bool(fit_seed)
        self.loss_fn = loss_fn
        self.batch = int(batch) if batch else None
        runner.batch = self.batch
        nets = runner.model.infection_networks.networks
        self.names = list(networks) if networks is not None else list(nets.keys())
        agent = runner.data["agent"]
        ops.require_cuda(agent.susceptibility, "data['agent'].susceptibility")
        self.device = agent.susceptibility.device
        init = [float(torch.as_tensor(nets[k].log_beta).detach().reshape(-1)[0]) for k in self.names]
        self.n_beta = len(init)
        self.seed_names = []
        if self.fit_seed:   # the log-fractions follow the log-betas: one per region, or one national value
            lf = runner.log_fraction_initial_cases
            lf = lf.detach().cpu().numpy() if torch.is_tensor(lf) else np.asarray(lf, dtype=np.float64)
            if runner.seed_by is None:
                self.seed_names = ["national"]
                init += [float(lf.reshape(-1)[0])]
            else:
                R = len(runner.seed_labels)
                self.seed_names = [str(v) for v in runner.seed_labels]
                init += [float(v) for v in np.broadcast_to(lf.reshape(-1)[:R] if lf.size >= R else lf, (R,))]
        self.log_beta = torch.tensor(init, dtype=torch.float32).to(self.device)
        if self.batch:
            self.log_beta = self.log_beta.repeat(self.batch, 1)          # [b, K]
        self.log_beta.requires_grad_(True)
        # the networks that are NOT calibrated keep their log-betas as constants of the graph: they must already
        # live on the device (a host-to-device copy cannot be captured)
        for k, net in nets.items():
            if k not in self.names:
                value = torch.as_tensor(net.log_beta).detach().to(device=self.device, dtype=torch.float32)
                net._parameters.pop("log_beta", None)
                net.log_beta = value
        self.warmup = warmup
        self.graph = None
        self.recapture(seed)

    def _iteration(self):
        nets = self.runner.model.infection_networks.networks
        for i, k in enumerate(self.names):
            # a network built with log_beta=nn.Parameter(...) holds it as a registered parameter, and nn.Module
            # refuses to assign a plain tensor over one: unregister it first
            nets[k]._parameters.pop("log_beta", None)
            nets[k].log_beta = self.log_beta[:, i] if self.batch else self.log_beta[i]
        if self.fit_seed:
            K = self.n_beta
            self.runner._parameters.pop("log_fraction_initial_cases", None)   # an nn.Parameter is replaced like log_beta
            if self.runner.seed_by is None:
                self.runner.log_fraction_initial_cases = self.log_beta[:, K] if self.batch else self.log_beta[K]
            else:
                self.runner.log_fraction_initial_cases = self.log_beta[:, K:] if self.batch else self.log_beta[K:]
        with ops.philox_seed(self.seed):
            results, is_infected = self.runner()
        loss = self.loss_fn(results)
        if self.batch and tuple(loss.shape) != (self.batch,):
            raise ValueError(f"batched window: loss_fn must return one loss per sample, shape ({self.batch},); "
                             f"got {tuple(loss.shape)}")
        loss.sum().backward()
        part = self.runner.data.__dict__.get("_gj_partition")
        if part is not None and part.world_size > 1:
            # geographic partition: every rank holds the d/dbeta terms of the groups it owns; the sum over ranks
            # is part of the captured iteration (one more NCCL kernel in the graph, no eager collective per replay);
            # with fit_seed the seeding gradients (each rank's own agents) are summed in the same all-reduce
            import torch.distributed as dist
            dist.all_reduce(self.log_beta.grad, group=part.process_group)
        return loss.detach(), results, is_infected

    def recapture(self, seed: int):
        """(Re)record the graph with Philox key ``seed``."""
        self.seed = int(seed)
        self.graph = None
        dev = self.device
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side), warnings.catch_warnings():
            # lazy initialisation (occupancy queries, workspaces, NCCL) happens here; the leaf was created on another
            # stream than this warm-up's, which autograd remarks on
            warnings.simplefilter("ignore", UserWarning)
            for _ in range(max(self.warmup, 1)):
                self.log_beta.grad = None
                self._iteration()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.log_beta.grad = None
        torch.cuda.empty_cache()               # the eager window's tape must not stay cached next to the graph's pool
        graph = torch.cuda.CUDAGraph()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", UserWarning)
            with torch.cuda.graph(graph):
                self.loss, self.results, self.is_infected = self._iteration()
        self.grads = self.log_beta.grad        # allocated in the graph's pool: refilled by every replay
        self.graph = graph
        return self

    @torch.no_grad()
    def __call__(self, log_beta: Optional[torch.Tensor] = None):
        """Replay with ``log_beta`` ([K], or [b, K] for a batched window; [K + R] / [b, K + R] with ``fit_seed``, the
        log-fractions last; any device; None = keep).  Returns (loss, d loss / d log_beta, results): static device
        tensors that the next replay overwrites."""
        if log_beta is not None:
            self.log_beta.copy_(log_beta.to(dtype=torch.float32), non_blocking=True)
        self.graph.replay()
        return self.loss, self.grads, self.results
