"""Batched evaluation of parameter samples (SURVEY.md §8f rank 4, BASELINE config 5: a calibration ensemble of
log-beta samples on one world, sharded across the GPUs of a box).

The reference evaluates one sample per Python-driven run (example_scripts/run_model.py:6-11).  Here every rank holds
a replica of the world and its own captured window (:class:`grad_june.graphed.GraphedRunner`); a batch ``[B, K]`` of
log-beta vectors is dealt out round-robin, each rank replays its samples back to back (one graph launch per sample)
and the losses and gradients are all-gathered — no collective on the data path.  With ``batch=b`` every replay steps
b of the rank's samples together ([N, b] batching, ``gj_step_forward_batch``): one read of the world's index data per
b samples; ``loss_fn`` then returns one loss per sample.
"""
from typing import Callable, Optional, Sequence

import torch

from .graphed import GraphedRunner


def ensemble_deal(n_samples: int, world_size: int, rank: int, batch: Optional[int] = None):
    """Which samples ``rank`` evaluates, and in which replays: sample i goes to rank i % world_size (round-robin), a
    rank's samples are taken ``batch`` at a time (one at a time without batching).  Returns (rows per rank in the
    gathered table — the last ranks' rows may be padding — and the list of replays, each a list of sample indices).
    Row j of rank r in the gathered table is sample j * world_size + r."""
    per = -(-n_samples // world_size)
    mine = [j * world_size + rank for j in range(per) if j * world_size + rank < n_samples]
    step = int(batch) if batch else 1
    return per, [mine[j0:j0 + step] for j0 in range(0, len(mine), step)]


class EnsembleEvaluator:
    def __init__(self, runner, loss_fn: Callable[[dict], torch.Tensor], networks: Optional[Sequence[str]] = None,
                 seed: int = 0, process_group=None, batch: Optional[int] = None):
        import torch.distributed as dist

        self.batch = int(batch) if batch else None
        self.graphed = GraphedRunner(runner, loss_fn, networks=networks, seed=seed, batch=self.batch)
        self.names = self.graphed.names
        self.group = process_group
        self.distributed = dist.is_available() and dist.is_initialized()
        self.rank = dist.get_rank(process_group) if self.distributed else 0
        self.world_size = dist.get_world_size(process_group) if self.distributed else 1

    @torch.no_grad()
    def __call__(self, log_betas: torch.Tensor):
        """``log_betas``: [B, K] (same on every rank).  Returns (losses [B], d loss / d log_beta [B, K]) on every rank."""
        import torch.distributed as dist

        dev = self.graphed.device
        log_betas = log_betas.to(device=dev, dtype=torch.float32)
        B, K = log_betas.shape
        per = -(-B // self.world_size)                       # samples per rank, the last ones padded
        mine = torch.zeros(per, K + 1, device=dev)
        if self.batch:
            b = self.batch
            _, replays = ensemble_deal(B, self.world_size, self.rank, b)
            j0 = 0
            for chunk in replays:                             # chunk: up to b sample indices of this rank
                n = len(chunk)
                lb = log_betas[torch.tensor(chunk, device=dev)]
                if n < b:                                     # the last replay is padded with copies of its first row
                    lb = torch.cat([lb, lb[:1].expand(b - n, K)])
                loss, grads, _ = self.graphed(lb)
                mine[j0:j0 + n, 0] = loss[:n]
                mine[j0:j0 + n, 1:] = grads[:n]
                j0 += n
        for j in range(per if not self.batch else 0):
            i = j * self.world_size + self.rank               # round-robin: sample i goes to rank i % world_size
            if i >= B:
                break
            loss, grads, _ = self.graphed(log_betas[i])
            mine[j, 0] = loss
            mine[j, 1:] = grads
        if self.world_size > 1:
            every = [torch.empty_like(mine) for _ in range(self.world_size)]
            dist.all_gather(every, mine, group=self.group)
            table = torch.stack(every, dim=1).reshape(per * self.world_size, K + 1)[:B]   # [j, rank] -> i
        else:
            table = mine[:B]
        return table[:, 0].clone(), table[:, 1:].clone()


class Calibrator:
    """Gradient-based calibration of the networks' log-betas (SURVEY.md 8f rank 4: the consumer of the hot path).

    The reference's workflow (example_scripts/run_model.py:5-11; docs: fit log_beta by back-propagating a loss on the
    simulated time series) as a loop: every iteration is ONE replay of the captured window (forward T steps +
    backward, :class:`grad_june.graphed.GraphedRunner`) followed by a torch optimiser step on the log-beta vector.
    The Philox key is fixed per capture (common random numbers: the loss surface the optimiser walks is deterministic);
    ``reseed_every`` re-captures with a new key every so many iterations (stochastic optimisation over the noise).

        cal = Calibrator(runner, loss_fn=lambda r: ((r["cases_per_timestep"] - target) ** 2).mean())
        history = cal.fit(50)              # pandas DataFrame: iteration, loss, log_beta_<network>..., grad_<network>...
                                           # (fit_seed=True: also log_fraction_<label>..., grad_log_fraction_<label>...)
        cal.save(history)                  # <save_path>/calibration.csv + the reference's results.csv of the last run
    """

    def __init__(self, runner, loss_fn: Callable[[dict], torch.Tensor], networks: Optional[Sequence[str]] = None,
                 lr: float = 0.05, optimizer: str = "adam", seed: int = 0, reseed_every: int = 0, fit_seed: bool = False):
        """``fit_seed=True`` also calibrates the initial-case log-fractions (one national value, or one per region of
        ``runner.seed_labels``): they sit after the log-betas in the parameter vector."""
        self.runner = runner
        self.graphed = GraphedRunner(runner, loss_fn, networks=networks, seed=seed, fit_seed=fit_seed)
        self.names = self.graphed.names
        self.seed_names = self.graphed.seed_names
        dev = self.graphed.device
        self.log_beta = self.graphed.log_beta.detach().clone().requires_grad_(True)
        opt = {"adam": torch.optim.Adam, "sgd": torch.optim.SGD}[optimizer.lower()]
        self.optimizer = opt([self.log_beta], lr=lr)
        self.seed, self.reseed_every, self.iteration = int(seed), int(reseed_every), 0
        self.device = dev

    def step(self):
        """One iteration: replay at the current log-betas, optimiser step.  Returns (loss, log_beta before the step,
        gradient) as host floats / lists."""
        if self.reseed_every and self.iteration and self.iteration % self.reseed_every == 0:
            self.seed += 1
            self.graphed.recapture(self.seed)
        loss, grads, _ = self.graphed(self.log_beta.detach())
        before = self.log_beta.detach().cpu().tolist()
        self.log_beta.grad = grads.detach().clone()
        self.optimizer.step()
        self.iteration += 1
        return float(loss), before, grads.detach().cpu().tolist()

    def fit(self, n_iterations: int, callback=None):
        import pandas as pd
        rows = []
        for _ in range(n_iterations):
            loss, lb, grads = self.step()
            row = {"iteration": self.iteration, "loss": loss}
            K = len(self.names)
            row.update({f"log_beta_{k}": v for k, v in zip(self.names, lb)})
            row.update({f"grad_{k}": v for k, v in zip(self.names, grads)})
            row.update({f"log_fraction_{k}": v for k, v in zip(self.seed_names, lb[K:])})
            row.update({f"grad_log_fraction_{k}": v for k, v in zip(self.seed_names, grads[K:])})
            rows.append(row)
            if callback is not None:
                callback(row)
        return pd.DataFrame(rows).set_index("iteration")

    def save(self, history):
        """calibration.csv next to the reference's results.csv / results_is_infected.csv (runner.py:185-196) of the
        last evaluated window."""
        path = self.runner.save_path
        path.mkdir(exist_ok=True, parents=True)
        history.to_csv(path / "calibration.csv")
        self.runner.save_results(self.graphed.results, self.graphed.is_infected)
        return path
