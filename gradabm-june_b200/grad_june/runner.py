"""Simulation driver (reference: grad_june/runner.py).

Builds model, world and timer from the YAML parameters, keeps a backup of the initial state so that
``runner()`` can be re-run for every calibration iteration, seeds the initial cases and loops the
fused step.  The per-step result reductions (cases, differentiable deaths, cases by age bin —
runner.py:167-171,198-224) are produced inside the step kernel, so the loop issues no extra passes
over the agents.
"""
import copy
from pathlib import Path

import numpy as np
import pandas as pd
import torch
import yaml

from . import ops
from .model import GradJune
from .partition import all_reduce_sum, label_union
from .paths import ensure_default_config
from .timer import Timer
from .transmission import PROFILE_KEYS, TransmissionSampler
from .utils import read_path
from .world import load_world, original_order, renumber_world

_STATE_KEYS = ("susceptibility", "is_infected", "infection_time", "transmission")
_SYMPTOM_KEYS = ("current_stage", "next_stage", "time_to_next_stage")


def agent_labels(values, n_agents):
    """A per-agent label attribute (1-D torch / numpy array of integers or strings) as a numpy array of ``n_agents``
    entries; a one-element array applies to every agent."""
    a = values.detach().cpu().numpy() if torch.is_tensor(values) else np.asarray(values)
    if a.ndim != 1 or a.shape[0] not in (1, n_agents):
        raise ValueError(f"a label attribute must be a 1-D array of 1 or {n_agents} entries, got shape {a.shape}")
    return np.broadcast_to(a, (n_agents,)) if a.shape[0] == 1 else a


def label_codes(labels, columns):
    """Column of every label in the sorted ``columns``; a label that is not a column raises."""
    codes = np.searchsorted(columns, labels)
    hit = codes < len(columns)
    hit[hit] = columns[codes[hit]] == labels[hit]
    if not hit.all():
        raise ValueError(f"label {labels[~hit][0]!r} is not one of the result columns")
    return codes


def seed_log_fractions(mapping, labels):
    """A per-region log-fraction mapping ``{label: value, ..., "default": value}`` (the YAML form) as a list in the
    order of the sorted ``labels``.  Labels the mapping does not list take ``default``; a label in the mapping that no
    agent carries raises, and so does a missing ``default`` when some label is not listed."""
    mapping = dict(mapping)
    default = mapping.pop("default", None)
    labels = np.asarray(labels)
    out = [None] * len(labels)
    for key, value in mapping.items():
        if labels.dtype.kind in "iu" and not isinstance(key, (int, np.integer)):
            try:
                key = int(key)
            except (TypeError, ValueError):
                raise ValueError(f"seeding: label {key!r} is not carried by any agent") from None
        elif labels.dtype.kind in "US" and not isinstance(key, str):
            key = str(key)
        i = int(np.searchsorted(labels, key))
        if i >= len(labels) or labels[i] != key:
            raise ValueError(f"seeding: label {key!r} is not carried by any agent")
        out[i] = float(value)
    missing = [labels[i] for i, v in enumerate(out) if v is None]
    if missing and default is None:
        raise ValueError(f"seeding: no log-fraction for label {missing[0]!r} and no 'default'")
    return [float(default) if v is None else v for v in out]


class Runner(torch.nn.Module):
    def __init__(self, model, data, timer, log_fraction_initial_cases, save_path, parameters,
                 age_bins=(0, 18, 65, 100), results_by=None, seed_by=None):
        """``seed_by`` (``infection_seed: {by: super_area}`` in the YAML): seed the initial cases per value of
        ``data["agent"][seed_by]`` (``runner.seed_labels``, the sorted distinct values over every rank of a partitioned
        world).  ``log_fraction_initial_cases`` is then a scalar (every region), a list or tensor of one value per
        region in ``seed_labels`` order ([b, R] or [R] when ``runner.batch = b``; may be an ``nn.Parameter``: the
        gradient reaches every region), or a mapping ``{label: value, "default": value}``.  A region's fraction below
        about 2^-24 (log-fraction < -7.2) rounds its q = 1 - fraction to exactly 1 in fp32: none of its agents is
        infected, and its gradient is NaN (the sampler's d/dq divides 0 by 0, as the reference's torch code does);
        the other regions' gradients are unaffected."""
        super().__init__()
        self.model = model
        self.data = data
        self.data_backup = self.backup_infection_data(data)
        self.timer = timer
        self.log_fraction_initial_cases = log_fraction_initial_cases
        self.device = model.device
        self.age_bins = torch.tensor(age_bins, device=self.device)
        self._age_bins_host = tuple(int(b) for b in age_bins)
        self.ethnicities = np.sort(np.unique(data["agent"].ethnicity))
        self.n_agents = data["agent"].id.shape[0]
        self.population_by_age = self.get_people_by_age()
        self.save_path = Path(save_path)
        self.input_parameters = parameters
        # results by label (``results_by: super_area``): cases and deaths per value of data["agent"][results_by] and
        # timestep, reduced inside the step kernels.  The columns are the sorted distinct values, over every rank of a
        # partitioned world.
        self.results_by = results_by
        self.result_labels = None
        if results_by is not None:
            labels = agent_labels(data["agent"][results_by], self.n_agents)
            self.result_labels = label_union(np.unique(labels), data.__dict__.get("_gj_partition"))
        # seeding by label: one initial-case fraction per value of data["agent"][seed_by]
        self.seed_by = seed_by
        self.seed_labels = None
        if seed_by is not None:
            if seed_by == results_by:
                self.seed_labels = self.result_labels
            else:
                labels = agent_labels(data["agent"][seed_by], self.n_agents)
                self.seed_labels = label_union(np.unique(labels), data.__dict__.get("_gj_partition"))
            if isinstance(log_fraction_initial_cases, dict):
                log_fraction_initial_cases = seed_log_fractions(log_fraction_initial_cases, self.seed_labels)
            self.log_fraction_initial_cases = log_fraction_initial_cases
            self._seed_fraction_shape(log_fraction_initial_cases)
        elif isinstance(log_fraction_initial_cases, dict):
            raise ValueError("a per-region log_fraction_initial_cases mapping needs infection_seed.by (seed_by)")
        # batched ensemble (SURVEY 8e-2): ``runner.batch = b`` makes ``forward()`` step b independent samples of the
        # epidemic at once — the networks' ``log_beta`` then hold b values each, the state tensors are [b, Np] and
        # every result series is [T+1, b].  All samples draw the same noise (common random numbers).
        self.batch = None
        self.restore_initial_data()

    @classmethod
    def from_file(cls, fpath=None):
        with open(fpath or ensure_default_config(), "r") as f:
            return cls.from_parameters(yaml.safe_load(f))

    @classmethod
    def from_parameters(cls, params):
        return cls(
            model=GradJune.from_parameters(params),
            data=cls.get_data(params),
            timer=Timer.from_parameters(params),
            log_fraction_initial_cases=params["infection_seed"]["log_fraction_initial_cases"],
            save_path=params["save_path"],
            parameters=params,
            age_bins=params.get("age_bins_to_save", (0, 18, 65, 100)),
            results_by=params.get("results_by"),
            seed_by=params["infection_seed"].get("by"),
        )

    @staticmethod
    def get_data(params, data=None):
        """World + freshly sampled per-agent profile parameters + initial state (runner.py:65-91).
        ``data`` may be passed directly instead of ``params['data_path']`` (synthetic worlds)."""
        device = params["system"]["device"]
        if data is None:
            data = load_world(read_path(params["data_path"]))
        data = data.to(device)
        # Worlds arrive numbered as the reference's loaders number them (by area and age): renumber the agents
        # household-contiguous inside their leisure cell so that the streaming layout tiers apply
        # (world.layout_order).  ``data["agent"].original_index`` keeps the loaded numbering; the noise stream is
        # keyed by it and ``Runner.forward`` returns ``is_infected`` in it.  ``system: {renumber_agents: false}``
        # keeps the loaded numbering (one part of a partitioned world is never renumbered on its own).
        if params["system"].get("renumber_agents", True) and "_gj_partition" not in data.__dict__ \
                and "_gj_block" not in data.__dict__:
            data = renumber_world(data)
        n_agents = len(data["agent"]["id"])
        values = TransmissionSampler.from_parameters(params)(n_agents)
        if "original_index" in data["agent"] and "_gj_partition" not in data.__dict__:
            values = values[:, data["agent"]["original_index"]]     # drawn per ORIGINAL agent: independent of the layout
        data["agent"].infection_parameters = {key: values[i, :].contiguous() for i, key in enumerate(PROFILE_KEYS)}
        data["agent"].transmission = torch.zeros(n_agents, device=device)
        data["agent"].susceptibility = torch.ones(n_agents, device=device)
        data["agent"].is_infected = torch.zeros(n_agents, device=device)
        data["agent"].infection_time = torch.zeros(n_agents, device=device)
        data["agent"].symptoms = {
            "current_stage": torch.ones(n_agents, dtype=torch.long, device=device),
            "next_stage": torch.ones(n_agents, dtype=torch.long, device=device),
            "time_to_next_stage": torch.zeros(n_agents, device=device),
        }
        return data

    def backup_infection_data(self, data):
        agent = data["agent"]
        backup = {key: agent[key].detach().clone() for key in _STATE_KEYS}
        backup["symptoms"] = {key: agent["symptoms"][key].detach().clone() for key in _SYMPTOM_KEYS}
        return backup

    def restore_initial_data(self):
        agent = self.data["agent"]
        for key in _STATE_KEYS:
            agent[key] = self.data_backup[key].detach().clone()
        for key in _SYMPTOM_KEYS:
            agent.symptoms[key] = self.data_backup["symptoms"][key].detach().clone()
        self.data["results"] = {"deaths_per_timestep": None}

    def _restore_for_window(self):
        """``restore_initial_data`` for ``forward()``: the fused step never writes its inputs in place, so the window
        can START from the backup tensors themselves instead of clones of them, with the stage arrays already in the
        fp32 the kernels read (the reference's initial stages are int64 ones; same values).  At 56 M agents this
        saves ~5 GB of copies and dtype conversions per window.  The backup is re-read (identity check) if the user
        replaced it."""
        key = tuple(id(self.data_backup[k]) for k in _STATE_KEYS) + \
            tuple((id(self.data_backup["symptoms"][k]), self.data_backup["symptoms"][k]._version) for k in _SYMPTOM_KEYS)
        key = key + (self.batch,)
        hit = self.__dict__.get("_window_start")
        if hit is None or hit[0] != key:
            state = {k: self.data_backup[k].detach() for k in _STATE_KEYS}
            sym = {k: self.data_backup["symptoms"][k].detach().to(torch.float32) for k in _SYMPTOM_KEYS}
            if self.batch:      # b copies of the initial state, rows padded to a multiple of four agents
                n = self.n_agents
                n_pad = (n + 3) // 4 * 4

                def rows(t):
                    out = torch.zeros(self.batch, n_pad, dtype=torch.float32, device=t.device)
                    out[:, :n] = t.to(torch.float32)
                    return out

                state = {k: rows(v) for k, v in state.items()}
                sym = {k: rows(v) for k, v in sym.items()}
            hit = self.__dict__["_window_start"] = (key, state, sym)
        agent = self.data["agent"]
        for k in _STATE_KEYS:
            agent[k] = hit[1][k]
        agent.symptoms = dict(hit[2])
        self.data["results"] = {"deaths_per_timestep": None}

    def _seed_fraction_shape(self, value):
        """Check a per-region log-fraction's shape; returns the number of values it holds per sample."""
        R = len(self.seed_labels)
        shape = tuple(value.shape) if torch.is_tensor(value) else np.shape(value)
        batch = self.__dict__.get("batch")
        if shape in ((), (1,), (R,)) or (batch and shape == (batch, R)):
            return R
        raise ValueError(f"seeding by {self.seed_by!r}: log_fraction_initial_cases must be a scalar or hold one value "
                         f"per region ({R}, or [b, {R}] batched), got shape {shape}")

    def _fraction_tensor(self):
        if self.seed_by is not None:
            return self._seed_fraction_tensor()
        fraction = 10.0 ** self.log_fraction_initial_cases
        dev = self.data["agent"].susceptibility.device
        if not torch.is_tensor(fraction):
            # a plain number: keep its device copy (no host-to-device copy per run; CUDA-graph capturable)
            key = (float(fraction), str(dev))
            if getattr(self, "_fraction_cache", (None, None))[0] != key:
                self._fraction_cache = (key, torch.tensor([float(fraction)], dtype=torch.float32).to(dev))
            return self._fraction_cache[1]
        return fraction.reshape(-1).to(device=dev, dtype=torch.float32)   # [1], or [b] per sample

    def _seed_fraction_tensor(self):
        """The per-region fractions 10^log_fraction on the device: [R] ([b, R] for a per-sample batch)."""
        lf = self.log_fraction_initial_cases
        R = len(self.seed_labels)
        self._seed_fraction_shape(lf)
        dev = self.data["agent"].susceptibility.device
        if not torch.is_tensor(lf):
            # plain numbers: evaluated like the national scalar (host fp64, then fp32), the device copy kept
            vals = np.broadcast_to(np.asarray(lf, dtype=np.float64), (R,) if np.ndim(lf) < 2 else np.shape(lf))
            key = (tuple(float(10.0 ** v) for v in vals.reshape(-1)), vals.shape, str(dev))
            if getattr(self, "_seed_fraction_cache", (None, None))[0] != key:
                self._seed_fraction_cache = (key, torch.tensor(key[0], dtype=torch.float32).reshape(vals.shape).to(dev))
            return self._seed_fraction_cache[1]
        fraction = (10.0 ** lf).to(device=dev, dtype=torch.float32)
        if fraction.numel() == 1:
            fraction = fraction.reshape(1).expand(R)
        return fraction.contiguous()

    def _seed_label_codes(self):
        """ops.SeedLabels of ``seed_by`` on the device (built once per label array and device; shares the device codes
        of ``results_by`` when both name the same attribute), or None."""
        if self.seed_by is None:
            return None
        values = self.data["agent"][self.seed_by]
        dev = self.data["agent"].susceptibility.device
        hit = self.__dict__.get("_seed_codes")
        if hit is None or hit[0] is not values or hit[1] != dev:
            if self.seed_by == self.results_by:
                codes = self._labels().codes
            else:
                codes = label_codes(agent_labels(values, self.n_agents), self.seed_labels)
            hit = self.__dict__["_seed_codes"] = (values, dev, ops.make_seed_labels(codes, len(self.seed_labels), dev))
        return hit[2]

    def _labels(self):
        """ops.Labels of ``results_by`` on the device (built once per label array and device, like
        ``_ethnicity_codes``), or None."""
        if self.results_by is None:
            return None
        values = self.data["agent"][self.results_by]
        dev = self.data["agent"].susceptibility.device
        hit = self.__dict__.get("_label_codes")
        if hit is None or hit[0] is not values or hit[1] != dev:
            codes = label_codes(agent_labels(values, self.n_agents), self.result_labels)
            hit = self.__dict__["_label_codes"] = (values, dev, ops.make_labels(codes, len(self.result_labels), dev))
        return hit[2]

    def set_initial_cases(self):
        """infect_fraction_of_people + first symptoms update (runner.py:138-149) as one fused call (with
        ``results_by``: returns (reductions, label table))."""
        out = self.model.step(self.data, self.timer, age_bins=self._age_bins_host, mode=ops.MODE_SEED,
                              seed_fraction=self._fraction_tensor(), label=self._labels(),
                              seed_label=self._seed_label_codes())
        return out[1] if self.results_by is None else out[1:]

    def forward(self):
        timer, model, data = self.timer, self.model, self.data
        timer.reset()
        if self.data["agent"].susceptibility.is_cuda:
            self._restore_for_window()
        elif self.batch:
            raise RuntimeError("batched ensembles run on a CUDA device only")
        else:
            self.restore_initial_data()
        label = self._labels()
        reds, tabs = [], []
        first = self.set_initial_cases()
        if label is None:
            reds.append(first)
        else:
            reds.append(first[0])
            tabs.append(first[1])
        dates = [timer.date]
        while timer.date < timer.final_date:
            next(timer)
            ahead = None
            if timer.date < timer.final_date:      # the schedule is known: tell the step what the next one will be
                ahead = copy.copy(timer)
                next(ahead)
            out = model.step(data, timer, age_bins=self._age_bins_host, want_probs=False, next_timer=ahead, label=label)
            data = out[0]
            reds.append(out[1])
            if label is not None:
                tabs.append(out[2])
            dates.append(timer.date)
        part = data.__dict__.get("_gj_partition")
        table = torch.stack(reds)                      # [T+1, 2 + n_bins]   (batched: [T+1, b, 2 + n_bins])
        table = all_reduce_sum(table, part)            # partitioned world: sum over ranks
        ex = data.__dict__.get("_gj_cache", {}).get("exchange")
        if ex is not None and not torch.cuda.is_current_stream_capturing():
            ex.check()      # a peer that never arrived at an exchange must not go unnoticed (once per window)
        cases_per_timestep = table[..., 0]
        data["results"]["deaths_per_timestep"] = table[..., 1]
        results = {
            "dates": dates,
            "cases_per_timestep": cases_per_timestep,
            "daily_cases_per_timestep": torch.diff(
                cases_per_timestep, dim=0, prepend=torch.zeros_like(cases_per_timestep[:1])),
            "deaths_per_timestep": data["results"]["deaths_per_timestep"],
        }
        for i, key in enumerate(self._age_bins_host[1:]):
            results[f"cases_by_age_{key:02d}"] = table[..., 2 + i]
        if label is not None:
            by = all_reduce_sum(torch.stack(tabs), part)   # [T+1, R, 2]   (batched: [T+1, b, R, 2])
            results[f"cases_by_{self.results_by}"] = by[..., 0]
            results[f"deaths_by_{self.results_by}"] = by[..., 1]
        is_infected = data["agent"].is_infected
        if is_infected.dim() == 2:                      # batched: [b, Np] -> [b, n_agents] in the loaded order
            is_infected = original_order(data, is_infected[:, : self.n_agents].t()).t()
            return results, is_infected
        return results, original_order(data, is_infected)

    def save_results(self, results, is_infected):
        self.save_path.mkdir(exist_ok=True, parents=True)
        by = () if self.results_by is None else (f"cases_by_{self.results_by}", f"deaths_by_{self.results_by}")
        df = pd.DataFrame(index=results["dates"])
        df.index.name = "date"
        for key, value in results.items():
            if key != "dates" and key not in by:
                df[key] = value.detach().cpu().numpy()
        df.to_csv(self.save_path / "results.csv")
        if by:      # long format: one row per (date, label)
            cases, deaths = (results[k].detach().cpu().numpy() for k in by)
            n_dates, n_labels = cases.shape
            pd.DataFrame({"date": np.repeat(np.asarray(results["dates"]), n_labels),
                          "label": np.tile(self.result_labels, n_dates),
                          "cases": cases.reshape(-1), "deaths": deaths.reshape(-1)}).to_csv(
                self.save_path / f"results_by_{self.results_by}.csv", index=False)
        pd.DataFrame({"is_infected": is_infected.detach().cpu().numpy()}).to_csv(
            self.save_path / "results_is_infected.csv")

    # --- reference helper reductions, kept for API parity (runner.py:198-242) ----------------------
    def store_differentiable_deaths(self, data):
        symptoms = data["agent"].symptoms
        dead = self.model.symptoms_updater.stages_ids[-1]
        deaths = ((symptoms["current_stage"] == dead) * symptoms["current_stage"] / dead).sum()
        prev = data["results"]["deaths_per_timestep"]
        data["results"]["deaths_per_timestep"] = deaths if prev is None else torch.hstack((prev, deaths))

    def _age_mask(self, i):
        age = self.data["agent"].age
        return (age < self.age_bins[i]) * (age > self.age_bins[i - 1])

    def get_cases_by_age(self, data):
        ret = torch.zeros(self.age_bins.shape[0] - 1, device=self.device)
        for i in range(1, self.age_bins.shape[0]):
            ret[i - 1] = (data["agent"].is_infected * self._age_mask(i)).sum()
        return ret

    def get_people_by_age(self):
        return {int(self.age_bins[i].item()): self._age_mask(i).sum() for i in range(1, self.age_bins.shape[0])}

    def get_cases_by_ethnicity(self, data):
        """runner.py:226-242, in one pass on the device: the per-agent ethnicity code is built once (the reference
        rebuilds a boolean mask from the numpy strings per ethnicity and call), the sums are one index_add —
        differentiable with respect to is_infected like the reference's masked sums."""
        agent = data["agent"]
        eth = agent.ethnicity
        hit = self.__dict__.get("_ethnicity_codes")
        if hit is None or hit[0] is not eth or hit[2] != agent.is_infected.device:
            labels = np.asarray(eth)
            n = agent.is_infected.shape[0]
            if labels.shape[0] != n:             # synthetic worlds carry one label for everybody
                labels = np.broadcast_to(labels[:1], (n,))
            codes = np.searchsorted(self.ethnicities, labels)
            hit = self.__dict__["_ethnicity_codes"] = (eth, torch.as_tensor(codes, dtype=torch.long).to(
                agent.is_infected.device), agent.is_infected.device)
        ret = torch.zeros(len(self.ethnicities), device=agent.is_infected.device, dtype=agent.is_infected.dtype)
        return ret.index_add(0, hit[1], agent.is_infected)
