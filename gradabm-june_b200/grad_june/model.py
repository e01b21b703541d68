"""One simulation timestep (reference: grad_june/model.py).

``GradJune.forward(data, timer)`` keeps the reference's contract — it returns the same ``data`` object
with ``transmission``, ``susceptibility``, ``is_infected``, ``infection_time`` and the symptoms dict
replaced by new (differentiable) tensors — but runs the whole step (transmission update, infection
networks under the active policies, Gumbel-softmax draw, state update, symptoms) as one fused
forward of ``gj_step_forward`` with a hand-written backward, instead of ~430 torch ops.
"""
import torch
import yaml

from . import ops
from .infection import IsInfectedSampler
from .infection_networks import InfectionNetworks
from .infection_networks.base import _quarantine_thresholds, beta_vector, leisure_table
from .paths import ensure_default_config
from .policies import Policies
from .symptoms import SymptomsUpdater
from .transmission import TransmissionUpdater, profile_packed, profile_tensors
from .partition import exchange_for
from .world import get_device_world


class GradJune(torch.nn.Module):
    def __init__(self, symptoms_updater=None, policies=None, infection_networks=None, device="cpu"):
        super().__init__()
        self.symptoms_updater = SymptomsUpdater.from_file() if symptoms_updater is None else symptoms_updater
        self.policies = Policies.from_file() if policies is None else policies
        self.infection_networks = InfectionNetworks.from_file() if infection_networks is None else infection_networks
        self.transmission_updater = TransmissionUpdater()
        self.is_infected_sampler = IsInfectedSampler()
        self.device = device

    @classmethod
    def from_file(cls, fpath=None):
        with open(fpath or ensure_default_config(), "r") as f:
            return cls.from_parameters(yaml.safe_load(f))

    @classmethod
    def from_parameters(cls, params):
        return cls(
            symptoms_updater=SymptomsUpdater.from_parameters(params),
            policies=Policies.from_parameters(params),
            infection_networks=InfectionNetworks.from_parameters(params),
            device=params["system"]["device"],
        )

    def infect_people(self, data, timer, new_infected):
        """model.py:90-110 (maximum variant: the gradient splits 1/2-1/2 where s - n == 0)."""
        agent = data["agent"]
        agent.susceptibility = torch.maximum(torch.tensor(0.0, device=agent.susceptibility.device),
                                             agent.susceptibility - new_infected)
        agent.is_infected = agent.is_infected + new_infected
        agent.infection_time = agent.infection_time + new_infected * (timer.now - agent.infection_time)

    # ------------------------------------------------------------------------------------------
    def _static(self, data, device):
        """Per-world constants of the step, rebuilt only when the world, the profile parameters, a leisure
        table or the symptoms tables are replaced."""
        world = get_device_world(data, device)
        prof = profile_tensors(data)
        nets = list(self.infection_networks.networks.values())
        tables = tuple((id(t), t._version) for t in (getattr(net, "leisure_probabilities", None) for net in nets)
                       if t is not None)
        key = (id(world), id(prof[4]), tables, tuple(id(net) for net in nets),
               self.symptoms_updater.symptoms_sampler.tables_key())
        cache = data.__dict__.setdefault("_gj_cache", {})
        hit = cache.get("static")
        if hit is None or hit[0] != key:
            maxinf, shape, rate, shift, k0 = prof
            table, rows = leisure_table(nets, device)
            static = ops.StepStatic(world=world, maxinf=maxinf, shape=shape, rate=rate, shift=shift, k0=k0,
                                    prof4=profile_packed(data), leisure_prob=table,
                                    symptoms=self.symptoms_updater.symptoms_sampler.tables(device),
                                    exchange=exchange_for(data, world))
            cache["static"] = hit = (key, static, rows)
        return hit[1], hit[2]

    def _spec(self, timer, rows, age_bins, mode, want_probs):
        policies = self.policies
        if mode == ops.MODE_SEED:
            nets, phases = [], ops.PHASE_SAMPLE | ops.PHASE_INFECT | ops.PHASE_SYMPTOMS
        else:
            nets, phases = self.infection_networks.active_networks(timer, policies), ops.PHASE_ALL
        spec = ops.StepSpec(
            now=timer.now, dt=timer.duration, day_type=0 if timer.day_type == "weekday" else 1,
            nets=[net.net_spec(rows.get(id(net), -1)) for net in nets],
            quarantine=_quarantine_thresholds(policies, timer), phases=phases, mode=mode,
            age_bins=tuple(int(b) for b in age_bins) if age_bins is not None else (),
            want_reductions=age_bins is not None, want_probs=want_probs)
        return spec, nets

    def step(self, data, timer, age_bins=None, mode=ops.MODE_STEP, seed_fraction=None, noise=None, want_probs=True,
             next_timer=None, label=None, seed_label=None):
        """Fused step; returns (data, reductions) where reductions = [cases, deaths, cases by age bin...]
        (None unless ``age_bins`` is given).  With ``label`` (:class:`grad_june.ops.Labels`) it returns
        (data, reductions, label_table): the post-step cases and deaths per label column, [n, 2] ([b, n, 2] batched),
        reduced inside the step kernels.  ``want_probs=False`` skips the two diagnostic per-agent outputs
        (``not_infected_probs``, ``new_infected``) that the reference keeps only as locals of its forward.
        ``seed_label`` (:class:`grad_june.ops.SeedLabels`, seeding step only): ``seed_fraction`` holds one fraction per
        region and every agent is seeded with its region's.
        ``next_timer``: the timer as it will be at the FOLLOWING call (the driver knows the schedule): the
        kernels then run that step's transmission pass inside this one (used only if the next call matches)."""
        agent = data["agent"]
        ops.require_cuda(agent.susceptibility, "data['agent'].susceptibility")
        dev = agent.susceptibility.device
        if mode == ops.MODE_STEP and self.infection_networks.has_custom(
                self.infection_networks.active_networks(timer, self.policies)):
            return self._step_modular(data, timer, age_bins, label)
        static, rows = self._static(data, dev)
        policies = self.policies
        spec, nets = self._spec(timer, rows, age_bins, mode, want_probs)
        next_spec = None
        if next_timer is not None and mode == ops.MODE_STEP:
            next_spec, _ = self._spec(next_timer, rows, age_bins, ops.MODE_STEP, want_probs)
        sym = agent["symptoms"]
        state = {"s": agent.susceptibility, "inf": agent.is_infected, "tinf": agent.infection_time,
                 "cur": sym["current_stage"], "nxt": sym["next_stage"], "ttn": sym["time_to_next_stage"]}
        beta = beta_vector(nets, policies, timer, dev) if nets else None
        out = ops.infection_step(static, spec, beta, state, seed_fraction=seed_fraction, noise=noise,
                                 next_spec=next_spec, label=label, seed_label=seed_label)
        if out["T"] is not None:
            agent.transmission = out["T"]
        agent.susceptibility = out["s"]
        agent.is_infected = out["inf"]
        agent.infection_time = out["tinf"]
        sym["current_stage"] = out["cur"]
        sym["next_stage"] = out["nxt"]
        sym["time_to_next_stage"] = out["ttn"]
        if out["n"] is not None:
            data["agent"]["new_infected"] = out["n"]
        if out["q"] is not None:
            data["agent"]["not_infected_probs"] = out["q"]
        if label is not None:
            return data, out["red"], out["red_label"]
        return data, out["red"]

    def _step_modular(self, data, timer, age_bins, label=None):
        """The reference's own sequencing (model.py:112-144), module by module, for steps with a user-defined network
        subclass (its masking hooks return arbitrary tensors, which the fused kernels cannot evaluate in registers):
        every module is still a CUDA kernel of the library (stand-alone phases), only the fusion is lost."""
        agent = data["agent"]
        agent.transmission = self.transmission_updater(data=data, timer=timer)
        q = self.infection_networks(data=data, timer=timer, policies=self.policies)
        n = self.is_infected_sampler(q)
        self.infect_people(data, timer, n)
        self.symptoms_updater(data=data, timer=timer, new_infected=n)
        agent["new_infected"], agent["not_infected_probs"] = n, q
        red = None
        if age_bins is not None:      # runner.py:167-171,198-224
            cur, inf, age = agent.symptoms["current_stage"], agent.is_infected, agent.age
            dead = float(len(self.symptoms_updater.stages_ids) - 1)
            red = [inf.sum(), ((cur == dead) * cur / dead).sum()]
            red += [(inf * ((age < hi) * (age > lo))).sum() for lo, hi in zip(age_bins[:-1], age_bins[1:])]
            red = torch.stack(red)
        if label is not None:         # the label table as index_add of the same per-agent terms
            cur, inf = agent.symptoms["current_stage"], agent.is_infected
            dead = float(len(self.symptoms_updater.stages_ids) - 1)
            idx = label.codes.long()
            cases = torch.zeros(label.n, dtype=inf.dtype, device=inf.device).index_add(0, idx, inf)
            deaths = (cur == dead) * cur / dead
            deaths = torch.zeros(label.n, dtype=deaths.dtype, device=deaths.device).index_add(0, idx, deaths)
            return data, red, torch.stack((cases, deaths.to(cases.dtype)), dim=1)
        return data, red

    def kernel_family(self, data, timer) -> str:
        """"throughput" or "reference-order": the kernel family the fused step at ``timer`` runs on with in-kernel
        noise (the throughput kernels need the household edge type on the RANGE tier or unquarantined, the leisure
        type on the CELL tier and plain kinds elsewhere — what :func:`grad_june.world.renumber_world` arranges)."""
        dev = data["agent"].susceptibility.device
        if self.infection_networks.has_custom(self.infection_networks.active_networks(timer, self.policies)):
            return "modular (user-defined network)"
        static, rows = self._static(data, dev)
        spec, _ = self._spec(timer, rows, None, ops.MODE_STEP, False)
        return ops.step_plan(static, spec)

    def forward(self, data, timer):
        return self.step(data, timer)[0]
