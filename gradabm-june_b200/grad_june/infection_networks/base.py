"""Infection networks: bipartite agent<->group pressure per venue type.

Module interface of the reference's ``grad_june/infection_networks/base.py`` — ``<X>Network(log_beta,
device)``, ``InfectionNetworks(device=, **networks)``, ``nets[name].log_beta`` assignable after
construction, ``nets(data=, timer=, policies=) -> not_infected_probs`` — over the CSR kernels: the
scatter / normalise / gather / exp(-sum beta dt pressure) chain of base.py:61-87,118-141 is the
NETWORKS phase of ``gj_step_forward``; only the scalar beta_eff = 10**log_beta * policy factors is
formed here with ordinary autograd so that log_beta (and the policies' beta factors) stay leaves.
"""
import re

import torch
import yaml

from .. import ops
from ..paths import ensure_default_config
from ..world import get_device_world


class InfectionNetwork(torch.nn.Module):
    kind = ops.KIND_PLAIN

    def __init__(self, log_beta, device="cpu"):
        super().__init__()
        self.device = device
        self.log_beta = log_beta if type(log_beta) == torch.nn.Parameter else torch.tensor(float(log_beta))
        self.name = self._get_name()

    @classmethod
    def from_parameters(cls, params):
        return cls(device=params["system"]["device"], **params["networks"][cls._get_name()])

    @classmethod
    def _get_name(cls):
        return "_".join(re.findall("[A-Z][^A-Z]*", cls.__name__)[:-1]).lower()

    # which edge set / group table the network runs on (leisure classes share "leisure")
    def edge_type(self):
        return self.name

    def _get_edge_index(self, data):
        return data["attends_" + self.edge_type()].edge_index

    def _get_reverse_edge_index(self, data):
        return data["rev_attends_" + self.edge_type()].edge_index

    def _get_people_per_group(self, data):
        return data[self.edge_type()]["people"]

    def beta_eff(self, policies, timer):
        """Scalar 10**log_beta times the active interaction-policy factors (base.py:36-40)."""
        beta = 10.0 ** self.log_beta
        if policies is not None and policies.interaction_policies:
            beta = policies.interaction_policies.apply(beta=beta, name=self.name, timer=timer)
        return beta

    def _get_beta(self, policies, timer, data):
        n_groups = len(data[self.edge_type()]["id"])
        return self.beta_eff(policies, timer) * torch.ones(n_groups, device=self.device)

    def net_spec(self, prob_row=-1):
        return ops.NetSpec(name=self.name, edge_type=self.edge_type(), kind=self.kind, prob_row=prob_row)

    # ---- the reference's per-agent masking hooks (base.py:47-59).  The built-in classes' versions are what the
    # kernels evaluate in registers from `kind`; a USER SUBCLASS that overrides one of them (or `forward`) is detected
    # (`is_custom`) and its networks then run through the modular path: the hook's tensors are scattered / gathered by
    # the same CSR kernels without any built-in mask (`_custom_pressure`), and the step is sequenced module by module
    # like the reference's GradJune.forward instead of as one fused call.
    def _agent_mask(self, data, policies, timer):
        qp = None if policies is None else policies.quarantine_policies
        return qp.quarantine_mask if qp else 1.0

    def _get_transmissions(self, data, policies, timer):
        return self._agent_mask(data, policies, timer) * data["agent"].transmission

    def _get_susceptibilities(self, data, policies, timer):
        return self._agent_mask(data, policies, timer) * data["agent"].susceptibility

    def is_custom(self):
        hooks = ("_get_transmissions", "_get_susceptibilities", "_agent_mask", "forward", "_get_beta")
        for name in hooks:
            owner = next(k for k in type(self).__mro__ if name in k.__dict__)
            if owner.__module__.split(".")[0] != __name__.split(".")[0]:
                return True
        return False

    def _custom_pressure(self, data, timer, policies, venue=None):
        """base.py:61-84 with the hooks' own tensors: C_g = sum of T'_a * beta_eff * pc_g over the members, P_a = C_g(a)
        * s'_a, through the stand-alone NETWORKS phase with no built-in mask (differentiable with respect to T', s'
        and beta_eff)."""
        agent = data["agent"]
        dev = agent.susceptibility.device
        world = get_device_world(data, dev)
        Tm = self._get_transmissions(data, policies, timer)
        sm = self._get_susceptibilities(data, policies, timer)
        spec = ops.StepSpec(now=timer.now, dt=timer.duration, day_type=0 if timer.day_type == "weekday" else 1,
                            nets=[ops.NetSpec(name=self.name, edge_type=self.edge_type(), kind=ops.KIND_HOUSEHOLD)],
                            quarantine=None, phases=ops.PHASE_NETWORKS, want_reductions=False, want_lam=True)
        from ..partition import exchange_for

        static = ops.StepStatic(world=world, exchange=exchange_for(data, world))
        beta = self.beta_eff(policies, timer).reshape(1).to(device=dev, dtype=torch.float32)
        out = ops.infection_step(static, spec, beta, {"s": ops._f32(sm, dev)}, T_in=ops._f32(Tm, dev), venue=venue)
        return out["lam"]

    def forward(self, data, timer, policies, venue=None):
        """Pressure this network alone exerts on every agent (the reference's per-network output).  ``venue``
        (:class:`grad_june.ops.Venue` of one row): the regional venue factor of this network's groups."""
        if self.is_custom():
            return self._custom_pressure(data, timer, policies, venue)
        out = _run_networks([self], data, timer, policies, self.device, want_lam=True, venue=venue)
        return out["lam"]


class HouseholdNetwork(InfectionNetwork):
    kind = ops.KIND_HOUSEHOLD   # ignores the quarantine mask (base.py:144-149)

    def _agent_mask(self, data, policies, timer):
        return 1.0


class CareHomeNetwork(InfectionNetwork):
    pass


class SchoolNetwork(InfectionNetwork):
    pass


class CompanyNetwork(InfectionNetwork):
    pass


class UniversityNetwork(InfectionNetwork):
    pass


def _quarantine_thresholds(policies, timer):
    if policies is None or not policies.quarantine_policies:
        return None
    return policies.quarantine_policies.active_thresholds(timer)


def leisure_table(networks, device):
    """Stack the leisure networks' [2,2,100] attendance tables -> ([n,2,2,100] tensor, row per network)."""
    rows, tabs = {}, []
    for net in networks:
        if net.kind in (ops.KIND_LEISURE, ops.KIND_CARE_VISIT):
            rows[id(net)] = len(tabs)
            tabs.append(ops._f32(net.leisure_probabilities, torch.device(device)))
    return (torch.stack(tabs).contiguous() if tabs else None), rows


def _interaction_active(policies, timer):
    ip = None if policies is None else policies.interaction_policies
    return bool(ip) and any(pol.is_active(timer.date) for pol in ip.policies)


def beta_vector(networks, policies, timer, device):
    """[K] vector of beta_eff = 10**log_beta * policy factors (base.py:36-42), differentiable wrt every
    log_beta / factor tensor.  A batched ensemble (``Runner.batch = b``) holds b values per log_beta: the result is
    then [b, K]."""
    if not networks:
        return torch.zeros(0, device=device)
    device = torch.device(device)
    lbs = [net.log_beta for net in networks]
    nb = max((lb.numel() for lb in lbs if torch.is_tensor(lb)), default=1)
    if nb > 1:      # batched ensemble: networks that are not calibrated broadcast their scalar
        cols = [net.beta_eff(policies, timer).to(device=device, dtype=torch.float32).reshape(-1).expand(nb)
                for net in networks]
        return torch.stack(cols, dim=1).contiguous()
    if (not _interaction_active(policies, timer)
            and all(torch.is_tensor(lb) and lb.device == device and lb.dtype == torch.float32 for lb in lbs)):
        # every log_beta already lives on the step's device: one stack + one pow instead of K of each
        # (same elementwise powf as the per-scalar evaluation)
        return 10.0 ** torch.stack([lb.reshape(()) for lb in lbs])
    # log_beta usually lives on the CPU while policy factors follow system.device: move each scalar first
    return torch.stack([net.beta_eff(policies, timer).reshape(()).to(device=device, dtype=torch.float32)
                        for net in networks])


def _run_networks(networks, data, timer, policies, device, want_lam=False, region=None, venue=None):
    agent = data["agent"]
    ops.require_cuda(agent.susceptibility, "data['agent'].susceptibility")
    dev = agent.susceptibility.device
    world = get_device_world(data, dev)
    table, rows = leisure_table(networks, dev)
    specs = [net.net_spec(rows.get(id(net), -1)) for net in networks]
    day_type = 0 if timer.day_type == "weekday" else 1
    spec = ops.StepSpec(now=timer.now, dt=timer.duration, day_type=day_type, nets=specs,
                        quarantine=_quarantine_thresholds(policies, timer), phases=ops.PHASE_NETWORKS,
                        want_reductions=False, want_lam=want_lam)
    state = {"s": agent.susceptibility}
    if spec.quarantine:
        state["cur"] = agent["symptoms"]["current_stage"]
    from ..partition import exchange_for

    static = ops.StepStatic(world=world, leisure_prob=table, exchange=exchange_for(data, world))
    return ops.infection_step(static, spec, beta_vector(networks, policies, timer, dev), state,
                              T_in=agent.transmission, region=region, venue=venue)


class InfectionNetworks(torch.nn.Module):
    def __init__(self, device="cpu", **kwargs):
        super().__init__()
        self.networks = torch.nn.ModuleDict(kwargs)
        self.device = device

    def __getitem__(self, item):
        return self.networks[item]

    @classmethod
    def from_parameters(cls, params):
        from .. import infection_networks as _module

        device = params["system"]["device"]
        nets = {}
        for key in params["networks"]:
            cls_name = "".join(word.title() for word in key.split("_")) + "Network"
            nets[key] = getattr(_module, cls_name).from_parameters(params)
        return cls(device=device, **nets)

    @classmethod
    def from_file(cls, fpath=None):
        with open(fpath or ensure_default_config(), "r") as f:
            return cls.from_parameters(yaml.safe_load(f))

    def active_networks(self, timer, policies):
        """Networks of this step in accumulation order: activity hierarchy minus closed venues
        (base.py:128-133)."""
        order = timer.get_activity_order()
        if policies is not None and policies.close_venue_policies:
            order = policies.close_venue_policies.apply(edge_types=order, timer=timer)
        return [self.networks[name] for name in order]

    def has_custom(self, nets=None):
        return any(net.is_custom() for net in (self.networks.values() if nets is None else nets))

    def forward(self, data, timer, policies, region=None, venue=None):
        """not_infected_probs of the step.  ``region`` (:class:`grad_june.ops.Region`): every agent's summed pressure is
        multiplied by its region's factor before the clamp (the regional policies active at this step).  ``venue``
        (:class:`grad_june.ops.Venue`): the regional venue factors of the step's networks, row k for the k-th."""
        policies.apply(timer=timer, data=data)
        nets = self.active_networks(timer, policies)
        if not self.has_custom(nets):
            return _run_networks(nets, data, timer, policies, self.device, region=region, venue=venue)["q"]
        # a user-defined network among them: network by network in the activity order, then the reference's clamp /
        # exp chain (base.py:133-140) in torch
        agent = data["agent"]
        lam = torch.zeros_like(agent.susceptibility)
        for k, net in enumerate(nets):
            kw = {} if venue is None else {"venue": venue.row(k)}
            lam = lam + net(data=data, timer=timer, policies=policies, **kw)
        if region is not None:
            lam = lam * region.factor.to(lam.device)[region.labels.codes.long()]
        lam = torch.clamp(lam, min=1e-6, max=100)
        return torch.clamp(torch.exp(-lam * timer.duration), min=0.0, max=1.0)
