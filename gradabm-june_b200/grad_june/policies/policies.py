"""Time-windowed policies (host side).

Only the date-window logic and the scalar beta multipliers live here; their effect on the per-agent
arithmetic (quarantine mask, closed venues, scaled beta) is applied inside the CUDA step kernels
from the scalars these classes produce.  Interface mirrors grad_june/policies/policies.py.
"""
import datetime

import torch
import yaml

from ..paths import ensure_default_config
from ..utils import read_date


class Policy(torch.nn.Module):
    def __init__(self, start_date, end_date, device):
        super().__init__()
        self.start_date = read_date(start_date)
        self.end_date = read_date(end_date)
        self.device = device

    def apply(self):
        raise NotImplementedError

    def is_active(self, date: datetime.datetime) -> bool:
        """Active on the half-open window [start_date, end_date)."""
        return self.start_date <= date < self.end_date


class PolicyCollection(torch.nn.Module):
    """Policies of one kind; truthy even when empty (nn.Module has no __len__), like the reference."""

    def __init__(self, policies):
        super().__init__()
        self.policies = torch.nn.ModuleList(policies)

    def __getitem__(self, idx):
        return self.policies[idx]


def _camel(name):
    return "".join(part.capitalize() or "_" for part in name.split("_"))


class Policies(torch.nn.Module):
    def __init__(self, interaction_policies=None, quarantine_policies=None, close_venue_policies=None,
                 regional_policies=None, venue_policies=None):
        super().__init__()
        self.interaction_policies = interaction_policies
        self.quarantine_policies = quarantine_policies
        self.close_venue_policies = close_venue_policies
        self.regional_policies = regional_policies
        self.venue_policies = venue_policies
        if regional_policies is not None:
            regional_policies.by()   # one region attribute per run
        if venue_policies is not None:
            venue_policies.by()

    @classmethod
    def from_policy_list(cls, policies):
        from . import CloseVenuePolicies, InteractionPolicies, QuarantinePolicies, RegionalPolicies, VenuePolicies

        policies = [] if policies is None else policies
        return cls(
            interaction_policies=InteractionPolicies(cls._get_policies_by_type(policies, "interaction")),
            quarantine_policies=QuarantinePolicies(cls._get_policies_by_type(policies, "quarantine")),
            close_venue_policies=CloseVenuePolicies(cls._get_policies_by_type(policies, "close_venue")),
            regional_policies=RegionalPolicies(cls._get_policies_by_type(policies, "regional")),
            venue_policies=VenuePolicies(cls._get_policies_by_type(policies, "venue")),
        )

    @classmethod
    def from_file(cls, fpath=None):
        with open(fpath or ensure_default_config(), "r") as f:
            return cls.from_parameters(yaml.safe_load(f))

    @classmethod
    def from_parameters(cls, params):
        device = params["system"]["device"]
        found = []
        for collection in params.get("policies", {}).values():
            for name, config in collection.items():
                found += cls._parse_policy_config(config, name=name, device=device)
        return cls.from_policy_list(found)

    @staticmethod
    def _parse_policy_config(config, name, device):
        from .. import policies as _module

        policy_class = getattr(_module, _camel(name))
        if "start_date" in config:
            return [policy_class(**config, device=device)]
        out = []
        for entry in config.values():
            if "start_date" not in entry or "end_date" not in entry:
                raise ValueError("policy config file not valid.")
            out.append(policy_class(**entry, device=device))
        return out

    @classmethod
    def _get_policies_by_type(cls, policies, type):
        return [p for p in policies if p.spec == type]

    def apply(self, data, timer):
        if self.quarantine_policies:
            self.quarantine_policies.apply(
                timer=timer, symptom_stages=data["agent"]["symptoms"]["current_stage"]
            )
