"""Regional social distancing: a per-region multiplier on every agent's force of infection.

While a ``RegionalSocialDistancing`` policy is active, agent a's summed pressure over the active networks is multiplied
by the factor of its region (the value of ``data["agent"][by]``) before the clamp.  The factor belongs to the receiving
agent's region and applies to every venue type: it models the region's compliance, not a venue's.  The factors of all
regional policies active at a step multiply.  The runner resolves the regions (``Runner.region_labels``) and passes
the product to the step kernels; see ``Runner`` and ``GradJune.step(region=...)``.
"""
import numpy as np
import torch

from .policies import Policy, PolicyCollection


class RegionalPolicy(Policy):
    spec = "regional"


class RegionalSocialDistancing(RegionalPolicy):
    """Active on ``[start_date, end_date)``; ``by`` names the per-agent region attribute (e.g. ``super_area``).
    ``beta_factors`` is a scalar (every region), a mapping ``{label: factor, ..., "default": factor}`` (the YAML
    form), or an [R] tensor in ``Runner.region_labels`` order ([b, R] batched; an ``nn.Parameter`` to fit it with
    autograd).  Factors must be >= 0."""

    def __init__(self, start_date, end_date, by, beta_factors, device):
        super().__init__(start_date=start_date, end_date=end_date, device=device)
        if not isinstance(by, str) or not by:
            raise ValueError(f"regional_social_distancing: 'by' must name an agent attribute, got {by!r}")
        self.by = by
        if torch.is_tensor(beta_factors):
            if beta_factors.dim() > 2 or bool((beta_factors.detach() < 0).any()):
                raise ValueError("regional_social_distancing: beta_factors must be >= 0 and hold [R] or [b, R] values")
        elif isinstance(beta_factors, dict):
            for key, value in beta_factors.items():
                _check_factor(value, key)
        elif np.ndim(beta_factors) == 0:
            _check_factor(beta_factors, "all")
        else:
            vals = np.asarray(beta_factors, dtype=np.float64)
            if vals.ndim > 2 or (vals < 0).any():
                raise ValueError("regional_social_distancing: beta_factors must be >= 0 and hold [R] or [b, R] values")
        self.beta_factors = beta_factors

    def factors(self, labels, device, batch=None):
        """The factor of every region of the sorted ``labels`` as an fp32 tensor on ``device``: [R], or [b, R] for a
        per-sample tensor of a batch of ``b``.  Differentiable with respect to a tensor ``beta_factors``."""
        from ..runner import seed_log_fractions

        R = len(labels)
        f = self.beta_factors
        if isinstance(f, dict):
            f = seed_log_fractions(f, labels, what="regional_social_distancing", value="factor")
        if torch.is_tensor(f):
            shape = tuple(f.shape)
            if shape not in ((), (1,), (R,)) and not (batch and shape == (batch, R)):
                raise ValueError(f"regional_social_distancing by {self.by!r}: beta_factors must be a scalar or hold one "
                                 f"value per region ({R}, or [b, {R}] batched), got shape {shape}")
            f = f.to(device=device, dtype=torch.float32)
            return f.reshape(1).expand(R) if f.numel() == 1 else f
        vals = np.asarray(f, dtype=np.float64)
        if vals.shape not in ((), (1,), (R,)) and not (batch and vals.shape == (batch, R)):
            raise ValueError(f"regional_social_distancing by {self.by!r}: beta_factors must be a scalar or hold one "
                             f"value per region ({R}, or [b, {R}] batched), got shape {vals.shape}")
        key = (vals.tobytes(), vals.shape, R, str(device))
        hit = self.__dict__.get("_factor_cache")
        if hit is None or hit[0] != key:
            t = torch.tensor(np.broadcast_to(vals, (R,)) if vals.ndim < 2 else vals, dtype=torch.float32).to(device)
            hit = self.__dict__["_factor_cache"] = (key, t)
        return hit[1]


def _check_factor(value, label, what="regional_social_distancing"):
    try:
        v = float(value)
    except (TypeError, ValueError):
        raise ValueError(f"{what}: factor of {label!r} is not a number: {value!r}") from None
    if not v >= 0.0:
        raise ValueError(f"{what}: factor of {label!r} must be >= 0, got {value!r}")


class RegionalPolicies(PolicyCollection):
    def by(self):
        """The region attribute of the regional policies (None without any); two different attributes raise."""
        names = {policy.by for policy in self.policies}
        if len(names) > 1:
            raise ValueError(f"every regional policy of a run must use the same 'by', got {sorted(names)}")
        return names.pop() if names else None

    def active(self, timer):
        return [policy for policy in self.policies if policy.is_active(timer.date)]

    def factor(self, timer, labels, device, batch=None):
        """Elementwise product of the factors of the policies active at ``timer`` ([R] or [b, R]), or None."""
        out = None
        for policy in self.active(timer):
            f = policy.factors(labels, device, batch)
            out = f if out is None else out * f
        return out


class VenuePolicy(Policy):
    spec = "venue"


class RegionalVenueDistancing(VenuePolicy):
    """Regional venue restrictions: while active (``[start_date, end_date)``), network k's beta at a group is multiplied
    by the factor of the group's region (the value of ``data[<edge type>][by]``, or the majority of its members' when
    the group carries none; see :func:`grad_june.world.group_labels`).  The factor belongs to the venue's location, not
    to the visitor's home, and a factor of 0 closes that venue type in that region.

    ``beta_factors`` maps a network name, or ``all`` (every network but ``household``), to a scalar, a mapping
    ``{label: factor, ..., "default": factor}`` (the YAML form, parsed like the per-region seed values) or an [R]
    tensor in ``Runner.venue_labels`` order ([b, R] batched; an ``nn.Parameter`` to fit it).  A network takes its
    own entry, else ``all``, else 1.  Factors must be >= 0.  Households, and any other network whose edge type runs on
    the RANGE tier, have no per-group pass: use :class:`RegionalSocialDistancing` for them."""

    def __init__(self, start_date, end_date, by, beta_factors, device):
        super().__init__(start_date=start_date, end_date=end_date, device=device)
        if not isinstance(by, str) or not by:
            raise ValueError(f"regional_venue_distancing: 'by' must name a group attribute, got {by!r}")
        if not isinstance(beta_factors, dict) or not beta_factors:
            raise ValueError("regional_venue_distancing: beta_factors must map network names (or 'all') to factors")
        if "household" in beta_factors:
            raise ValueError("regional_venue_distancing: households have no per-venue pass; use "
                             "regional_social_distancing for them")
        self.by = by
        self.beta_factors = {}
        for name, f in beta_factors.items():
            _check_venue_entry(name, f)
            self.beta_factors[str(name)] = f
        # nn.Parameter entries registered so that .parameters() finds them
        self._params = torch.nn.ParameterDict({k: v for k, v in self.beta_factors.items()
                                               if isinstance(v, torch.nn.Parameter)})

    def entry(self, name):
        """The entry that applies to network ``name`` (its own, else ``all`` unless it is the household network), or
        None (factor 1)."""
        if name in self.beta_factors:
            return name
        if name != "household" and "all" in self.beta_factors:
            return "all"
        return None

    def factors(self, key, labels, device, batch=None):
        """Entry ``key``'s factor of every region of the sorted ``labels`` as an fp32 tensor on ``device``: [R], or
        [b, R] for a per-sample tensor of a batch of ``b``.  Differentiable with respect to a tensor entry."""
        from ..runner import seed_log_fractions

        R = len(labels)
        f = self.beta_factors[key]
        what = f"regional_venue_distancing ({key})"
        if isinstance(f, dict):
            f = seed_log_fractions(f, labels, what=what, value="factor")
        if torch.is_tensor(f):
            shape = tuple(f.shape)
            if shape not in ((), (1,), (R,)) and not (batch and shape == (batch, R)):
                raise ValueError(f"{what} by {self.by!r}: a factor must be a scalar or hold one value per region "
                                 f"({R}, or [b, {R}] batched), got shape {shape}")
            f = f.to(device=device, dtype=torch.float32)
            return f.reshape(1).expand(R) if f.numel() == 1 else f
        vals = np.asarray(f, dtype=np.float64)
        if vals.shape not in ((), (1,), (R,)) and not (batch and vals.shape == (batch, R)):
            raise ValueError(f"{what} by {self.by!r}: a factor must be a scalar or hold one value per region "
                             f"({R}, or [b, {R}] batched), got shape {vals.shape}")
        cache = self.__dict__.setdefault("_factor_cache", {})
        ck = (key, vals.tobytes(), vals.shape, R, str(device))
        t = cache.get(key)
        if t is None or t[0] != ck:
            t = cache[key] = (ck, torch.tensor(np.broadcast_to(vals, (R,)) if vals.ndim < 2 else vals,
                                               dtype=torch.float32).to(device))
        return t[1]


def _check_venue_entry(name, f):
    what = f"regional_venue_distancing ({name})"
    if torch.is_tensor(f):
        if f.dim() > 2 or bool((f.detach() < 0).any()):
            raise ValueError(f"{what}: factors must be >= 0 and hold [R] or [b, R] values")
    elif isinstance(f, dict):
        for key, value in f.items():
            _check_factor(value, key, what)
    elif np.ndim(f) == 0:
        _check_factor(f, "all", what)
    else:
        vals = np.asarray(f, dtype=np.float64)
        if vals.ndim > 2 or (vals < 0).any():
            raise ValueError(f"{what}: factors must be >= 0 and hold [R] or [b, R] values")


class VenuePolicies(PolicyCollection):
    def by(self):
        """The group attribute of the venue policies (None without any); two different attributes raise."""
        names = {policy.by for policy in self.policies}
        if len(names) > 1:
            raise ValueError(f"every regional venue policy of a run must use the same 'by', got {sorted(names)}")
        return names.pop() if names else None

    def active(self, timer):
        return [policy for policy in self.policies if policy.is_active(timer.date)]

    def covered(self, names):
        """The networks among ``names`` that some venue policy has an entry for."""
        return [n for n in names if any(policy.entry(n) is not None for policy in self.policies)]

    def table(self, timer, names, labels, device, batch=None):
        """The factor table of the step at ``timer`` for its networks ``names`` (step order): [K, R] ([b, K, R] when
        an entry holds one row per sample), the product over the active policies; None when no active policy has an
        entry for any of the networks."""
        R = len(labels)
        rows = [None] * len(names)
        for policy in self.active(timer):
            for k, name in enumerate(names):
                key = policy.entry(name)
                if key is None:
                    continue
                f = policy.factors(key, labels, device, batch)
                rows[k] = f if rows[k] is None else rows[k] * f
        if all(r is None for r in rows):
            return None
        lead = next((tuple(r.shape[:-1]) for r in rows if r is not None and r.dim() == 2), ())
        one = torch.ones(lead + (R,), dtype=torch.float32, device=device)
        return torch.stack([one if r is None else r.expand(lead + (R,)) for r in rows], dim=-2)
