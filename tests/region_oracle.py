"""Regional transmission factor in the oracle: ``regional_factor(factor_of)`` hooks ``O.not_infected_probs`` (the way
``helpers.perturb_q`` does) and multiplies the oracle's summed pressure by a per-agent factor before the clamp, so
``lam_raw`` is the product.  A per-region factor gathered per agent gives, through autograd, d/dfactor per region."""
import torch

from oracle import gj_oracle as O


class regional_factor:
    """``factor_of(spec)``: the per-agent factor of the step ([N], any float dtype), or None outside every window."""

    def __init__(self, factor_of):
        self.factor_of = factor_of

    def __enter__(self):
        self.orig = O.not_infected_probs

        def hooked(world, spec, T, s, current_stage, return_pressure=False):
            qmask = O.quarantine_mask(current_stage, spec.quarantine)
            lam = torch.zeros(world.n_agents, dtype=T.dtype, device=T.device)
            for net in spec.nets:
                lam = lam + O.network_pressure(world, net, T, s, qmask, spec.day_type)
            m = self.factor_of(spec)
            if m is not None:
                lam = lam * m.to(lam.dtype)
            lam_raw = lam
            lam = torch.clamp(lam, min=1e-6, max=100)
            q = torch.clamp(torch.exp(-lam * spec.dt), min=0.0, max=1.0)
            return (q, lam_raw) if return_pressure else q
        O.not_infected_probs = hooked
        return self

    def __exit__(self, *a):
        O.not_infected_probs = self.orig
