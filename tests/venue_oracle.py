"""Regional venue factor in the oracle: ``venue_factor(factor_of)`` replaces the ``ones(G)`` of the oracle's per-group
beta (``O.network_pressure``, the reference's ``_get_beta`` vector, base.py:36-42) by the factor of each group's region,
so the group value is ``(beta * f[code]) * pc`` and autograd gives d/dfactor per region."""
from oracle import gj_oracle as O


class venue_factor:
    """``factor_of(spec, net)``: network ``net``'s per-group factor at step ``spec`` ([G] tensor), or None (factor 1)."""

    def __init__(self, factor_of):
        self.factor_of = factor_of

    def __enter__(self):
        self.orig = O.network_pressure
        orig = self.orig
        factor_of = self.factor_of

        class _Hooked:
            spec = None

        def not_infected_probs(world, spec, T, s, current_stage, return_pressure=False):
            _Hooked.spec = spec
            return self.orig_probs(world, spec, T, s, current_stage, return_pressure)

        def network_pressure(world, net, T, s, qmask, day_type):
            f = factor_of(_Hooked.spec, net)
            if f is None:
                return orig(world, net, T, s, qmask, day_type)
            et = world.edges[net.edge_type]
            beta = net.beta * f.to(T.dtype)                                             # base.py:41, per group
            beta = beta * O.p_contact(et.people.to(T.device), T)
            if net.kind == O.KIND_HOUSEHOLD:
                Tm, sm = T, s
            elif net.kind == O.KIND_PLAIN:
                Tm, sm = qmask * T, qmask * s
            else:
                lm = net.prob.to(T.dtype)[day_type, world.sex, world.age]
                Tm = qmask * lm * T
                sm = qmask * lm * s
                if net.kind == O.KIND_CARE_VISIT:
                    sm = sm * (world.age > 75)
            cum = O.propagate(et.src, et.dst, Tm, beta)
            return O.propagate(et.dst, et.src, cum, sm)

        self.orig_probs = O.not_infected_probs
        O.not_infected_probs = not_infected_probs
        O.network_pressure = network_pressure
        return self

    def __exit__(self, *a):
        O.network_pressure = self.orig
        O.not_infected_probs = self.orig_probs
