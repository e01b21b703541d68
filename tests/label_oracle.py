"""The oracle's trajectory (``oracle.gj_oracle.run``, same step order) with a per-label table of the result series:
cases and deaths per label column and timestep, each one ``index_add`` of the national reduction's per-agent terms in
the oracle's dtype, differentiable like the national series."""
import torch

from oracle import gj_oracle as O


def by_label(state, sym, label, n_labels):
    """[n_labels] cases and deaths per label column (label[a] = agent a's column)."""
    dead = sym.n_stages - 1
    cur, inf = state["current_stage"], state["is_infected"]
    idx = torch.as_tensor(label, dtype=torch.long, device=inf.device)
    cases = torch.zeros(n_labels, dtype=inf.dtype, device=inf.device).index_add(0, idx, inf)
    d = ((cur == dead) * cur / dead).to(inf.dtype)
    return cases, torch.zeros(n_labels, dtype=inf.dtype, device=inf.device).index_add(0, idx, d)


def run_with_labels(world, params, sym, log_fraction, steps, noises, label, age_bins=(0, 18, 65, 100),
                    dtype=torch.float32):
    """``O.run`` plus ``cases_by_label`` / ``deaths_by_label`` [T+1, max(label) + 1]."""
    n_labels = int(torch.as_tensor(label).max()) + 1
    st = O.initial_state(world.n_agents, dtype, world.age.device)
    O.seed(world, st, log_fraction, 0.0, sym, noises[0])
    rows = [(st["is_infected"].sum(), O.deaths(st, sym), O.cases_by_age(world, st, age_bins),
             *by_label(st, sym, label, n_labels))]
    for spec, noise in zip(steps, noises[1:]):
        O.step(world, st, params, spec, sym, noise)
        rows.append((st["is_infected"].sum(), O.deaths(st, sym), O.cases_by_age(world, st, age_bins),
                     *by_label(st, sym, label, n_labels)))
    cols = [torch.stack(c) for c in zip(*rows)]
    return {"cases_per_timestep": cols[0], "deaths_per_timestep": cols[1], "cases_by_age": cols[2],
            "cases_by_label": cols[3], "deaths_by_label": cols[4], "state": st}
