"""Seeding by label in the oracle: ``oracle.gj_oracle.seed`` broadcasts a per-agent log-fraction, so a per-region
log-fraction gathered per agent gives, through autograd, d/dlog_fraction per region."""
import torch


def seed_log_fraction(log_fraction, label):
    """Per-agent log-fractions ``log_fraction[label]``: ``log_fraction`` [R] per region, ``label`` [N] each agent's
    region."""
    idx = torch.as_tensor(label, dtype=torch.long, device=log_fraction.device)
    return log_fraction[idx]
