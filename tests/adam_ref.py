"""Reference computations for the fused Adam step (test infrastructure).

* `adam_update`: one torch.optim.Adam step (amsgrad=False, maximize=False, L2 weight decay added to the gradient and not
  written back) over flat fp64 arrays, with the bias corrections computed from the step count as torch's non-capturable
  Adam does on the host.
* `clip_adam`: clip_grad_norm_ (q_learner.py:104, np_oracle.clip_grad_norm) over the trained parameters followed by
  `adam_update`; a frozen prefix (freeze_agent_weights) has no gradient, stays out of the norm and is not stepped.
"""
from __future__ import annotations

import numpy as np

from oracle import np_oracle as O

BETAS = (0.9, 0.999)
EPS = 1e-8


def adam_update(p, g, m, v, step, lr, betas=BETAS, eps=EPS, weight_decay=0.0):
    """(p, exp_avg, exp_avg_sq, step) after one step from gradient g (all flat fp64 arrays but `step`, an int)."""
    b1, b2 = betas
    g = g + weight_decay * p if weight_decay else g
    t = step + 1
    m = b1 * m + (1.0 - b1) * g
    v = b2 * v + (1.0 - b2) * g * g
    p = p - (lr / (1.0 - b1 ** t)) * m / (np.sqrt(v) / np.sqrt(1.0 - b2 ** t) + eps)
    return p, m, v, t


def clip_adam(p, g, m, v, step, lr, clip, n_frozen=0, betas=BETAS, eps=EPS, weight_decay=0.0):
    """(norm, clipped gradient, p, exp_avg, exp_avg_sq, step): the fused step over flat fp64 arrays.  The clipped gradient
    is zero on the frozen prefix, whose parameters and state are returned unchanged."""
    p, m, v, g = (np.array(x, dtype=np.float64) for x in (p, m, v, g))
    g[:n_frozen] = 0.0
    norm, (gc,) = O.clip_grad_norm([g[n_frozen:]], clip)
    g[n_frozen:] = gc
    s = slice(n_frozen, None)
    p[s], m[s], v[s], t = adam_update(p[s], g[s], m[s], v[s], step, lr, betas, eps, weight_decay)
    return norm, g, p, m, v, t
