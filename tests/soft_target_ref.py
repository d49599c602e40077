"""Reference of the soft target update (test infrastructure): the three fp32 torch ops of a per-tensor Polyak loop,
`target.data.copy_(target.data * (1.0 - tau) + param.data * tau)` with a Python-float tau, which the SOFT optimiser
kernels reproduce bit for bit (c1 = fp32(1 - tau) with the subtraction in double, c2 = fp32(tau), no FMA)."""
import numpy as np
import torch as th


def blend_(target, param, tau):
    """In place on fp32 tensors (any device): target <- fp32(fp32(target * (1 - tau)) + fp32(param * tau))."""
    target.copy_(target * (1.0 - tau) + param * tau)
    return target


def blend_np(target, param, tau):
    """The same arithmetic in numpy float32 (every operation rounded to fp32, no contraction)."""
    c1, c2 = np.float32(1.0 - tau), np.float32(tau)
    t, p = np.asarray(target, np.float32), np.asarray(param, np.float32)
    return (t * c1).astype(np.float32) + (p * c2).astype(np.float32)


def blend_modules_(target_modules, modules, tau):
    """blend_ over every parameter of each (target, online) module pair, in place."""
    with th.no_grad():
        for tm, m in zip(target_modules, modules):
            for tp, p in zip(tm.parameters(), m.parameters()):
                blend_(tp.data, p.data, tau)
