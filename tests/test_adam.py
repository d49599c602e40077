"""Adam in the fused learner step (`args.optimizer: "adam"`), host side: the fp64 reference of tests/adam_ref.py against a
stock torch.optim.Adam in float64, FusedAdam's torch state-dict format in both directions, the optimiser selection and
its rejections, and the mal_adam_t ABI."""
import ctypes as C

import numpy as np
import pytest
import torch as th

from ma_league_b200 import _native as nat
from ma_league_b200.learners.learner import FusedAdam, FusedRMSprop
from tests import adam_ref as R


def _params(seed, shapes=((7, 5), (5,), (3, 7), (3,))):
    g = th.Generator().manual_seed(seed)
    return [th.randn(s, generator=g, dtype=th.float64) for s in shapes]


@pytest.mark.parametrize("clip", [100.0, 0.5])
@pytest.mark.parametrize("weight_decay", [0.0, 1e-4])
@pytest.mark.parametrize("n_frozen_params", [0, 2])
def test_reference_equals_torch_adam_float64(clip, weight_decay, n_frozen_params):
    """5 chained steps of clip_grad_norm_ + torch.optim.Adam against adam_ref.clip_adam; both clip branches are taken."""
    ps = [p.clone().requires_grad_(i >= n_frozen_params) for i, p in enumerate(_params(0))]
    trained = [p for p in ps if p.requires_grad]
    opt = th.optim.Adam(trained, lr=1e-3, weight_decay=weight_decay)
    n_frozen = sum(p.numel() for p in ps[:n_frozen_params])
    flat = np.concatenate([p.detach().numpy().ravel() for p in ps])
    m, v, step = np.zeros_like(flat), np.zeros_like(flat), 0
    gen = th.Generator().manual_seed(1)
    for i in range(5):
        grads = [th.randn(p.shape, generator=gen, dtype=th.float64) * (i + 1) for p in ps]
        for p, g in zip(trained, grads[n_frozen_params:]):
            p.grad = g.clone()
        norm_t = float(th.nn.utils.clip_grad_norm_(trained, clip))
        opt.step()
        g_flat = np.concatenate([g.numpy().ravel() for g in grads])
        norm, g_clip, flat, m, v, step = R.clip_adam(flat, g_flat, m, v, step, 1e-3, clip, n_frozen,
                                                     weight_decay=weight_decay)
        assert abs(norm - norm_t) <= 1e-12 * norm_t
        assert (norm > clip) == (clip < 1.0)
        got = np.concatenate([p.detach().numpy().ravel() for p in ps])
        np.testing.assert_allclose(got, flat, rtol=1e-12, atol=1e-15)
        np.testing.assert_allclose(np.concatenate([p.grad.numpy().ravel() for p in trained]), g_clip[n_frozen:],
                                   rtol=1e-12, atol=0)
        st = [opt.state[p] for p in trained]
        np.testing.assert_allclose(np.concatenate([s["exp_avg"].numpy().ravel() for s in st]), m[n_frozen:], rtol=1e-12)
        np.testing.assert_allclose(np.concatenate([s["exp_avg_sq"].numpy().ravel() for s in st]), v[n_frozen:], rtol=1e-12)
        assert all(float(s["step"]) == step for s in st)
    assert not m[:n_frozen].any() and not v[:n_frozen].any()


def _stock_after_steps(params, n, lr=1e-3, weight_decay=0.0):
    opt = th.optim.Adam(params, lr=lr, weight_decay=weight_decay)
    gen = th.Generator().manual_seed(2)
    for _ in range(n):
        for p in params:
            p.grad = th.randn(p.shape, generator=gen)
        opt.step()
    return opt


def test_state_dict_matches_stock_adam_and_round_trips():
    ps = [p.float() for p in _params(3)]
    stock = _stock_after_steps([p.clone() for p in ps], 3, weight_decay=1e-4)
    ref = stock.state_dict()
    fused = FusedAdam(ps, lr=1e-3, weight_decay=1e-4)
    fused.load_state_dict(ref)                                    # a stock checkpoint loads ...
    P = sum(p.numel() for p in ps)
    assert fused._steps == 3 and float(fused.flat_state[2 * P]) == 3.0
    assert int(fused.flat_state[2 * P + 1:].view(th.int32)[0]) == 0
    for p in ps:                                                  # ... into views of the one flat buffer
        st = fused.state[p]
        assert st["exp_avg"].untyped_storage().data_ptr() == fused.flat_state.untyped_storage().data_ptr()
        assert st["exp_avg_sq"].untyped_storage().data_ptr() == fused.flat_state.untyped_storage().data_ptr()
    sd = fused.state_dict()                                       # ... and writes torch's format back
    assert sd["param_groups"] == ref["param_groups"]
    assert sd["state"].keys() == ref["state"].keys()
    for k, st in ref["state"].items():
        assert sd["state"][k].keys() == st.keys()
        for name, val in st.items():
            assert sd["state"][k][name].dtype == val.dtype and sd["state"][k][name].device == val.device, name
            assert th.equal(sd["state"][k][name], val), (k, name)
    # a FusedAdam checkpoint continues a stock Adam exactly like the stock checkpoint
    a, b = [p.clone() for p in ps], [p.clone() for p in ps]
    oa, ob = th.optim.Adam(a, lr=1e-3), th.optim.Adam(b, lr=1e-3)
    oa.load_state_dict(ref)
    ob.load_state_dict(sd)
    for x, y in zip(a, b):
        x.grad = th.ones_like(x)
        y.grad = th.ones_like(y)
    oa.step()
    ob.step()
    assert all(th.equal(x, y) for x, y in zip(a, b))
    assert fused.param_groups[0]["weight_decay"] == 1e-4
    h = fused.hyper(5e-4, 10.0)
    assert (h.lr, h.beta1, h.beta2, h.eps, h.weight_decay) == (5e-4, 0.9, 0.999, 1e-8, 1e-4)


def test_fresh_state_dict_has_zero_state():
    ps = [p.float() for p in _params(4)]
    sd = FusedAdam(ps, lr=1e-3).state_dict()
    g = sd["param_groups"][0]
    assert g["lr"] == 1e-3 and g["betas"] == (0.9, 0.999) and g["eps"] == 1e-8 and g["weight_decay"] == 0
    assert not g["amsgrad"] and not g["maximize"]
    for st in sd["state"].values():
        assert set(st) == {"step", "exp_avg", "exp_avg_sq"} and float(st["step"]) == 0.0
        assert not st["exp_avg"].any() and not st["exp_avg_sq"].any()


def test_rejections():
    ps = [p.float() for p in _params(5)]
    fused = FusedAdam(ps, lr=1e-3)
    with pytest.raises(nat.MalError):
        fused.step()
    ams = th.optim.Adam([p.clone() for p in ps], lr=1e-3, amsgrad=True)
    with pytest.raises(nat.MalError, match="amsgrad"):
        fused.load_state_dict(ams.state_dict())
    rms = th.optim.RMSprop([p.clone() for p in ps], lr=1e-3)
    before = fused.flat_state.clone()
    with pytest.raises(nat.MalError):
        fused.load_state_dict(rms.state_dict())
    assert th.equal(fused.flat_state, before) and fused.param_groups[0]["betas"] == (0.9, 0.999)   # nothing half-loaded
    fr = FusedRMSprop(ps, lr=1e-3, alpha=0.99, eps=1e-5)
    sq = fr.flat_sq.clone()
    with pytest.raises(nat.MalError):
        fr.load_state_dict(_stock_after_steps([p.clone() for p in ps], 1).state_dict())
    assert th.equal(fr.flat_sq, sq) and fr.param_groups[0]["alpha"] == 0.99


def _cpu_learner(**over):
    from tests.gpu_helpers import build_system
    return build_system(3, 9, 32, 48, 4, 6, "qmix", True, device="cpu", **over).learner


def test_build_optimizer_selects_by_args_optimizer():
    assert isinstance(_cpu_learner().optimiser, FusedRMSprop)                       # key absent: unchanged
    assert isinstance(_cpu_learner(optimizer="rmsprop").optimiser, FusedRMSprop)
    L = _cpu_learner(optimizer="adam", lr=1e-3)
    assert isinstance(L.optimiser, FusedAdam) and L._adam() is not None
    g = L.optimiser.param_groups[0]
    assert g["lr"] == 1e-3 and g["weight_decay"] == 0 and g["betas"] == (0.9, 0.999) and g["eps"] == 1e-8
    assert L.optimiser.flat_state.numel() == nat.adam_state_floats(sum(p.numel() for p in L.parameters()))
    assert _cpu_learner(optimizer="adam", weight_decay=1e-4).optimiser.param_groups[0]["weight_decay"] == 1e-4
    assert _cpu_learner(optimizer="rmsprop")._adam() is None
    for bad in ("adamw", "Adam", "sgd", 1):
        with pytest.raises(nat.MalError, match="optimizer"):
            _cpu_learner(optimizer=bad)


def test_adam_struct_matches_c():
    import os
    import subprocess
    import tempfile
    from tests.helpers import ROOT
    prog = r'''
    #include <stdio.h>
    #include <stddef.h>
    #include "mal_b200.h"
    int main(void) { printf("%zu %zu %d\n", sizeof(mal_adam_t), offsetof(mal_adam_t, clip), (int)MAL_ADAM_STATE_FLOATS(10)); return 0; }'''
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, "s.c")
        open(src, "w").write(prog)
        exe = os.path.join(d, "s")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), src, "-o", exe])
        size, off, floats = [int(x) for x in subprocess.check_output([exe]).split()]
    assert size == C.sizeof(nat.AdamHyper) and off == nat.AdamHyper.clip.offset and floats == nat.adam_state_floats(10)
