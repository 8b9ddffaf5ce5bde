"""CPU checks of the optimizer row (SURVEY §8(f)-3): the Adam arithmetic of `k_adam_flat` (host build of
gsb200_math.cuh) against torch.optim.Adam as the reference configures it (eps 1e-15, per-field lr), and the restated
learning-rate schedules against utils/schedulers.py (imported from $GSB200_REFERENCE when set, otherwise the values it
computed, tests/golden/schedulers_ref.npz)."""
import ctypes
import math
import sys

import pytest
import torch

from gsgen_b200 import optim
from tests.util import RefValues, fp


def test_adam_arithmetic_matches_torch(hostmath):
    g = torch.Generator().manual_seed(3)
    n = 4099
    p0 = torch.randn(n, generator=g)
    p_ref = p0.clone().requires_grad_()
    opt = torch.optim.Adam([{"params": [p_ref], "lr": 0.005}], lr=0.0, eps=1e-15)
    p, m, v = p0.clone(), torch.zeros(n), torch.zeros(n)
    hostmath.hm_adam.argtypes = [ctypes.c_longlong] + [ctypes.c_void_p] * 4 + [ctypes.c_double] * 4 + \
        [ctypes.c_longlong, ctypes.c_float]
    for step in range(1, 9):
        grad = torch.randn(n, generator=g) * (10.0 ** float(torch.randint(-6, 2, (1,), generator=g)))
        grad[::7] = 0.0  # culled Gaussians: exact zeros
        lr = 0.005 * (0.9 ** step)
        opt.param_groups[0]["lr"] = lr
        p_ref.grad = grad.clone()
        opt.step()
        hostmath.hm_adam(n, fp(p), fp(grad), fp(m), fp(v), lr, 0.9, 0.999, 1e-15, step, 1.0)
        st = opt.state[p_ref]
        # fp32 rounding (FMA contraction differs between the two builds); 0.9 m + 0.1 g may cancel, hence the atol
        assert torch.allclose(m, st["exp_avg"], rtol=2e-6, atol=2e-7 * float(st["exp_avg"].abs().max()))
        assert torch.allclose(v, st["exp_avg_sq"], rtol=2e-6, atol=1e-38)
        # the update is lr-sized: compare the parameters relative to the accumulated step length
        assert float((p - p_ref.detach()).abs().max()) <= 2e-6 * 0.005 * step + 1e-7 * float(p0.abs().max())
    assert torch.isfinite(p).all()


def test_adam_grad_scale_is_a_gradient_prefactor(hostmath):
    g = torch.Generator().manual_seed(4)
    n = 257
    grad = torch.randn(n, generator=g)
    out = []
    for scale, gr in ((0.125, grad), (1.0, grad * 0.125)):
        p, m, v = torch.ones(n), torch.zeros(n), torch.zeros(n)
        hostmath.hm_adam.argtypes = [ctypes.c_longlong] + [ctypes.c_void_p] * 4 + [ctypes.c_double] * 4 + \
            [ctypes.c_longlong, ctypes.c_float]
        hostmath.hm_adam(n, fp(p), fp(gr.contiguous()), fp(m), fp(v), 0.01, 0.9, 0.999, 1e-15, 1, scale)
        out.append((p, m, v))
    for a, b in zip(*out):
        assert torch.equal(a, b)  # 0.125 is a power of two: bit-identical


PINNED = {  # utils/schedulers.py evaluated in the dev container (conf/base.yaml:13-22 entries)
    ("exp", 0.005, 3.0e-05, 15000): {0: 0.005000000000000002, 1: 0.00499829495884606, 7500: 0.00038729833462074144,
                                     15000: 2.9999999999999977e-05, 20000: 2.9999999999999977e-05},
    ("exp", 0.003, 0.001, 15000): {0: 0.002999999999999999, 3000: 0.00240822468528069, 15000: 0.0010000000000000002},
    ("cosine", 0.01, 0.001, 1000): {0: 0.010000000000000002, 250: 0.008681980515339464, 500: 0.0055000000000000005,
                                    1000: 0.001},
}


@pytest.mark.parametrize("key", list(PINNED))
def test_lr_schedules_pinned(key):
    kind, a, b, steps = key
    sched = optim.make_scheduler([a, b, steps, kind], max_steps=15000)
    for step, want in PINNED[key].items():
        assert math.isclose(sched(step), want, rel_tol=1e-12), (key, step, sched(step), want)
    assert optim.make_scheduler(0.003, 15000)(1234) == 0.003


def test_lr_schedules_match_reference_module():
    rv = RefValues("schedulers_ref")
    ref = None
    if rv.live:
        sys.path.insert(0, rv.src)
        try:
            import importlib
            ref = importlib.import_module("utils.schedulers")
        finally:
            sys.path.pop(0)
    for kind in ("exp", "cosine", "nothing"):
        for (a, b, steps) in ((0.005, 3e-5, 15000), (0.003, 0.001, 15000), (1e-4, 1e-6, 777)):
            ours = optim.lr_schedulers[kind](steps, a, b)
            theirs = ref.lr_schedulers[kind](steps, a, b) if ref else None
            for step in (0, 1, 13, steps // 3, steps - 1, steps, steps + 50 if kind != "cosine" else steps):
                want = float(rv(f"{kind}_{a}_{b}_{steps}_{step}", lambda: float(theirs(step))))
                assert math.isclose(ours(step), want, rel_tol=1e-12), (kind, a, b, steps, step)
    # warm-up branch
    ours = optim.exp_decay(1000, 1e-2, 1e-4, warmup_steps=100)
    theirs = ref.exp_decay(1000, 1e-2, 1e-4, warmup_steps=100) if ref else None
    for step in (0, 50, 99, 100, 500):
        assert math.isclose(ours(step), float(rv(f"warmup_{step}", lambda: float(theirs(step)))), rel_tol=1e-12)
    rv.save()
