"""Background models (gsgen_b200/backgrounds.py) against the reference's OWN classes (gs/backgrounds.py compiled out of
the file with `ast` where the reference is at $GSB200_REFERENCE; elsewhere against their draws stored in
tests/golden/backgrounds_ref.npz) draw for draw, and their wiring into
the trainer-facing renderer (`cfg.background` -> setup_bg, `.bg`, train / eval, checkpoint `bg` state)."""
import ast
import os
import random

import pytest
import torch
import torch.nn as nn

from gsgen_b200 import backgrounds as B
from tests.util import RefValues


class Cfg(dict):
    __getattr__ = dict.__getitem__


def _ref_classes(rv):
    from einops import repeat

    path = os.path.join(rv.src, "gs", "backgrounds.py")
    ns = {"torch": torch, "nn": nn, "random": random, "repeat": repeat, "tcnn_capable": False}
    tree = ast.parse(open(path).read())
    for node in tree.body:
        if isinstance(node, ast.ClassDef):
            exec(compile(ast.Module(body=[node], type_ignores=[]), path, "exec"), ns)
    return ns


@pytest.mark.parametrize("kind,extra", [("random", dict(range=[0.2, 0.9])), ("fixed", dict(color=[0.1, 0.5, 0.9])),
                                        ("random", dict(range=[0.0, 1.0], random_aug=True, random_aug_prob=0.5))])
def test_backgrounds_match_reference_draw_for_draw(kind, extra):
    rv = RefValues("backgrounds_ref")
    cfg = Cfg(type=kind, device="cpu", random_aug=False, random_aug_prob=0.0)
    cfg.update(extra)
    ref = None
    if rv.live:
        ns = _ref_classes(rv)
        ref = {"random": ns["RandomBackground"], "fixed": ns["FixedBackground"]}[kind](cfg)
    ours = B.make_background(cfg)
    dirs = torch.randn(5, 7, 3, generator=torch.Generator().manual_seed(5))
    tag = f"{kind}_{'_'.join(f'{k}={v}' for k, v in sorted(extra.items()))}"

    def draw(model):
        random.seed(11); torch.manual_seed(11)
        return model(dirs)

    for m, mode in enumerate((True, False, True)):
        ours.train(mode)
        if ref is not None:
            ref.train(mode)
        for i in range(6):
            a = torch.from_numpy(rv(f"{tag}_{m}_{i}", lambda: draw(ref)))
            b = draw(ours)
            assert a.shape == b.shape == (5, 7, 3) and torch.equal(a, b)
    if kind == "fixed":  # the colour is a parameter: gradient of sum(bg * w) is the sum of w over the pixels
        w = torch.randn(5, 7, 3)
        (ours(dirs) * w).sum().backward()
        assert torch.allclose(ours.bg_color.grad, w.sum(dim=(0, 1)))
        assert set(ours.state_dict()) == set(rv(f"{tag}_state", lambda: sorted(ref.state_dict()))) == {"bg_color"}
    rv.save()


def test_learned_const_and_unknown_types():
    bg = B.make_background({"type": "learned_const", "initial_color": [0.3, 0.4, 0.5]})
    out = bg(torch.zeros(4, 6, 3))
    assert out.shape == (4, 6, 3) and torch.equal(out[2, 3], torch.tensor([0.3, 0.4, 0.5])) and bg.bg_color.requires_grad
    with pytest.raises(NotImplementedError):
        B.make_background({"type": "mlp"})
    with pytest.raises(NotImplementedError):
        B.make_background({"type": "sky"})


def test_renderer_builds_its_background_from_cfg(oracle_mod):
    from gsgen_b200.splatting import GaussianSplattingRenderer
    from gsgen_b200.store import quat_to_rotmat

    g = torch.Generator().manual_seed(0)
    N = 40
    init = {"mean": torch.randn(N, 3, generator=g), "qvec": torch.randn(N, 4, generator=g),
            "svec": torch.rand(N, 3, generator=g) * 0.1 + 0.01, "color": torch.rand(N, 3, generator=g) * 0.8 + 0.1,
            "alpha": torch.rand(N, generator=g) * 0.8 + 0.1}
    cfg = {"background": {"type": "fixed", "color": [0.2, 0.3, 0.4], "device": "cpu", "random_aug": False,
                          "random_aug_prob": 0.0}}
    r = GaussianSplattingRenderer(cfg, init, device="cpu", render_fn=lambda *a, **k: None)
    assert isinstance(r.bg, B.FixedBackground) and r.bg is r.background
    r.eval()
    assert not r.bg.training
    r.train()
    assert r.bg.training
    assert "bg_color" in r.get_params_for_save()["bg"]
    # the attributes guidance / export code reads (gs/gaussian_splatting.py:146-156)
    assert torch.allclose(r.cov, r.svec.unsqueeze(-2) * quat_to_rotmat(r.qvec))
    assert torch.equal(r.principal_axis, r.rotmat) and r.cov.shape == (N, 3, 3)
    # no cfg.background and no argument: black (None), as before
    r2 = GaussianSplattingRenderer({}, init, device="cpu", render_fn=lambda *a, **k: None)
    assert r2.bg is None


def test_background_parameters_are_optimised_with_the_renderer(oracle_mod):
    """the reference's Adam holds a "bg" param group with its own schedule (gs/gaussian_splatting.py:383-419,
    conf/base.yaml:26): a FIXED background's colour is a parameter and trains (conf/renderer/regular.yaml)"""
    from gsgen_b200.optim import CompanionAdam
    from gsgen_b200.splatting import GaussianSplattingRenderer

    g = torch.Generator().manual_seed(0)
    N = 30
    init = {"mean": torch.randn(N, 3, generator=g), "qvec": torch.randn(N, 4, generator=g),
            "svec": torch.rand(N, 3, generator=g) * 0.1 + 0.01, "color": torch.rand(N, 3, generator=g) * 0.8 + 0.1,
            "alpha": torch.rand(N, generator=g) * 0.8 + 0.1}
    cfg = {"background": {"type": "fixed", "color": [0.2, 0.3, 0.4], "device": "cpu", "random_aug": False,
                          "random_aug_prob": 0.0}}
    r = GaussianSplattingRenderer(cfg, init, device="cpu", render_fn=lambda *a, **k: None)
    lr = {"mean": 1e-3, "qvec": 1e-3, "svec": 1e-3, "color": 1e-2, "alpha": 1e-2}
    r.setup_lr(lr)
    with pytest.raises(RuntimeError, match="bg"):
        r.set_optimizer({"type": "Adam", "opt_args": {"eps": 1e-15}})
    r.setup_lr(dict(lr, bg=[0.003, 0.0003, 100, "exp"]))
    opt = r.set_optimizer({"type": "Adam", "opt_args": {"eps": 1e-15}})
    (comp,) = opt.companions
    assert isinstance(comp, CompanionAdam) and comp.params[0] is r.bg.bg_color
    # one update of the companion = torch.optim.Adam on a twin parameter with the scheduled lr
    w = torch.randn(4, 5, 3, generator=g)
    twin = torch.nn.Parameter(r.bg.bg_color.detach().clone())
    ref = torch.optim.Adam([twin], lr=0.0, eps=1e-15)
    for step in (0, 50):
        for p_, bgimg in ((r.bg.bg_color, r.bg(torch.zeros(4, 5, 3))), (twin, twin.reshape(1, 1, 3).expand(4, 5, 3))):
            p_.grad = None
            (bgimg * w).sum().backward()
        used = comp.step(step)
        ref.param_groups[0]["lr"] = float(comp.scheduler(step))
        ref.step()
        assert used == pytest.approx(float(comp.scheduler(step))) and torch.equal(r.bg.bg_color.detach(), twin.detach())
    assert comp.scheduler(0) == pytest.approx(0.003) and comp.scheduler(100) == pytest.approx(0.0003, rel=1e-6)
    opt.flat_grad.fill_(1.0)
    opt.zero_grad()  # FlatAdam.zero_grad reaches the companion
    assert r.bg.bg_color.grad is None or float(r.bg.bg_color.grad.abs().max()) == 0.0
    assert float(opt.flat_grad.abs().max()) == 0.0
    # a background without parameters needs no lr
    r2 = GaussianSplattingRenderer({"background": {"type": "random", "device": "cpu"}}, init, device="cpu",
                                   render_fn=lambda *a, **k: None)
    r2.setup_lr(lr)
    assert not getattr(r2.set_optimizer({"type": "Adam", "opt_args": {"eps": 1e-15}}), "companions", [])


def test_checkpoint_round_trip_restores_cfg_and_background(tmp_path):
    """vis.py:17 `GaussianSplattingRenderer.load(None, ckpt).to("cuda")`: the configuration and the background state
    come out of the checkpoint (gs/gaussian_splatting.py:312-339)"""
    from gsgen_b200.splatting import GaussianSplattingRenderer

    g = torch.Generator().manual_seed(3)
    N = 25
    init = {"mean": torch.randn(N, 3, generator=g), "qvec": torch.randn(N, 4, generator=g),
            "svec": torch.rand(N, 3, generator=g) * 0.1 + 0.01, "color": torch.rand(N, 3, generator=g) * 0.8 + 0.1,
            "alpha": torch.rand(N, generator=g) * 0.8 + 0.1}
    cfg = {"T_thresh": 2e-4, "background": {"type": "fixed", "color": [0.2, 0.3, 0.4], "device": "cpu",
                                            "random_aug": False, "random_aug_prob": 0.0}}
    r = GaussianSplattingRenderer(cfg, init, device="cpu", render_fn=lambda *a, **k: None)
    with torch.no_grad():
        r.bg.bg_color.copy_(torch.tensor([0.9, 0.8, 0.7]))  # a trained background colour
    fake = lambda *a, **k: None
    # renderer-only checkpoint
    p1 = str(tmp_path / "renderer.pt")
    torch.save(r.get_params_for_save(), p1)
    a = GaussianSplattingRenderer.load(None, p1, device="cpu", render_fn=fake)
    # trainer checkpoint (params + the experiment cfg with its `renderer` block)
    p2 = str(tmp_path / "trainer.pt")
    torch.save({"params": r.get_params_for_save(), "cfg": {"renderer": cfg, "max_steps": 10}, "step": 5}, p2)
    b = GaussianSplattingRenderer.load({"T_thresh": 1e-4}, p2, device="cpu", render_fn=fake)
    for x in (a, b):
        assert x.N == N and torch.equal(x.mean.detach(), r.mean.detach())
        assert isinstance(x.bg, B.FixedBackground) and torch.equal(x.bg.bg_color.detach(), torch.tensor([0.9, 0.8, 0.7]))
    assert a.cfg["T_thresh"] == 2e-4 and b.cfg["T_thresh"] == 1e-4  # the argument overrides the stored value
    assert a.to("cpu") is a  # same device: nothing moves
