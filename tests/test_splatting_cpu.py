"""The trainer-facing `gsgen_b200.splatting.GaussianSplattingRenderer` (store + fused view + flat Adam wiring) on CPU,
with the CPU oracle plugged in as `render_fn`: one view against the fixture the reference's OWN `render_one` produced
(tests/golden/render_one_ref.npz), then the trainer's call sequence -- forward(batch), backward, post_backward,
densify(step), prune(step), checkpoint -- for its bookkeeping.  (The CUDA `render_fn` and `FlatAdam.step` are covered by
the -m gpu tests; they cannot run here.)"""
import os

import numpy as np
import pytest
import torch

from gsgen_b200.camera import CameraInfo
from gsgen_b200.splatting import GaussianSplattingRenderer
from tests.util import ocam_of

GOLD = os.path.join(os.path.dirname(__file__), "golden", "render_one_ref.npz")
LR = {"mean": [0.005, 3.0e-05, 15000, "exp"], "svec": [0.003, 0.001, 15000, "exp"], "qvec": 0.003, "color": 0.01,
      "alpha": 0.003}


class _Aux(dict):
    """the product's aux exposes a full-size mean2d gradient after the backward; the oracle a masked one"""

    def __getitem__(self, k):
        if k == "mean2d_grad":
            g = torch.zeros(self["mask"].shape[0], 2)
            g[self["mask"]] = self["mean2d_masked"].grad
            return g
        return super().__getitem__(k)


def _oracle_render_fn(oracle_mod):
    def render_fn(mean, qvec, svec, alpha, c2w, cam, color=None, bg=None, rgb_only=False, raw_params=False,
                  frustum_radius=6.0, tile_radius=6.0, T_thresh=1e-4, skip_frustum_culling=False, depth_detach=True,
                  grad_sink=None, slot=0):
        assert raw_params and not skip_frustum_culling
        out = oracle_mod.render_view(mean, qvec, torch.exp(svec), torch.sigmoid(alpha), c2w, ocam_of(cam),
                                     color=torch.sigmoid(color), bg=bg, rgb_only=rgb_only, depth_detach=depth_detach,
                                     frustum_radius=frustum_radius, tile_radius=tile_radius, thresh=T_thresh)
        a = out["aux"]
        radii = torch.zeros(mean.shape[0])
        cov = a["cov2d"].detach()
        m = (cov[:, 0, 0] + cov[:, 1, 1]) / 2
        radii[a["mask"]] = m + torch.sqrt((m * m - torch.det(cov)).clamp(min=0))
        out["aux"] = _Aux(mask=a["mask"], mean2d_masked=a["mean2d"], radii2d=radii, N_with_dub=a["D"])
        out.setdefault("T", None)
        return out

    return render_fn


@pytest.fixture(scope="module")
def gold():
    z = np.load(GOLD)
    return {k: torch.from_numpy(z[k]) for k in z.files}


def _renderer(gold, tag, oracle_mod, cfg=None, **kw):
    init = {k: gold[f"{tag}_in_{k}"] for k in ("mean", "qvec", "svec", "color", "alpha")}
    bg = gold[f"{tag}_in_bg"]
    r = GaussianSplattingRenderer(cfg or {}, init, device="cpu", background=lambda rays: bg,
                                  render_fn=_oracle_render_fn(oracle_mod), **kw)
    fx, fy, cx, cy, w, h, near, far = gold[f"{tag}_cam"].tolist()
    return r, CameraInfo(fx, fy, cx, cy, int(w), int(h), near, far)


@pytest.mark.parametrize("tag", ["a", "b"])
def test_one_view_matches_the_reference_render_one(gold, oracle_mod, tag):
    r, cam = _renderer(gold, tag, oracle_mod)
    r.setup_lr(LR)
    r.set_optimizer({"type": "Adam", "opt_args": {"eps": 1e-15}})
    out = r.render_one(gold[f"{tag}_c2w"], cam, use_bg=True, rgb_only=False)
    for k in ("rgb", "depth", "opacity", "z_var"):
        ref = gold[f"{tag}_{k}"]
        assert torch.allclose(out[k].reshape(ref.shape), ref, rtol=1e-4, atol=2e-5), k  # log/exp round trip of the leaves
    sum((out[k].reshape(gold[f"{tag}_w_{k}"].shape) * gold[f"{tag}_w_{k}"]).sum()
        for k in ("rgb", "depth", "opacity", "z_var")).backward()
    # gradients arrive in the arena, w.r.t. the RAW leaves: chain rule of the reference's activated-leaf gradients
    s, a, c = gold[f"{tag}_in_svec"], gold[f"{tag}_in_alpha"].reshape(-1), gold[f"{tag}_in_color"]
    want = {"mean": gold[f"{tag}_grad_mean"], "qvec": gold[f"{tag}_grad_qvec"], "svec": gold[f"{tag}_grad_svec"] * s,
            "alpha": gold[f"{tag}_grad_alpha"].reshape(-1) * a * (1 - a), "color": gold[f"{tag}_grad_color"] * c * (1 - c)}
    for k, ref in want.items():
        got = r.store.grad_views[k]
        assert float((got - ref).norm() / ref.norm()) < 2e-4, k
    r.post_backward()
    mask = gold[f"{tag}_mask"]
    assert torch.equal(r.store.cnt, mask.float())
    assert torch.allclose(r.store.mean_2d_grad_accum, torch.zeros(r.N).index_put((mask,), gold[f"{tag}_mean2d_grad"].norm(dim=-1)),
                          rtol=1e-3, atol=1e-7)
    assert torch.allclose(r.store.max_radii2d, gold[f"{tag}_max_radii2d"], rtol=1e-4, atol=1e-8)


def test_trainer_call_sequence(gold, oracle_mod, tmp_path):
    cfg = {"densify": dict(enabled=True, type="official", warm_up=2, end=100, period=2, mean2d_thresh=1e-9,
                           split_thresh=0.02, n_splits=2, split_shrink=0.8, use_legacy=False),
           "prune": dict(enabled=True, warm_up=0, end=100, period=2, radii2d_thresh=0.0, alpha_thresh=0.05,
                         radii3d_thresh=0.0)}
    r, cam = _renderer(gold, "a", oracle_mod, cfg=cfg)
    r.setup_lr(LR)
    opt = r.set_optimizer({"type": "Adam", "opt_args": {"eps": 1e-15}})
    assert opt.eps == 1e-15 and opt.flat_param.data_ptr() == r.store.flat_param.data_ptr()
    c2w = gold["a_c2w"]
    batch = {"c2w": torch.stack([c2w, c2w]), "camera_info": [cam, cam]}
    torch.manual_seed(0)
    sizes = []
    for step in range(4):
        r.update(step)
        assert opt.train_step == step
        out = r(batch, use_bg=True, rgb_only=False)
        assert out["rgb"].shape == (2, cam.h, cam.w, 3) and out["z_var"].shape == (2, cam.h, cam.w, 1)
        out["rgb"].sum().backward()
        assert float(r.store.flat_grad.abs().max()) > 0
        # optimizer.step() needs the CUDA library: not run here (tests/test_optim_gpu.py, tests/test_train_step_gpu.py)
        r.post_backward()
        if step < 2:  # two views per step accumulate until densify() resets the statistics (:816-817)
            assert float(r.store.cnt.max()) == 2.0 * (step + 1)
        n0 = r.N
        r.densify(step)
        r.prune(step)
        sizes.append((n0, r.N))
        assert opt.flat_param.data_ptr() == r.store.flat_param.data_ptr()  # the optimizer follows re-allocations
        opt.zero_grad()
        assert float(r.store.flat_grad.abs().max()) == 0
    assert sizes[0][0] == sizes[0][1] and sizes[1][0] == sizes[1][1] == sizes[0][0]  # steps 0, 1: nothing due
    assert sizes[2][1] != sizes[2][0]  # step 2: warm-up reached, period 2 -> densify + prune ran
    assert r.mean.shape[0] == r.N and r.svec.shape == (r.N, 3) and float(r.alpha.min()) > 0
    # eval mode renders without touching the gradient arena or the statistics
    r.eval()
    img = r.render_one(c2w, cam, rgb_only=True)["rgb"]
    assert img.shape == (cam.h, cam.w, 3) and float(r.store.flat_grad.abs().max()) == 0 and not r._pending
    # checkpoint round trip under the reference's keys
    path = str(tmp_path / "ck.pt")
    torch.save({"params": r.get_params_for_save(), "cfg": {}, "step": 3}, path)
    r2 = GaussianSplattingRenderer.load({}, path, device="cpu", render_fn=_oracle_render_fn(oracle_mod))
    assert r2.N == r.N and torch.equal(r2.mean.detach(), r.mean.detach())
    assert torch.allclose(r2.svec.detach(), r.svec.detach())


def test_auxiliary_losses_match_the_reference_methods(gold, oracle_mod):
    """alpha / mean / scale penalties and auxiliary_loss against the reference's own method definitions
    (gs/gaussian_splatting.py:950-1013, :1115-1122) and its schedule helper C (utils/misc.py:218-250), executed with
    `ast` on a stand-in object where the reference is at $GSB200_REFERENCE; elsewhere against the values they computed
    (tests/golden/aux_losses_ref.npz)."""
    import ast
    import types

    from gsgen_b200.splatting import scheduled_value
    from tests.util import RefValues

    rv = RefValues("aux_losses_ref")

    def defs(path, names, ns, in_class=None):
        if not rv.live:
            return ns
        tree = ast.parse(open(os.path.join(rv.src, path)).read())
        body = tree.body
        if in_class:
            body = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == in_class).body
        for node in body:
            if isinstance(node, ast.FunctionDef) and node.name in names:
                node.returns, node.decorator_list = None, []
                for a in node.args.args:
                    a.annotation = None
                exec(compile(ast.Module(body=[node], type_ignores=[]), path, "exec"), ns)
        return ns

    ns = defs("utils/misc.py", ["C"], {"np": np, "Any": object, "to_primitive": lambda v: list(v)})
    for i, (spec, step) in enumerate(((3.5, 10), ([0, 1.0, 5.0, 100], 25), ([10, 2.0, 0.5, 60], 5), ([1.0, 3.0, 50], 20))):
        assert scheduled_value(spec, step) == pytest.approx(float(rv(f"C_{i}", lambda: ns["C"](spec, step, None))))
    names = ["alpha_penalty_loss", "mean_penalty_loss", "scale_penalty_loss", "auxiliary_loss"]
    ns = defs("gs/gaussian_splatting.py", names, dict(ns, torch=torch), in_class="GaussianSplattingRenderer")

    class W:
        def __init__(self):
            self.s = {}

        def add_scalar(self, k, v, step=None):
            self.s[k] = float(v)

    NS = types.SimpleNamespace
    for kind_a, kind_m in (("center_weighted", "weighted_l2"), ("uniform_l2", "uniform_l1")):
        pen = {"alpha": {"type": kind_a, "value": [0, 10.0, 100.0, 200]}, "mean": {"type": kind_m, "value": 0.5},
               "scale": {"value": 2.0}}
        r, cam = _renderer(gold, "a", oracle_mod, cfg={"penalty": pen})
        step = 50
        w_ours, w_ref = W(), W()
        ours = r.auxiliary_loss(step, w_ours)
        ours.backward()
        g_ours = {k: r.store.grad_views[k].clone() for k in ("mean", "svec", "alpha")}
        # the reference's methods on a stand-in that exposes the same activated views of fresh leaves
        leaves = {k: r.store.params[k].detach().clone().requires_grad_() for k in ("mean", "svec", "alpha")}

        def reference_loss():
            ref_self = NS(cfg=NS(penalty=NS(alpha=NS(**pen["alpha"]), mean=NS(**pen["mean"]), scale=NS(**pen["scale"]))),
                          mean=leaves["mean"], alpha=torch.sigmoid(leaves["alpha"]), svec=torch.exp(leaves["svec"]))
            ref_self.cfg.penalty.__iter__ = None
            for n in names[:3]:
                setattr(ref_self, n, types.MethodType(ns[n], ref_self))

            class Pen(dict):  # `for key in self.cfg.penalty` + attribute access
                __getattr__ = dict.__getitem__

            ref_self.cfg = NS(penalty=Pen({k: NS(**v) for k, v in pen.items()}))
            ref = ns["auxiliary_loss"](ref_self, step, w_ref)
            ref.backward()
            return float(ref)

        tag = f"{kind_a}_{kind_m}"
        assert float(ours) == pytest.approx(float(rv(tag + "_loss", reference_loss)), rel=1e-6)
        for k in g_ours:
            assert torch.allclose(g_ours[k], torch.from_numpy(rv(f"{tag}_grad_{k}", lambda: leaves[k].grad)),
                                  rtol=1e-5, atol=1e-9), k
        ref_keys = [str(k) for k in rv(tag + "_scalar_keys", lambda: sorted(w_ref.s))]
        assert sorted(w_ours.s) == ref_keys
        for k in ref_keys:
            assert w_ours.s[k] == pytest.approx(float(rv(f"{tag}_scalar_{k}", lambda: w_ref.s[k])), rel=1e-6), k
    rv.save()
    # log(): smoke (tags the reference writes)
    w = W()
    w.h = {}
    w.add_histogram = lambda k, v, step=None: w.h.__setitem__(k, len(v))
    r.log(w, 3)
    assert "renderer/num_gaussians" in w.s and "renderer/alpha/grad_max" in w.s and "hists/max_radii2d" in w.h
    # the tag set of the reference's log / log_bounds / log_grad_bounds / log_statistics (:1477-1549) for one rendered view
    r.render_one(gold["a_c2w"], cam, rgb_only=True)
    assert r.total_dub_gaussians == int(gold["a_N_with_dub"])
    w2 = W()
    w2.h = {}
    w2.add_histogram = lambda k, v, step=None: w2.h.__setitem__(k, len(v))
    r.log(w2, 3)
    want = {"renderer/num_gaussians", "renderer/n_gaussians_with_dub"} | {
        f"renderer/{f}/{k}" for f in ("mean", "qvec", "svec", "color", "alpha") for k in ("min", "max", "mean", "grad_min", "grad_max")}
    assert want <= set(w2.s), want - set(w2.s)
    assert {"hists/mean", "hists/svec_min", "hists/svec_max", "hists/alpha", "hists/grad_mean", "hists/max_radii2d"} <= set(w2.h)
    assert not r.is_densifying and "hists/cnt" not in w2.h  # no densify block in this cfg (:163-169, :1486-1487)


def test_render_one_overrides_recolour_a_view(gold, oracle_mod):
    """render_one(..., overrides={"color": activated}) (gs/gaussian_splatting.py:1179-1183, utils/relight.py:64): the
    view equals the one of a renderer whose colour leaf IS that colour, gradients reach the override tensor and -- for
    the fields that were not overridden -- the arena"""
    def fn(mean, qvec, svec, alpha, c2w, cam, color=None, bg=None, rgb_only=False, raw_params=False, grad_sink=None,
           slot=0, frustum_radius=6.0, tile_radius=6.0, T_thresh=1e-4, skip_frustum_culling=False, depth_detach=True):
        s, a, c = (torch.exp(svec), torch.sigmoid(alpha), torch.sigmoid(color)) if raw_params else (svec, alpha, color)
        out = oracle_mod.render_view(mean, qvec, s, a, c2w, ocam_of(cam), color=c, bg=bg, rgb_only=rgb_only,
                                     depth_detach=depth_detach, frustum_radius=frustum_radius, tile_radius=tile_radius,
                                     thresh=T_thresh)
        au = out["aux"]
        out["aux"] = _Aux(mask=au["mask"], mean2d_masked=au["mean2d"], radii2d=torch.zeros(mean.shape[0]),
                          N_with_dub=au["D"])
        out.setdefault("T", None)
        return out

    init = {k: gold[f"a_in_{k}"] for k in ("mean", "qvec", "svec", "color", "alpha")}
    fx, fy, cx, cy, w, h, near, far = gold["a_cam"].tolist()
    cam = CameraInfo(fx, fy, cx, cy, int(w), int(h), near, far)
    c2w = gold["a_c2w"]
    g = torch.Generator().manual_seed(9)
    new_color = (torch.rand(init["color"].shape, generator=g) * 0.9 + 0.05).requires_grad_()
    r = GaussianSplattingRenderer({}, init, device="cpu", render_fn=fn)
    r.store.zero_grad()
    img = r.render_one(c2w, cam, use_bg=False, rgb_only=True, overrides={"color": new_color})["rgb"]
    r2 = GaussianSplattingRenderer({}, dict(init, color=new_color.detach()), device="cpu", render_fn=fn)
    ref = r2.render_one(c2w, cam, use_bg=False, rgb_only=True)["rgb"]
    assert torch.allclose(img, ref, atol=2e-6) and float((img - r.render_one(c2w, cam, use_bg=False, rgb_only=True)["rgb"]).abs().max()) > 1e-3
    img.sum().backward()
    assert new_color.grad is not None and float(new_color.grad.abs().max()) > 0
    assert float(r.store.grad_views["mean"].abs().max()) > 0  # not overridden: gradient lands in the arena
    assert float(r.store.grad_views["color"].abs().max()) == 0  # overridden: the colour leaf took no part
    with pytest.raises(RuntimeError):
        r.render_one(c2w, cam, overrides={"sh": new_color})
