"""Every renderer configuration the reference ships (conf/renderer/*.yaml, plus the `renderer:` blocks of the top-level
experiment files) drives `gsgen_b200.splatting.GaussianSplattingRenderer` through the trainer's call sequence on the CPU
(oracle as `render_fn`, brute-force search as `knn_fn`): construction incl. `setup_bg`, `setup_lr` / `set_optimizer`,
one batch forward + backward + `post_backward`, `auxiliary_loss`, and `densify(step)` / `prune(step)` at
a step where the config's own gates fire.  The yaml files are read where they lie when $GSB200_REFERENCE names the
reference (and then written to $GSB200_GOLDEN_OUT/shipped_renderer_configs.json when that is set); elsewhere their parsed
contents come from tests/golden/shipped_renderer_configs.json.  OmegaConf interpolations (`${device}`, `${max_steps}`) are resolved by hand.  What it pins: no shipped key is
unsupported or mis-read (densify types official / all / scale / compatness / shrink_then_compatness, the three prune
rules, penalty schedules, background types) -- the numerical parity of each piece is pinned elsewhere."""
import glob
import json
import os

import pytest
import torch
import yaml

from gsgen_b200.scenes import make_scene
from tests.test_splatting_cpu import _oracle_render_fn
from tests.util import GOLDEN

REF = os.environ.get("GSB200_REFERENCE")
CONF = os.path.join(REF, "conf") if REF else None
STORED = os.path.join(GOLDEN, "shipped_renderer_configs.json")
MAX_STEPS = 5000


def _resolve(x):
    if isinstance(x, dict):
        return {k: _resolve(v) for k, v in x.items()}
    if isinstance(x, list):
        return [_resolve(v) for v in x]
    if isinstance(x, str) and x.startswith("${"):
        key = x[2:-1]
        return {"device": "cpu", "max_steps": MAX_STEPS}.get(key, x)
    return x


def _read_configs():
    """{"<file relative to conf/>|<key or empty>": the renderer block as parsed}"""
    out = {}
    for path in sorted(glob.glob(os.path.join(CONF, "renderer", "*.yaml"))):
        d = yaml.safe_load(open(path))
        if isinstance(d, dict):  # (short.yaml is an empty file)
            out[os.path.relpath(path, CONF) + "|"] = d
    for path in sorted(glob.glob(os.path.join(CONF, "*.yaml"))):
        try:
            d = yaml.safe_load(open(path))
        except Exception:
            continue
        if isinstance(d, dict) and isinstance(d.get("renderer"), dict) and "densify" in d["renderer"]:
            out[os.path.relpath(path, CONF) + "|renderer"] = d["renderer"]
    out_dir = os.environ.get("GSB200_GOLDEN_OUT")
    if out_dir:
        os.makedirs(out_dir, exist_ok=True)
        json.dump(out, open(os.path.join(out_dir, os.path.basename(STORED)), "w"), indent=1, sort_keys=True)
    return out


CONFIGS = _read_configs() if CONF and os.path.isdir(CONF) else json.load(open(STORED))


# (None, None): no configuration file at all -- the renderer's own defaults (no densify, no prune, no background)
@pytest.mark.parametrize("rel,sub", [(None, None)] + [(k.split("|")[0], k.split("|")[1] or None) for k in CONFIGS])
def test_shipped_renderer_config_drives_the_renderer(oracle_mod, rel, sub):
    from gsgen_b200.splatting import GaussianSplattingRenderer

    cfg = _resolve(CONFIGS[f"{rel}|{sub or ''}"]) if rel is not None else {}
    if cfg.get("background", {}).get("type") == "mlp":
        cfg["background"] = dict(cfg["background"], type="fixed", color=[0.0, 0.0, 0.0])  # tinycudann: outside the path
    sc = make_scene("c1", N=300, reso=48)
    init = {"mean": sc.mean, "qvec": sc.qvec, "svec": sc.svec * 3.0, "color": sc.color.clamp(0.05, 0.95),
            "alpha": sc.alpha}
    r = GaussianSplattingRenderer(cfg, init, device="cpu", render_fn=_oracle_render_fn(oracle_mod),
                                  knn_fn=oracle_mod.knn_points)
    if "background" in cfg:
        assert r.bg is not None
    r.setup_lr({"mean": 1e-3, "qvec": 1e-3, "svec": 1e-3, "color": 1e-2, "alpha": 1e-2, "bg": 3e-3})
    r.set_optimizer({"type": "Adam", "opt_args": {"eps": 1e-15}})
    cam, c2w = sc.cams[0], sc.c2ws[0]
    dens, prune = cfg.get("densify", {}), cfg.get("prune", {})
    # a step at which this config's own gates fire (both period multiples, inside both windows, where possible)
    step = None
    for s in range(0, MAX_STEPS + 1, 100):
        ok_d = (not dens.get("enabled")) or (dens["warm_up"] <= s <= dens["end"] and s % dens["period"] == 0)
        ok_p = (not prune.get("enabled")) or (prune["warm_up"] <= s <= prune["end"] and s != 0 and s % prune["period"] == 0)
        if ok_d and ok_p and s > 0:
            step = s
            break
    assert step is not None, (rel, dens, prune)
    r.update(step)
    r.optimizer.zero_grad()
    out = r({"c2w": c2w[None], "camera_info": [cam]}, use_bg=True, rgb_only=False)
    loss = out["rgb"].square().mean() + out["opacity"].mean() * 0.1
    aux_loss = r.auxiliary_loss(step, None)
    (loss + aux_loss).backward()
    r.post_backward()  # (optimizer.step() is the CUDA kernel: tests/test_optim_gpu.py, tests/test_train_step_gpu.py)
    n0 = r.N
    res_d = r.densify(step)
    res_p = r.prune(step)
    if dens.get("enabled"):
        assert res_d is not None, (rel, step)
        assert r.store.cnt.shape[0] == r.N
    else:
        assert res_d is None
    if prune.get("enabled"):
        assert res_p is not None
    else:
        assert res_p is None
    assert r.N > 0 and all(r.store.params[f].shape[0] == r.N for f in ("mean", "qvec", "svec", "color", "alpha"))
    # the renderer keeps working on the new arena
    r.optimizer.zero_grad()
    out = r({"c2w": c2w[None], "camera_info": [cam]}, use_bg=True, rgb_only=True)
    out["rgb"].mean().backward()
    r.post_backward()
    assert torch.isfinite(out["rgb"]).all() and r.N >= 1
