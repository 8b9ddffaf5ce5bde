"""`GaussianSplattingRenderer` as the reference's trainer sees it (SURVEY.md §8(b), "autograd surface above"), built
from the pieces of this package:

    reference (gs/gaussian_splatting.py)                         here
    ---------------------------------------------------------    ------------------------------------------------------
    raw leaves as nn.Parameters, activations in properties       `GaussianStore` capacity arena (raw leaves are views of it)
    render_one: ~60 torch kernels + 5 `_gs` calls per view       `rasterizer.render_view(raw_params=True, grad_sink=...)`
    forward(batch): sequential views, stack_dicts (:1426-1460)   `__call__(batch)`
    set_optimizer / update_lr: torch Adam, one group per field   `FlatAdam` over the arena, per-field lr schedules
    post_backward -> update_densify_info (:464-469, :1471-1476)  `post_backward()`
    densify(step) / prune(step) with optimizer surgery           `store.densify_step / prune_step` (row operations)
    get_params_for_save / load (:294-339)                        same keys

The trainer loop of the reference (`trainer.py:575-617`) then reads:

    renderer.update(step); out = renderer(batch, use_bg, rgb_only); loss.backward()
    renderer.optimizer.step(); renderer.post_backward(); renderer.densify(step); renderer.prune(step)
    renderer.optimizer.zero_grad()

Only the default configuration of the reference is covered: exp / sigmoid / sigmoid activations, RGB colours (no PBR
shading, no learned normals), a constant or per-pixel background, and `normal_as_rgb` (normals estimated from the means,
rendered as colours: gsgen_b200/normals.py).  `render_fn` exists so that this host logic can be
exercised without a GPU (the test-suite plugs in the CPU oracle); the default is the CUDA path and there is no
fallback.
"""
from __future__ import annotations

from typing import Callable, Dict, Optional, Sequence

import torch
import torch.nn.functional as F

from .store import GaussianStore, quat_to_rotmat

FIELDS = ("mean", "qvec", "svec", "color", "alpha")  # self.fields of the reference (:241-258)


def _get(cfg, key, default=None):
    if cfg is None:
        return default
    if hasattr(cfg, "get"):
        return cfg.get(key, default)
    return getattr(cfg, key, default)


def scheduled_value(value, step, max_steps=None) -> float:
    """utils/misc.py:218-250 `C(value, step)`: a number, or [start_step, start_value, end_value, end_step] (3 entries:
    start_step = 0) linearly interpolated and clamped; a FLOAT end_step means a fraction of max_steps."""
    if isinstance(value, (int, float)):
        return value
    value = list(value)
    if len(value) == 3:
        value = [0] + value
    if len(value) != 4:
        raise TypeError(f"Scalar specification only supports a number or a list of 3 / 4 entries, got {value}")
    start_step, start_value, end_value, end_step = value
    if isinstance(end_step, int):
        current = step
    else:
        if max_steps is None:
            raise ValueError("max_steps must be specified when using float step")
        current = end_step * max_steps
    return start_value + (end_value - start_value) * max(min(1.0, (current - start_step) / (end_step - start_step)), 0.0)


def _scalar(writer, tag, value, step):
    if writer is not None and hasattr(writer, "add_scalar"):
        writer.add_scalar(tag, value.item() if torch.is_tensor(value) else value, step)


def stack_dicts(dicts: Sequence[Dict[str, torch.Tensor]]) -> Dict[str, torch.Tensor]:
    """utils/misc.py:180-184"""
    return {k: torch.stack([d[k] for d in dicts], dim=0) for k in dicts[0].keys()}


class GaussianSplattingRenderer:
    """cfg: mapping with the renderer keys the hot path consumes (conf/renderer/base.yaml): tile_size (16),
    frustum_culling_radius, tile_culling_radius, T_thresh, depth_detach, skip_frustum_culling, densify{...},
    prune{...}.  initial_values: {"mean","qvec","svec","color","alpha"[, "raw"]} -- activated values unless raw
    (initialize(), :166-191)."""

    def __init__(self, cfg, initial_values: Dict[str, torch.Tensor], device="cuda", capacity: Optional[int] = None,
                 background=None, render_fn: Optional[Callable] = None, group=None, knn_fn: Optional[Callable] = None):
        self.cfg = cfg
        self.device = torch.device(device)
        if _get(cfg, "tile_size", 16) != 16:
            raise RuntimeError("tile_size must be 16")
        for key, want in (("svec_act", "exp"), ("alpha_act", "sigmoid"), ("color_act", "sigmoid")):
            if _get(cfg, key, want) != want:
                raise NotImplementedError(f"{key}={_get(cfg, key)}: the fused front end implements {want}")
        raw = bool(initial_values.get("raw", False))
        f32 = lambda t: torch.as_tensor(t, dtype=torch.float32)
        leaves = {"mean": f32(initial_values["mean"]), "qvec": f32(initial_values["qvec"])}
        svec, color, alpha = f32(initial_values["svec"]), f32(initial_values["color"]), f32(initial_values["alpha"])
        leaves["svec"] = svec if raw else torch.log(svec)              # inv_activations["exp"]
        leaves["color"] = color if raw else torch.logit(color)         # inv_activations["sigmoid"]
        leaves["alpha"] = (alpha if raw else torch.logit(alpha)).reshape(-1)
        self.store = GaussianStore(leaves, None, self.device, capacity=capacity, group=group, knn_fn=knn_fn)
        # None (black), a [3] tensor, or callable(rays_d[H,W,3]) -> [H,W,3]; with none given, cfg.background builds the
        # reference's background module (setup_bg, :207-218; gsgen_b200/backgrounds.py)
        if background is None and _get(cfg, "background", None) is not None:
            from .backgrounds import make_background

            background = make_background(_get(cfg, "background")).to(self.device)
        self.background = background
        self.training = True
        self.step = 0
        self.optimizer = None
        self._lr_cfg = None
        self._pending = []  # (mask, aux) of the views rendered since the last post_backward
        if render_fn is None:
            from .rasterizer import render_view as render_fn  # the CUDA path; raises without libgsb200.so / a GPU
        self._render_fn = render_fn

    # ---- the attributes the reference exposes ------------------------------------------------------------
    @property
    def N(self) -> int:
        return self.store.N

    mean = property(lambda self: self.store.params["mean"])
    qvec = property(lambda self: self.store.params["qvec"])
    svec_before_activation = property(lambda self: self.store.params["svec"])
    color_before_activation = property(lambda self: self.store.params["color"])
    alpha_before_activation = property(lambda self: self.store.params["alpha"])
    svec = property(lambda self: torch.exp(self.store.params["svec"]))
    color = property(lambda self: torch.sigmoid(self.store.params["color"]))
    alpha = property(lambda self: torch.sigmoid(self.store.params["alpha"]))
    rotmat = property(lambda self: quat_to_rotmat(self.store.params["qvec"]))  # :150-152 (kornia quat -> R)
    principal_axis = rotmat                                                     # :146-148
    # `cov` is qsvec2rotmat_batched(qvec, svec) in the reference (:154-156, utils/transforms.py:34-46):
    # `svec.unsqueeze(-2) * R_q`, i.e. the rotation matrix with column j scaled by svec[j] (M = R diag(s)) -- not a
    # covariance matrix, despite the name
    cov = property(lambda self: self.svec.unsqueeze(-2) * quat_to_rotmat(self.store.params["qvec"]))
    bg = property(lambda self: self.background)                                 # the attribute name the reference uses

    @property
    def normal(self) -> torch.Tensor:
        """:1189-1196, the `normal_type: "estimated"` branch: one normal per Gaussian from the means,
        `estimate_normal(self.mean, **cfg.normal)` (the function's defaults where cfg has no `normal` block); the
        gradient reaches `mean` through it.  `knn_fn` (CPU test-suite) feeds it as it feeds the compactness rules."""
        from .normals import estimate_normal

        c = _get(self.cfg, "normal", None)
        return estimate_normal(self.mean, neighborhood_size=_get(c, "neighborhood_size", 50),
                               disambiguate_directions=_get(c, "disambiguate_directions", True), knn=self.store.knn_fn)

    def update_normal(self) -> torch.Tensor:
        """:1185-1187.  The reference assigns to the read-only `normal` property there (an AttributeError on an
        nn.Module, so its normal_as_rgb path never ran); here it returns the estimate the property defines."""
        return self.normal

    @property
    def is_densifying(self) -> bool:
        """:163-169"""
        d = _get(self.cfg, "densify", None)
        return bool(d is not None and _get(d, "enabled", False) and _get(d, "warm_up", 0) < self.step < _get(d, "end", 0))

    def train(self, mode: bool = True):
        self.training = mode
        if isinstance(self.background, torch.nn.Module):  # nn.Module.train() reaches the background in the reference
            self.background.train(mode)
        return self

    def eval(self):
        return self.train(False)

    # ---- optimizer -----------------------------------------------------------------------------------------
    def setup_lr(self, lr_cfg):
        """cfg.lr (conf/base.yaml:12-26): field -> number | [start, end, steps, type]; `bg` is the background's group"""
        self._bg_lr = _get(lr_cfg, "bg")
        self._lr_cfg = {f: _get(lr_cfg, f) for f in FIELDS}
        missing = [f for f, v in self._lr_cfg.items() if v is None]
        if missing:
            raise RuntimeError(f"no learning rate for {missing}")

    def set_optimizer(self, opt_cfg=None, step: int = 0):
        """cfg.optimizer (conf/base.yaml:8-11): type Adam, opt_args {eps: 1e-15}"""
        if self._lr_cfg is None:
            raise RuntimeError("call setup_lr(cfg.lr) first (trainer.py:162-163)")
        if _get(opt_cfg, "type", "Adam") != "Adam":
            raise NotImplementedError("only Adam (the reference's optimizer surgery is Adam-only too, :421-423)")
        args = _get(opt_cfg, "opt_args", None) or {}
        self.optimizer = self.store.make_optimizer(self._lr_cfg, max_steps=_get(opt_cfg, "max_steps", 15000),
                                                   betas=tuple(_get(args, "betas", (0.9, 0.999))),
                                                   eps=float(_get(args, "eps", 1e-8)))
        # the background's parameters are param group "bg" of the same Adam in the reference (:383-396); here they are
        # the only parameters outside the arena and ride along as a companion of the flat optimizer
        bg_params = [p for p in self.background.parameters()] if isinstance(self.background, torch.nn.Module) else []
        if bg_params:
            if getattr(self, "_bg_lr", None) is None:
                raise RuntimeError("no learning rate for 'bg' (cfg.lr.bg, conf/base.yaml:26): the background module "
                                   "has parameters")
            from .optim import CompanionAdam

            self.optimizer.companions = [CompanionAdam(
                bg_params, self._bg_lr, max_steps=_get(opt_cfg, "max_steps", 15000),
                betas=tuple(_get(args, "betas", (0.9, 0.999))), eps=float(_get(args, "eps", 1e-8)))]
        self.optimizer.train_step = step
        self.store.zero_grad()
        return self.optimizer

    def update(self, step: int):
        """update(step) -> update_lr(step) (:451-462): the schedules are evaluated at the trainer's step"""
        self.step = step
        if self.optimizer is not None:
            self.optimizer.train_step = step

    # ---- rendering -----------------------------------------------------------------------------------------
    def _bg_image(self, camera_info, c2w, use_bg: bool):
        H, W = camera_info.h, camera_info.w
        if not use_bg or self.background is None:
            return None
        if callable(self.background):
            return self.background(camera_info.get_rays_d(c2w).to(self.device)).contiguous()
        return self.background.to(self.device).reshape(1, 1, 3).expand(H, W, 3).contiguous()

    def render_one(self, c2w, camera_info, use_bg: bool = True, rgb_only: bool = False, overrides=None,
                   return_T: bool = False):
        """render_one (:1198-1421), same positional order.  `overrides`: {field: ACTIVATED tensor} replacing
        `self.<field>` for this view (get_with_overrides :1179-1183; utils/relight.py:64 re-colours a scene with it) --
        the view then runs on activated values (`raw_params=False`), gradients flow to the leaves through torch's own
        exp / sigmoid and to the override tensors directly."""
        p = self.store.params
        leaves, raw = (p["mean"], p["qvec"], p["svec"], p["alpha"], p["color"]), True
        if overrides:
            unknown = [k for k in overrides if k not in FIELDS]
            if unknown:
                raise RuntimeError(f"overrides for unknown fields {unknown}")
            act = {f: (overrides[f] if f in overrides else getattr(self, f)) for f in FIELDS}
            leaves, raw = (act["mean"], act["qvec"], act["svec"], act["alpha"], act["color"]), False
        return self._render(leaves, raw, raw, c2w, camera_info, use_bg, rgb_only, return_T)

    def _render(self, leaves, raw: bool, sink: bool, c2w, camera_info, use_bg, rgb_only, return_T):
        """one view of (mean, qvec, svec, alpha, color): raw leaves (activations in the kernels) or activated values;
        `sink`: gradients go straight into the arena's flat gradient buffer (only when every leaf IS an arena leaf)"""
        out = self._render_fn(
            leaves[0], leaves[1], leaves[2], leaves[3], c2w, camera_info, color=leaves[4],
            bg=self._bg_image(camera_info, c2w, use_bg), rgb_only=rgb_only, raw_params=raw,
            frustum_radius=_get(self.cfg, "frustum_culling_radius", 6.0),
            tile_radius=_get(self.cfg, "tile_culling_radius", 6.0), T_thresh=_get(self.cfg, "T_thresh", 1e-4),
            skip_frustum_culling=_get(self.cfg, "skip_frustum_culling", False),
            depth_detach=_get(self.cfg, "depth_detach", True),
            # (the flat gradient sink holds gradients w.r.t. the RAW leaves: only the raw-leaf path may write into it)
            grad_sink=self.store.grad_views if (self.training and sink) else None,
            # one library context per in-flight view: the views of a batch are all rendered before ONE loss.backward()
            # (trainer.py:575-599), and a context keeps a view's binning + splat records until its backward has run
            slot=len(self._pending) if self.training else 0)
        aux = out["aux"]
        try:  # `self.total_dub_gaussians = N_with_dub` (:1264); -1 while unresolved in the asynchronous count mode
            self.total_dub_gaussians = int(aux["N_with_dub"])
        except (KeyError, TypeError, ValueError):
            self.total_dub_gaussians = None
        if self.training:
            self._pending.append(aux)  # mask + mean2d gradient are read in post_backward (:1246-1250)
        res = {"rgb": out["rgb"]}
        if not rgb_only:  # (the reference's eval-mode `out = out.clamp(0, 1)` at :1405-1406 rebinds a local AFTER
            # outputs["rgb"] was stored, so the returned image is never clamped -- reproduced by not clamping)
            res.update(depth=out["depth"], opacity=out["opacity"], z_var=out["z_var"])
        if return_T:
            res["T"] = out["T"]
        return res

    def __call__(self, batch, use_bg: bool = True, rgb_only: bool = False):
        """forward(batch) (:1426-1460): batch["c2w"] [bs,3,4] (host or device), batch["camera_info"] list"""
        c2ws, infos = batch["c2w"], batch["camera_info"]
        if not _get(self.cfg, "normal_as_rgb", False):
            return stack_dicts([self.render_one(c2ws[i], infos[i], use_bg, rgb_only) for i in range(len(infos))])
        # cfg.normal_as_rgb (:1427-1430, :1462-1463): the normals, estimated once per batch, replace the colours of
        # every view; the composited colour is normalised back to a direction and mapped to [0, 1]
        # The views run on the raw arena leaves with the colour leaf replaced by logit((n + 1) / 2) -- the kernels'
        # sigmoid gives the colour back to fp32 rounding (logit clamped at 1e-6 from 0 and 1, where a normal component
        # is exactly -1 or 1) -- and without the flat gradient sink, so autograd takes the colour gradient to the
        # normals and from there to `mean`, and the colour leaf gets none.  Same image as
        # render_one(overrides={"color": (n + 1) / 2}) to ~1e-6, on the raw-leaf path every render_fn provides.
        p = self.store.params
        col = torch.logit((self.update_normal() + 1.0) * 0.5, eps=1e-6)
        leaves = (p["mean"], p["qvec"], p["svec"], p["alpha"], col)
        out = stack_dicts([self._render(leaves, True, False, c2ws[i], infos[i], use_bg, rgb_only, False)
                           for i in range(len(infos))])
        out["rgb"] = (F.normalize(out["rgb"], dim=-1, eps=1e-6) + 1.0) / 2.0
        return out

    forward = __call__

    # ---- after the backward pass ---------------------------------------------------------------------------
    def post_backward(self):
        """update_densify_info for every view of the step (:464-469, :1471-1476)"""
        if self.training:
            for aux in self._pending:
                self.store.update_densify_info(aux["mask"], aux["mean2d_grad"], aux.get("radii2d"))
        self._pending = []

    def densify(self, step: int):
        return self.store.densify_step(step, _get(self.cfg, "densify", {"enabled": False}))

    def prune(self, step: int):
        return self.store.prune_step(step, _get(self.cfg, "prune", {"enabled": False}))

    # called directly by the trainer's up-sampling fine-tune stage (trainer.py:799-801)
    def densify_by_compatness(self, K: int = 1) -> int:
        """:682-694"""
        return self.store.densify_by_compatness(K=K)

    def reset_densify_info(self):
        """:476-479"""
        self.store.reset_densify_info()

    # ---- auxiliary losses (gs/gaussian_splatting.py:950-1122) ----------------------------------------------
    def _penalty_cfg(self, key):
        pen = _get(self.cfg, "penalty", None)
        return None if pen is None else _get(pen, key, None)

    def alpha_penalty_loss(self, step, writer=None):
        """:950-970 -- "uniform_l1" | "uniform_l2" | "center_weighted" (the shipped configs, conf/renderer/*.yaml:50-53)"""
        c = self._penalty_cfg("alpha")
        w = scheduled_value(_get(c, "value", 0.0), step) if c is not None else 0.0
        if not w > 0.0:
            return torch.zeros_like(self.alpha[0], requires_grad=False)
        kind = _get(c, "type")
        if kind == "uniform_l1":
            pen = torch.mean(self.alpha)
        elif kind == "uniform_l2":
            pen = torch.mean(self.alpha ** 2)
        elif kind == "center_weighted":
            pen = torch.mean(self.mean.detach().norm(dim=-1) * self.alpha)
        else:
            raise ValueError(f"Unknown alpha penalty type: {kind}")
        _scalar(writer, "auxiliary/alpha_penalty", pen, step)
        _scalar(writer, "auxiliary/alpha_penalty_weight", w, step)
        return w * pen

    def mean_penalty_loss(self, step, writer=None):
        """:972-999"""
        c = self._penalty_cfg("mean")
        w = scheduled_value(_get(c, "value", 0.0), step) if c is not None else 0.0
        if not w > 0.0:
            return torch.zeros_like(self.alpha[0], requires_grad=False)
        kind, r = _get(c, "type"), self.mean.norm(dim=-1)
        if kind == "uniform_l1":
            pen = torch.mean(r)
        elif kind == "uniform_l2":
            pen = torch.mean(r ** 2)
        elif kind == "weighted_l1":
            pen = torch.mean(r.detach() * r)
        elif kind == "weighted_l2":
            pen = torch.mean(r.detach() ** 2 * r ** 2)
        else:
            raise ValueError(f"Unknown mean penalty type: {kind}")
        _scalar(writer, "auxiliary/mean_penalty", pen, step)
        _scalar(writer, "auxiliary/mean_penalty_weight", w, step)
        return w * pen

    def scale_penalty_loss(self, step, writer=None):
        """:1001-1013 (total volume prod(svec).sum())"""
        c = self._penalty_cfg("scale")
        w = scheduled_value(_get(c, "value", 0.0), step) if c is not None else 0.0
        if not w:
            return torch.zeros_like(self.alpha[0], requires_grad=False)
        volume = self.svec.prod(dim=-1).sum()
        _scalar(writer, "auxiliary/scale_penalty", volume, step)
        _scalar(writer, "auxiliary/scale_penalty_weight", w, step)
        return w * volume

    def NN_penalty_loss(self, step, writer=None):
        """:1032-1046: mean distance to the nearest other Gaussian (the neighbour is found under no_grad and enters as
        a constant, utils/ops.py:103-114); the search is gsb200_knn (csrc/knn.cu)."""
        from .knn import nearest_neighbor

        c = self._penalty_cfg("NN")
        w = scheduled_value(_get(c, "value", 0.0), step) if c is not None else 0.0
        if not w > 0.0:
            return torch.zeros_like(self.alpha[0], requires_grad=False)
        nn_pos, _ = nearest_neighbor(self.mean, knn=self.store._knn())
        pen = torch.mean((self.mean - nn_pos).norm(dim=-1))
        _scalar(writer, "auxiliary/NN_penalty", pen, step)
        _scalar(writer, "auxiliary/NN_penalty_weight", w, step)
        return w * pen

    def compat_penalty_loss(self, step, writer=None):
        """:1048-1094: the gap between every Gaussian's "surface" and its nearest neighbour's along the line of centres
        (utils/ops.py:137-158), where there is one -- "l1" mean gap or "l2" mean squared gap over ALL Gaussians."""
        from .knn import distance_to_gaussian_surface, nearest_neighbor

        c = self._penalty_cfg("compat")
        w = scheduled_value(_get(c, "value", 0.0), step) if c is not None else 0.0
        if not w > 0.0:
            return torch.zeros_like(self.alpha[0], requires_grad=False)
        _, idx = nearest_neighbor(self.mean, knn=self.store._knn())
        svec, rotmat, mean = self.svec, self.rotmat, self.mean
        nn_svec, nn_rotmat, nn_pos = svec[idx], rotmat[idx], mean[idx]
        nn_surface = distance_to_gaussian_surface(nn_pos, nn_svec, nn_rotmat, mean)
        surface = distance_to_gaussian_surface(mean, svec, rotmat, nn_pos)
        dist_to_nn = torch.norm(nn_pos - mean, dim=-1)
        mask = (surface + nn_surface) < dist_to_nn
        kind = _get(c, "type")
        if kind == "l1":
            pen = torch.mean((dist_to_nn - surface - nn_surface) * mask)
        elif kind == "l2":
            pen = torch.mean((dist_to_nn - surface - nn_surface) ** 2 * mask)
        else:
            raise ValueError(f"Unknown compat penalty type: {kind}")
        _scalar(writer, "auxiliary/compat_penalty", pen, step)
        _scalar(writer, "auxiliary/effective_rate", torch.sum(mask).item() / self.N, step)
        _scalar(writer, "auxiliary/compat_penalty_weight", w, step)
        return w * pen

    def auxiliary_loss(self, step, writer=None):
        """:1115-1122: the sum of `<key>_penalty_loss` over cfg.penalty.  Not built: `move` (the reference reads
        `self.prev_mean`, which nothing ever sets, :1015-1030) and the PBR ones (normal, specular: fields outside the
        hot path); they raise here."""
        loss = 0.0
        pen = _get(self.cfg, "penalty", None) or {}
        for key in (pen.keys() if hasattr(pen, "keys") else vars(pen)):
            fn = getattr(self, f"{key}_penalty_loss", None)
            if fn is None:
                raise NotImplementedError(f"penalty '{key}' is not part of the rasterizer hot path")
            loss = loss + fn(step, writer)
        if torch.is_tensor(loss):
            _scalar(writer, "auxiliary/total", loss, step)
        return loss

    # ---- logging (gs/gaussian_splatting.py:1477-1565) --------------------------------------------------------
    @torch.no_grad()
    def log(self, writer, step):
        """scalars / histograms the reference writes: parameter bounds, gradient bounds, learning rates, densification
        statistics.  `writer`: anything with add_scalar / add_histogram (tensorboard SummaryWriter)."""
        _scalar(writer, "renderer/num_gaussians", self.N, step)
        if getattr(self, "total_dub_gaussians", None) is not None:  # (:1493-1495) N_with_dub of the last rendered view
            _scalar(writer, "renderer/n_gaussians_with_dub", self.total_dub_gaussians, step)
        st = self.store
        for field in FIELDS:
            v = getattr(self, field)
            _scalar(writer, f"renderer/{field}/min", v.abs().min(), step)
            _scalar(writer, f"renderer/{field}/max", v.abs().max(), step)
            _scalar(writer, f"renderer/{field}/mean", v.mean(), step)
            g = st.grad_views[field]
            _scalar(writer, f"renderer/{field}/grad_min", g.abs().min(), step)
            _scalar(writer, f"renderer/{field}/grad_max", g.abs().max(), step)
        if self.optimizer is not None:
            for name, lr in self.optimizer.lr_at(self.step).items():
                _scalar(writer, f"lr/{name}", lr, step)
            for c in getattr(self.optimizer, "companions", ()):  # the "bg" param group (:1551-1558)
                _scalar(writer, "lr/bg", float(c.scheduler(self.step)), step)
        if hasattr(writer, "add_histogram"):
            writer.add_histogram("hists/mean", self.mean.norm(dim=-1).cpu().numpy(), step)
            writer.add_histogram("hists/svec_min", self.svec.min(dim=-1)[0].cpu().numpy(), step)
            writer.add_histogram("hists/svec_max", self.svec.max(dim=-1)[0].cpu().numpy(), step)
            writer.add_histogram("hists/alpha", self.alpha.cpu().numpy(), step)
            writer.add_histogram("hists/grad_mean", st.grad_views["mean"].norm(dim=-1).cpu().numpy(), step)
            writer.add_histogram("hists/max_radii2d", st.max_radii2d.cpu().numpy(), step)
            if self.is_densifying:  # (:1486-1487)
                writer.add_histogram("hists/grad_mean2d", st.mean_2d_grad_accum.cpu().numpy(), step)
                writer.add_histogram("hists/cnt", st.cnt.cpu().numpy(), step)

    # ---- checkpoints ---------------------------------------------------------------------------------------
    def get_params_for_save(self):
        """gs/gaussian_splatting.py:294-303: the raw leaves + `cfg` + `bg` (the reference's `load` does
        OmegaConf.create(ckpt["cfg"]) and utils/export.to_ply / to_splat read ckpt["cfg"]["prompt"]).  Optimizer state is
        not part of a renderer checkpoint in the reference either."""
        params = self.store.get_params_for_save()
        cfg = self.cfg
        if hasattr(cfg, "items"):  # a plain container (OmegaConf.to_container in the reference)
            cfg = {k: (dict(v) if hasattr(v, "items") else v) for k, v in cfg.items()}
        params["cfg"] = cfg if cfg is not None else {}
        bg = self.background
        params["bg"] = bg.state_dict() if hasattr(bg, "state_dict") else ({} if bg is None or callable(bg)
                                                                           else {"color": torch.as_tensor(bg).cpu()})
        return params

    @classmethod
    def load(cls, cfg, ckpt, device="cuda", **kw) -> "GaussianSplattingRenderer":
        """`load(cfg, ckpt)` (:312-339): a path or dict; a renderer-only checkpoint (the params incl. its own `cfg`) or a
        trainer checkpoint (`{"params", "cfg": {... "renderer": ...}}`).  The configuration stored in the checkpoint is
        the base, `cfg` (may be None, as in vis.py:17) overrides it key by key; the background's state is restored when
        it fits (the reference only prints a message when it does not)."""
        if not isinstance(ckpt, dict):
            ckpt = torch.load(ckpt, map_location="cpu")
        stored = ckpt.get("cfg") or {}
        if "params" in ckpt:
            stored = _get(stored, "renderer", None) or {}
            ckpt = ckpt["params"]
            stored = _get(ckpt, "cfg", None) or stored  # (our get_params_for_save keeps the renderer cfg with the params)
        merged = dict(stored.items()) if hasattr(stored, "items") else {}
        if cfg is not None:
            merged.update(dict(cfg.items()) if hasattr(cfg, "items") else vars(cfg))
        r = cls(merged, dict({k: ckpt[k] for k in FIELDS}, raw=True), device, **kw)
        bg_state = ckpt.get("bg") if hasattr(ckpt, "get") else None
        if bg_state and isinstance(r.background, torch.nn.Module):
            try:
                r.background.load_state_dict(bg_state)
            except Exception:  # "the background will be randomly initialized" (:333-337)
                pass
        return r

    def to(self, device) -> "GaussianSplattingRenderer":
        """nn.Module.to as vis.py:17 uses it (`load(None, ckpt).to("cuda")`): the arena moves to `device` (parameters,
        gradients, Adam moments, statistics); an optimizer has to be set again afterwards, as after a fresh load"""
        device = torch.device(device)
        if device.type == self.device.type and (device.index is None or device.index == self.device.index):
            return self
        old = self.store
        names = list(old._field)
        new = GaussianStore({n: old.params[n].detach() for n in names}, old.C, device, capacity=old.cap, group=old.group,
                            knn_fn=old.knn_fn)
        for src, dst in zip(old._buffers()[1:], new._buffers()[1:]):
            for n in names:
                new._rows(dst, n, new.N).copy_(old._rows(src, n, old.N))
        for a in ("mean_2d_grad_accum", "cnt", "max_radii2d"):
            setattr(new, a, getattr(old, a).to(device))
        self.store, self.device, self.optimizer = new, device, None
        if isinstance(self.background, torch.nn.Module):
            self.background.to(device)
        elif torch.is_tensor(self.background):
            self.background = self.background.to(device)
        self._pending = []
        return self
