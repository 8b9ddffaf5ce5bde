"""Shared helpers of the parity tests."""
import ctypes
import hashlib
import os
import re
import zlib

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

# Tolerances stated by BASELINE.json north_star: images within 1e-4 abs (fp32), gradients within 1e-3 rel.
IMG_ATOL = 1e-4
GRAD_RTOL = 1e-3


def note(line: str):
    """a measured number a test wants kept (timings, diff statistics): printed, and appended to $GSB200_TEST_NOTES when
    set (the GPU run scripts point it into gpurun_out/ so the line survives pytest's output capture)"""
    print("\n" + line)
    path = os.environ.get("GSB200_TEST_NOTES")
    if path:
        with open(path, "a") as f:
            f.write(line + "\n")


def fp(t):
    return ctypes.cast(t.data_ptr(), ctypes.POINTER(ctypes.c_float))


def ip(t):
    return ctypes.cast(t.data_ptr(), ctypes.POINTER(ctypes.c_int32))


def load_golden(name):
    path = os.path.join(GOLDEN, name + ".npz")
    if not os.path.exists(path):
        return None
    z = np.load(path)
    return {k: torch.from_numpy(z[k]) for k in z.files}


def golden_names():
    if not os.path.isdir(GOLDEN):
        return []
    # rasterizer fixtures are named g<k>_*.npz (tests/golden/make_golden.py); other fixtures share the directory
    return sorted(f[:-4] for f in os.listdir(GOLDEN) if f.endswith(".npz") and re.match(r"g\d+_", f))


def assert_image_close(ours, ref, margin=None, atol=IMG_ATOL, what="image", max_flip_frac=2e-3, flip_margin=2e-3):
    """|ours-ref| <= atol everywhere, EXCEPT at pixels where the reference itself sits on a discontinuity:
    the `a*G < 1/255 -> skip` test (A.6) makes the output jump by up to ~1/255*T when a*G crosses the threshold
    in the last ulp, so two correct implementations can legitimately differ there.  `margin` (from the oracle)
    is min over the pixel's evaluated pairs of |a*G*255 - 1|; a violation is accepted only if that pixel's margin
    is < flip_margin, the error is bounded by the size of one blend step, and such pixels are rare."""
    ours, ref = ours.detach().float().cpu(), ref.detach().float().cpu()
    assert ours.shape == ref.shape, (ours.shape, ref.shape)
    assert torch.isfinite(ours).all(), f"{what}: non-finite values"
    err = (ours - ref).abs()
    if err.dim() == 3:
        err = err.amax(dim=-1)
    bad = err > atol
    nbad = int(bad.sum())
    if nbad == 0:
        return float(err.max())
    assert margin is not None, f"{what}: {nbad} pixels exceed {atol} (max {float(err.max()):.3e})"
    m = margin.reshape(err.shape)
    not_explained = bad & ~(m < flip_margin)
    assert int(not_explained.sum()) == 0, (
        f"{what}: {int(not_explained.sum())} pixels exceed {atol} away from any 1/255 threshold "
        f"(max err {float(err[not_explained].max()):.3e})")
    assert float(err.max()) <= 8e-3, f"{what}: threshold-flip error {float(err.max()):.3e} larger than one blend step"
    assert nbad <= max(4, max_flip_frac * err.numel()), f"{what}: too many threshold-flip pixels ({nbad})"
    return float(err.max())


def assert_grad_close(ours, ref, rtol=GRAD_RTOL, what="grad", floor=1e-6):
    """Relative error of the whole tensor in the max norm and in the l2 norm, both <= rtol (x a small factor for
    l-inf).  Per-element relative error is meaningless for sums of thousands of signed fp32 atomics."""
    ours, ref = ours.detach().double().cpu().reshape(-1), ref.detach().double().cpu().reshape(-1)
    assert ours.shape == ref.shape, (ours.shape, ref.shape)
    assert torch.isfinite(ours).all(), f"{what}: non-finite values"
    scale = max(float(ref.abs().max()), floor)
    linf = float((ours - ref).abs().max()) / scale
    l2 = float((ours - ref).norm()) / max(float(ref.norm()), floor)
    assert l2 <= rtol, f"{what}: relative l2 error {l2:.3e} > {rtol} (linf {linf:.3e})"
    assert linf <= 5 * rtol, f"{what}: relative max error {linf:.3e} > {5 * rtol}"
    return l2


def ocam_of(cam):
    import oracle

    return oracle.Cam(cam.fx, cam.fy, cam.cx, cam.cy, cam.w, cam.h, cam.near_plane, cam.far_plane)


def classify_image_diff(ours, ref, margin_fn, exact_fn=None, atol=IMG_ATOL, what="image", flip_margin=2e-3,
                        max_flip_frac=2e-3, report=None, exact_self_fn=None):
    """Full-size parity of two fp32 implementations of the same composite (ours vs the reference extension).

    Every pixel with |ours - ref| > atol must be EXPLAINED, by one of
      (flip)     the pixel sits on the reference's `a*G < 1/255 -> skip` discontinuity: the oracle's margin
                 min|a*G*255 - 1| over the pixel's evaluated pairs is < flip_margin (error bounded by one blend step);
      (rounding) the two fp32 results straddle the real-arithmetic value: |ours - exact| <= atol where `exact` is the
                 fp64 arbiter (oracle.composite_sh_fwd_exact) -- i.e. OURS is within tolerance of the true value and
                 the remainder is the reference's own fp32 rounding (its `radial` formula, kernels.h:172-193, cancels
                 for thin Gaussians).
      (projection) only when the two sides composite DIFFERENT per-Gaussian inputs (the fused view against the reference
                 pipeline: each side projects the Gaussians itself, in fp32, with its own operation order): the pixel is
                 explained if OURS equals the fp64 composite of ITS OWN projected inputs (`exact_self_fn`) within atol, or
                 sits on a 1/255 threshold of those inputs.  For sub-pixel, thin splats (C5) the conic amplifies an ulp of
                 the projected covariance to ~1e-3 in a*G, enough to move a pair across the threshold although both
                 projections agree to fp32 rounding (checked separately by the caller).
    margin_fn() -> margin[H,W]; exact_fn() / exact_self_fn() -> (exact[H,W,3] f64, margin_exact[H,W]); all lazy.
    Returns a dict of counts (also appended to `report` when given)."""
    ours_c, ref_c = ours.detach().float().cpu(), ref.detach().float().cpu()
    assert ours_c.shape == ref_c.shape, (ours_c.shape, ref_c.shape)
    assert torch.isfinite(ours_c).all(), f"{what}: non-finite values"
    err = (ours_c - ref_c).abs()
    epix = err.amax(dim=-1) if err.dim() == 3 else err
    bad = epix > atol
    res = {"what": what, "pixels": int(epix.numel()), "max_abs_diff": float(epix.max()), "over_atol": int(bad.sum()),
           "atol": atol, "flip_explained": 0, "rounding_explained": 0, "unexplained": 0}
    if res["over_atol"]:
        margin = margin_fn().reshape(epix.shape)
        flip = bad & (margin < flip_margin)
        rest = bad & ~flip
        if int(rest.sum()) and exact_fn is not None:
            exact, margin_x = exact_fn()
            ex_err = (ours_c.double() - exact.reshape(ours_c.shape)).abs()
            ex_pix = ex_err.amax(dim=-1) if ex_err.dim() == 3 else ex_err
            ref_ex = (ref_c.double() - exact.reshape(ours_c.shape)).abs()
            ref_pix = ref_ex.amax(dim=-1) if ref_ex.dim() == 3 else ref_ex
            flip_x = rest & (margin_x.reshape(epix.shape) < flip_margin)
            flip = flip | flip_x
            rest = rest & ~flip_x
            rounding = rest & (ex_pix <= atol)
            res["rounding_explained"] = int(rounding.sum())
            res["ours_vs_exact_max_at_rounding"] = float(ex_pix[rounding].max()) if int(rounding.sum()) else 0.0
            res["ref_vs_exact_max_at_rounding"] = float(ref_pix[rounding].max()) if int(rounding.sum()) else 0.0
            res["ours_vs_exact_max_all"] = float(ex_pix.max())
            res["ref_vs_exact_max_all"] = float(ref_pix.max())
            rest = rest & ~rounding
        if int(rest.sum()) and exact_self_fn is not None:
            ex_s, margin_s = exact_self_fn()
            es = (ours_c.double() - ex_s.reshape(ours_c.shape)).abs()
            es_pix = es.amax(dim=-1) if es.dim() == 3 else es
            proj = rest & ((es_pix <= atol) | (margin_s.reshape(epix.shape) < flip_margin))
            res["projection_explained"] = int(proj.sum())
            res["ours_vs_exact_of_own_inputs_max"] = float(es_pix[proj].max()) if int(proj.sum()) else 0.0
            res["ours_vs_exact_of_own_inputs_max_all"] = float(es_pix.max())
            rest = rest & ~proj
        res["flip_explained"] = int(flip.sum())
        res["flip_max_err"] = float(epix[flip].max()) if int(flip.sum()) else 0.0
        res["unexplained"] = int(rest.sum())
        res["unexplained_max_err"] = float(epix[rest].max()) if int(rest.sum()) else 0.0
    if report is not None:
        report.append(res)
    assert res["unexplained"] == 0, f"{what}: {res}"
    assert res.get("flip_max_err", 0.0) <= 8e-3, f"{what}: threshold-flip error larger than one blend step: {res}"
    assert res["flip_explained"] <= max(4, max_flip_frac * epix.numel()), f"{what}: too many flip pixels: {res}"
    return res


def load_ref_ext():
    """The unmodified reference `_gs` extension (oracle/_ref/_gs.so, built by oracle/build_ref.sh from the reference's
    sources), or None where it has not been built."""
    import sys

    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.exists(os.path.join(ref_dir, "_gs.so")):
        return None
    if ref_dir not in sys.path:
        sys.path.insert(0, ref_dir)
    import _gs

    return _gs


class RefGolden:
    """The reference extension's side of a full-size comparison.

    live (`ext` is the extension): each of its outputs is compared whole, as the reference's own numbers, and a fixed
    seeded sample of it is kept; save() writes the samples to $GSB200_GOLDEN_OUT/<name>.npz when that is set.  Stored
    (`ext` is None): the same comparison runs on that sample, read from tests/golden/<name>.npz, against the same
    elements of ours.  Integer results (masks, tile ranges, sorted ids) are pinned whole by their SHA-256."""

    N_PIX = 384  # sampled pixels per image
    N_EL = 384  # sampled elements per gradient tensor

    def __init__(self, name, ext):
        self.name, self.ext, self.rec = name, ext, {}
        self.z = None if ext is not None else np.load(os.path.join(GOLDEN, name + ".npz"))

    @property
    def live(self):
        return self.ext is not None

    def _idx(self, key, n, k):
        g = torch.Generator().manual_seed(zlib.crc32(f"{self.name}/{key}".encode()))
        return torch.randperm(n, generator=g)[:min(k, n)].sort().values

    def stored(self, key):
        return torch.from_numpy(self.z[key])

    @staticmethod
    def _sha(t):
        return np.frombuffer(hashlib.sha256(t.detach().cpu().contiguous().numpy().tobytes()).digest(), np.uint8)

    def scalar(self, key, fn):
        """a number the comparison derives from the reference's output (e.g. an image's scale)"""
        if self.live:
            self.rec[key] = np.float64(fn())
        return float(self.rec[key] if self.live else self.z[key])

    def equal(self, key, ours, ref=None):
        if self.live:
            assert torch.equal(ours, ref), key
            self.rec[key + "_sha"] = self._sha(ref)
        else:
            assert np.array_equal(self._sha(ours), self.z[key + "_sha"]), f"{key}: differs from the reference"

    def sorted_ids(self, key, ids, depth, ref=None):
        """tile-sorted Gaussian ids: equal to the reference's, except inside runs of identical (tile, depth) keys"""
        idx = self._idx(key, ids.numel(), self.N_EL)
        if self.live:
            self.rec[key + "_sha"] = self._sha(ref)
            self.rec[key] = ref.cpu()[idx].numpy()
            rids = ref
        elif np.array_equal(self._sha(ids), self.z[key + "_sha"]):
            return
        else:
            ids, rids = ids[idx.to(ids.device)], self.stored(key).to(ids.device)
        neq = ids != rids
        if bool(neq.any()):
            assert torch.equal(depth.view(-1)[ids[neq].long()], depth.view(-1)[rids[neq].long()]), key

    def image(self, key, ours, ref, margin_fn, exact_fn=None, exact_self_fn=None, **kw):
        """classify_image_diff (tests/util.py) on the whole image, or on the stored pixels"""
        H, W = ours.shape[0], ours.shape[1]
        idx = self._idx(key, H * W, self.N_PIX)
        if self.live:
            self.rec[key] = ref.detach().float().cpu().reshape(H * W, -1)[idx].numpy()
            return classify_image_diff(ours, ref, margin_fn, exact_fn, what=key, exact_self_fn=exact_self_fn, **kw)
        pick = lambda t: t.detach().cpu().reshape(H * W, -1)[idx].unsqueeze(1)  # [S, 1, channels]: one pixel per row
        pick_m = lambda m: m.reshape(H * W)[idx].unsqueeze(1)

        def wrap(fn):
            return None if fn is None else (lambda: (lambda e, m: (pick(e), pick_m(m)))(*fn()))

        return classify_image_diff(pick(ours), self.stored(key).unsqueeze(1), lambda: pick_m(margin_fn()), wrap(exact_fn),
                                   what=key + " (stored pixels)", exact_self_fn=wrap(exact_self_fn), **kw)

    def grad(self, key, ours, ref=None, rtol=GRAD_RTOL):
        """assert_grad_close on the whole tensor, or on the stored elements"""
        idx = self._idx(key, ours.numel(), self.N_EL)
        if self.live:
            self.rec[key] = ref.detach().float().cpu().reshape(-1)[idx].numpy()
            return assert_grad_close(ours, ref, rtol, what=key)
        return assert_grad_close(ours.detach().cpu().reshape(-1)[idx], self.stored(key), rtol, what=key + " (stored elements)")

    def save(self):
        out = os.environ.get("GSB200_GOLDEN_OUT")
        if self.live and out:
            os.makedirs(out, exist_ok=True)
            np.savez_compressed(os.path.join(out, self.name + ".npz"), **self.rec)


class RefValues:
    """Values computed by the reference's own Python definitions, for the tests that execute them out of its files.

    Live when $GSB200_REFERENCE names a checkout of the reference: the test executes the definitions (`src` is that
    directory) and every value passes through; save() writes them to $GSB200_GOLDEN_OUT/<name>.npz when that is set.
    Otherwise each value comes from tests/golden/<name>.npz, recorded that way."""

    def __init__(self, name):
        src = os.environ.get("GSB200_REFERENCE")
        self.name, self.rec = name, {}
        self.src = src if src and os.path.isdir(src) else None
        self.z = None if self.live else np.load(os.path.join(GOLDEN, name + ".npz"))

    @property
    def live(self):
        return self.src is not None

    def __call__(self, key, fn):
        """fn() -> the reference's value (live); returned as an ndarray either way"""
        if self.live:
            v = fn()
            self.rec[key] = np.asarray(v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else v)
            return self.rec[key]
        return self.z[key]

    def save(self):
        out = os.environ.get("GSB200_GOLDEN_OUT")
        if self.live and out:
            os.makedirs(out, exist_ok=True)
            path = os.path.join(out, self.name + ".npz")
            old = dict(np.load(path)) if os.path.exists(path) else {}
            np.savez_compressed(path, **dict(old, **self.rec))
