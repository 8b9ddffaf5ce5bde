"""The float64 composite reference of tests/kernel_edges.py against the CPU oracle on the constructed edge cases, and
the case builders against what they claim (list lengths, termination points, threshold margins, tile-grid sizes).

This pins `composite_ref64` to the oracle, which the real reference extension pins (test_golden.py), so that the GPU
tests (test_kernel_edges_gpu.py) can hold the kernels to an independent plain-definition reference."""
import pytest
import torch

from tests import kernel_edges as ke
from tests.util import assert_grad_close


def _cases():
    out = [("lengths", t) for t in ke.THRESHES] + [("termination", t) for t in ke.THRESHES]
    out += [("geometry", hw) for hw in ke.GEOMETRIES] + [("grazing", None)]
    return out


CASES = _cases()
_cache = {}


def make_case(family, arg):
    key = (family, arg)
    if key not in _cache:
        if family == "lengths":
            _cache[key] = ke.lengths_case(arg)
        elif family == "termination":
            _cache[key] = ke.termination_case(arg)
        elif family == "geometry":
            _cache[key] = ke.geometry_case(*arg)
        elif family == "grazing":
            _cache[key] = ke.grazing_case()
        else:
            _cache[key] = ke.degenerate_case()
    return _cache[key]


def case_id(c):
    return f"{c[0]}-{c[1]}".replace(" ", "").replace("(", "").replace(")", "").replace(",", "x")


def cfg_of(c):
    return dict(H=c["H"], W=c["W"], n_tiles_h=c["n_tiles_h"], n_tiles_w=c["n_tiles_w"], psx=c["psx"], psy=c["psy"],
                thresh=c["thresh"])


def split_kind(kind):
    """'sh3bg' -> ('sh', 3, True)"""
    if kind.startswith("sh"):
        return "sh", int(kind[2]), kind.endswith("bg")
    return kind, None, kind == "rgb"


def inputs(c, kind):
    """payload, gout and reference keyword arguments of one payload kind"""
    base, C, bg = split_kind(kind)
    H, W = c["H"], c["W"]
    if base == "rgb":
        return c["color"], c["gout"], dict(kind="rgb", bg=c["bg"])
    if base == "scalar":
        return c["scalar"], c["gout"][..., 0].contiguous(), dict(kind="scalar")
    sh = c["sh"][..., :C * C].contiguous()
    return sh, c["gout"], dict(kind="sh", c2w9=c["c2w9"], C=C, bg_rgb=c["bg_rgb"] if bg else None)


def ref64(c, kind, grads=True, **kw):
    pay, gout, rk = inputs(c, kind)
    return ke.composite_ref64(c["mean2d"], c["cov2d"], pay, c["alpha"], c["start"], c["end"], c["ids"], c["topleft"],
                              c["psx"], c["psy"], c["H"], c["W"], c["thresh"], gout=gout if grads else None, **rk, **kw)


def oracle_run(oracle, c, kind):
    """the oracle's image (with the background term) and gradients for the same loss sum(out * gout)"""
    pay, gout, rk = inputs(c, kind)
    cfg = cfg_of(c)
    a = (c["mean2d"], c["cov2d"].contiguous(), pay, c["alpha"], c["start"], c["end"], c["ids"])
    if rk["kind"] == "rgb":
        out, T, _ = oracle.composite_rgb_fwd(*a, c["topleft"], cfg)
        fin = out + T.unsqueeze(-1) * c["bg"]
        gm, gc, gp, ga = oracle.composite_rgb_bwd(*a, fin, gout, c["topleft"], cfg)
        return dict(out=fin, g_mean2d=gm, g_cov2d=gc, g_pay=gp, g_alpha=ga, g_bg=gout * T.unsqueeze(-1))
    if rk["kind"] == "scalar":
        out, T = oracle.composite_scalar_fwd(*a, c["topleft"], cfg)
        gm, gc, gp, ga = oracle.composite_scalar_bwd(*a, out, gout, c["topleft"], cfg)
        return dict(out=out, g_mean2d=gm, g_cov2d=gc, g_pay=gp, g_alpha=ga)
    C, bg_rgb = rk["C"], rk["bg_rgb"]
    out, T, _ = oracle.composite_sh_fwd(*a, c["topleft"], c["c2w9"], C, cfg, bg_rgb)
    exact, _, _ = oracle.composite_sh_fwd_exact(*a, c["topleft"], c["c2w9"], C, cfg, bg_rgb)
    gm, gc, gp, ga = oracle.composite_sh_bwd(*a, out, gout, c["topleft"], c["c2w9"], C, cfg)
    return dict(out=out, exact=exact, g_mean2d=gm, g_cov2d=gc, g_pay=gp, g_alpha=ga)


def kinds_for(i):
    return (ke.KINDS[i % len(ke.KINDS)], ke.KINDS[(i + 5) % len(ke.KINDS)])


@pytest.mark.parametrize("i", range(len(CASES)), ids=[case_id(c) for c in CASES])
def test_ref64_matches_oracle(oracle_mod, i):
    """images to 1e-5 away from the two discontinuities (SH: to 1e-9 against the oracle's fp64 arbiter), gradients to
    1e-4 relative; the SH gradients of the grazing case are not compared (the oracle's SH path evaluates the
    reference's fp32 `radial`, which cancels for the axis ratios up to 10^3 built there, DESIGN.md §2)."""
    c = make_case(*CASES[i])
    for kind in kinds_for(i):
        r = ref64(c, kind)
        o = oracle_run(oracle_mod, c, kind)
        ok = ke.flip_free(r)
        if "exact" in o:
            err = (r["out"] - o["exact"]).abs().amax(-1)
            assert float(err[ok].max() if ok.any() else 0.0) <= 1e-9, (kind, float(err[ok].max()))
        else:
            err = (r["out"] - o["out"].double()).abs()
            err = err.amax(-1) if err.dim() == 3 else err
            assert float(err[ok].max() if ok.any() else 0.0) <= 1e-5, (kind, float(err[ok].max()))
        if kind.startswith("sh") and CASES[i][0] == "grazing":
            continue
        # at thresh 0 the termination case composites on behind T ~ 1e-10; the oracle's backward, like the reference's,
        # takes the remaining colour as a difference of fp32 running sums ((F - Cacc) / (1 - aG)), which has cancelled to
        # noise there: measured 5.5e-4 relative l2 on g_mean2d (SH C=2)
        rtol = 2e-3 if CASES[i] == ("termination", 0.0) else 1e-4
        for k in ("g_mean2d", "g_cov2d", "g_pay", "g_alpha", "g_bg"):
            if k in o and k in r:
                assert_grad_close(r[k], o[k], rtol=rtol, what=f"{CASES[i]} {kind} {k}", floor=1e-9)


def test_lengths_case_lists_and_hits():
    c = ke.lengths_case()
    r = ref64(c, "rgb", grads=False, keep_masks=True)
    lens = torch.where(c["start"] >= 0, c["end"] - c["start"], torch.zeros_like(c["start"]))
    for t, n in c["meta"]["lengths"].items():
        assert int(lens[t]) == n
        m = r["masks"][t].view(4, 4, 2, 8, n)  # [warp row, px row, warp col, px col, entry]
        if n >= 31:
            assert bool(m.any(dim=(1, 3, 4)).all()), f"tile {t}: a warp without hits"
    assert sorted(c["meta"]["lengths"].values()) == list(ke.LENGTHS)
    assert torch.equal(r["stop"], pixel_lengths(c))  # thresh 1e-4 stops nowhere: every entry is evaluated


def pixel_lengths(c):
    lens = torch.where(c["start"] >= 0, c["end"] - c["start"], torch.zeros_like(c["start"])).long()
    lens = lens.view(c["n_tiles_h"], 1, c["n_tiles_w"], 1).expand(-1, 16, -1, 16)
    return lens.reshape(c["n_tiles_h"] * 16, c["n_tiles_w"] * 16)[: c["H"], : c["W"]]


def test_termination_case_stops_where_it_claims():
    c = ke.termination_case(1e-4)
    r = ref64(c, "rgb", grads=False, keep_masks=True)
    assert bool(ke.flip_free(r).all())
    mods = set()
    for (t, row), s in c["meta"]["stops"].items():
        ty, tx = divmod(t, c["n_tiles_w"])
        blk = r["stop"][ty * 16 + 4 * row: ty * 16 + 4 * row + 4, tx * 16: tx * 16 + 16]
        assert bool((blk == s).all()), ((t, row), s, blk.unique())
    for t, B in c["meta"]["batches"].items():
        rows = {row: s for (tt, row), s in c["meta"]["stops"].items() if tt == t}
        assert {(s - 1) // B for s in rows.values()} == {0, 1}  # rows of one CTA stop in batch 0 and in batch 1
        assert (B + B // 2 + 1) in rows.values()                # ... one inside the batch prefetched during batch 0
        m = r["masks"][t].view(4, 4, 2, 8, -1)
        for row, s in rows.items():
            for wc in range(2):
                hits = m[row, :, wc, :, :].reshape(32, -1).any(0)
                for Bk in ke.BATCHES:  # hits of the warp in its last batch, for every kernel's batch size
                    b0 = (s - 1) // Bk * Bk
                    mods.add(int(hits[b0:s].sum()) % 4)
    assert {1, 2, 3} <= mods, mods


@pytest.mark.parametrize("thresh", ke.THRESHES)
def test_termination_thresholds(thresh):
    """0: never terminates; 1.0: every pixel stops after its first blend; 1.5: done before the first entry"""
    c = ke.termination_case(thresh)
    r = ref64(c, "rgb", grads=False)
    lens = pixel_lengths(c)
    if thresh == 0.0:
        assert torch.equal(r["stop"], lens)
    elif thresh > 1.0:
        assert int(r["stop"].max()) == 0 and bool((r["T"] == 1).all())
    elif thresh == 1.0:
        assert bool((r["T"] < 1).all()) and bool((r["stop"] < lens).all())


def test_grazing_case_sits_on_the_threshold():
    c = ke.grazing_case()
    r = ref64(c, "rgb", grads=False)
    band = (r["margin"] > 1e-5) & (r["margin"] < 5e-3)
    hit = 0
    for t, info in c["meta"]["targets"].items():
        ty, tx = divmod(t, c["n_tiles_w"])
        w = info["warp"]
        y0, x0 = ty * 16 + (w >> 1) * 4, tx * 16 + (w & 1) * 8
        m = r["margin"][y0:y0 + 4, x0:x0 + 8]
        hit += int(bool(band[y0:y0 + 4, x0:x0 + 8].any()))
        assert abs(float(m.min()) - info["margin"]) < 0.05 * info["margin"] + 1e-6, (t, info, float(m.min()))
    assert hit >= 0.9 * len(c["meta"]["targets"])
    assert max(i["ratio"] for i in c["meta"]["targets"].values()) > 300


def test_binning_cases_straddle_the_key_width():
    """the grids sit on both sides of 65 536 tiles, also with the padding key of the asynchronous mode (T + 1)"""
    k16 = set()
    for name, (th, tw, N) in ke.BIN_GRIDS.items():
        c = ke.binning_case(name)
        T = th * tw
        assert th <= 65535 and tw <= 65535
        k16.add((T <= 65536, T + 1 <= 65536))
        if N > 1:
            assert int(c["counts"][0]) == T
        if N >= 32:
            assert bool((c["counts"][: N // 32 * 32].view(-1, 32) == 0).any(1).all())  # zero counts in every warp
            d = c["depth"].view(-1)
            assert bool((d < 0).any()) and len(torch.unique(d)) < N
            assert bool((torch.signbit(d) & (d == 0)).any()) and bool((~torch.signbit(d) & (d == 0)).any())
    assert k16 == {(True, True), (True, False), (False, False)}


def test_binning_cases_match_their_count(oracle_mod):
    for name in ke.BIN_GRIDS:
        c = ke.binning_case(name)
        ids, start, end = oracle_mod.tile_culling_aabb_start_end(c["tl"], c["br"], c["depth"], c["n_tiles_h"],
                                                                 c["n_tiles_w"], c["D"])
        assert ids.numel() == c["D"]
