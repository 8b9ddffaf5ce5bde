"""Small host-side functions the product mirrors from the reference, checked against the reference's own definitions
executed with `ast` out of the files where the reference is at $GSB200_REFERENCE, and otherwise against the values they
computed, stored in tests/golden/host_mirrors_ref.npz (tests/util.py::RefValues)."""
import ast
import os

import numpy as np
import pytest
import torch

from tests.util import RefValues


@pytest.fixture(scope="module")
def rv():
    r = RefValues("host_mirrors_ref")
    yield r
    r.save()


def _defs(rv, path, names, ns):
    if not rv.live:
        return ns
    tree = ast.parse(open(os.path.join(rv.src, path)).read())
    for node in tree.body:
        if isinstance(node, ast.FunctionDef) and node.name in names:
            node.returns, node.decorator_list = None, []
            for a in node.args.args:
                a.annotation = None
            exec(compile(ast.Module(body=[node], type_ignores=[]), path, "exec"), ns)
    return ns


def test_step_check(rv):
    from gsgen_b200.renderer import step_check

    ref = _defs(rv, "gs/renderer.py", ["step_check"], {}).get("step_check")
    for step in (0, 1, 99, 100, 300):
        for size in (0, 1, 100):
            for z in (False, True):
                assert step_check(step, size, z) == rv(f"step_check_{step}_{size}_{z}", lambda: ref(step, size, z))


def test_look_at_pose(rv):
    from gsgen_b200.camera import get_c2w_from_up_and_look_at, orbit_c2w

    ref = _defs(rv, "data/__init__.py", ["get_c2w_from_up_and_look_at"], {"np": np}).get("get_c2w_from_up_and_look_at")
    rng = np.random.default_rng(0)
    for i in range(20):
        up, look, pos = rng.standard_normal(3), rng.standard_normal(3) * 0.1, rng.standard_normal(3) * 2.0
        assert np.array_equal(get_c2w_from_up_and_look_at(up.copy(), look.copy(), pos.copy()),
                              rv(f"look_at_{i}", lambda: ref(up.copy(), look.copy(), pos.copy())))
    # the orbit pose of the benchmark scenes = CameraPoseProvider's convention (data/__init__.py:151-205): up +z,
    # look at the centre from d * (cos e cos a, cos e sin a, sin e)
    d, e, a = 2.5, np.deg2rad(15.0), np.deg2rad(30.0)
    pos = d * np.array([np.cos(e) * np.cos(a), np.cos(e) * np.sin(a), np.sin(e)])
    want = rv("look_at_orbit", lambda: ref(np.array([0.0, 0.0, 1.0]), np.zeros(3), pos))
    assert np.allclose(orbit_c2w(2.5, 15.0, 30.0).numpy()[:3, :4], want, atol=1e-6)


def test_sh_dc_initialisation(rv):
    """sh_renderer.py:38-43: DC coefficient = logit(rgb) / Y_0, higher orders zero (ours adds seeded noise on top so that
    view dependence is exercised; noise=0 must reproduce the reference)."""
    from scipy.special import logit

    from gsgen_b200.scenes import init_sh_coeffs

    ns = {"torch": torch, "sh_base": 0.28209479177387814,
          "inv_activations": {"sigmoid": lambda x: torch.logit(x) if isinstance(x, torch.Tensor) else logit(x)}}
    ref = _defs(rv, "gs/sh_renderer.py", ["init_sh_coeffs"], ns).get("init_sh_coeffs")
    rgb = torch.rand(50, 3, generator=torch.Generator().manual_seed(0)).clamp(0.02, 0.98)
    ours = init_sh_coeffs(rgb, 4, torch.Generator().manual_seed(1), noise=0.0)
    assert torch.allclose(ours, torch.from_numpy(rv("init_sh_coeffs", lambda: ref(None, rgb, 4))), rtol=1e-6, atol=1e-7)


def test_viewer_camera_helpers(rv):
    """gsgen_b200.viewer.get_c2w / qvec2rotmat and CameraInfo.from_fov_camera against the reference's definitions
    (utils/viewer/viser_viewer.py:14-19, utils/transforms.py:12-31, utils/camera.py:316-325)."""
    import types

    from gsgen_b200.camera import CameraInfo
    from gsgen_b200.viewer import get_c2w, qvec2rotmat

    ns = _defs(rv, "utils/transforms.py", ["qvec2rotmat"], {"np": np})
    ns = _defs(rv, "utils/viewer/viser_viewer.py", ["get_c2w"], ns)
    rng = np.random.default_rng(1)
    for i in range(10):
        q = rng.standard_normal(4)
        q /= np.linalg.norm(q)
        pos = rng.standard_normal(3)
        assert np.allclose(qvec2rotmat(q), rv(f"qvec2rotmat_{i}", lambda: ns["qvec2rotmat"](q)), atol=1e-15)
        cam = types.SimpleNamespace(wxyz=q, position=pos)
        assert np.array_equal(get_c2w(q, pos), rv(f"get_c2w_{i}", lambda: ns["get_c2w"](cam)))
    # from_fov_camera is a classmethod of the reference's CameraInfo: execute its body on a stand-in class
    ns2 = {"np": np}
    if rv.live:
        tree = ast.parse(open(os.path.join(rv.src, "utils/camera.py")).read())
        cls = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "CameraInfo")
        fn = next(n for n in cls.body if isinstance(n, ast.FunctionDef) and n.name == "from_fov_camera")
        fn.decorator_list = []
        exec(compile(ast.Module(body=[fn], type_ignores=[]), "utils/camera.py", "exec"), ns2)
    for fov, aspect, reso in ((0.9, 1.6, 512), (1.2, 0.75, 300), (0.5, 1.0, 64)):
        want = rv(f"from_fov_camera_{fov}_{aspect}_{reso}",
                  lambda: ns2["from_fov_camera"](lambda *a: a, fov, aspect, reso, 0.01, 100.0))
        got = CameraInfo.from_fov_camera(fov, aspect, reso, 0.01, 100.0)
        assert (got.fx, got.fy, got.cx, got.cy, got.w, got.h, got.near_plane, got.far_plane) == tuple(want.tolist())


def test_camera_info_resolution_changes_and_intrinsics(rv):
    """CameraInfo.downsample / upsample / set_reso / get_camera_intrinsic / from_fov_camera against the reference's own
    class (utils/camera.py:219-368), attribute for attribute"""
    import torch.nn.functional as F

    from gsgen_b200.camera import CameraInfo

    Ref = None
    if rv.live:
        tree = ast.parse(open(os.path.join(rv.src, "utils/camera.py")).read())
        node = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "CameraInfo")
        ns = {"np": np, "torch": torch, "F": F, "console": None}
        exec(compile(ast.Module(body=[node], type_ignores=[]), "utils/camera.py", "exec"), ns)
        Ref = ns["CameraInfo"]
    KEYS = ("fx", "fy", "cx", "cy", "w", "h", "yfov", "aspect", "near_plane", "far_plane")
    attrs = lambda b, keys=KEYS: [float(getattr(b, k)) for k in keys]

    def same(key, a, b, keys=KEYS, rel=1e-12):
        for k, want in zip(keys, rv(key, lambda: attrs(b, keys))):
            assert float(getattr(a, k)) == (float(want) if rel is None else pytest.approx(float(want), rel=rel)), (key, k)

    for i, args in enumerate(((400.0, 410.0, 256.0, 250.0, 512, 500, 0.01, 100.0),
                              (128.0, 128.0, 64.0, 64.0, 128, 128, 0.1, 10.0))):
        a, b = CameraInfo(*args), (Ref(*args) if Ref else None)
        same(f"cam{i}", a, b)
        for j, (op, arg) in enumerate((("downsample", 2), ("upsample", 2), ("set_reso", 96), ("upsample", 3),
                                       ("downsample", 4))):
            getattr(a, op)(arg)
            if b is not None:
                getattr(b, op)(arg)
            same(f"cam{i}_op{j}", a, b)
        assert torch.equal(a.get_camera_intrinsic("cpu"),
                           torch.from_numpy(rv(f"cam{i}_intrinsic", lambda: b.get_camera_intrinsic("cpu"))))
    a = CameraInfo.from_fov_camera(0.9, 1.5, 300, 0.01, 100.0)
    same("from_fov_camera", a, Ref.from_fov_camera(0.9, 1.5, 300, 0.01, 100.0) if Ref else None)
    a = CameraInfo.from_reso(64)
    # (the reference's from_reso hard-codes near 0.01 / far 1000)
    same("from_reso", a, Ref.from_reso(64) if Ref else None, keys=("fx", "fy", "cx", "cy", "w", "h"), rel=None)
