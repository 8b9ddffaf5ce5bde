"""Generate the shading golden fixture from the UNMODIFIED reference code (TEST INFRASTRUCTURE; runs in the dev
container only, needs /root/reference).

Executed as they are (parsed with `ast`, compiled into a scratch namespace, nothing of the source is written anywhere):
  utils/ops.py  angle_bisector, compute_shaded_color
Inputs: seeded Gaussians (means, unit normals, colours), a camera position and several lights, including a light and a
camera on the normal's line (bisector parallel / antiparallel to it, |dot| clamped at 1).
Result: tests/golden/shaded_color_ref.npz
"""
import ast
import os

import numpy as np
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
REF_OPS = "/root/reference/utils/ops.py"
OPS = ["angle_bisector", "compute_shaded_color"]


def load(namespace):
    tree = ast.parse(open(REF_OPS).read())
    for node in tree.body:
        if isinstance(node, ast.FunctionDef) and node.name in OPS:
            exec(compile(ast.Module(body=[node], type_ignores=[]), REF_OPS, "exec"), namespace)
    assert all(n in namespace for n in OPS)


def main():
    ns = {"torch": torch, "F": F}
    load(ns)
    g = torch.Generator().manual_seed(11)
    n = 512
    mean = torch.randn(n, 3, generator=g) * 0.5
    normal = F.normalize(torch.randn(n, 3, generator=g), dim=-1)
    color = torch.rand(n, 3, generator=g)
    cam_pos = torch.tensor([3.0, 0.0, 1.0])
    lights = torch.tensor([[3.0, 0.0, 3.0], [0.0, 3.0, 3.0], [-3.0, -1.0, 3.0], [3.0, 0.0, 1.0]])
    light_colors = torch.tensor([[1.0, 1.0, 1.0], [1.0, 0.5, 0.25], [0.2, 0.9, 0.4], [1.0, 1.0, 1.0]])
    # row 0 faces the camera and the light of index 3 head-on (both along +x from the origin)
    mean[0] = 0.0
    normal[0] = torch.tensor([1.0, 0.0, 0.0])
    out = {"mean": mean.numpy(), "normal": normal.numpy(), "color": color.numpy(), "cam_pos": cam_pos.numpy(),
           "lights": lights.numpy(), "light_colors": light_colors.numpy()}
    shaded, bis = [], []
    for lp, lc in zip(lights, light_colors):
        shaded.append(ns["compute_shaded_color"](lp, lc, normal, color, mean, cam_pos).numpy())
        bis.append(ns["angle_bisector"](lp - mean, cam_pos - mean).numpy())
    out["shaded"] = np.stack(shaded)
    out["bisector"] = np.stack(bis)
    np.savez_compressed(os.path.join(HERE, "shaded_color_ref.npz"), **out)


if __name__ == "__main__":
    main()
