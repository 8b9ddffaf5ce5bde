"""Time the normal estimate (gsb200_estimate_normals / _backward) on 1 M points.

    python tools/normals_bench.py [--n 1000000] [--repeats 20] [--warmup 3] [--out FILE]

Clouds: uniform in the unit ball, and a sphere shell of radius 1 with 1 % radial noise; K = 10, 30, 50.  For each it
times the forward alone (grid build + fused query / PCA, no [N,K] output) and forward + backward (neighbour indices
saved, gradient scattered back) with CUDA events, and reports the median over the repeats after warm-up.  Prints the
GPU name and its power limit with the numbers and one JSON line at the end.  There is no reference timing: the
reference's pytorch3d path is not installed here.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gsgen_b200.normals import estimate_normal  # noqa: E402


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip() or None
    except Exception:
        return None


def cloud(kind, n, g):
    v = torch.randn(n, 3, generator=g)
    v = v / v.norm(dim=1, keepdim=True)
    if kind == "ball":
        return v * torch.rand(n, 1, generator=g) ** (1 / 3)
    return v * (1 + 0.01 * torch.randn(n, 1, generator=g))


def median_ms(fn, repeats, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(repeats):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return sorted(times)[len(times) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--repeats", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    res = {"gpu": torch.cuda.get_device_name(dev), "power_limit": power_limit(), "n": a.n, "repeats": a.repeats,
           "rows": []}
    print(f"# {res['gpu']}, power limit {res['power_limit']}, N = {a.n}, median of {a.repeats} after {a.warmup}")
    g = torch.Generator().manual_seed(0)
    for kind in ("ball", "shell"):
        pts = cloud(kind, a.n, g).to(dev)
        grad = torch.randn(a.n, 3, device=dev)
        for K in (10, 30, 50):
            fwd = median_ms(lambda: estimate_normal(pts, K), a.repeats, a.warmup)
            p = pts.clone().requires_grad_()

            def fwd_bwd():
                p.grad = None
                (estimate_normal(p, K) * grad).sum().backward()

            fb = median_ms(fwd_bwd, a.repeats, a.warmup)
            row = {"cloud": kind, "K": K, "forward_ms": round(fwd, 3), "forward_backward_ms": round(fb, 3)}
            res["rows"].append(row)
            print(f"{kind:6s} K={K:2d}  forward {fwd:8.3f} ms   forward+backward {fb:8.3f} ms")
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
