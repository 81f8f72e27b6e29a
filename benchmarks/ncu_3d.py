"""A few launches of the 3D (NeRF-shape, cfg4) kernels for an ncu capture.
    ncu --set full ... python benchmarks/ncu_3d.py [--sorted TILE_POINTS] [--what fwd|bwd|both]"""
import argparse
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from shacira_b200 import _lib  # noqa: E402
from shacira_b200.grids import geometric_resolutions  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--sorted", type=int, default=0)
ap.add_argument("--what", default="both")
ap.add_argument("--reps", type=int, default=2)
args = ap.parse_args()
L, BW, C, F, S = 16, 19, 1, 4, 4096 * 128
dev = torch.device("cuda", 0)
res = geometric_resolutions(16, 2048, L)
sizes = [min(2 ** BW, r ** 3) for r in res]
first = [0]
for s in sizes[:-1]:
    first.append(first[-1] + s)
T = sum(sizes)
torch.manual_seed(7)
lat = (torch.rand((T, C), device=dev) - 0.5) * 16
A = torch.randn((1, C, F), device=dev) * 0.1
shift = torch.randn((1, F), device=dev) * 0.05
coords = torch.rand((S, 3), device=dev) * 2 - 1
g = torch.randn((S, L * F), device=dev)
for _ in range(args.reps):
    if args.sorted:
        plan = _lib.Plan(coords, tile_points=args.sorted)
        f, z = _lib.latent_forward_planned_z(plan, lat, first, res, BW, A, shift, F, True, True)
        if args.what != "fwd":
            _lib.latent_backward_planned_z(plan, g, z, first, res, BW, A, C, F, T, True)
    else:
        f, z = _lib.latent_forward(coords, lat, first, res, BW, A, shift, F, True, True)
        if args.what != "fwd":
            _lib.latent_backward(coords, g, z, first, res, BW, A, C, F, T, True)
torch.cuda.synchronize()
