"""Where the tiled / sorted paths start to pay: fwd and bwd device time against the batch size, planned vs point-parallel.
2D: BASELINE cfg2 grid (16 levels 16->512, 2^16, C=F=1), plan cached (static coordinates) -- and the one-off plan build
for callers whose coordinates change. 3D: BASELINE cfg4 grid (C=1 -> F=4), plan re-binned every step (NeRF samples).
One JSON line per (dim, N). The switches PLAN_MIN_POINTS / PLAN_MIN_POINTS_3D (grid_ops.py) are set from this sweep."""
import ctypes
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from shacira_b200 import _lib  # noqa: E402
from shacira_b200.grids import geometric_resolutions  # noqa: E402

dev = torch.device("cuda", 0)
lib = _lib.load()


def timed(fn, iters=12, warm=3):
    for i in range(warm):
        fn(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3


def layout(res, bw, dim):
    sizes = [min(2 ** bw, r ** dim) for r in res]
    first = [0]
    for s in sizes[:-1]:
        first.append(first[-1] + s)
    return first, sum(sizes)


def sweep(dim, L, bw, rmax, C, F, ns):
    res = geometric_resolutions(16, rmax, L)
    first, T = layout(res, bw, dim)
    torch.manual_seed(0)
    lat = (torch.rand((T, C), device=dev) - 0.5) * 16
    A = torch.randn((1, C, F), device=dev) * 0.1
    S = torch.randn((1, F), device=dev) * 0.05
    for n in ns:
        sets = [dict(c=torch.rand((n, dim), device=dev) * 2 - 1, g=torch.randn((n, L * F), device=dev)) for _ in range(3)]
        zs = [_lib.latent_forward(s["c"], lat, first, res, bw, A, S, F, True, True)[1] for s in sets]
        r = {"dim": dim, "n": n}
        r["pp_fwd_us"] = timed(lambda i: _lib.latent_forward(sets[i % 3]["c"], lat, first, res, bw, A, S, F, True, True))
        r["pp_bwd_us"] = timed(lambda i: _lib.latent_backward(sets[i % 3]["c"], sets[i % 3]["g"], zs[i % 3], first, res, bw, A, C, F, T, True))
        plans = [_lib.Plan(s["c"]) for s in sets]
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        r["plan_us"] = timed(lambda i: _lib._check(lib.shacira_plan_rebuild(plans[i % 3].handle, dim, _lib._ptr(sets[i % 3]["c"]), n, 0, st)))
        r["tiles"] = plans[0].info()["ntiles"]
        if dim == 2:
            r["tiled_fwd_us"] = timed(lambda i: _lib.latent_forward_planned(plans[i % 3], lat, first, res, bw, A, S, F, True))
            r["tiled_bwd_us"] = timed(lambda i: _lib.latent_backward_planned(plans[i % 3], sets[i % 3]["g"], lat, first, res, bw, A, C, F, T, True, True))
        else:
            zp = [_lib.latent_forward_planned_z(plans[k], lat, first, res, bw, A, S, F, True, True)[1] for k in range(3)]
            r["tiled_fwd_us"] = timed(lambda i: _lib.latent_forward_planned_z(plans[i % 3], lat, first, res, bw, A, S, F, True, True))
            r["tiled_bwd_us"] = timed(lambda i: _lib.latent_backward_planned_z(plans[i % 3], sets[i % 3]["g"], zp[i % 3], first, res, bw, A, C, F, T, True))
        r["pp_us"] = r["pp_fwd_us"] + r["pp_bwd_us"]
        r["tiled_static_us"] = r["tiled_fwd_us"] + r["tiled_bwd_us"]
        r["tiled_rebinned_us"] = r["tiled_static_us"] + r["plan_us"]
        print(json.dumps(r), flush=True)
        for p in plans:
            p.close()


sweep(2, 16, 16, 512, 1, 1, [1 << k for k in range(12, 19)])
sweep(3, 16, 19, 2048, 1, 4, [1 << k for k in range(13, 20)])
