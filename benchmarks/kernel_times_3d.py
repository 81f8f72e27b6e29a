"""Device time of the 3D kernels at the NeRF shape (BASELINE cfg4: 2^19 samples, 16 levels 16->2048, 2^19-row
tables, C=1 -> F=4) and the plain HashGrid shape (F=2): CUDA events around 20 launches after 5 warm-ups, four rotating
input sets (4 x 160 MB > L2).

    python benchmarks/kernel_times_3d.py [--n 524288] [--bw 19]
"""
import argparse
import ctypes
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from shacira_b200 import _lib  # noqa: E402
from shacira_b200.grids import geometric_resolutions  # noqa: E402


def timed(fn, iters=20, warm=5):
    for i in range(warm):
        fn(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3  # us


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 19)
    ap.add_argument("--bw", type=int, default=19)
    ap.add_argument("--rmax", type=int, default=2048)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    L, BW, S = 16, args.bw, args.n
    res = geometric_resolutions(16, args.rmax, L)
    sizes = [min(2 ** BW, r ** 3) for r in res]
    first = [0]
    for s in sizes[:-1]:
        first.append(first[-1] + s)
    T = sum(sizes)
    lib = _lib.load()
    fi, _ = _lib._i32_array(first)
    rs, _ = _lib._i32_array(res)
    P = _lib._ptr
    torch.manual_seed(0)
    out = {"n": S, "bw": BW, "rows": T}
    for name, C, F in (("latent_c1_f4", 1, 4), ("plain_f2", 2, 2)):
        sets = [dict(coords=torch.rand((S, 3), device=dev) * 2 - 1, g=torch.randn((S, L * F), device=dev)) for _ in range(4)]
        lat = (torch.rand((T, C), device=dev) - 0.5) * 16
        A = torch.randn((1, C, F), device=dev) * 0.1
        shift = torch.zeros((1, F), device=dev)
        feats = torch.empty((S, L * F), device=dev)
        z = torch.empty((S, L * C), device=dev)
        gl = torch.zeros((T, C), device=dev)
        gA = torch.zeros((L, C, F), device=dev)
        gS = torch.zeros((L, F), device=dev)
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        if name.startswith("latent"):
            fwd = lambda i: _lib._check(lib.shacira_latent_forward(3, P(sets[i % 4]["coords"]), S, P(lat), fi, rs, L, BW, C, F, 1,
                                                                   P(A), P(shift), 0, P(feats), P(z), st))
            bwd = lambda i: _lib._check(lib.shacira_latent_backward(3, P(sets[i % 4]["coords"]), S, P(sets[i % 4]["g"]), P(z), fi,
                                                                    rs, L, BW, C, F, P(A), 0, T, 1, P(gl), P(gA), P(gS), st))
            bwd_nodec = lambda i: _lib._check(lib.shacira_latent_backward(3, P(sets[i % 4]["coords"]), S, P(sets[i % 4]["g"]), None, fi,
                                                                          rs, L, BW, C, F, P(A), 0, T, 1, P(gl), None, None, st))
            out[name] = {"fwd_us": timed(fwd), "bwd_us": timed(bwd), "bwd_nodec_us": timed(bwd_nodec)}
        else:
            fwd = lambda i: _lib._check(lib.shacira_hashgrid_forward(3, P(sets[i % 4]["coords"]), S, P(lat), fi, rs, L, BW, F,
                                                                     P(feats), st))
            bwd = lambda i: _lib._check(lib.shacira_hashgrid_backward(3, P(sets[i % 4]["coords"]), S, P(sets[i % 4]["g"]), fi, rs, L,
                                                                      BW, F, T, 1, P(gl), st))
            out[name] = {"fwd_us": timed(fwd), "bwd_us": timed(bwd)}
        del sets
    # packed exponential integration (SURVEY 8 f-3): 4096 rays x 128 samples, RGB
    R, per = 4096, S // 4096
    feats3 = torch.rand((S, 3), device=dev)
    tau = torch.rand((S,), device=dev) ** 3
    starts = (torch.arange(R + 1, device=dev, dtype=torch.int32) * per).contiguous()
    w = torch.empty((S,), device=dev)
    ray = torch.empty((R, 3), device=dev)
    alpha = torch.empty((R,), device=dev)
    g_ray = torch.randn((R, 3), device=dev)
    g_w = torch.randn((S,), device=dev)
    g_f = torch.empty((S, 3), device=dev)
    g_t = torch.empty((S,), device=dev)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    ifwd = lambda i: _lib._check(lib.shacira_integrate_forward(P(feats3), P(tau), P(starts), R, 3, P(w), P(ray), P(alpha), st))
    ibwd = lambda i: _lib._check(lib.shacira_integrate_backward(P(feats3), P(tau), P(w), P(starts), R, 3, P(g_ray), P(g_w),
                                                                P(g_f), P(g_t), st))
    out["integrate_rgb"] = {"rays": R, "samples": S, "fwd_us": timed(ifwd), "bwd_us": timed(ibwd)}
    # sample generation (SURVEY 8 f-3): 4096 rays against a dense 8^3 grid (the reference's make_dense level 3),
    # 16 stratified samples per intersected cell -- DDA count + fill + fused voxel-sample kernel
    from shacira_b200 import render
    occ = torch.ones((8, 8, 8), dtype=torch.uint8, device=dev)
    org = torch.randn((4096, 3), device=dev)
    org = org / org.norm(dim=1, keepdim=True) * 3.0
    dirs = -org + (torch.rand((4096, 3), device=dev) - 0.5)
    dirs = dirs / dirs.norm(dim=1, keepdim=True)
    box = {}

    def march(i):
        box["r"] = render.raymarch_voxel(occ, org, dirs, 16)
    t_march = timed(march)
    out["raymarch_voxel"] = {"rays": 4096, "grid": "8^3 dense", "samples_per_cell": 16,
                             "samples": int(box["r"][1].shape[0]), "us": t_march,
                             "note": "includes the one host sync that sizes the outputs"}
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
