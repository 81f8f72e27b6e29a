"""Evaluation side of the native image fit on the GPU: render time and the cost of best-state tracking.

  render   shacira_fit_render (image_fit.render_image: grid -> MLP -> RGB in one kernel) against
           mlp(grid.interpolate(coords)) (tiled forward writing [N, 16] feature rows + three PyTorch linear layers) on
           the same coordinates, at the Kodak shape (393 216 px) and 2 x 2 upsampled (1 572 864 px). CUDA events around
           a CUDA graph of K launches, best of 5 replays (the method of benchmarks/kernel_times.py). L2 is NOT flushed
           between launches: the 256 KB table and the weights stay resident, as they do when a trainer evaluates.
  recipe   step time of the reference's recipe through ImageFitStep, graph-replayed, SGA and STE phases separately,
           three fits in flight on one GPU, track_best off and on ALTERNATED within the run (rounds off, on, off, on).

Prints one JSON line with the card's name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "benchmarks"))
import fit_image  # noqa: E402
from shacira_b200 import _lib, grid_ops  # noqa: E402
from shacira_b200.image_fit import ImageFitStep, _render, lambda_at, render_image, temperature_at  # noqa: E402


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [s.strip() for s in out.split(",")]
    return {"gpu": name, "power_limit": power, "sm_clock_max": clock}


def graph_time_us(fn, K, stream):
    with torch.cuda.stream(stream):
        for _ in range(3):
            fn()
        stream.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=stream):
            for _ in range(K):
                fn()
        g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        best = 1e9
        for _ in range(5):
            e0.record()
            g.replay()
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1) / K * 1e3)
    return round(best, 2)


def render_times(dev, K, fit_steps):
    grid, mlp, coords, gt, fs = fit_image._native_setup(0, dev)
    for it in range(fit_steps):   # a trained-looking model (the kernel's time does not depend on it)
        fs.set_lambda(1e-3)
        if it + 1 in (1, 2, 5, 10):
            fs.update_div()
        fs.step()
    fs.close()
    h, w = 2 * fit_image.H, 2 * fit_image.W
    ys, xs = torch.meshgrid(torch.arange(h), torch.arange(w), indexing="ij")
    up = torch.stack([(ys.reshape(-1) + 0.5) / h * 2 - 1, (xs.reshape(-1) + 0.5) / w * 2 - 1], 1).float().to(dev)
    out = {}
    stream = torch.cuda.Stream(device=dev)
    for name, c in (("kodak_393216px", coords), ("upsampled_2x2_1572864px", up)):
        n = c.shape[0]
        rgb, _ = render_image(grid, mlp, c)            # builds / caches the plan and its node table
        with torch.no_grad():
            ref = mlp(grid.interpolate(c, 0))
        err = float((rgb - ref).abs().max())
        plan = grid_ops.plan_for(c)
        A, shift = grid.latent_dec.affine_map()
        A, shift = A.detach().contiguous(), shift.detach().contiguous()
        fi, _ = _lib._i32_array(grid._first_idx())
        rs, L = _lib._i32_array(grid.resolutions)
        lin = [mlp[0], mlp[2], mlp[4]]
        lat = grid.codebook.data
        sse = torch.zeros((), dtype=torch.int64, device=dev)
        tgt = torch.rand(n, 3, device=dev)

        def kernel():
            _render(plan, lat, fi, rs, L, int(grid.codebook_bitwidth), A, shift, lin, rgb, None, None)

        def kernel_psnr():
            _render(plan, lat, fi, rs, L, int(grid.codebook_bitwidth), A, shift, lin, None, tgt, sse)

        def torch_path():
            with torch.no_grad():
                mlp(grid.interpolate(c, 0))

        out[name] = {"render_kernel_us": graph_time_us(kernel, K, stream),
                     "render_kernel_psnr_only_us": graph_time_us(kernel_psnr, K, stream),
                     "interpolate_plus_torch_mlp_us": graph_time_us(torch_path, K, stream),
                     "max_abs_diff_vs_torch_path": err}
    return out


def recipe_round(dev, track, seeds, sga_steps, ste_steps, temperature=0.1, decay_period=0.9):
    """fit_native_recipe's timed structure (graph per fit and phase, one stream per fit), with track_best on or off."""
    fits = []
    for s in seeds:
        grid, mlp, coords, gt, fs0 = fit_image._native_setup(s, dev, device_noise=True, sga=True)
        fs0.close()
        fits.append(ImageFitStep(grid, mlp, coords, gt, lr=1e-3, grid_lr=2e-2, ldec_lr=1e-2, prob_lr=1e-4,
                                 weight_decay=0.0, weight_decay_decoder=1e-2, device_noise=True, noise_seed=10_000 + s,
                                 track_best=track))
    streams = [torch.cuda.Stream(device=dev) for _ in seeds]
    total = int(round(sga_steps / decay_period))

    def host_side(k, it):
        fs = fits[k]
        fs.set_lambda(lambda_at(it, total))
        if fs.sga:
            fs.set_temperature(temperature_at(it, total, temperature, decay_period))
        if it + 1 in (1, 2, 5, 10):
            fs.update_div()

    def capture():
        graphs = []
        for k in range(len(seeds)):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=streams[k]):
                fits[k].step()
            graphs.append(g)
        return graphs

    def timed(graphs, a, b, warm=20):
        def run(x, y):
            for it in range(x, y):
                for k in range(len(seeds)):
                    with torch.cuda.stream(streams[k]):
                        host_side(k, it)
                        graphs[k].replay()
        run(a, a + warm)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        run(a + warm, b)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / (b - a - warm) * 1e3 / len(seeds)

    for k in range(len(seeds)):
        with torch.cuda.stream(streams[k]):
            for it in range(3):
                host_side(k, it)
                fits[k].step()
    torch.cuda.synchronize()
    ms_sga = timed(capture(), 3, 3 + sga_steps)
    for f in fits:
        f.set_sga(False)
    ms_ste = timed(capture(), 3 + sga_steps, 3 + sga_steps + ste_steps)
    best = [float(f.best_loss()) for f in fits] if track else None
    last = [float(f.rgb_loss()) for f in fits]
    for f in fits:
        f.close()
    return ms_sga, ms_ste, best, last


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--K", type=int, default=200, help="render launches per graph")
    ap.add_argument("--sga-steps", type=int, default=300)
    ap.add_argument("--ste-steps", type=int, default=300)
    ap.add_argument("--rounds", type=int, default=2, help="off/on pairs of the recipe timing")
    ap.add_argument("--fits", type=int, default=3, help="fits in flight per GPU")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"benchmark": "fit_eval", **card(), "l2_flushed": False, "render_launches_per_graph": args.K}
    res["render"] = render_times(dev, args.K, 50)
    seeds = list(range(args.fits))
    arms = {False: {"sga": [], "ste": []}, True: {"sga": [], "ste": []}}
    extra = {}
    for r in range(args.rounds):
        for track in (False, True):
            ms_sga, ms_ste, best, last = recipe_round(dev, track, seeds, args.sga_steps, args.ste_steps)
            arms[track]["sga"].append(round(ms_sga * 1e3, 2))
            arms[track]["ste"].append(round(ms_ste * 1e3, 2))
            if track:
                extra["best_loss_vs_last_loss"] = [[b, l] for b, l in zip(best, last)]
    res["recipe"] = {
        "fits_in_flight": args.fits, "sga_steps_timed": args.sga_steps - 20, "ste_steps_timed": args.ste_steps - 20,
        "us_per_step_sga_track_off": arms[False]["sga"], "us_per_step_sga_track_on": arms[True]["sga"],
        "us_per_step_ste_track_off": arms[False]["ste"], "us_per_step_ste_track_on": arms[True]["ste"],
        "median_delta_us_sga": round(float(np.median(arms[True]["sga"]) - np.median(arms[False]["sga"])), 2),
        "median_delta_us_ste": round(float(np.median(arms[True]["ste"]) - np.median(arms[False]["ste"])), 2),
        **extra}
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
