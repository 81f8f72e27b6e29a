"""NeRF decoder heads: the tcgen05 kernels against the same heads in PyTorch fp32 and under autocast bf16.

S = 2^19 samples at (IN, H, E) = (64, 128, 27) (cfg4: 16 levels x F = 4) and (96, 128, 27) (nerf_lego.yaml: 24 levels
x F = 4). feats is 128 / 192 MB, larger than the 126 MB L2, so every pass streams it from HBM. Each arm is warmed up,
then timed with CUDA events over --iters launches. Achieved TFLOP/s use the FLOP count below (useful products only,
no padding); bytes are the HBM traffic the kernels need at least. A separate torch.profiler pass lists each arm's kernels.

    python benchmarks/nerf_heads.py --out profiles/r06_nerf_heads.json
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

H, D, E = 128, 16, 27
PEAK_TFLOPS = 2250.0      # dense bf16, HGX B200 data sheet, one GPU at 1000 W
PEAK_TBS = 7.7            # HBM3e


def flops_per_sample(in_dim):
    """Forward: the five products. Forward + backward (recompute, input gradients, weight gradients): four times."""
    fwd = 2 * (in_dim * H + H * D + (D + E) * H + H * H + H * 3)
    return fwd, 4 * fwd


def bytes_moved(S, in_dim, arm):
    """Least HBM traffic: feats read (twice for forward + backward: the forward and the backward's recompute), ridx,
    outputs, and for the backward the output gradients in and g_X out. vemb and the weights are L2-sized."""
    fwd = S * (in_dim * 4 + 4 + 4 * 4)
    if arm == "fwd":
        return fwd
    return fwd + S * (in_dim * 4 + 4 + 4 * 4 + in_dim * 4)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in out.split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:  # the number stands only with the card beside it
        return dict(name=torch.cuda.get_device_name(0), power_limit="unknown (%r)" % e)


def time_arm(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(iters):
        fn()
    stop.record()
    torch.cuda.synchronize()
    return start.elapsed_time(stop) * 1e3 / iters   # us


def profile_arm(fn, out_dir, tag):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    rows = []
    for ev in prof.key_averages():
        if ev.device_type.name == "CUDA" and ev.count:
            rows.append(dict(kernel=ev.key[:120], calls=ev.count, us=round(ev.device_time_total, 2)))
    rows.sort(key=lambda r: -r["us"])
    return rows


def bench(in_dim, S, iters, warmup):
    from shacira_b200.nerf_heads import NerfHeads
    torch.manual_seed(0)
    dev = torch.device("cuda", 0)
    dd = nn.Sequential(nn.Linear(in_dim, H), nn.ReLU(), nn.Linear(H, D)).to(dev)
    dc = nn.Sequential(nn.Linear(D + E, H), nn.ReLU(), nn.Linear(H, H), nn.ReLU(), nn.Linear(H, 3)).to(dev)
    heads = NerfHeads(dd, dc)
    feats = torch.randn(S, in_dim, device=dev, requires_grad=True)
    R = S // 64
    vemb = torch.randn(R, E, device=dev)
    ridx = torch.arange(R, device=dev, dtype=torch.int32).repeat_interleave(64)
    gd, grgb = torch.randn(S, 1, device=dev), torch.randn(S, 3, device=dev)

    def kernel_fwd():
        with torch.no_grad():
            heads(feats, vemb, ridx)

    def kernel_fwd_bwd():
        density, rgb = heads(feats, vemb, ridx)
        torch.autograd.backward([density, rgb], [gd, grgb])

    def torch_heads(autocast):
        def fn():
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
                d = dd(feats)
                rgb = torch.sigmoid(dc(torch.cat([d, vemb[ridx]], 1)))
                density = torch.relu(d[:, :1])
            torch.autograd.backward([density.float(), rgb.float()], [gd, grgb])
        return fn

    fwd_flops, fb_flops = flops_per_sample(in_dim)
    arms = {"kernel_fwd": (kernel_fwd, fwd_flops * S, bytes_moved(S, in_dim, "fwd")),
            "kernel_fwd_bwd": (kernel_fwd_bwd, fb_flops * S, bytes_moved(S, in_dim, "fwd_bwd")),
            "torch_fp32_fwd_bwd": (torch_heads(False), fb_flops * S * 3 / 4, bytes_moved(S, in_dim, "fwd_bwd")),
            "torch_autocast_bf16_fwd_bwd": (torch_heads(True), fb_flops * S * 3 / 4, bytes_moved(S, in_dim, "fwd_bwd"))}
    res = dict(in_dim=in_dim, hidden=H, emb=E, samples=S, feats_mbytes=S * in_dim * 4 / 2 ** 20, arms={})
    for name, (fn, flops, nbytes) in arms.items():
        us = time_arm(fn, iters, warmup)
        t_flop, t_byte = flops / (PEAK_TFLOPS * 1e12) * 1e6, nbytes / (PEAK_TBS * 1e12) * 1e6
        res["arms"][name] = dict(
            us=round(us, 2), flops=flops, bytes=nbytes, tflops=round(flops / us / 1e6, 2),
            tflops_share_of_2250=round(flops / us / 1e6 / PEAK_TFLOPS, 4), tb_per_s=round(nbytes / us / 1e6, 3),
            bytes_share_of_7_7=round(nbytes / us / 1e6 / PEAK_TBS, 4), bound="flops" if t_flop > t_byte else "bytes",
            lower_bound_us=round(max(t_flop, t_byte), 2))
    res["note"] = ("the PyTorch arms store activations instead of recomputing them: their FLOP count is 3/4 of the "
                   "kernel's forward + backward")
    res["profile"] = {name: profile_arm(fn, None, name)[:12] for name, (fn, _, _) in arms.items()}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=1 << 19)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("benchmarks/nerf_heads.py needs a CUDA device")
    out = dict(card=card(), iters=args.iters, warmup=args.warmup,
               runs=[bench(in_dim, args.samples, args.iters, args.warmup) for in_dim in (64, 96)])
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
