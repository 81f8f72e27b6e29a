"""Kodak-shape image INR fit (BASELINE cfg2 / cfg3): end-to-end PSNR / bpp parity and fits/hour.

The fit follows the reference's ImageTrainer (wisp/trainers/image_trainer.py:269-359, SURVEY section 8 appendix):
768x512 synthetic image, full-image steps on shuffled pixel-centre coordinates (y, x); 2D LatentGrid (16 levels
16->512, 2^16 rows, C = F = 1, single affine decoder with shift, norm='max' at iterations 1,2,5,10), MLP
16->16->16->3 ReLU, Adam groups {decoder lr 1e-3, grid lr 2e-2, latent_dec lr 1e-2 wd 1e-2, prob_model lr 1e-4
wd 1e-2}, loss = mse + lambda(epoch) * bits / rows with lambda cosine 1e-3 -> 1e-4, num_prob_layers = 2, noise
every step. SGA is OFF (it is RNG-bound; SURVEY 8d asks for SGA-off parity runs).

  --impl ours   shacira_b200.grids.LatentGrid (fused + tiled kernels)
  --impl native shacira_b200.image_fit.ImageFitStep: the whole training step (grid, MLP + loss, bit-rate loss, every
                gradient, Adam for every parameter group) as 11 native launches, no autograd
  --impl ref    the reference path restated with ITS OWN CUDA kernels (oracle/_ref): table-side
                round/decode in torch, repeat(1,2), one kernel launch per level, torch ent_loss  -- the checker
  --graph       capture the whole training step (grid, MLP, loss, backward, Adam) in one CUDA graph
  --images K    fit K images (seeds 0..K-1), sharded round-robin over the ranks (torchrun): fits/hour

Prints one JSON line: PSNR (clamped, uint8-quantised like ops/image/metrics.py:39-57), bpp (entropy of the
rounded latents + 32 bit per decoder/MLP parameter, image_trainer.py:162-168), ms/step, fits/hour
(60 000-step fits, the reference's kodak.yaml budget).
"""
import argparse
import json
import math
import os
import sys
import time

import numpy as np
import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from shacira_b200.image_fit import lambda_at, temperature_at   # noqa: E402  the recipe's schedules

H, W = 512, 768
LATENT_SCALE = 20.0


def synthetic_image(seed):
    g = torch.Generator().manual_seed(seed)
    ys, xs = torch.meshgrid(torch.linspace(0, 1, H), torch.linspace(0, 1, W), indexing="ij")
    img = torch.zeros(H, W, 3)
    for k in range(6):  # smooth multi-scale pattern + mild noise, in [0, 1]
        fx, fy, ph = torch.rand(3, generator=g) * torch.tensor([6.0 + 6 * k, 6.0 + 6 * k, 6.28])
        col = torch.rand(3, generator=g)
        img += (torch.sin(2 * math.pi * (fx * xs + fy * ys) + ph)[..., None] * 0.5 + 0.5) * col / (k + 1)
    img = img / img.amax()
    img = (img + 0.02 * torch.randn(H, W, 3, generator=g)).clamp(0, 1)
    return img


def make_data(seed, dev):
    img = synthetic_image(seed)
    ys, xs = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    coords = torch.stack([(ys.reshape(-1) / H - 0.5) * 2, (xs.reshape(-1) / W - 0.5) * 2], 1).float()
    perm = torch.randperm(H * W, generator=torch.Generator().manual_seed(seed))  # multi_image_dataset.py:156-158
    return coords[perm].contiguous().to(dev), img.reshape(-1, 3)[perm].contiguous().to(dev)


DEC = dict(ldecode_enabled=True, ldecode_type="single", use_sga=False, diff_sampling=True, use_shift=True,
           ldecode_matrix="sq", latent_dim=1, norm="max", norm_every=10, ldec_std=0.1, decay_period=0.9, temperature=0.1)
ENT = dict(num_prob_layers=2, entropy_reg=1e-3, entropy_reg_end=1e-4, entropy_reg_sched="cosine", noise_freq=1)


class RefGrid(nn.Module):
    """The reference's LatentGrid.interpolate / ent_loss restated around the reference's own kernels."""

    def __init__(self, ours):
        super().__init__()
        from oracle import build_ref
        self.ref = build_ref.load()
        assert self.ref is not None, "oracle/_ref/wisp_ref_ops.so missing"
        self.codebook = nn.Parameter(ours.codebook.detach().clone())
        import copy
        self.latent_dec = copy.deepcopy(ours.latent_dec)
        self.prob_model = copy.deepcopy(ours.prob_model)
        self.register_buffer("first_idx", ours.codebook_lod_first_idx.clone())   # device tensor, as the reference passes it
        self.resolutions, self.bw = list(ours.resolutions), ours.codebook_bitwidth
        ref, grid_self = self.ref, self
        res, bw = self.resolutions, self.bw

        class Fn(torch.autograd.Function):  # wisp/ops/grid.py:135-176
            @staticmethod
            def forward(ctx, coords, table):
                ctx.save_for_backward(coords, table)
                return ref.hashgrid_interpolate2d_cuda(coords, table, grid_self.first_idx, res, bw)

            @staticmethod
            def backward(ctx, g):
                coords, table = ctx.saved_tensors
                return None, ref.hashgrid_interpolate2d_backward_cuda(coords, g.contiguous(), table, grid_self.first_idx,
                                                                      res, bw, table.shape[1], False)
        self.fn = Fn

    def interpolate(self, coords, lod_idx):
        table = self.latent_dec(self.codebook).repeat(1, 2)       # latent_grid.py:359-363
        return self.fn.apply(coords, table)[:, ::2]                # :370

    def ent_loss(self, noise):
        weight = self.codebook + noise                             # latent_grid.py:132-136
        prob = self.prob_model(weight + 0.5) - self.prob_model(weight - 0.5)
        bits = torch.sum(torch.clamp(-1.0 * torch.log(prob + 1e-10) / np.log(2.0), 0, 50))
        return bits / self.codebook.shape[0], bits


def clamped_psnr(pred, gt):
    a = (torch.clamp(pred, 0, 1) * 255).to(torch.uint8).float()
    b = (torch.clamp(gt, 0, 1) * 255).to(torch.uint8).float()
    mse = torch.mean((a - b) ** 2).item()
    return 20 * np.log10(255.0) - 10 * np.log10(max(mse, 1e-12))


def _native_setup(seed, dev, device_noise=False, sga=False):
    from shacira_b200.grids import LatentGrid
    from shacira_b200.image_fit import ImageFitStep
    torch.manual_seed(seed)
    dec = dict(DEC)
    dec["use_sga"] = bool(sga)    # kodak.yaml:43: the reference's recipe; off after decay_period (image_trainer.py:136)
    grid = LatentGrid.from_geometric(feature_dim=1, num_lods=16, latent_dim=1, multiscale_type="cat", resolution_dim=2,
                                     feature_std=0.1, codebook_bitwidth=16, min_grid_res=16, max_grid_res=512,
                                     init_grid="uniform", conf_latent_decoder=dec, conf_entropy_reg=dict(ENT))
    mlp = nn.Sequential(nn.Linear(16, 16), nn.ReLU(), nn.Linear(16, 16), nn.ReLU(), nn.Linear(16, 3))
    with torch.no_grad():
        grid.codebook.mul_(LATENT_SCALE)
    grid, mlp = grid.to(dev), mlp.to(dev)
    coords, gt = make_data(seed, dev)
    fs = ImageFitStep(grid, mlp, coords, gt, lr=1e-3, grid_lr=2e-2, ldec_lr=1e-2, prob_lr=1e-4, weight_decay=0.0,
                      weight_decay_decoder=1e-2, device_noise=device_noise, noise_seed=10_000 + seed)
    return grid, mlp, coords, gt, fs


def _native_metrics(seed, grid, mlp, coords, gt, fs, ms_per_step):
    rgb_loss = float(fs.rgb_loss())
    fs.close()
    with torch.no_grad():
        pred = mlp(grid.interpolate(coords, 0))
        psnr = clamped_psnr(pred, gt)
        q = torch.round(grid.codebook.detach()[:, 0]).long()
        _, counts = torch.unique(q, return_counts=True)
        p = counts / counts.sum()
        latent_bits = float(torch.sum(torch.clamp(-torch.log(p + 1e-10) / np.log(2.0), 0, 1000) * counts))
        n_other = sum(p.numel() for p in mlp.parameters()) + sum(p.numel() for p in grid.latent_dec.parameters())
        bpp = (latent_bits + 32 * n_other) / (H * W)
    return dict(seed=seed, psnr=psnr, bpp=bpp, latent_bits=latent_bits, ms_per_step=ms_per_step, rgb_loss=rgb_loss)


def fit_native_recipe(seeds, steps, dev, decay_period=0.9, temperature=0.1):
    """The reference's recipe (kodak.yaml:43-52): SGA with the exponential temperature schedule while
    epoch / max_epochs <= decay_period, straight-through rounding afterwards; len(seeds) independent fits in flight, one
    stream and one CUDA graph per image and PHASE (a captured graph holds its quantiser). The two phases are timed
    separately: fits/hour weights them decay_period : 1 - decay_period."""
    fits = [_native_setup(s, dev, device_noise=True, sga=True) for s in seeds]
    streams = [torch.cuda.Stream(device=dev) for _ in seeds]
    switch = int(math.floor(decay_period * steps))      # epochs 1..switch sample with SGA (epoch = it + 1)

    def host_side(k, it):
        fs = fits[k][4]
        fs.set_lambda(lambda_at(it, steps))
        if fs.sga:
            fs.set_temperature(temperature_at(it, steps, temperature, decay_period))
        if it + 1 in (1, 2, 5, 10):
            fs.update_div()

    def capture():
        graphs = []
        for k in range(len(seeds)):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=streams[k]):
                fits[k][4].step()
            graphs.append(g)
        return graphs

    def run(graphs, a, b):
        for it in range(a, b):
            for k in range(len(seeds)):
                with torch.cuda.stream(streams[k]):
                    host_side(k, it)
                    graphs[k].replay()

    def timed(graphs, a, b):
        warm = min(20, max(0, (b - a) // 4))
        run(graphs, a, a + warm)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        run(graphs, a + warm, b)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / max(1, b - a - warm) * 1e3 / len(seeds)

    for k in range(len(seeds)):                         # eager warm-up (allocator, plan, Adam state)
        with torch.cuda.stream(streams[k]):
            for it in range(3):
                host_side(k, it)
                fits[k][4].step()
    torch.cuda.synchronize()
    ms_sga = timed(capture(), 3, switch)
    for f in fits:
        f[4].set_sga(False)
    ms_ste = timed(capture(), switch, steps)
    out = []
    for s, f in zip(seeds, fits):
        m = _native_metrics(s, *f, decay_period * ms_sga + (1 - decay_period) * ms_ste)
        m.update(ms_per_step_sga=ms_sga, ms_per_step_ste=ms_ste, sga_steps=switch, ste_steps=steps - switch)
        out.append(m)
    return out


def fit_native_many(seeds, steps, dev, use_graph, noise_cpu):
    """Fit len(seeds) independent images AT ONCE on one GPU through shacira_b200.image_fit.ImageFitStep (the whole
    training step as 11 native launches), one stream and one CUDA graph per image. Independent INRs share nothing, and
    every kernel of the step alone leaves most of the SMs' issue slots idle (ncu: 35-50 % busy), so two or three fits in
    flight overlap each other's latency. `ms_per_step` is wall time per step of the whole group divided by the group
    size, i.e. the throughput figure that fits/hour is made of."""
    fits = [_native_setup(s, dev, device_noise=not noise_cpu) for s in seeds]
    gens = [torch.Generator().manual_seed(10_000 + s) for s in seeds]
    streams = [torch.cuda.Stream(device=dev) for _ in seeds]

    def host_side(k, it):
        fs = fits[k][4]
        fs.set_lambda(lambda_at(it, steps))
        if noise_cpu:
            fs.draw_noise(gens[k])      # otherwise the bit-rate kernel draws its own noise (device_noise)
        if it + 1 in (1, 2, 5, 10):
            fs.update_div()

    graphs, start_it = [None] * len(seeds), 0
    if use_graph:
        for k in range(len(seeds)):
            with torch.cuda.stream(streams[k]):
                for it in range(3):
                    host_side(k, it)
                    fits[k][4].step()
        torch.cuda.synchronize()
        for k in range(len(seeds)):
            graphs[k] = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graphs[k], stream=streams[k]):
                fits[k][4].step()
        start_it = 3

    def run_steps(a, b):
        for it in range(a, b):
            for k in range(len(seeds)):
                with torch.cuda.stream(streams[k]):
                    host_side(k, it)
                    if graphs[k] is not None:
                        graphs[k].replay()
                    else:
                        fits[k][4].step()

    # the first replays are not timed: graph upload, and SM clocks that have dropped while the process was busy
    # elsewhere (measured in bench.py: a 400-step fit right after the PCIe-bound host-buffer phase ran 1.7x slower)
    warm = min(50, max(0, (steps - start_it) // 8))
    run_steps(start_it, start_it + warm)
    start_it += warm
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    run_steps(start_it, steps)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    ms = dt / (steps - start_it) * 1e3 / len(seeds)
    return [_native_metrics(s, *f, ms) for s, f in zip(seeds, fits)]


def fit_native(seed, steps, dev, use_graph, noise_cpu):
    return fit_native_many([seed], steps, dev, use_graph, noise_cpu)[0]


def fit_native_sga(seed, steps, dev, decay_period=0.9):
    """The recipe fit of fit(..., sga=True) through ImageFitStep: same CPU-drawn bit-rate noise and SGA draws (injected)."""
    grid, mlp, coords, gt, fs = _native_setup(seed, dev, device_noise=False, sga=True)
    gen = torch.Generator().manual_seed(10_000 + seed)
    sga_gen = torch.Generator().manual_seed(20_000 + seed)
    T = grid.codebook.shape[0]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for it in range(steps):
        fs.set_lambda(lambda_at(it, steps))
        fs.draw_noise(gen)
        if it + 1 in (1, 2, 5, 10):
            fs.update_div()
        on = it < int(decay_period * steps)
        if on != fs.sga:
            fs.set_sga(on)
        fs.set_temperature(temperature_at(it, steps, 0.1, decay_period), refresh=True)
        fs.sga_uniforms = torch.rand((T, 1, 2), generator=sga_gen).to(dev) if on else None
        fs.step()
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) / steps * 1e3
    return _native_metrics(seed, grid, mlp, coords, gt, fs, ms)


def fit(seed, impl, steps, dev, use_graph, noise_cpu, fused_mlp=False, sga=False, decay_period=0.9):
    """sga=True: the reference's recipe -- SGA sampling (temperature schedule of image_trainer.py:131-137) while
    it / steps <= decay_period, straight-through rounding afterwards -- with the U(0,1) draws of every step taken from a
    CPU generator and INJECTED into each arm, so that the arms differ by float ordering only. The "ref" arm then runs the
    torch definition of the sample (latent_decoders.FORCE_TORCH_SGA) in front of the reference's own kernels."""
    if impl == "native":
        return fit_native_sga(seed, steps, dev, decay_period) if sga else fit_native(seed, steps, dev, use_graph, noise_cpu)
    from shacira_b200 import grid_ops
    from shacira_b200.grids import LatentGrid
    torch.manual_seed(seed)
    grid = LatentGrid.from_geometric(feature_dim=1, num_lods=16, latent_dim=1, multiscale_type="cat", resolution_dim=2,
                                     feature_std=0.1, codebook_bitwidth=16, min_grid_res=16, max_grid_res=512,
                                     init_grid="uniform", conf_latent_decoder=dict(DEC), conf_entropy_reg=dict(ENT))
    mlp = nn.Sequential(nn.Linear(16, 16), nn.ReLU(), nn.Linear(16, 16), nn.ReLU(), nn.Linear(16, 3))
    with torch.no_grad():
        # SGA-off runs start with every latent rounding to 0 at the reference's feature_std = 0.1 and frequently
        # never leave that state (both arms collapse identically); SURVEY 8d: scale the latents so that rounding
        # is non-trivial from step 0.
        grid.codebook.mul_(LATENT_SCALE)
    grid, mlp = grid.to(dev), mlp.to(dev)
    grid.noise_on_device = not noise_cpu
    if impl == "ref":
        grid = RefGrid(grid).to(dev)
    coords, gt = make_data(seed, dev)
    T = grid.codebook.shape[0]
    cap = dict(capturable=True) if use_graph else {}
    if fused_mlp:
        cap["fused"] = True   # one multi-tensor Adam kernel per group instead of ~10 elementwise launches
    table_opt = None
    if fused_mlp and impl == "ours":
        from shacira_b200._lib import TableAdam
        table_opt = TableAdam(grid.codebook, lr=2e-2)     # SURVEY 8 f-4: one kernel for the 375 k-row table
    groups = [dict(params=list(mlp.parameters()), lr=1e-3, weight_decay=0.0)] + \
             ([] if table_opt else [dict(params=[grid.codebook], lr=2e-2, weight_decay=0.0)]) + [
              dict(params=[p for p in grid.latent_dec.parameters() if p.requires_grad], lr=1e-2, weight_decay=1e-2),
              dict(params=list(grid.prob_model.parameters()), lr=1e-4, weight_decay=1e-2)]
    opt = torch.optim.Adam(groups, eps=1e-8, **cap)
    lam = torch.zeros((), device=dev)
    noise_gen = torch.Generator().manual_seed(10_000 + seed)
    noise_buf = torch.zeros((T, 1), device=dev)
    out = {}
    sga_gen = torch.Generator().manual_seed(20_000 + seed)
    if sga:
        assert not use_graph
        from shacira_b200 import latent_decoders
        grid.latent_dec.diff_sampling = True

    def train_step():
        opt.zero_grad(set_to_none=use_graph)   # captured step: gradients are re-created from the graph's pool, no fills
        if sga:
            latent_decoders.FORCE_TORCH_SGA = impl == "ref"
        feats = grid.interpolate(coords, 0)
        if sga:
            latent_decoders.FORCE_TORCH_SGA = False
        if fused_mlp:   # SURVEY 8 f-1: MLP + MSE + all their gradients in one kernel
            rgb_loss, pred = grid_ops.mlp_mse_loss(feats, gt, mlp)
        else:
            pred = mlp(feats)
            rgb_loss = ((pred - gt) ** 2).mean()
        if impl == "ref":
            avg_bits, bits = grid.ent_loss(noise_buf)
        else:
            grid.noise = noise_buf
            grid.noise_freq = 2                      # odd idx: use the preset grid.noise (filled below)
            avg_bits, bits = grid.ent_loss(1)
        loss = rgb_loss + lam * avg_bits
        loss.backward()
        opt.step()
        if table_opt is not None:
            table_opt.step()
            grid.codebook.grad = None
        out["pred"], out["rgb_loss"], out["bits"] = pred.detach(), rgb_loss.detach(), bits.detach()

    def host_side(it):
        # schedules and the noise draw happen outside the (possibly captured) device step
        lam.fill_(lambda_at(it, steps))   # schedulers.py:26-27
        if noise_cpu:
            noise_buf.copy_(torch.rand((T, 1), generator=noise_gen) - 0.5)
        else:
            noise_buf.uniform_(-0.5, 0.5)
        if it + 1 in (1, 2, 5, 10):                  # norm_every % total_iterations == 0 (reversed modulo, Q7)
            with torch.no_grad():
                w = grid.codebook
                grid.latent_dec.div.data.copy_(torch.max(torch.abs(w.min(dim=0)[0]), torch.abs(w.max(dim=0)[0])))
        if sga:
            on = it < int(decay_period * steps)
            grid.latent_dec.use_sga = on
            grid.latent_dec.temperature = temperature_at(it, steps, 0.1, decay_period)
            grid.latent_dec.sga_uniforms = torch.rand((T, 1, 2), generator=sga_gen).to(dev) if on else None

    graph = None
    if use_graph:
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            for it in range(3):                      # warm-up on a side stream (allocator, plan, Adam state)
                host_side(it)
                train_step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            train_step()
        start_it = 3
    else:
        start_it = 0
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for it in range(start_it, steps):
        host_side(it)
        if graph is not None:
            graph.replay()
        else:
            train_step()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    with torch.no_grad():
        pred = mlp(grid.interpolate(coords, 0))
        psnr = clamped_psnr(pred, gt)
        q = torch.round(grid.codebook.detach()[:, 0]).long()
        _, counts = torch.unique(q, return_counts=True)
        p = counts / counts.sum()
        latent_bits = float(torch.sum(torch.clamp(-torch.log(p + 1e-10) / np.log(2.0), 0, 1000) * counts))
        n_other = sum(p.numel() for p in mlp.parameters()) + sum(p.numel() for p in grid.latent_dec.parameters())
        bpp = (latent_bits + 32 * n_other) / (H * W)
    return dict(seed=seed, psnr=psnr, bpp=bpp, latent_bits=latent_bits, ms_per_step=dt / (steps - start_it) * 1e3,
                rgb_loss=float(out["rgb_loss"]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--impl", default="ours", choices=["ours", "ref", "native"])
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--images", type=int, default=1)
    ap.add_argument("--graph", action="store_true")
    ap.add_argument("--noise-cpu", action="store_true", help="draw the entropy noise with the CPU generator (parity runs)")
    ap.add_argument("--fused-mlp", action="store_true", help="fused decoder MLP + MSE kernel (SURVEY 8 f-1) and fused Adam")
    ap.add_argument("--concurrent", type=int, default=1, help="--impl native: independent images fitted at once per GPU")
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from shacira_b200 import dp
    mine = dp.shard_units(args.images, rank, world)      # independent images: round-robin, no collective
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    if args.impl == "native" and args.concurrent > 1:
        results = []
        for i in range(0, len(mine), args.concurrent):
            results += fit_native_many(mine[i:i + args.concurrent], args.steps, dev, args.graph, args.noise_cpu)
    else:
        results = [fit(s, args.impl, args.steps, dev, args.graph, args.noise_cpu, args.fused_mlp) for s in mine]
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    allres = dp.gather_results(dict(rank=rank, wall=wall, fits=results))
    if rank == 0:
        wall = max(r["wall"] for r in allres)
        fits = [f for r in allres for f in r["fits"]]
        ms = float(np.mean([f["ms_per_step"] for f in fits]))
        print(json.dumps({"workload": "Kodak-shape image INR fit (BASELINE cfg2/cfg3)", "impl": args.impl,
                          "n_gpus": world, "images": args.images, "steps_per_fit": args.steps, "concurrent_per_gpu": args.concurrent, "cuda_graph": args.graph, "fused_mlp": args.fused_mlp,
                          "ms_per_step": ms, "psnr": [round(f["psnr"], 3) for f in fits], "bpp": [round(f["bpp"], 4) for f in fits],
                          "wall_s": wall,
                          "fits_per_hour_at_60000_steps": world * 3600.0 / (60000 * ms * 1e-3) if fits else None}), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
