#!/usr/bin/env python
"""bench.py -- latent hash-grid fwd+bwd throughput (BASELINE.json metric) on N B200s.

    python bench.py --gpus N --steps K --warmup W            # this package (CUDA, C-ABI)
    python bench.py --steps K --dump-outputs DIR             # + what the last timed step computes, DIR/<name>.npy
    python bench.py --impl reference --steps K --warmup W    # the reference's path on the host cores
    python bench.py --impl reference-gpu                     # the reference's own CUDA kernels (oracle/_ref)

Workload (BASELINE.json configs[1], SURVEY 8d cfg2): the Kodak-shape image INR grid -- 768x512
pixel-centre coordinates in reference (y, x) order shuffled by randperm, 2D LatentGrid, 16 levels
16->512, 2^16-row tables (374 612 rows), latent_dim = feature_dim = 1, affine per-table decoder
with shift, straight-through rounding. One STEP = one forward + one backward of the latent grid
over the full 393 216-point batch: quantise + decode + interpolate, then the scatter-add to the
latents plus the decoder's scale/shift gradients. Synthetic, seeded data; random-init parameters
(latents scaled so that rounding is non-trivial).

Multi-GPU (N > 1, torchrun): every rank fits its own independent image (different shuffle,
different latents) -- the path shards by independent units, there is no data-path collective,
scaling is weak. Timing is on the device (CUDA events), barrier + synchronize on both sides, max
over ranks.

The JSON line also carries: `roofline` (dominant kernel, algorithmic bytes / measured launch time
against the measured HBM copy peak), `kernels` (every kernel of the step), `entropy` (the fused
bit-rate kernel, reported beside the step), `cpu_baseline` (the oracle port on this box's host
cores), `e2e` (the same fwd+bwd through the host-buffer C-ABI session, PCIe copies inside the timed region),
`clocks`, `gpu_launches`.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the tree as it found it (it may be read-only)

H, W = 512, 768
NUM_LODS, BITWIDTH, MIN_RES, MAX_RES = 16, 16, 16, 512
LATENT_DIM, FEATURE_DIM, DIM = 1, 1, 2
ROTATE = 4  # independent input/output buffer sets cycled through so that no step finds its streams in L2


def algorithmic_bytes_per_point(D, L, C, F):
    """SURVEY 8d: fwd [4D + 2^D*L*C*4 + 4*L*F] + bwd [4D + 4*L*F + 2^D*L*C*4]."""
    one = 4 * D + (2 ** D) * L * C * 4 + 4 * L * F
    return one, one


def make_workload(seed):
    b = np.exp((np.log(MAX_RES) - np.log(MIN_RES)) / (NUM_LODS - 1))  # latent_grid.py:280-281
    res = [int(1 + np.floor(MIN_RES * (b ** l))) for l in range(NUM_LODS)]
    sizes, first, T = oracle_layout(res)
    rng = np.random.default_rng(seed)
    ys, xs = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    coords = np.stack([(ys.reshape(-1) / H - 0.5) * 2, (xs.reshape(-1) / W - 0.5) * 2], 1).astype(np.float32)
    sets = []
    for r in range(ROTATE):
        perm = rng.permutation(coords.shape[0])
        sets.append(dict(coords=np.ascontiguousarray(coords[perm]),
                         grad_out=rng.standard_normal((coords.shape[0], NUM_LODS * FEATURE_DIM)).astype(np.float32)))
    latents = ((rng.random((T, LATENT_DIM), dtype=np.float32) - 0.5) * 16).astype(np.float32)  # U(-8, 8)
    scale = (rng.standard_normal((1, LATENT_DIM, FEATURE_DIM)) * 0.1).astype(np.float32)
    shift = (rng.standard_normal((1, FEATURE_DIM)) * 0.05).astype(np.float32)
    noise = (rng.random((T, LATENT_DIM), dtype=np.float32) - 0.5).astype(np.float32)
    prob = (rng.standard_normal((4, 3, LATENT_DIM)) * 0.3).astype(np.float32)
    return dict(res=res, first=first, T=T, sets=sets, latents=latents, A=scale, shift=shift, noise=noise, prob=prob)


def oracle_layout(res):
    sizes = [min(2 ** BITWIDTH, r ** DIM) for r in res]
    first = [0]
    for s in sizes[:-1]:
        first.append(first[-1] + s)
    return sizes, first, sum(sizes)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def recorded_traffic():
    """dram bytes per launch of the dominant kernel from the committed ncu capture, if any."""
    path = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f)
    return {}


class ClockSampler:
    """Polls NVML during the timed region: SM clock and clock-event (throttle) reasons."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _poll(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    bits = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if bits & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.0005)

    def start(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._poll, daemon=True)
            self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
# the reference arm / CPU baseline: the oracle port on the host cores
# ------------------------------------------------------------------------------------------------
def cpu_step(wl, s, want_entropy=False):
    """One step of the reference's path restated on the CPU: table-side round + decode (torch), then the
    reference's interpolation forward and backward (oracle/hashgrid_oracle.c, OpenMP). F == 1 is padded to
    2 and strided back exactly like LatentGrid.interpolate (latent_grid.py:361-363,370)."""
    import torch
    import oracle
    from oracle import latent_oracle as lo
    cb = torch.from_numpy(wl["latents"])
    table = lo.decode_single(lo.ste_round(cb), torch.ones(LATENT_DIM), torch.from_numpy(wl["A"][0]),
                             torch.from_numpy(wl["shift"]))
    table2 = table.repeat(1, 2).numpy()
    feats = oracle.forward(s["coords"], table2, wl["first"], wl["res"], BITWIDTH)[:, ::2]
    g2 = np.zeros((s["coords"].shape[0], NUM_LODS * 2), dtype=np.float32)
    g2[:, ::2] = s["grad_out"]
    gtab = oracle.backward(s["coords"], g2, wl["T"], wl["first"], wl["res"], BITWIDTH, 2)
    glat = gtab.sum(1, keepdims=True) * wl["A"][0, 0, 0]  # straight-through + d decode / d latent
    ent = None
    if want_entropy:
        p = wl["prob"]
        params = {"f%d" % (i + 1): (torch.from_numpy(p[i, 0:1]), torch.from_numpy(p[i, 1:2]),
                                    torch.from_numpy(p[i, 2:3]) if i < 3 else None) for i in range(4)}
        ent = lo.ent_loss(cb, torch.from_numpy(wl["noise"]), params, 2)[1].item()
    return feats, glat, ent


def run_cpu(wl, steps, warmup):
    import oracle
    oracle.use_all_cores()   # torchrun exports OMP_NUM_THREADS=1; the CPU arm gets every host core
    n = wl["sets"][0]["coords"].shape[0]
    for i in range(warmup):
        cpu_step(wl, wl["sets"][i % ROTATE])
    t0 = time.perf_counter()
    for i in range(steps):
        cpu_step(wl, wl["sets"][i % ROTATE])
    dt = time.perf_counter() - t0
    t1 = time.perf_counter()
    cpu_step(wl, wl["sets"][0], want_entropy=True)
    t_with_ent = time.perf_counter() - t1
    return {"mpts": n * steps / dt / 1e6, "ms_per_step": dt / steps * 1e3, "threads": oracle.num_threads(),
            "entropy_ms": max(0.0, t_with_ent * 1e3 - dt / steps * 1e3)}


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    wl = make_workload(0)
    n = wl["sets"][0]["coords"].shape[0]
    steps, warmup = args.steps, args.warmup
    r = run_cpu(wl, steps, warmup)
    line = {
        "impl": "reference", "metric": "latent hash-grid fwd+bwd Mpoints/s per GPU", "value": r["mpts"],
        "unit": "Mpoints/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(),
        "cpu_baseline": {"value": r["mpts"], "unit": "Mpoints/s", "cores": r["threads"], "kind": "port",
                         "sample": "%d steps x full %d-point batch (fwd+bwd incl. table decode), OpenMP oracle port; "
                                   "the reference has no CPU implementation of this path" % (steps, n)},
        "e2e": {"value": r["mpts"], "unit": "Mpoints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "entropy": {"ms": r["entropy_ms"], "impl": "torch CPU restatement of ent_loss forward (no backward)"},
        "host_cpus": os.cpu_count(),
    }
    print(json.dumps(line), flush=True)
    return 0


def workload_config():
    return {"workload": "BASELINE cfg2: Kodak-shape 768x512 image INR grid, 2D LatentGrid, 16 levels 16->512, "
                        "2^16-row tables (374612 rows), C=F=1, affine decoder, STE rounding; 393216 points/step",
            "points_per_step": H * W, "levels": NUM_LODS, "bitwidth": BITWIDTH, "latent_dim": LATENT_DIM,
            "feature_dim": FEATURE_DIM, "step": "latent grid forward + backward (latents + decoder grads)",
            "l2": "inputs larger than L2: %d rotating input/output sets (~%d MB) cycled between steps" % (
                ROTATE, ROTATE * (H * W * (8 + 3 * 64)) // (1 << 20)),
            "parallelism": "independent images, one per GPU, no collective"}


# ------------------------------------------------------------------------------------------------
# this package
# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-plan", action="store_true", help="point-parallel kernels instead of the tiled path")
    ap.add_argument("--no-graph", action="store_true", help="launch from the host loop instead of replaying a CUDA graph")
    ap.add_argument("--no-fit", action="store_true", help="skip the short Kodak-shape fit (fits/hour, second half of the metric)")
    ap.add_argument("--no-nerf", action="store_true", help="skip the NeRF-shape ray-batch data-parallel step (cfg4)")
    ap.add_argument("--no-ref-gpu", action="store_true", help="skip timing the reference's own CUDA kernels (oracle/_ref)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computes (rank 0): feature rows, latent gradient and the "
                         "shared decoder's scale / shift gradients, as DIR/<name>.npy in float32; the seeded inputs "
                         "are the same in every run, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours only")
    if args.impl == "reference":
        return reference_arm(args)
    if args.impl == "reference-gpu":
        return reference_gpu_arm(args)

    import torch
    import torch.distributed as dist
    from shacira_b200 import _lib

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback "
                         "(use --impl reference for the host-core baseline)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()
    steps, warmup = args.steps, max(args.warmup, 3)

    wl = make_workload(rank)  # every rank: its own image (independent unit)
    n, T, L = H * W, wl["T"], NUM_LODS
    d = lambda a: torch.from_numpy(a).to(dev)
    sets = [dict(coords=d(s["coords"]), grad_out=d(s["grad_out"])) for s in wl["sets"]]
    latents, A, shift = d(wl["latents"]), d(wl["A"]), d(wl["shift"])
    noise, prob = d(wl["noise"]), d(wl["prob"])
    first, res = wl["first"], wl["res"]

    # static coordinates: one spatial plan per coordinate set, built once (an image fit reuses it for
    # every step); its build time is reported as plan_ms and is NOT part of the timed steps.
    plan_ms = None
    if not args.no_plan:
        for s in sets:
            s["plan"] = _lib.Plan(s["coords"])
        torch.cuda.synchronize()
        # device time of binning one coordinate set (3 kernels; the allocation is reused by plan_rebuild)
        import ctypes as _ct
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        st_cur = _ct.c_void_p(torch.cuda.current_stream().cuda_stream)
        p0.record()
        for s in sets:
            _lib._check(_lib.load().shacira_plan_rebuild(s["plan"].handle, DIM, _lib._ptr(s["coords"]), n, 0, st_cur))
        p1.record()
        torch.cuda.synchronize()
        plan_ms = p0.elapsed_time(p1) / len(sets)

    # Outputs are preallocated and the C-ABI is called directly: the timed region holds kernel launches
    # only (no allocator, no Python tensor plumbing). The K timed steps are captured into ONE CUDA graph
    # and replayed, so the device never waits for the host between launches.
    import ctypes
    lib = _lib.load()
    fi, _ = _lib._i32_array(first)
    rs, _ = _lib._i32_array(res)
    P = _lib._ptr
    for s in sets:
        s["feats"] = torch.empty((n, L * FEATURE_DIM), device=dev)
        s["z"] = torch.empty((n, L * LATENT_DIM), device=dev)
        s["gl"] = torch.empty((T, LATENT_DIM), device=dev)
    gA = torch.zeros((L, LATENT_DIM, FEATURE_DIM), device=dev)
    gS = torch.zeros((L, FEATURE_DIM), device=dev)

    def fwd(i, st):
        s = sets[i % ROTATE]
        if args.no_plan:
            rc = lib.shacira_latent_forward(DIM, P(s["coords"]), n, P(latents), fi, rs, L, BITWIDTH, LATENT_DIM,
                                            FEATURE_DIM, 1, P(A), P(shift), 0, P(s["feats"]), P(s["z"]), st)
        else:
            rc = lib.shacira_latent_forward_planned(s["plan"].handle, P(latents), fi, rs, L, BITWIDTH, LATENT_DIM,
                                                    FEATURE_DIM, 1, P(A), P(shift), 0, P(s["feats"]), st)
        _lib._check(rc)

    def bwd(i, st):
        s = sets[i % ROTATE]
        if args.no_plan:
            rc = lib.shacira_latent_backward(DIM, P(s["coords"]), n, P(s["grad_out"]), P(s["z"]), fi, rs, L, BITWIDTH,
                                             LATENT_DIM, FEATURE_DIM, P(A), 0, T, 1, P(s["gl"]), P(gA), P(gS), st)
        else:
            rc = lib.shacira_latent_backward_planned(s["plan"].handle, P(s["grad_out"]), P(latents), fi, rs, L,
                                                     BITWIDTH, LATENT_DIM, FEATURE_DIM, 1, P(A), 0, T, 1, P(s["gl"]),
                                                     P(gA), P(gS), st)
        _lib._check(rc)

    def step(i, st):
        fwd(i, st)
        bwd(i, st)

    stream = torch.cuda.Stream(device=dev)

    def make_graph(fn, count):
        """`count` consecutive calls of fn(i, stream) captured into one CUDA graph on `stream`."""
        if args.no_graph:
            return None
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=stream):
            st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            for i in range(count):
                fn(i, st)
        return g

    def run(fn, count, graph):
        if graph is not None:
            graph.replay()
        else:
            st = ctypes.c_void_p(stream.cuda_stream)
            for i in range(count):
                fn(i, st)

    with torch.cuda.stream(stream):
        st0 = ctypes.c_void_p(stream.cuda_stream)
        for i in range(warmup):
            step(i, st0)
        stream.synchronize()
        launches_per_step0 = _lib.launch_count()
        step(0, st0)
        launches_per_step = _lib.launch_count() - launches_per_step0
        g_step, g_fwd, g_bwd = make_graph(step, steps), make_graph(fwd, steps), make_graph(bwd, steps)
        run(step, steps, g_step)  # one untimed replay (graph upload)
        stream.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        sampler = ClockSampler(local)
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sampler.start()
        start.record()
        run(step, steps, g_step)
        stop.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        total_ms = start.elapsed_time(stop)
        outputs = None
        if args.dump_outputs and rank == 0:
            # The decoder gradients are accumulated into across steps (the timed loop never clears them), so the last
            # timed step runs once more, untimed, from zeroed ones. One shared decoder: only the sum over the L rows is
            # defined, and that sum is what a caller receives (grid_ops.LatentHashGrid.backward).
            gA.zero_()
            gS.zero_()
            step(steps - 1, st0)
            stream.synchronize()
            last = sets[(steps - 1) % ROTATE]
            outputs = {"feats": last["feats"].clone(), "grad_latents": last["gl"].clone(),
                       "grad_A": gA.sum(0, keepdim=True), "grad_shift": gS.sum(0, keepdim=True)}
        # per-kernel launch durations, measured live with CUDA events over K back-to-back launches each
        def timed(fn, graph):
            run(fn, steps, graph)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run(fn, steps, graph)
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / steps
        fwd_ms, bwd_ms = timed(fwd, g_fwd), timed(bwd, g_bwd)
        clocks = sampler.stop()  # sampled across the timed step replay and the per-kernel replays
    launches = launches_per_step * steps
    t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())

    # the fused bit-rate kernel, reported beside the step (table-side: once per step, not per point);
    # graph-replayed like the step so that the number is device time, not Python launch overhead
    ent_bits = torch.empty((1 + L,), dtype=torch.float64, device=dev)
    ent_gl = torch.empty((T, LATENT_DIM), device=dev)
    ent_gp = torch.empty((4, 3, LATENT_DIM), device=dev)
    ent_scratch = torch.zeros(int(lib.shacira_entropy_scratch_bytes(LATENT_DIM, L)), dtype=torch.uint8, device=dev)

    def ent(i, st):
        _lib._check(lib.shacira_entropy_bits(P(latents), P(noise), T, LATENT_DIM, P(prob), 2, fi, L, P(ent_bits),
                                             P(ent_gl), P(ent_gp), P(ent_scratch), ent_scratch.numel(), st))

    with torch.cuda.stream(stream):
        ent(0, ctypes.c_void_p(stream.cuda_stream))
        stream.synchronize()
        g_ent = make_graph(ent, 20)
        run(ent, 20, g_ent)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run(ent, 20, g_ent)
        e1.record()
        torch.cuda.synchronize()
        ent_ms = e0.elapsed_time(e1) / 20

    # end to end: the host-buffer C-ABI (shacira_host_session_*), pinned host memory, every copy inside the timed region.
    # One coordinate set (an image fit has static coordinates: uploaded and binned once, before the loop); per step the
    # host hands over the current table + decoder (they change every step of a fit) and the upstream gradient rows, and
    # receives the feature rows, the table gradient and the decoder gradients. Two steps in flight.
    pin = lambda a: torch.from_numpy(a).pin_memory()
    h_coords = pin(wl["sets"][0]["coords"])
    h_gout = [pin(wl["sets"][k]["grad_out"]) for k in range(2)]
    h_lat, h_A, h_shift = pin(wl["latents"]), pin(wl["A"]), pin(wl["shift"])
    h_feats = [torch.empty((n, L * FEATURE_DIM), dtype=torch.float32).pin_memory() for _ in range(2)]
    h_gl = [torch.empty((T, LATENT_DIM), dtype=torch.float32).pin_memory() for _ in range(2)]
    h_gA = [torch.empty((L, LATENT_DIM, FEATURE_DIM), dtype=torch.float32).pin_memory() for _ in range(2)]
    h_gS = [torch.empty((L, FEATURE_DIM), dtype=torch.float32).pin_memory() for _ in range(2)]
    sess = _lib.HostSession(h_coords, T, first, res, BITWIDTH, LATENT_DIM, FEATURE_DIM, device=dev)
    e2e_steps = max(4, min(steps, 100))

    def e2e_run(count):
        pending = None
        for i in range(count):
            sess.set_table(h_lat, h_A, h_shift, True)
            slot = sess.step(h_gout[i % 2], h_feats[i % 2], h_gl[i % 2], h_gA[i % 2], h_gS[i % 2])
            if pending is not None:
                sess.wait(pending)       # the host consumes step i-1's results while step i is in flight
            pending = slot
        sess.wait(pending)

    e2e_run(6)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    e2e_run(e2e_steps)
    e2e_s = time.perf_counter() - t0  # the last wait synchronises
    sess.close()
    te = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_s = float(te.item())
    h2d = 4 * (T * LATENT_DIM + n * L * FEATURE_DIM + A.numel() + shift.numel())
    d2h = 4 * (n * L * FEATURE_DIM + T * LATENT_DIM + L * LATENT_DIM * FEATURE_DIM + L * FEATURE_DIM)

    # Second half of BASELINE.json's metric: Kodak-shape INR fits/hour. Every rank fits its own image (independent
    # units, no collective) for a short fixed budget with the whole training step -- grid, fused decoder MLP + MSE,
    # bit-rate loss, Adam -- in one CUDA graph; fits/hour extrapolates to the reference's 60 000-step fits.
    kodak_fit = None
    if not args.no_fit and not args.no_plan:
        try:
            sys.path.insert(0, os.path.join(ROOT, "benchmarks"))
            import fit_image
            # The reference's recipe (kodak.yaml:43-52): SGA sampling with the exponential temperature schedule while
            # epoch / max_epochs <= 0.9, straight-through rounding for the last 10 %. Both phases are measured
            # (CUDA-graph replay, one graph per phase) and fits/hour weights them 0.9 / 0.1.
            one = fit_image.fit_native_recipe([rank], 400, dev)[0]
            # throughput form (BASELINE cfg3: 24 independent images over the GPUs): three fits in flight per GPU,
            # one stream + one CUDA graph each -- independent INRs overlap each other's latency
            group = fit_image.fit_native_recipe([3 * rank, 3 * rank + 1, 3 * rank + 2], 400, dev)[0]
            tf = torch.tensor([one["ms_per_step_sga"], one["ms_per_step_ste"], group["ms_per_step_sga"],
                               group["ms_per_step_ste"]], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(tf, op=dist.ReduceOp.MAX)
            s1, t1, s3, t3 = [float(v) for v in tf.tolist()]
            w1, w3 = 0.9 * s1 + 0.1 * t1, 0.9 * s3 + 0.1 * t3
            kodak_fit = {"recipe": "SGA (temperature 1.0 -> 0.1, exponential) for 90 % of the steps, then STE rounding; "
                                   "kodak.yaml:43-52, image_trainer.py:131-137",
                         "ms_per_step_sga": s1, "ms_per_step_ste": t1, "ms_per_step": w1,
                         "steps_measured": {"sga": one["sga_steps"], "ste": one["ste_steps"]}, "steps_per_fit": 60000,
                         "fits_per_hour_one_fit_per_gpu": world * 3600.0 / (60000 * w1 * 1e-3),
                         "concurrent_fits_per_gpu": 3, "ms_per_step_sga_per_fit_concurrent": s3,
                         "ms_per_step_ste_per_fit_concurrent": t3, "ms_per_step_per_fit_concurrent": w3,
                         "fits_per_hour": world * 3600.0 / (60000 * w3 * 1e-3),
                         "psnr_after_400_steps": one["psnr"], "bpp_after_400_steps": one["bpp"],
                         "note": "step times extrapolated to the reference's 60 000-step fits; the per-epoch size() / "
                                 "PSNR / best-state bookkeeping of ImageTrainer is not part of the step",
                         "step": "shacira_b200.image_fit.ImageFitStep: 3 launches per step in one CUDA graph per phase -- the "
                                 "tile-resident fused kernel (grid forward + tensor-core decoder MLP / MSE + grid "
                                 "backward, shacira_fit_tile_step), the bit-rate kernel beside it, and ONE optimizer "
                                 "launch (Adam of every parameter group + the next step's SGA sample, "
                                 "shacira_fit_optimizer_step); independent images, no collective"}
        except Exception as e:  # the headline metric must not depend on the extra measurement
            kodak_fit = {"unavailable": repr(e)[:200]}

    # End to end at the level the path is meant to be used at (the base contract's wording: that step's inputs from
    # pinned host memory in, the step's loss out): the natively fused fit step keeps table, decoder, MLP and optimizer
    # state on the device, so per step only the batch's targets cross PCIe (4.7 MB) and 8 bytes of loss come back --
    # against 53 MB per step when a host-side consumer wants the feature rows (the `e2e` entry above).
    e2e_fit = fit_tile = None
    if not args.no_fit and not args.no_plan:
        try:
            import fit_image
            grid_f, mlp_f, coords_f, gt_f, fs = fit_image._native_setup(1000 + rank, dev, device_noise=True, sga=True)
            h_gt = [gt_f.cpu().pin_memory(), gt_f.flip(0).cpu().pin_memory()]
            loss_host = torch.zeros(2, dtype=torch.float64).pin_memory()
            fs.set_lambda(5e-4)
            fs.set_temperature(0.5)
            fstream = torch.cuda.Stream(device=dev)
            cstream = torch.cuda.Stream(device=dev)      # uploads: step i + 1's targets travel while step i runs
            tbuf = [fs.target, torch.empty_like(fs.target)]
            gfit, uploaded, consumed = [], [torch.cuda.Event(), torch.cuda.Event()], [torch.cuda.Event(), torch.cuda.Event()]
            with torch.cuda.stream(fstream):
                for _ in range(3):
                    fs.step()
                fstream.synchronize()
                for b in range(2):                       # one captured step per target buffer
                    fs.target = tbuf[b]
                    g_ = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g_, stream=fstream):
                        fs.step()
                    gfit.append(g_)
                fs.target = tbuf[0]

                loss_dev = fs.mlp_out[:2].view(torch.float64)                    # views made once: the loop is host bound
                loss_slot = [loss_host[0:1], loss_host[1:2]]
                cctx = torch.cuda.stream(cstream)

                def fit_e2e(count):
                    for b in range(2):
                        consumed[b].record(fstream)
                    for i in range(count):
                        b = i & 1
                        with cctx:
                            cstream.wait_event(consumed[b])                     # the step that last read this buffer is done
                            tbuf[b].copy_(h_gt[b], non_blocking=True)           # this step's targets, host -> device
                            uploaded[b].record(cstream)
                        fstream.wait_event(uploaded[b])
                        gfit[b].replay()
                        consumed[b].record(fstream)
                        loss_slot[b].copy_(loss_dev, non_blocking=True)
                        if i % 8 == 7:
                            fstream.synchronize()                               # the host reads the losses in small batches
                    fstream.synchronize()

                fit_e2e(16)
                if world > 1:
                    dist.barrier()
                # three timed batches, the median one reported: this leg is bound by the HOST side of the loop (six CUDA calls
                # per step from Python) and its wall clock is jittery (0.16 ... 0.45 ms per step seen for one batch)
                fit_steps, batches = 100, []
                for _ in range(3):
                    t0 = time.perf_counter()
                    fit_e2e(fit_steps)
                    batches.append(time.perf_counter() - t0)
                fit_s = sorted(batches)[1]
            tfit = torch.tensor([fit_s], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(tfit, op=dist.ReduceOp.MAX)
            fit_s = float(tfit.item())
            # the fused tile kernel of that step alone (SURVEY 8 row f-1: grid forward + decoder MLP / MSE + grid backward
            # in one launch, feature rows never in HBM): device time over a graph of 20 launches
            try:
                Pp, lin = _lib._ptr, fs.lin
                sh = fs.layer.shift.data if fs.has_shift else None

                def tile_step(st_):
                    _lib._check(lib.shacira_fit_tile_step(
                        fs.plan.handle, Pp(fs.grid.codebook.data), fs.fi, fs.rs, fs.L, fs.bw, 1, Pp(fs.A), Pp(sh),
                        Pp(fs.target), Pp(lin[0].weight.data), Pp(lin[0].bias.data), Pp(lin[1].weight.data),
                        Pp(lin[1].bias.data), Pp(lin[2].weight.data), Pp(lin[2].bias.data), fs.T, Pp(fs.g_grid),
                        Pp(fs.g_dec), Pp(fs.g_dec[fs.L:]), Pp(fs.mlp_out), st_))
                with torch.cuda.stream(fstream):
                    tile_step(ctypes.c_void_p(fstream.cuda_stream))
                    fstream.synchronize()
                    gt_ = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(gt_, stream=fstream):
                        for _ in range(20):
                            tile_step(ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
                    gt_.replay()
                    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    ev0.record()
                    gt_.replay()
                    ev1.record()
                    fstream.synchronize()
                    tile_ms = ev0.elapsed_time(ev1) / 20
                bpp_alg = sum(algorithmic_bytes_per_point(DIM, L, LATENT_DIM, FEATURE_DIM))
                fit_tile = {"ms": tile_ms, "what": "shacira_fit_tile_step: grid forward + decoder MLP / MSE + grid backward, one launch",
                            "algorithmic_GBs": bpp_alg * n / tile_ms / 1e6, "bytes_per_point": bpp_alg,
                            "dram_bytes_per_launch_ncu": 22004480,
                            "note": "ncu: 22 MB of DRAM traffic per launch (profiles/r02r_ncu_fit_fused_summary.txt) against "
                                    "~170 MB for the three launches it replaces (96 us); bound by instruction issue / "
                                    "latency of the MLP and lerp chains at 16 warps per SM, not by memory"}
            except Exception as e:
                fit_tile = {"unavailable": repr(e)[:200]}
            fs.close()
            e2e_fit = {"value": n * world * fit_steps / fit_s / 1e6, "unit": "Mpoints/s", "ms_per_step": fit_s / fit_steps * 1e3,
                       "h2d_bytes_per_step": int(gt_f.numel() * 4), "d2h_bytes_per_step": 8, "steps": fit_steps,
                       "batches_ms_per_step": [round(b / fit_steps * 1e3, 4) for b in batches],
                       "api": "shacira_b200.image_fit.ImageFitStep (SGA phase, CUDA graph): targets from pinned host "
                              "memory every step (two device buffers: the next step's upload runs beside this step), loss "
                              "read back; grid fwd + bwd + decoder MLP / MSE + bit-rate loss + Adam per step"}
        except Exception as e:
            e2e_fit = {"unavailable": repr(e)[:200]}

    # BASELINE cfg4 (the other half of the north_star): NeRF-shape ray-batch data parallel step at this N -- grid
    # forward + backward on 4096 rays x 128 samples per rank, then the NCCL all-reduce of the gradient arena.
    nerf = None
    if not args.no_nerf:
        try:
            sys.path.insert(0, os.path.join(ROOT, "benchmarks"))
            import nerf_dp
            nerf = nerf_dp.run(dev, rank, world, steps=30, warmup=5)
            peak_n, _ = measured_peaks()
            nerf["roofline"] = {"bound": "hbm", "achieved": nerf["alg_GBs_per_gpu"], "peak": peak_n, "unit": "GB/s",
                                "frac": nerf["alg_GBs_per_gpu"] / peak_n,
                                "note": "1560 algorithmic B/sample (SURVEY 8d) x samples per rank / step time incl. the "
                                        "per-step binning and the exchange; measured HBM copy peak"}
        except Exception as e:
            nerf = {"unavailable": repr(e)[:200]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    peak, peak_src = measured_peaks()
    bf, bb = algorithmic_bytes_per_point(DIM, L, LATENT_DIM, FEATURE_DIM)
    kernels = {
        "latent_fwd": {"ms": fwd_ms, "algorithmic_GBs": bf * n / fwd_ms / 1e6, "bytes_per_point": bf},
        "latent_bwd": {"ms": bwd_ms, "algorithmic_GBs": bb * n / bwd_ms / 1e6, "bytes_per_point": bb},
    }
    dom = "latent_bwd" if bwd_ms >= fwd_ms else "latent_fwd"
    traffic = recorded_traffic()
    roofline = {"bound": "hbm", "kernel": dom, "achieved": kernels[dom]["algorithmic_GBs"], "peak": peak,
                "unit": "GB/s", "frac": kernels[dom]["algorithmic_GBs"] / peak,
                "traffic": traffic.get(dom), "peak_source": peak_src,
                "step_achieved": (bf + bb) * n * steps / total_ms / 1e6,
                "step_frac": (bf + bb) * n * steps / total_ms / 1e6 / peak}
    value = n * world * steps / (total_ms * 1e-3) / 1e6
    line = {
        "metric": "latent hash-grid fwd+bwd Mpoints/s per GPU", "value": value, "unit": "Mpoints/s", "n_gpus": world,
        "steps": steps, "warmup": warmup, "ms_per_step": total_ms / steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(),
        "per_gpu": value / world, "roofline": roofline, "kernels": kernels,
        "entropy": {"ms": ent_ms, "rows": T, "GBs": 12.0 * T * LATENT_DIM / ent_ms / 1e6,
                    "note": "fused bit-rate fwd+bwd kernel, 12 B/entry algorithmic"},
        "e2e": {"value": n * world * e2e_steps / e2e_s / 1e6, "unit": "Mpoints/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "steps": e2e_steps, "ms_per_step": e2e_s / e2e_steps * 1e3,
                "api": "shacira_host_session_* (C-ABI, pinned host buffers in and out, two steps in flight; static "
                       "coordinate set uploaded and binned once; table + decoder + gradient rows up, feature rows + "
                       "table / decoder gradients down every step)"},
        "e2e_fit": e2e_fit, "fit_tile_kernel": fit_tile, "gpu_launches": int(launches), "clocks": clocks,
        "path": "point-parallel (no plan)" if args.no_plan else "tiled (spatial plan, built once per coordinate set)",
        "kodak_fit": kodak_fit, "nerf_dp": nerf, "plan_ms": plan_ms, "launch": "host loop" if args.no_graph else "one CUDA graph of K steps, replayed",
    }
    if not args.no_ref_gpu:
        # REF-GPU (SURVEY 2a: the bar is "the reference's own SIMT kernels compiled for sm_100a on the same box"):
        # same standing as the cpu_baseline leg -- the checker's build is timed, never used by the product path
        line["ref_gpu_baseline"] = time_reference_kernels(wl, dev, sets, latents, A, shift, steps=10, warmup=3)
    if not args.no_cpu_baseline:
        r = run_cpu(make_workload(0), 3, 1)
        line["cpu_baseline"] = {"value": r["mpts"], "unit": "Mpoints/s", "cores": r["threads"], "kind": "port",
                                "sample": "3 steps x full %d-point batch (fwd+bwd incl. table decode) after 1 warm-up; "
                                          "OpenMP oracle port of the reference kernels" % n,
                                "host_cpus": os.cpu_count()}
    if outputs is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, t in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), t.cpu().numpy())
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def reference_gpu_arm(args):
    """`--impl reference-gpu`: the reference's own CUDA kernels on this GPU (REF-GPU in BASELINE.md), a
    separate invocation so that the default run never touches oracle/."""
    import torch
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    dev = torch.device("cuda", 0)
    wl = make_workload(0)
    d = lambda a: torch.from_numpy(a).to(dev)
    sets = [dict(coords=d(s["coords"]), grad_out=d(s["grad_out"])) for s in wl["sets"]]
    r = time_reference_kernels(wl, dev, sets, d(wl["latents"]), d(wl["A"]), d(wl["shift"]), args.steps, args.warmup)
    r.update({"impl": "reference-gpu", "metric": "latent hash-grid fwd+bwd Mpoints/s per GPU", "n_gpus": 1,
              "config": workload_config()})
    print(json.dumps(r), flush=True)
    return 0


def time_reference_kernels(wl, dev, sets, latents, A, shift, steps=20, warmup=5):
    """The reference's own path on this GPU: table-side decode with torch ops, repeat(1,2), then its
    CUDA kernels (oracle/_ref, one launch per level), backward through the same kernels. Baseline only."""
    try:
        import torch
        from oracle import build_ref
        ref = build_ref.load()
        if ref is None:
            return {"unavailable": "oracle/_ref/wisp_ref_ops.so not built"}
        first_dev = torch.tensor(wl["first"], dtype=torch.int32, device=dev)
        n = H * W

        def ref_step(i):
            s = sets[i % ROTATE]
            table = (torch.round(latents) / 1.0) @ A[0] + shift
            table2 = table.repeat(1, 2)
            feats = ref.hashgrid_interpolate2d_cuda(s["coords"], table2, first_dev, wl["res"], BITWIDTH)[:, ::2]
            g2 = torch.zeros((n, NUM_LODS * 2), device=dev)
            g2[:, ::2] = s["grad_out"]
            gt = ref.hashgrid_interpolate2d_backward_cuda(s["coords"], g2, table2, first_dev, wl["res"], BITWIDTH, 2, False)
            return feats, gt.sum(1, keepdim=True) * A[0, 0, 0]

        for i in range(max(warmup, 3)):
            ref_step(i)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k = steps
        e0.record()
        for i in range(k):
            ref_step(i)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / k
        return {"value": n / ms / 1e3, "unit": "Mpoints/s", "ms_per_step": ms,
                "what": "reference CUDA kernels compiled for sm_100a + torch table decode, same workload, same GPU"}
    except Exception as e:  # baseline only: never fail the bench over it
        return {"unavailable": repr(e)[:200]}


if __name__ == "__main__":
    sys.exit(main())
