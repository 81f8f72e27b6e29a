"""A/B of two (or more) builds of the library on the flagship workload, alternated in one session.

    python benchmarks/tiled_prefetch_ab.py --lib parent=PATH.so --lib new=shacira_b200/libshacira_b200.so \
        [--rounds 3] [--out profiles/r05_tiled_prefetch_ab.json]

Every round runs, for each build in turn (selected with SHACIRA_LIB, each in its own process): `bench.py --gpus 1`,
`benchmarks/kernel_times.py` (tiled forward / backward alone) and `benchmarks/dropin_times.py` (the reference's F = 2
call pattern). It also records the card, its power limit, and for each tiled kernel a build launches at the flagship
shape the dynamic shared memory of that launch and the resident CTAs per SM the CUDA occupancy calculator gives."""
import argparse
import ctypes
import glob
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TILED = ("latent_fwd_tiled_kernel", "latent_bwd_tiled_kernel")


def probe():
    """Runs the flagship forward + backward once under torch.profiler and prints, for each tiled kernel launched, the
    shared memory the trace reports for that launch (static + dynamic)."""
    import torch
    sys.path.insert(0, ROOT)
    import bench
    from shacira_b200 import _lib
    dev = torch.device("cuda", 0)
    wl = bench.make_workload(0)
    d = lambda a: torch.from_numpy(a).to(dev)
    coords, g = d(wl["sets"][0]["coords"]), d(wl["sets"][0]["grad_out"])
    lat, A, S = d(wl["latents"]), d(wl["A"]), d(wl["shift"])
    plan = _lib.Plan(coords)
    run_once = lambda: (_lib.latent_forward_planned(plan, lat, wl["first"], wl["res"], bench.BITWIDTH, A, S, 1, True),
                        _lib.latent_backward_planned(plan, g, lat, wl["first"], wl["res"], bench.BITWIDTH, A, 1, 1,
                                                     wl["T"], True, True))
    run_once()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        run_once()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        events = json.load(open(path))["traceEvents"]
    out = {}
    for e in events:
        if e.get("cat") == "kernel" and any(t in e["name"] for t in TILED):
            out[e["name"]] = e["args"]["shared memory"]
    print(json.dumps(out))


def occupancy(lib_path):
    """For each tiled kernel the flagship step launches with this build: its dynamic shared memory (the launch's
    shared memory from the trace minus the kernel's static shared memory) and the CTAs per SM that
    cuOccupancyMaxActiveBlocksPerMultiprocessor gives for it, on the library's own sm_100a cubins."""
    launched = run(["benchmarks/tiled_prefetch_ab.py", "--probe"], lib_path)
    cu = ctypes.CDLL("libcuda.so.1")
    assert cu.cuInit(0) == 0
    ctx = ctypes.c_void_p()
    assert cu.cuDevicePrimaryCtxRetain(ctypes.byref(ctx), 0) == 0
    assert cu.cuCtxSetCurrent(ctx) == 0
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        subprocess.run(["cuobjdump", "-xelf", "all", os.path.abspath(lib_path)], cwd=tmp, check=True,
                       stdout=subprocess.DEVNULL)
        for cubin in sorted(glob.glob(os.path.join(tmp, "*.cubin"))):
            mod = ctypes.c_void_p()
            if cu.cuModuleLoad(ctypes.byref(mod), cubin.encode()) != 0:
                continue
            count = ctypes.c_uint()
            assert cu.cuModuleGetFunctionCount(ctypes.byref(count), mod) == 0
            fns = (ctypes.c_void_p * count.value)()
            assert cu.cuModuleEnumerateFunctions(fns, count, mod) == 0
            for fn in fns:
                name = ctypes.c_char_p()
                assert cu.cuFuncGetName(ctypes.byref(name), ctypes.c_void_p(fn)) == 0
                if not any(t in name.value.decode() for t in TILED):
                    continue
                pretty = subprocess.run(["c++filt", name.value.decode()], capture_output=True, text=True).stdout.strip()
                if pretty not in launched:
                    continue
                static = ctypes.c_int()
                assert cu.cuFuncGetAttribute(ctypes.byref(static), 1, ctypes.c_void_p(fn)) == 0  # SHARED_SIZE_BYTES
                dyn = launched[pretty] - static.value
                assert dyn >= 0, (pretty, launched[pretty], static.value)
                n = ctypes.c_int()
                assert cu.cuOccupancyMaxActiveBlocksPerMultiprocessor(ctypes.byref(n), ctypes.c_void_p(fn), 128,
                                                                      ctypes.c_size_t(dyn)) == 0
                out[pretty.split("(")[0]] = {"dynamic_smem": dyn, "static_smem": static.value, "ctas_per_sm": n.value}
            cu.cuModuleUnload(mod)
    missing = set(k.split("(")[0] for k in launched) - set(out)
    assert not missing, "launched kernels not found in %s: %s" % (lib_path, missing)
    return out


def last_json(text):
    for line in reversed(text.strip().splitlines()):
        if line.startswith("{"):
            return json.loads(line)
    raise RuntimeError("no JSON line in:\n" + text[-2000:])


def run(cmd, lib_path, extra_env=None):
    env = dict(os.environ, SHACIRA_LIB=os.path.abspath(lib_path), **(extra_env or {}))
    r = subprocess.run([sys.executable] + cmd, cwd=ROOT, env=env, capture_output=True, text=True)
    if r.returncode:
        raise RuntimeError("%s failed (%d):\n%s" % (" ".join(cmd), r.returncode, (r.stdout + r.stderr)[-3000:]))
    return last_json(r.stdout)


def compare_outputs(libs, runs=4):
    """`bench.py --dump-outputs`, `runs` times for every build. Every run of every build is compared with the first
    build's first run: feats must be bit-identical; a gradient may differ by as much as the first build's own runs
    differ among themselves (the cross-tile float REDs are the only order-dependent step)."""
    import numpy as np
    names = list(libs)
    with tempfile.TemporaryDirectory() as tmp:
        dirs = []
        for r in range(runs):
            for name in (names if r % 2 == 0 else names[::-1]):
                d = os.path.join(tmp, "%s_%d" % (name, r))
                run(["bench.py", "--gpus", "1", "--steps", "20", "--warmup", "5", "--no-cpu-baseline", "--no-ref-gpu",
                     "--no-fit", "--no-nerf", "--dump-outputs", d], libs[name])
                dirs.append((name, r, d))
        ref = [d for name, r, d in dirs if name == names[0] and r == 0][0]
        out = {}
        for name, r, d in dirs:
            if d == ref:
                continue
            for f in sorted(os.listdir(ref)):
                a, b = np.load(os.path.join(ref, f)), np.load(os.path.join(d, f))
                one = out.setdefault(name, {}).setdefault(f[:-4], {"runs": 0, "bit_identical_runs": 0, "max_abs_diff": 0.0})
                one["runs"] += 1
                one["bit_identical_runs"] += a.tobytes() == b.tobytes()
                one["max_abs_diff"] = max(one["max_abs_diff"],
                                          float(np.max(np.abs(a.astype(np.float64) - b.astype(np.float64)))))
    return {"reference": names[0] + " run 0", "against_reference": out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", metavar="NAME=PATH")
    ap.add_argument("--probe", action="store_true", help=argparse.SUPPRESS)   # one process per build, see occupancy()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_tiled_prefetch_ab.json"))
    args = ap.parse_args()
    if args.probe:
        return probe()
    if not args.lib:
        ap.error("--lib NAME=PATH is required")
    libs = dict(s.split("=", 1) for s in args.lib)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    res = {"gpu": q, "occupancy": {k: occupancy(v) for k, v in libs.items()}, "rounds": []}
    print(json.dumps({"gpu": q, "occupancy": res["occupancy"]}), flush=True)
    for r in range(args.rounds):
        order = list(libs) if r % 2 == 0 else list(reversed(libs))
        for name in order:
            b = run(["bench.py", "--gpus", "1", "--steps", str(args.steps), "--warmup", "20", "--no-cpu-baseline",
                     "--no-ref-gpu"], libs[name])
            k = run(["benchmarks/kernel_times.py"], libs[name],
                    {"ONLY": "fwd_tiled,bwd_tiled_dec,bwd_tiled_dec_bounded,fwd_tiled_sorted_io,step_tiled"})
            dr = run(["benchmarks/dropin_times.py"], libs[name])
            one = {"round": r, "lib": name, "ms_per_step": b["ms_per_step"],
                   "kernels_ms": {kk: v.get("ms") for kk, v in b.get("kernels", {}).items()},
                   "kodak_fit": b.get("kodak_fit"), "nerf_dp_ms_per_step": (b.get("nerf_dp") or {}).get("ms_per_step"),
                   "e2e_fit_ms_per_step": (b.get("e2e_fit") or {}).get("ms_per_step"),
                   "kernel_times_us": k, "dropin_f2_us": {"fwd": dr["fwd_us"], "bwd": dr["bwd_us"]}}
            res["rounds"].append(one)
            print(json.dumps({x: one[x] for x in ("round", "lib", "ms_per_step", "kernels_ms", "kernel_times_us",
                                                  "dropin_f2_us", "nerf_dp_ms_per_step", "e2e_fit_ms_per_step")}),
                  flush=True)
    res["outputs"] = compare_outputs(libs)
    print(json.dumps({"outputs": res["outputs"]}), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
