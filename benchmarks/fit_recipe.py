"""The reference's image-fit recipe two ways, alternated in one run: the host-driven loop (fit_image.fit_native_recipe:
lambda / temperature fills on the host before every graph replay of ONE step) against image_fit.fit_image / fit_images
(the schedule advanced by the optimizer launch, graphs of `--chunk` steps), each at 1 and 3 fits in flight.

Per arm: device ms per step of the SGA and straight-through phases (host loop: wall time around synchronised replays,
as fit_native_recipe reports it; fit_image: CUDA events on each fit's stream, divided by the fits in flight), host CPU
seconds per step of the whole call (time.process_time, set-up and graph capture included), PSNR and bpp of every fit
(host loop: the final state; fit_image: the best state it restores). The GPU's name and power limit are read in the
same run. Prints one JSON object; --out also writes it to a file.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "benchmarks"))

import fit_image  # noqa: E402
from shacira_b200 import image_fit  # noqa: E402


def gpu_info():
    out = dict(name=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        out["nvidia_smi"] = q
    except Exception as e:   # the name above still identifies the card
        out["nvidia_smi_error"] = repr(e)[:200]
    return out


def host_loop(seeds, steps, dev):
    t0 = time.process_time()
    res = fit_image.fit_native_recipe(seeds, steps, dev)
    cpu = time.process_time() - t0
    return dict(arm="host_loop", in_flight=len(seeds), ms_per_step_sga=res[0]["ms_per_step_sga"],
                ms_per_step_ste=res[0]["ms_per_step_ste"], host_cpu_s_per_step=cpu / (steps * len(seeds)),
                psnr=[r["psnr"] for r in res], bpp=[r["bpp"] for r in res])


def device_loop(seeds, steps, dev, chunk):
    models = []
    for s in seeds:
        grid, mlp, coords, gt, fs = fit_image._native_setup(s, dev, device_noise=True, sga=True)
        fs.close()
        models.append((grid, mlp, coords, gt))
    recipe = image_fit.ImageRecipe(epochs=steps)
    t0 = time.process_time()
    res = image_fit.fit_images(models, recipe, in_flight=len(seeds), chunk=chunk,
                               noise_seeds=[10_000 + s for s in seeds])
    cpu = time.process_time() - t0
    per = lambda p: max(r["device_ms"][p] for r in res) / (res[0]["steps"][p] * len(seeds))
    return dict(arm="fit_image", in_flight=len(seeds), ms_per_step_eager=per("eager"), ms_per_step_sga=per("sga"),
                ms_per_step_ste=per("ste"), host_cpu_s_per_step=cpu / (steps * len(seeds)),
                psnr=[r["psnr"] for r in res], bpp=[r["size"]["empirical_entropy_bpp"] for r in res],
                file_bpp=[r["size"]["file_bpp"] for r in res], best_step=[r["best_step"] for r in res])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--chunk", type=int, default=100)
    ap.add_argument("--rounds", type=int, default=2, help="alternations of the two arms")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    runs = []
    for r in range(args.rounds):
        for k in (1, 3):
            seeds = list(range(k))
            arms = (host_loop, device_loop) if r % 2 == 0 else (device_loop, host_loop)
            for arm in arms:
                res = arm(seeds, args.steps, dev) if arm is host_loop else arm(seeds, args.steps, dev, args.chunk)
                res["round"] = r
                runs.append(res)
                print(json.dumps(res), flush=True)
    out = dict(workload="Kodak-shape image fit, reference recipe (SGA -> STE at 90 %%), %d steps" % args.steps,
               gpu=gpu_info(), chunk=args.chunk, runs=runs)
    print(json.dumps(out), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
