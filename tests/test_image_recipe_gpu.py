"""The image-fit recipe on the device: the scheduled optimizer launch (ImageFitStep.set_schedule / history,
shacira_fit_optimizer_step_sched) and fit_image / fit_images, on the Kodak shape (BASELINE cfg2 / cfg3).

The fit kernel adds with float atomics, so two runs of one fit agree to rounding only. Bit-identity is therefore
checked launch against launch from one cloned state, and whole fits against the spread of repeated runs or the
project's parity gates (PSNR +-0.05 dB, bpp +-1 %)."""
import dataclasses
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "benchmarks"))

DEV = torch.device("cuda", 0)
PSNR_GATE, BPP_GATE = 0.05, 0.01


def _setup(seed, sga=True, device_noise=True, track_best=False):
    import fit_image
    from shacira_b200.image_fit import ImageFitStep, ImageRecipe
    grid, mlp, coords, gt, fs = fit_image._native_setup(seed, DEV, device_noise=device_noise, sga=sga)
    if track_best:
        fs.close()
        fs = ImageFitStep(grid, mlp, coords, gt, noise_seed=10_000 + seed, track_best=True,
                          **dataclasses.replace(ImageRecipe(), device_noise=device_noise).step_kwargs())
    return grid, mlp, coords, gt, fs


def _kodak24(seed):
    """The reference's own Kodak configuration (kodak.yaml): 24 levels 16 -> 512, 2^11 table, MLP 24 -> 16 -> 16 -> 3;
    ImageFitStep runs it on the three-kernel path."""
    import fit_image
    from shacira_b200.grids import LatentGrid
    torch.manual_seed(seed)
    dec = dict(fit_image.DEC, use_sga=True)
    grid = LatentGrid.from_geometric(feature_dim=1, num_lods=24, latent_dim=1, multiscale_type="cat", resolution_dim=2,
                                     feature_std=0.1, codebook_bitwidth=11, min_grid_res=16, max_grid_res=512,
                                     init_grid="uniform", conf_latent_decoder=dec, conf_entropy_reg=dict(fit_image.ENT))
    nn = torch.nn
    mlp = nn.Sequential(nn.Linear(24, 16), nn.ReLU(), nn.Linear(16, 16), nn.ReLU(), nn.Linear(16, 3))
    with torch.no_grad():
        grid.codebook.mul_(fit_image.LATENT_SCALE)
    coords, gt = fit_image.make_data(seed, DEV)
    return grid.to(DEV), mlp.to(DEV), coords, gt


def _f32(x):
    return np.float32(x).view(np.int32)


def test_schedule_values_over_a_full_kodak_schedule(lib):
    """60 000 launches: every lambda / temperature the launch wrote equals lambda_at / temperature_at rounded to float32
    to <= 1 ulp (CUDA's double cos / exp may differ from the host's in the last double bit)."""
    from shacira_b200 import _lib
    from shacira_b200.image_fit import ImageRecipe, lambda_at, temperature_at
    grid, mlp, coords, gt, fs = _setup(1)
    recipe = ImageRecipe()
    fs.set_schedule(recipe)
    n, per_graph = recipe.epochs, 1000
    prefetch = fs.sga and fs.opt_fused and fs.sga_uniforms is None
    fs.step()                                                        # warm-up; draws the first SGA sample
    torch.cuda.synchronize()
    side = torch.cuda.Stream(device=DEV)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):                           # the optimizer launch alone, 1000 times
        for _ in range(per_graph):
            fs._optimize(prefetch, fs.dw, fs.ent_in_opt, _lib._stream())
    for _ in range((n - 1) // per_graph + 1):
        g.replay()
    torch.cuda.synchronize()
    h = fs.history()
    assert h["lam"].shape[0] == n
    lam = h["lam"].cpu().numpy().view(np.int32).astype(np.int64)
    tau = h["temperature"].cpu().numpy().view(np.int32).astype(np.int64)
    want_lam = np.array([_f32(lambda_at(it, n)) for it in range(n)], dtype=np.int64)
    want_tau = np.array([_f32(temperature_at(it, n)) for it in range(n)], dtype=np.int64)
    d_lam, d_tau = np.abs(lam - want_lam), np.abs(tau - want_tau)
    print("schedule values not bit-identical: lambda %d / %d, temperature %d / %d"
          % (int((d_lam != 0).sum()), n, int((d_tau != 0).sum()), n))
    assert int(d_lam.max()) <= 1 and int(d_tau.max()) <= 1
    # past the log's capacity the record is dropped and the schedule still advances
    assert int(fs.step_small) == n + 1
    assert abs(int(_f32(float(fs.lam))) - int(_f32(lambda_at(n + 1, n)))) <= 1
    fs.close()


@pytest.mark.parametrize("sga", [True, False])
def test_scheduled_launch_equals_the_host_set_launch(lib, monkeypatch, sga):
    """From one cloned state: the scheduled launch and shacira_fit_optimizer_step_best, with lambda and T set on the host
    to the values the log reports for that step, give bit-identical tables, moments, segments, w_hat / dw, counters and
    snapshot. The bit-rate loss runs in its own kernel (its folded form adds partials with shared-memory atomics)."""
    from shacira_b200 import _lib
    from shacira_b200.image_fit import ImageRecipe
    monkeypatch.setenv("SHACIRA_FIT_ENT_FUSED", "0")
    grid, mlp, coords, gt, fs = _setup(8, sga=sga, track_best=True)
    assert not fs.ent_in_opt
    fs.set_schedule(ImageRecipe(epochs=40, div_epochs=()))
    for _ in range(6):
        fs.step()
    fs.best_loss_t.fill_(float("inf"))                               # so that both launches take the snapshot
    torch.cuda.synchronize()
    tensors = [t for t in vars(fs).values() if isinstance(t, torch.Tensor)] + list(fs._keep) + list(fs._seg_params) + \
        list(fs.best_segs) + [grid.codebook.data, grid.latent_dec.div.data]
    saved = [t.clone() for t in tensors]
    prefetch = fs.sga and fs.opt_fused and fs.sga_uniforms is None
    gmul = fs.dw if fs.sga else None
    with torch.cuda.device(DEV):
        fs._optimize(prefetch, gmul, fs.ent_in_opt, _lib._stream())
    torch.cuda.synchronize()
    rec = fs.log[6].clone()
    assert float(rec[0]) == float(fs.rgb_loss()) and float(rec[1]) == float(fs.total_bits())
    with_sched = [t.clone() for t in tensors]
    assert int(fs.best_step_t) == 6 and int(fs.step_small) == 7
    for t, s in zip(tensors, saved):
        t.copy_(s)
    sched, fs.sched = fs.sched, None
    fs.set_lambda(float(rec[2]))
    fs.set_temperature(float(rec[3]))
    with torch.cuda.device(DEV):
        fs._optimize(prefetch, gmul, fs.ent_in_opt, _lib._stream())
    torch.cuda.synchronize()
    fs.sched = sched
    skip = {id(fs.lam), id(fs.temperature), id(fs.log)}               # the scheduled launch wrote the next values
    compared = 0
    for t, w in zip(tensors, with_sched):
        if id(t) not in skip:
            assert torch.equal(t, w)
            compared += 1
    assert compared > 30
    fs.close()


def test_history_is_rgb_loss_and_total_bits(lib):
    from shacira_b200.image_fit import ImageRecipe
    grid, mlp, coords, gt, fs = _setup(4, track_best=True)
    recipe = ImageRecipe(epochs=30, div_epochs=(1, 2, 5, 10))
    fs.set_schedule(recipe)
    losses, bits = [], []
    for it in range(30):
        if it + 1 in recipe.div_epochs:
            fs.update_div()
        fs.step()
        losses.append(fs.rgb_loss().item())
        bits.append(fs.total_bits().item())
    h = fs.history()
    assert h["rgb_loss"].shape[0] == 30
    assert np.array_equal(h["rgb_loss"].cpu().numpy(), np.array(losses, dtype=np.float32))
    assert np.array_equal(h["bits"].cpu().numpy(), np.array(bits, dtype=np.float32))
    fs.close()


def _host_hooked(seed, steps, epochs):
    from shacira_b200.image_fit import lambda_at, temperature_at
    grid, mlp, coords, gt, fs = _setup(seed)
    lam, tau, loss = [], [], []
    for it in range(steps):
        fs.set_lambda(lambda_at(it, epochs))
        fs.set_temperature(temperature_at(it, epochs))
        lam.append(float(fs.lam))
        tau.append(float(fs.temperature))
        fs.step()
        loss.append(fs.rgb_loss().item())
    fs.close()
    return np.array(lam, np.float32), np.array(tau, np.float32), np.array(loss, np.float64)


def test_graph_of_k_scheduled_steps_equals_host_hooked_steps(lib):
    from shacira_b200.image_fit import ImageRecipe
    seed, warm, k = 12, 3, 50
    recipe = ImageRecipe(epochs=warm + k, div_epochs=())
    grid, mlp, coords, gt, fs = _setup(seed)
    fs.set_schedule(recipe)
    for _ in range(warm):                                            # eager warm-up (plan, allocator)
        fs.step()
    torch.cuda.synchronize()
    side = torch.cuda.Stream(device=DEV)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        for _ in range(k):
            fs.step()
    g.replay()
    torch.cuda.synchronize()
    h = {key: v.cpu().numpy() for key, v in fs.history().items()}
    fs.close()
    lam1, tau1, loss1 = _host_hooked(seed, warm + k, recipe.epochs)
    lam2, tau2, loss2 = _host_hooked(seed, warm + k, recipe.epochs)
    assert np.array_equal(h["lam"].view(np.int32), lam1.view(np.int32))
    assert np.array_equal(h["temperature"].view(np.int32), tau1.view(np.int32))
    spread = float(np.abs(loss1 - loss2).max())
    diff = float(np.abs(h["rgb_loss"].astype(np.float64) - loss1).max())
    # a floor of a few float32 ulps of the loss, should the two host-hooked runs happen to agree exactly
    floor = 4 * float(np.spacing(np.float32(loss1.max())))
    print("graph vs host-hooked: max |d loss| %.3e, host-hooked spread %.3e" % (diff, spread))
    assert diff <= max(2 * spread, floor)


@pytest.fixture(scope="module")
def e2e(lib):
    """fit_image and fit_native_recipe (the host-driven loop) on one seed, 400 epochs."""
    import fit_image
    from shacira_b200.image_fit import ImageRecipe
    from shacira_b200.image_fit import fit_image as fit
    seed = 0
    recipe = ImageRecipe(epochs=400)
    grid, mlp, coords, gt, fs = _setup(seed)
    fs.close()
    res = fit(grid, mlp, coords, gt, recipe, chunk=64, noise_seed=10_000 + seed)
    host = fit_image.fit_native_recipe([seed], recipe.epochs, DEV)[0]
    return grid, mlp, coords, gt, res, host


def test_fit_image_matches_the_host_driven_recipe(e2e):
    grid, mlp, coords, gt, res, host = e2e
    print("fit_image: psnr %.4f bpp %.4f best_step %d | host loop: psnr %.4f bpp %.4f"
          % (res["psnr"], res["size"]["empirical_entropy_bpp"], res["best_step"], host["psnr"], host["bpp"]))
    assert abs(res["psnr"] - host["psnr"]) <= PSNR_GATE
    assert abs(res["size"]["empirical_entropy_bpp"] / host["bpp"] - 1) <= BPP_GATE
    assert res["steps"] == {"eager": 10, "sga": 350, "ste": 40}
    assert set(res["device_ms"]) == {"eager", "sga", "ste"} and all(v > 0 for v in res["device_ms"].values())
    assert res["size"]["file_bytes"] == len(res["blob"])


def test_fit_image_best_state(e2e):
    from shacira_b200 import codec
    from shacira_b200.grids import LatentGrid
    from shacira_b200.image_fit import render_image
    import fit_image
    grid, mlp, coords, gt, res, host = e2e
    loss = res["history"]["rgb_loss"].cpu().numpy()
    assert loss.shape[0] == 400
    assert res["best_step"] == int(np.argmin(np.where(np.isnan(loss), np.inf, loss)))
    assert res["best_loss"] == float(loss[res["best_step"]])
    _, psnr = render_image(grid, mlp, coords, target=gt)              # the modules hold the restored best state
    assert float(psnr) == res["psnr"]
    grid2 = LatentGrid.from_geometric(feature_dim=1, num_lods=16, latent_dim=1, multiscale_type="cat", resolution_dim=2,
                                      feature_std=0.1, codebook_bitwidth=16, min_grid_res=16, max_grid_res=512,
                                      init_grid="uniform", conf_latent_decoder=dict(fit_image.DEC),
                                      conf_entropy_reg=dict(fit_image.ENT)).to(DEV)
    mlp2 = torch.nn.Sequential(torch.nn.Linear(16, 16), torch.nn.ReLU(), torch.nn.Linear(16, 16), torch.nn.ReLU(),
                               torch.nn.Linear(16, 3)).to(DEV)
    codec.load_into(codec.decode_model(res["blob"]), grid2, mlp2)
    a, pa = render_image(grid, mlp, coords, target=gt)
    b, pb = render_image(grid2, mlp2, coords, target=gt)
    assert torch.equal(a, b) and float(pa) == float(pb)


def test_fit_images_in_flight_match_fits_alone(lib):
    """Three fits in flight, one of them the reference's 24-level configuration on the three-kernel path: each within
    the parity gates of the same fit run alone."""
    from shacira_b200.image_fit import ImageRecipe, fit_image, fit_images
    recipe = ImageRecipe(epochs=400)

    def models():
        out = []
        for seed in (20, 21):
            grid, mlp, coords, gt, fs = _setup(seed)
            fs.close()
            out.append((grid, mlp, coords, gt))
        out.append(_kodak24(22))
        return out

    together = fit_images(models(), recipe, in_flight=3, noise_seeds=[1, 2, 3])
    alone = [fit_image(*m, recipe, noise_seed=s) for m, s in zip(models(), [1, 2, 3])]
    for t, a in zip(together, alone):
        print("in flight: psnr %.4f bpp %.4f | alone: psnr %.4f bpp %.4f"
              % (t["psnr"], t["size"]["empirical_entropy_bpp"], a["psnr"], a["size"]["empirical_entropy_bpp"]))
        assert abs(t["psnr"] - a["psnr"]) <= PSNR_GATE
        assert abs(t["size"]["empirical_entropy_bpp"] / a["size"]["empirical_entropy_bpp"] - 1) <= BPP_GATE
        assert t["steps"] == a["steps"] == {"eager": 10, "sga": 350, "ste": 40}


def test_schedule_needs_the_one_launch_optimizer(lib, monkeypatch):
    from shacira_b200 import _lib
    from shacira_b200.image_fit import ImageFitStep, ImageRecipe
    grid, mlp, coords, gt, fs = _setup(2)
    with pytest.raises(_lib.ShaciraError, match="set_schedule"):
        fs.history()
    fs.close()
    monkeypatch.setenv("SHACIRA_FIT_OPT_FUSED", "0")
    fs = ImageFitStep(grid, mlp, coords, gt)
    with pytest.raises(_lib.ShaciraError, match="one-launch"):
        fs.set_schedule(ImageRecipe())
    fs.close()


def test_fit_image_without_div_epochs_or_ste_phase(lib):
    """No div epochs: one eager step still runs before the SGA graph is captured. decay_period = 1: the fit never
    switches to STE, and the result is still evaluated on the rounded model."""
    from shacira_b200.image_fit import ImageRecipe, _clamped_psnr, fit_image
    grid, mlp, coords, gt = _kodak24(23)
    res = fit_image(grid, mlp, coords, gt, ImageRecipe(epochs=60, div_epochs=(), decay_period=1.0), chunk=16)
    assert res["steps"] == {"eager": 1, "sga": 59}
    assert not grid.latent_dec.use_sga
    assert res["history"]["rgb_loss"].shape[0] == 60
    with torch.no_grad():
        psnr = float(_clamped_psnr(mlp(grid.interpolate(coords, 0)), gt))
    assert psnr == res["psnr"]
