"""Evaluation side of the native image fit: the forward-only render kernel (shacira_fit_render via
image_fit.render_image / ImageFitStep.render) and the best-state snapshot inside the optimizer launch
(ImageFitStep(track_best=True)), on the Kodak shape (BASELINE cfg2).

The fused fit kernel adds its per-node gradients and its SSE with float atomics, so two runs of the same fit agree to
rounding, not bit for bit. The snapshot is therefore checked against a host oracle that watches the SAME run (reads
rgb_loss() after every step and clones the parameters before it), and "training is unchanged" compares the optimizer
launch with and without the snapshot from one identical state."""
import math
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "benchmarks"))

DEV = torch.device("cuda", 0)


def _fit(seed=3, sga=False, device_noise=False, track_best=True):
    import fit_image
    grid, mlp, coords, gt, fs = fit_image._native_setup(seed, DEV, device_noise=device_noise, sga=sga)
    if track_best:
        fs.close()
        from shacira_b200.image_fit import ImageFitStep
        fs = ImageFitStep(grid, mlp, coords, gt, lr=1e-3, grid_lr=2e-2, ldec_lr=1e-2, prob_lr=1e-4, weight_decay=0.0,
                          weight_decay_decoder=1e-2, device_noise=device_noise, noise_seed=10_000 + seed,
                          track_best=True)
    return grid, mlp, coords, gt, fs


def _hooks(fs, it, steps, gen=None):
    fs.set_lambda(1e-4 + 0.5 * (1e-3 - 1e-4) * (1 + math.cos(math.pi * it / steps)))
    if gen is not None:
        fs.draw_noise(gen)
    if it + 1 in (1, 2, 5, 10):
        fs.update_div()


def _state(fs):
    """Every parameter the snapshot covers, cloned: table, segment params (segment order), div, A."""
    return ([fs.grid.codebook.data.clone()] + [p.clone() for p in fs._seg_params] +
            [fs.grid.latent_dec.div.data.clone(), fs.A.clone()])


def _ref_rgb(grid, mlp, coords, dtype=torch.float32):
    with torch.no_grad():
        feats = grid.interpolate(coords, 0)
        if dtype == torch.float64:
            import copy
            return copy.deepcopy(mlp).double()(feats.double())
        return mlp(feats)


def _short_fit(steps=20, seed=3):
    grid, mlp, coords, gt, fs = _fit(seed=seed)
    gen = torch.Generator().manual_seed(7)
    for it in range(steps):
        _hooks(fs, it, steps, gen)
        fs.step()
    torch.cuda.synchronize()
    return grid, mlp, coords, gt, fs


@pytest.fixture(scope="module")
def fitted(lib):
    out = _short_fit()
    yield out
    out[4].close()


def _coord_sets(coords):
    h, w = 2 * 512, 2 * 768
    ys, xs = torch.meshgrid(torch.arange(h), torch.arange(w), indexing="ij")
    up = torch.stack([(ys.reshape(-1) + 0.5) / h * 2 - 1, (xs.reshape(-1) + 0.5) / w * 2 - 1], 1).float()
    g = torch.Generator().manual_seed(11)
    rnd = torch.rand(300_001, 2, generator=g) * 2 - 1                 # N not a multiple of 64, uneven tiles
    quad = -torch.rand(200_003, 2, generator=g)                        # one quadrant: three quarters of the tiles empty
    return {"kodak": coords, "upsampled_2x": up.to(DEV), "random": rnd.to(DEV), "empty_tiles": quad.to(DEV)}


@pytest.mark.parametrize("which", ["kodak", "upsampled_2x", "random", "empty_tiles"])
def test_render_matches_interpolate_and_mlp(fitted, which):
    from shacira_b200.image_fit import render_image
    grid, mlp, coords, gt, fs = fitted
    c = _coord_sets(coords)[which]
    rgb, psnr = render_image(grid, mlp, c)
    assert psnr is None and rgb.shape == (c.shape[0], 3)
    want32 = _ref_rgb(grid, mlp, c)
    want64 = _ref_rgb(grid, mlp, c, torch.float64)
    assert float((rgb.double() - want64).abs().max()) <= 1e-5
    assert float((rgb - want32).abs().max()) <= 1e-5
    if which == "kodak":   # the step's own sorted-I/O plan, rows back in the caller's order
        rgb_fs, _ = fs.render(target=False)
        assert float((rgb_fs - want32).abs().max()) <= 1e-5


def test_psnr_is_the_exact_uint8_sse(fitted):
    import fit_image
    from shacira_b200 import _lib, grid_ops
    from shacira_b200.image_fit import _render, render_image
    grid, mlp, coords, gt, fs = fitted
    rgb, psnr = fs.render(target=True)
    q = lambda v: (torch.clamp(v, 0, 1) * 255).to(torch.uint8).long()   # fit_image.clamped_psnr's quantisation
    sse = int(((q(rgb) - q(gt)) ** 2).sum())
    assert int(fs.sse_u8) == sse
    want = fit_image.clamped_psnr(_ref_rgb(grid, mlp, coords), gt)
    assert abs(float(psnr) - want) <= 1e-3
    rgb2, psnr2 = render_image(grid, mlp, coords, target=gt)          # original-order plan, same numbers
    assert abs(float(psnr2) - float(psnr)) <= 1e-9 and float((rgb2 - rgb).abs().max()) <= 1e-5
    # rgb = NULL: PSNR without writing the image
    sse_only = torch.zeros((), dtype=torch.int64, device=DEV)
    plan = grid_ops.plan_for(coords)
    A, shift = grid.latent_dec.affine_map()
    _render(plan, grid.codebook.data, _lib._i32_array(grid._first_idx())[0], _lib._i32_array(grid.resolutions)[0], 16,
            int(grid.codebook_bitwidth), A.detach().contiguous(), shift.detach(), fs.lin, None, gt, sse_only)
    assert int(sse_only) == sse


def _oracle_run(fs, steps, switch=None, sga_gen=None, gen=None, graph=False, poison_after=None):
    """Steps of `fs` with the host oracle: parameters cloned before each step, rgb_loss() read after it."""
    T = fs.T
    losses, states = [], []
    g = None
    for it in range(steps):
        _hooks(fs, it, steps, gen)
        if switch is not None:
            on = it < switch
            if on != fs.sga:
                fs.set_sga(on)
                g = None
            fs.set_temperature(max(0.1, math.exp(-math.log(10.0) * (it + 1) / steps / 0.9)), refresh=sga_gen is not None)
            if sga_gen is not None:
                fs.sga_uniforms = torch.rand((T, 1, 2), generator=sga_gen).to(DEV) if on else None
        if poison_after is not None and it == poison_after:
            fs.target[0, 0] = float("nan")
        states.append(_state(fs))
        if graph:
            if g is None:
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                side = torch.cuda.Stream(device=DEV)
                side.wait_stream(torch.cuda.current_stream())
                # capture records the step; the first replay runs it
                with torch.cuda.graph(g, stream=side):
                    fs.step()
            g.replay()
        else:
            fs.step()
        losses.append(float(fs.rgb_loss()))
    return np.array(losses, dtype=np.float32), states


def _check_against_oracle(fs, losses, states):
    """`losses` / `states` cover every step of the fit (best_step counts from its first step)."""
    finite = np.where(np.isnan(losses), np.inf, losses)
    k = int(np.argmin(finite))                     # first argmin
    assert float(fs.best_loss()) == float(losses[k]) and fs.best_loss().dtype == torch.float32
    assert int(fs.best_step()) == k
    fs.restore_best()
    for got, want in zip(_state(fs), states[k]):
        assert torch.equal(got, want)
    return k


def test_snapshot_matches_host_oracle_across_sga_switch(lib):
    grid, mlp, coords, gt, fs = _fit(seed=5, sga=True)
    steps, switch = 60, 40
    losses, states = _oracle_run(fs, steps, switch=switch, sga_gen=torch.Generator().manual_seed(21),
                                 gen=torch.Generator().manual_seed(22))
    k = _check_against_oracle(fs, losses, states)
    assert 0 <= k < steps
    fs.close()


def test_snapshot_keeps_an_earlier_state(lib):
    """Later steps against a different target are worse: restore_best goes back to an earlier state."""
    grid, mlp, coords, gt, fs = _fit(seed=6)
    losses, states = _oracle_run(fs, 15, gen=torch.Generator().manual_seed(23))
    fs.target.copy_(torch.rand_like(fs.target))
    more, more_states = _oracle_run(fs, 5, gen=torch.Generator().manual_seed(24))
    k = _check_against_oracle(fs, np.concatenate([losses, more]), states + more_states)
    assert k < 15
    fs.close()


def test_snapshot_under_graph_replay(lib):
    """In-kernel draws (bit-rate noise, SGA sample) under CUDA-graph replay, SGA -> STE: the snapshot of the replayed
    launches equals the host oracle's view of the same run."""
    grid, mlp, coords, gt, fs = _fit(seed=7, sga=True, device_noise=True)
    warm, warm_states = _oracle_run(fs, 3)         # eager warm-up (plan, node table, allocator), watched too
    losses, states = _oracle_run(fs, 40, switch=30, graph=True)
    _check_against_oracle(fs, np.concatenate([warm, losses]), warm_states + states)
    fs.close()


def test_snapshot_does_not_change_training(lib, monkeypatch):
    """The optimizer launch with and without the snapshot, from one identical state: every parameter, Adam moment,
    counter and the next SGA sample come out bit for bit the same. The bit-rate loss runs in its own kernel here: folded
    into the launch, its per-CTA partial sums are added with shared-memory atomics (order dependent in the last bits),
    so the launch itself would not repeat bit for bit."""
    monkeypatch.setenv("SHACIRA_FIT_ENT_FUSED", "0")
    grid, mlp, coords, gt, fs = _fit(seed=8, sga=True, device_noise=True)
    assert not fs.ent_in_opt
    for it in range(6):
        _hooks(fs, it, 6)
        fs.step()
    fs.best_loss_t.fill_(float("inf"))               # so that the launch below takes its snapshot
    torch.cuda.synchronize()
    tensors = [t for t in vars(fs).values() if isinstance(t, torch.Tensor)] + list(fs._keep) + list(fs._seg_params) + \
        [grid.codebook.data, grid.latent_dec.div.data]
    saved = [t.clone() for t in tensors]
    prefetch = fs.sga and fs.opt_fused and fs.sga_uniforms is None
    from shacira_b200 import _lib
    with torch.cuda.device(DEV):
        fs._optimize(prefetch, fs.dw if fs.sga else None, fs.ent_in_opt, _lib._stream())
    torch.cuda.synchronize()
    with_snap = [t.clone() for t in tensors]
    assert int(fs.best_step_t) == 6                  # the snapshot was taken by this launch
    for t, s in zip(tensors, saved):
        t.copy_(s)
    fs.track_best = False
    with torch.cuda.device(DEV):
        fs._optimize(prefetch, fs.dw if fs.sga else None, fs.ent_in_opt, _lib._stream())
    torch.cuda.synchronize()
    skip = {id(fs.best_loss_t), id(fs.best_step_t), id(fs.best_table), id(fs.best_div), id(fs.best_A)}
    # bit for bit means equal bytes: buffers this path never writes (feats, gfeat: torch.empty) can hold NaN garbage,
    # which torch.equal calls unequal to itself
    as_bytes = lambda x: x.contiguous().view(-1).view(torch.uint8)
    for t, w in zip(tensors, with_snap):
        if id(t) not in skip:
            assert torch.equal(as_bytes(t), as_bytes(w))
    fs.close()


def test_nan_step_is_never_selected(lib):
    grid, mlp, coords, gt, fs = _fit(seed=9)
    losses, states = _oracle_run(fs, 14, gen=torch.Generator().manual_seed(25), poison_after=9)
    assert np.isnan(losses[9:]).all()
    k = _check_against_oracle(fs, losses, states)
    assert k < 9
    assert all(bool(torch.isfinite(t).all()) for t in _state(fs))
    fs.close()


def test_render_of_the_best_state_reproduces_its_loss(lib):
    grid, mlp, coords, gt, fs = _fit(seed=10)
    losses, states = _oracle_run(fs, 30, gen=torch.Generator().manual_seed(26))
    fs.restore_best()
    rgb, _ = fs.render(target=False)
    mse = float(((rgb.double() - gt.double()) ** 2).mean())
    assert abs(mse - float(fs.best_loss())) <= 1e-6 * float(fs.best_loss())
    fs.close()


def test_codec_round_trip_renders_bit_for_bit(fitted):
    import fit_image
    from shacira_b200 import codec
    from shacira_b200.grids import LatentGrid
    from shacira_b200.image_fit import render_image
    grid, mlp, coords, gt, fs = fitted
    blob = codec.encode_model(grid, mlp)
    grid2 = LatentGrid.from_geometric(feature_dim=1, num_lods=16, latent_dim=1, multiscale_type="cat", resolution_dim=2,
                                      feature_std=0.1, codebook_bitwidth=16, min_grid_res=16, max_grid_res=512,
                                      init_grid="uniform", conf_latent_decoder=dict(fit_image.DEC),
                                      conf_entropy_reg=dict(fit_image.ENT)).to(DEV)
    mlp2 = torch.nn.Sequential(torch.nn.Linear(16, 16), torch.nn.ReLU(), torch.nn.Linear(16, 16), torch.nn.ReLU(),
                               torch.nn.Linear(16, 3)).to(DEV)
    codec.load_into(codec.decode_model(blob), grid2, mlp2)
    a, pa = render_image(grid, mlp, coords, target=gt)
    b, pb = render_image(grid2, mlp2, coords, target=gt)
    assert torch.equal(a, b) and float(pa) == float(pb)


def test_track_best_needs_the_one_launch_optimizer(lib, monkeypatch):
    import fit_image
    from shacira_b200 import _lib
    from shacira_b200.image_fit import ImageFitStep
    grid, mlp, coords, gt, fs = fit_image._native_setup(2, DEV)
    with pytest.raises(_lib.ShaciraError, match="best_loss|track_best"):
        fs.best_loss()
    fs.close()
    monkeypatch.setenv("SHACIRA_FIT_OPT_FUSED", "0")
    with pytest.raises(_lib.ShaciraError, match="track_best"):
        ImageFitStep(grid, mlp, coords, gt, track_best=True)
