"""Argument validation of the render kernel's and the best-state optimizer launch's entry points (shacira_fit_render,
shacira_fit_optimizer_step_best) and of render_image's shape check. CPU only: validation runs before any CUDA call."""
import ctypes

import pytest
import torch


def _levels(vals):
    return (ctypes.c_int32 * len(vals))(*vals)


FAKE = ctypes.c_void_p(256)   # never dereferenced: every case fails validation first


def _render(L, plan=None, num_lods=16, res=None, rgb=FAKE, target=None, sse=None, W1=FAKE):
    res = res or [16 * (k + 1) for k in range(num_lods)]
    first = [0] * len(res)
    return L.shacira_fit_render(plan, FAKE, _levels(first), _levels(res), num_lods, 14, FAKE, None, W1, FAKE, FAKE,
                                FAKE, FAKE, FAKE, rgb, target, sse, None)


def test_fit_render_validates_before_any_cuda_call(lib):
    L = lib.load()
    assert _render(L, num_lods=8) == lib.ERR_UNSUPPORTED
    assert b"16 levels" in L.shacira_last_error()
    assert _render(L, W1=None) == lib.ERR_INVALID_ARGUMENT
    assert _render(L, rgb=None) == lib.ERR_INVALID_ARGUMENT
    assert b"nothing to compute" in L.shacira_last_error()
    assert _render(L, target=FAKE, sse=None) == lib.ERR_INVALID_ARGUMENT
    assert b"sse_u8" in L.shacira_last_error()
    assert _render(L) == lib.ERR_INVALID_ARGUMENT
    assert b"plan is NULL" in L.shacira_last_error()
    assert _render(L, res=[16] * 15 + [1 << 20]) == lib.ERR_INVALID_ARGUMENT   # a level past the 2D coordinate range


def _opt_best(lib, snap, A_out=FAKE):
    L = lib.load()
    f = ctypes.c_float
    seg = lib.AdamSeg()   # the `scale` segment (param == scale) that A_out needs
    seg.param = seg.grad = seg.exp_avg = seg.exp_avg_sq = FAKE.value
    seg.n, seg.grad_rows, seg.div_group = 1, 1, 1
    return L.shacira_fit_optimizer_step_best(
        ctypes.byref(seg), 1, FAKE, FAKE, None, None, None, f(1.0), FAKE, FAKE, 1024, f(1e-2), f(0.0), f(0.9), f(0.999), f(1e-8),
        FAKE, FAKE, FAKE, FAKE, A_out, 1, 1, None, 0, 0, None, None, None, None, 0, None, 0, None, None, None, None, 0,
        FAKE, snap, None)


def test_fit_optimizer_step_best_validates_the_descriptor(lib):
    L = lib.load()
    assert _opt_best(lib, None) == lib.ERR_INVALID_ARGUMENT
    assert b"descriptor is NULL" in L.shacira_last_error()
    snap = lib.FitSnapshot()
    assert _opt_best(lib, ctypes.byref(snap)) == lib.ERR_INVALID_ARGUMENT
    assert b"sse / count" in L.shacira_last_error()
    snap.sse, snap.count, snap.best_loss, snap.best_step, snap.table = 256, 3 * 4096, 256, 256, 256
    assert _opt_best(lib, ctypes.byref(snap)) == lib.ERR_INVALID_ARGUMENT   # div / A of the snapshot missing
    assert b"div and A" in L.shacira_last_error()
    snap.div, snap.A = 256, 256
    assert _opt_best(lib, ctypes.byref(snap), A_out=None) == lib.ERR_INVALID_ARGUMENT
    snap.count = 0
    assert _opt_best(lib, ctypes.byref(snap)) == lib.ERR_INVALID_ARGUMENT


def test_snapshot_struct_matches_the_header(lib):
    # 4 pointers + int64 + MAX_ADAM_SEGS pointers + 2 pointers on LP64
    assert ctypes.sizeof(lib.FitSnapshot) == 8 * (5 + lib.MAX_ADAM_SEGS + 2)


def _grid(num_lods=16, latent_dim=1):
    from shacira_b200.grids import LatentGrid
    dec = dict(ldecode_enabled=True, ldecode_type="single", use_sga=False, diff_sampling=True, use_shift=True,
               ldecode_matrix="sq", latent_dim=latent_dim, norm="max", norm_every=10, ldec_std=0.1, decay_period=0.9,
               temperature=0.1)
    ent = dict(num_prob_layers=2, entropy_reg=1e-3, entropy_reg_end=1e-4, entropy_reg_sched="cosine", noise_freq=1)
    return LatentGrid.from_geometric(feature_dim=1, num_lods=num_lods, latent_dim=latent_dim, multiscale_type="cat",
                                     resolution_dim=2, feature_std=0.1, codebook_bitwidth=12, min_grid_res=16,
                                     max_grid_res=256, init_grid="uniform", conf_latent_decoder=dec,
                                     conf_entropy_reg=ent)


def _mlp(inp=16, out=3):
    nn = torch.nn
    return nn.Sequential(nn.Linear(inp, 16), nn.ReLU(), nn.Linear(16, 16), nn.ReLU(), nn.Linear(16, out))


@pytest.mark.parametrize("case", ["levels", "latent_dim", "mlp_out"])
def test_render_image_rejects_other_model_shapes(lib, case):
    from shacira_b200.image_fit import render_image
    grid = _grid(num_lods=8) if case == "levels" else _grid(latent_dim=2) if case == "latent_dim" else _grid()
    mlp = _mlp(inp=8) if case == "levels" else _mlp(out=4) if case == "mlp_out" else _mlp()
    with pytest.raises(lib.ShaciraError, match="render_image"):
        render_image(grid, mlp, torch.zeros(4, 2))
