"""The 3D (NeRF-shape) path on a B200: lane-pair kernels (two lanes per sample, grid3d_kernels.cuh), tile-sorted
plans with the coarse levels accumulated per tile, against the C oracle (oracle/hashgrid_oracle.c restates
hashgrid_interpolate_cuda.cu:47-109,143-271) and the round-1 point-parallel kernels.
Tolerances: forward 1e-5 (and bit-identical to the point-parallel kernel), gradients 1e-4 -- per LEVEL."""
import numpy as np
import pytest
import torch

import oracle
from helpers import level_rel_err, level_rms_err, make_case, rel_err
from test_tiled_gpu import _case, _check_decoder_grads, _dev, _oracle_fwd_bwd

pytestmark = pytest.mark.gpu
FWD_TOL, BWD_TOL = 1e-5, 1e-4

CASES = [
    # L, bw, rmin, rmax, n, C, F, per_level, kind
    (16, 19, 16, 2048, 1 << 17, 1, 4, False, "uniform"),     # BASELINE cfg4 grid
    (24, 19, 16, 512, 70000, 1, 4, False, "arbitrary"),      # the reference's nerf_lego.yaml grid (24 levels)
    (8, 14, 8, 128, 30000, 2, 2, True, "arbitrary"),         # per-level decoders, two latent channels
    (5, 12, 4, 40, 1003, 1, 1, False, "uniform"),            # ragged: L % 4 != 0, n % 16 != 0
    (16, 19, 16, 2048, 70001, 2, 8, False, "clustered"),     # every sample in one tile: the tile's batch loop
    (3, 10, 4, 600, 5000, 1, 2, False, "uniform"),           # hashed level with res >= 257
]


def _sizes(c):
    return oracle.level_layout(c["res"], c["bw"], 3)[0]


@pytest.mark.parametrize("L,bw,rmin,rmax,n,C,F,per_level,kind", CASES)
def test_lane_pair_forward_backward(lib, L, bw, rmin, rmax, n, C, F, per_level, kind):
    c = _case(3, L, bw, rmin, rmax, n, C, F, seed=31 + L + C + F, per_level=per_level, kind=kind)
    coords, lat, A, S, g = _dev(c["coords"]), _dev(c["lat"]), _dev(c["A"]), _dev(c["S"]), _dev(c["g"])
    want_f, want_gl, want_gA, want_gS = _oracle_fwd_bwd(c)
    sizes = _sizes(c)
    # round-1 point-parallel kernels: the in-library yardstick for bit-identity. The library routes a table that is
    # not 16-byte aligned there; 8 bytes off keeps the C = 2 rows aligned for that kernel's float2 loads.
    buf = torch.empty(lat.numel() + 2, device=lat.device)
    lat_u = buf[2:].view_as(lat).copy_(lat)
    f_pp, z_pp = lib.latent_forward(coords, lat_u, c["first"], c["res"], bw, A, S, F, True, True)
    # unplanned lane-pair kernels
    f, z = lib.latent_forward(coords, lat, c["first"], c["res"], bw, A, S, F, True, True)
    assert torch.equal(f, f_pp) and torch.equal(z, z_pp)
    assert rel_err(f.cpu().numpy(), want_f) <= FWD_TOL
    gl, gA, gS = lib.latent_backward(coords, g, z, c["first"], c["res"], bw, A, C, F, c["T"], True)
    assert level_rel_err(gl.cpu().numpy(), want_gl, c["first"], sizes) <= BWD_TOL
    _check_decoder_grads(c, gA, gS, want_gA, want_gS)
    # planned: tile-sorted samples, staged coarse levels
    plan = lib.Plan(coords)
    fp, zp = lib.latent_forward_planned_z(plan, lat, c["first"], c["res"], bw, A, S, F, True, True)
    assert torch.equal(fp, f_pp)
    assert torch.equal(zp, z_pp[plan.perm_tensor()])
    glp, gAp, gSp = lib.latent_backward_planned_z(plan, g, zp, c["first"], c["res"], bw, A, C, F, c["T"], True)
    assert level_rel_err(glp.cpu().numpy(), want_gl, c["first"], sizes) <= BWD_TOL
    assert level_rms_err(glp.cpu().numpy(), want_gl, c["first"], sizes) <= BWD_TOL
    _check_decoder_grads(c, gAp, gSp, want_gA, want_gS)
    glq, _, _ = lib.latent_backward_planned_z(plan, g, None, c["first"], c["res"], bw, A, C, F, c["T"], False)
    assert level_rel_err(glq.cpu().numpy(), want_gl, c["first"], sizes) <= BWD_TOL
    plan.close()


def test_full_size_nerf_batch_backward_per_level(lib):
    """BASELINE cfg4 at full size: 2^19 samples, 16 levels 16 -> 2048, 2^19-row tables, C = 1 -> F = 4; every level's
    gradient against the oracle."""
    c = _case(3, 16, 19, 16, 2048, 1 << 19, 1, 4, seed=5, kind="uniform")
    coords, lat, A, S, g = _dev(c["coords"]), _dev(c["lat"]), _dev(c["A"]), _dev(c["S"]), _dev(c["g"])
    want_f, want_gl, want_gA, want_gS = _oracle_fwd_bwd(c)
    sizes = _sizes(c)
    plan = lib.Plan(coords)
    assert plan.info()["tiles_per_axis"] == 16
    f, z = lib.latent_forward_planned_z(plan, lat, c["first"], c["res"], 19, A, S, 4, True, True)
    assert rel_err(f.cpu().numpy(), want_f) <= FWD_TOL
    gl, gA, gS = lib.latent_backward_planned_z(plan, g, z, c["first"], c["res"], 19, A, 1, 4, c["T"], True)
    assert level_rel_err(gl.cpu().numpy(), want_gl, c["first"], sizes) <= BWD_TOL
    assert level_rms_err(gl.cpu().numpy(), want_gl, c["first"], sizes) <= 1e-5
    _check_decoder_grads(c, gA, gS, want_gA, want_gS)
    plan.close()


@pytest.mark.parametrize("F", [1, 2])
def test_plain_table_3d_takes_the_lane_pair_kernels_bit_exactly(lib, F):
    """wisp._C.ops.hashgrid_interpolate_cuda on a plain table: identity decoder inside the lane-pair kernels."""
    c = make_case(3, 16, 19, 16, 2048, 50000, F, seed=77 + F, coord_kind="arbitrary")
    want = oracle.forward(c["coords"], c["table"], c["first_idx"], c["resolutions"], 19)
    before = lib.launch_count()
    got = lib.hashgrid_forward(_dev(c["coords"]), _dev(c["table"]), c["first_idx"], c["resolutions"], 19)
    assert lib.launch_count() - before == 1
    assert np.array_equal(got.cpu().numpy().view(np.uint32), want.view(np.uint32))
    want_g = oracle.backward(c["coords"], c["grad_out"], c["T"], c["first_idx"], c["resolutions"], 19, F)
    got_g = lib.hashgrid_backward(_dev(c["coords"]), _dev(c["grad_out"]), c["first_idx"], c["resolutions"], 19, F, c["T"])
    assert level_rel_err(got_g.cpu().numpy(), want_g, c["first_idx"], c["sizes"]) <= BWD_TOL


def test_latent_grid_3d_autograd_uses_the_sorted_path(lib, monkeypatch):
    """LatentGrid.interpolate on a NeRF-size batch: plan re-binned per coordinate set, z saved in sorted order,
    gradients equal to the unplanned path; a second backward under retain_graph still sees its own plan."""
    from shacira_b200 import grid_ops
    c = _case(3, 16, 19, 16, 2048, 1 << 17, 1, 4, seed=9, kind="uniform")
    lat = _dev(c["lat"]).requires_grad_(True)
    A = _dev(c["A"]).requires_grad_(True)
    S = _dev(c["S"]).requires_grad_(True)
    coords, g = _dev(c["coords"]), _dev(c["g"])
    grid_ops.clear_plans()
    monkeypatch.setattr(grid_ops, "PLAN_MIN_POINTS_3D", 1)   # the mechanism, not the crossover, is under test
    builds = grid_ops.plan_stats["builds"]
    feats = grid_ops.latent_hashgrid(coords, lat, A, S, c["first"], c["res"], 19, True)
    assert grid_ops.plan_stats["builds"] == builds + 1
    feats.backward(g, retain_graph=True)
    g1 = lat.grad.clone()
    # other coordinate sets come and go while the graph is alive: its plan must not be re-binned under it
    for k in range(12):
        other = torch.rand((1 << 17, 3), device="cuda") * 2 - 1
        grid_ops.latent_hashgrid(other, lat.detach(), A.detach(), S.detach(), c["first"], c["res"], 19, True)
    lat.grad = None
    feats.backward(g)
    assert torch.allclose(lat.grad, g1, rtol=0, atol=1e-4 * float(g1.abs().max()))
    monkeypatch.setenv("SHACIRA_DISABLE_PLAN_3D", "1")
    lat2 = _dev(c["lat"]).requires_grad_(True)
    f2 = grid_ops.latent_hashgrid(coords, lat2, A.detach(), S.detach(), c["first"], c["res"], 19, True)
    assert torch.equal(f2, feats.detach())
    f2.backward(g)
    sizes = _sizes(c)
    assert level_rel_err(g1.cpu().numpy(), lat2.grad.cpu().numpy(), c["first"], sizes) <= BWD_TOL
    grid_ops.clear_plans()


def test_non_finite_gradient_reaches_the_table_3d(lib):
    """An Inf / NaN upstream gradient must poison the rows it touches (the reference's float atomics would)."""
    c = _case(3, 16, 19, 16, 2048, 70000, 1, 4, seed=3, kind="uniform")
    coords, lat, A, S = _dev(c["coords"]), _dev(c["lat"]), _dev(c["A"]), _dev(c["S"])
    for bad in (float("inf"), float("nan")):
        g = _dev(c["g"]).clone()
        g[123, :] = bad
        plan = lib.Plan(coords)
        gl, _, _ = lib.latent_backward_planned_z(plan, g, None, c["first"], c["res"], 19, A, 1, 4, c["T"], False)
        sizes = _sizes(c)
        for l, (f0, s0) in enumerate(zip(c["first"], sizes)):
            assert not torch.isfinite(gl[f0:f0 + s0]).all(), "level %d lost a non-finite gradient" % l
        plan.close()
