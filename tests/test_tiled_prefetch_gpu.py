"""The 2D tiled kernels' asynchronous requests: the forward's permutation entries and coordinates one batch ahead, and
the backward's gradient pieces one level chunk ahead, both through thread-private shared-memory slots. Each case
covers a shape those pipelines treat differently: no next chunk (L = 4), five chunks (L = 20), other slot sizes
(F = 2, 4), several forward batches and register batches per tile, several kBatch spans per tile, per-level decoders,
the bounded entry, non-finite gradient rows, and a forward whose shared memory leaves no room for the slots."""
import numpy as np
import pytest
import torch

from helpers import rel_err
from test_tiled_gpu import BWD_TOL, _case, _check_decoder_grads, _dev, _oracle_fwd_bwd

pytestmark = pytest.mark.gpu

CASES = [
    # L, bw, rmin, rmax, n, C, F, per_level, tile_points, bounded
    (4, 14, 16, 128, 30000, 1, 1, False, 0, False),       # one level chunk: nothing requested ahead
    (20, 14, 16, 512, 60000, 1, 1, False, 0, False),      # five chunks
    (16, 14, 16, 512, 40000, 1, 2, False, 0, False),      # two points per thread, two 16-byte pieces per chunk
    (16, 14, 16, 512, 40000, 2, 2, True, 0, False),       # scatter-g with per-level decoders
    (16, 14, 16, 512, 200000, 1, 4, True, 0, False),      # one point per thread, four pieces per chunk
    (16, 14, 16, 512, 40000, 1, 4, True, 0, False),       # node boxes too large for the slots: the register loop
    (16, 14, 16, 512, 60000, 1, 1, False, 700, False),    # tiles above 384 points: several batches per tile
    (16, 14, 16, 512, 100000, 1, 1, False, 6000, False),  # tiles above 2048 points: several kBatch spans
    (16, 14, 16, 512, 60000, 1, 1, True, 700, True),      # bounded entry, per-level decoders
    (12, 14, 16, 256, 60000, 1, 2, False, 6000, True),    # bounded, several spans, F = 2
]


@pytest.mark.parametrize("L,bw,rmin,rmax,n,C,F,per_level,tile_points,bounded", CASES)
def test_prefetched_tiles_match(lib, L, bw, rmin, rmax, n, C, F, per_level, tile_points, bounded):
    c = _case(2, L, bw, rmin, rmax, n, C, F, seed=L + 10 * F + C, per_level=per_level, kind="uniform")
    # an offset keeps the shift gradient (a sum of n zero-mean terms per level) from cancelling to a value far below
    # the fixed-point quantisation of the tiles' node sums, against which a relative error would measure nothing
    c["g"] += np.float32(0.5)
    coords, lat, A, S, g = _dev(c["coords"]), _dev(c["lat"]), _dev(c["A"]), _dev(c["S"]), _dev(c["g"])
    plan = lib.Plan(coords, tile_points)
    _, _, off = plan.arrays()
    if tile_points:
        assert np.diff(off).max() > min(tile_points, 2048)
    feats = lib.latent_forward_planned(plan, lat, c["first"], c["res"], bw, A, S, F, True)
    feats_pp, _ = lib.latent_forward(coords, lat, c["first"], c["res"], bw, A, S, F, True, True)
    assert torch.equal(feats, feats_pp)
    _, want_gl, want_gA, want_gS = _oracle_fwd_bwd(c)
    level_max = _dev(np.abs(c["g"]).max(0).astype(np.float32)) if bounded else None
    gl, gA, gS = lib.latent_backward_planned(plan, g, lat, c["first"], c["res"], bw, A, C, F, c["T"], True, True,
                                             level_max=level_max)
    assert rel_err(gl.cpu().numpy(), want_gl) <= BWD_TOL
    _check_decoder_grads(c, gA, gS, want_gA, want_gS)
    plan.close()


def test_forward_without_room_for_point_slots(lib):
    """C = 4, F = 8, per-level decoders, 28 levels: node box and decoder take 45 184 B of shared memory, so the point
    slots would pass the 48 KB limit; the forward loads the points directly instead."""
    c = _case(2, 28, 14, 16, 512, 60000, 4, 8, seed=5, per_level=True, kind="uniform")
    coords, lat, A, S = _dev(c["coords"]), _dev(c["lat"]), _dev(c["A"]), _dev(c["S"])
    plan = lib.Plan(coords)
    assert plan.info()["tiles_per_axis"] == 16
    feats = lib.latent_forward_planned(plan, lat, c["first"], c["res"], 14, A, S, 8, True)
    feats_pp, _ = lib.latent_forward(coords, lat, c["first"], c["res"], 14, A, S, 8, True, True)
    assert torch.equal(feats, feats_pp)
    want_f, _, _, _ = _oracle_fwd_bwd(c)
    assert rel_err(feats.cpu().numpy(), want_f) <= 1e-5
    plan.close()


@pytest.mark.parametrize("bad", [np.inf, np.nan])
@pytest.mark.parametrize("level", [1, 6])   # in the first level chunk, and in one requested ahead
def test_non_finite_rows_poison_only_their_level(lib, bad, level):
    c = _case(2, 8, 12, 16, 128, 20000, 1, 1, seed=12, kind="uniform")
    coords, lat, A = _dev(c["coords"]), _dev(c["lat"]), _dev(c["A"])
    g = c["g"].copy()
    g[321, level] = bad
    plan = lib.Plan(coords)
    gl, _, _ = lib.latent_backward_planned(plan, _dev(g), lat, c["first"], c["res"], 12, A, 1, 1, c["T"], True, True)
    a, b = c["first"][level], c["first"][level + 1]
    assert bool(torch.isnan(gl[a:b]).any())
    assert bool(torch.isfinite(gl[:a]).all()) and bool(torch.isfinite(gl[b:]).all())
    plan.close()
