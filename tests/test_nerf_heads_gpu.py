"""NeRF decoder heads on the tensor cores against a float64 oracle that rounds to bf16 at exactly the contract's points
(DESIGN section 9), plus determinism, NaN isolation, the density-only kernel, CUDA-graph capture and a NeRF-shape fit."""
import os
import sys

import pytest
import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "benchmarks"))

pytestmark = pytest.mark.gpu
GATE = 3e-4
DEV = torch.device("cuda", 0)
NAMES = ("W1", "b1", "W2", "b2", "W3", "b3", "W4", "b4", "W5", "b5")


def make_heads(in_dim, emb=27, seed=0):
    torch.manual_seed(seed)
    dd = nn.Sequential(nn.Linear(in_dim, 128), nn.ReLU(), nn.Linear(128, 16))
    dc = nn.Sequential(nn.Linear(16 + emb, 128), nn.ReLU(), nn.Linear(128, 128), nn.ReLU(), nn.Linear(128, 3))
    with torch.no_grad():
        for m in list(dd) + list(dc):
            if isinstance(m, nn.Linear):
                m.bias.uniform_(-0.2, 0.2)
    return dd.to(DEV), dc.to(DEV)


def make_inputs(S, in_dim, emb=27, seed=1, bad_ridx=True):
    g = torch.Generator().manual_seed(seed)
    lengths = torch.randint(1, 48, (S // 4 + 2,), generator=g)          # rays of varying length
    ridx = torch.repeat_interleave(torch.arange(lengths.numel()), lengths)[:S].to(torch.int32)
    R = int(ridx.max()) + 1 if S else 1
    if bad_ridx and S >= 3:
        ridx[S // 3] = -1
        ridx[-1] = R + 5
    feats = torch.randn(S, in_dim, generator=g)
    vemb = torch.randn(R, emb, generator=g)
    # Output gradients with a mean, as a photometric loss gives early in a fit. With zero-mean gradients the weight and
    # bias gradients at S = 2^19 are sums of random-sign terms that cancel to ~1/700 of their absolute size; then a
    # handful of ReLU decisions at pre-activations within a bf16 ulp of zero (upstream rounding of the kernel's fp32
    # values against the oracle's fp64 ones) move them by ~1e-3, which says nothing about the kernel's arithmetic.
    gd = 0.5 + torch.randn(S, 1, generator=g)
    grgb = 0.5 + torch.randn(S, 3, generator=g)
    return [t.to(DEV) for t in (feats, vemb, ridx, gd, grgb)]


def oracle(params, feats, vemb, ridx, gdens, grgb, rounded=True):
    """float64 restatement; b() rounds the fp32 value to bf16 (RNE) when `rounded`."""
    b = (lambda t: t.float().to(torch.bfloat16).double()) if rounded else (lambda t: t)
    W1, b1, W2, b2, W3, b3, W4, b4, W5, b5 = [p.detach().double() for p in params]
    X = feats.double()
    R = vemb.shape[0]
    ok = (ridx >= 0) & (ridx < R)
    Vr = torch.where(ok[:, None], vemb.double()[ridx.long().clamp(0, R - 1)], torch.zeros((), dtype=torch.float64,
                                                                                          device=X.device))
    z1 = b(X) @ b(W1).T + b1
    h1 = z1.clamp_min(0)
    d = b(h1) @ b(W2).T + b2
    density = d[:, :1].clamp_min(0)
    u = torch.cat([b(d), b(Vr)], 1)
    z2 = u @ b(W3).T + b3
    h2 = z2.clamp_min(0)
    z3 = b(h2) @ b(W4).T + b4
    h3 = z3.clamp_min(0)
    o = b(h3) @ b(W5).T + b5
    rgb = torch.sigmoid(o)
    go = grgb.double() * rgb * (1 - rgb)
    gW5, gb5 = b(go).T @ b(h3), go.sum(0)
    gz3 = (b(go) @ b(W5)) * (z3 > 0)
    gW4, gb4 = b(gz3).T @ b(h2), gz3.sum(0)
    gz2 = (b(gz3) @ b(W4)) * (z2 > 0)
    gW3, gb3 = b(gz2).T @ u, gz2.sum(0)
    gd = (b(gz2) @ b(W3))[:, :16].clone()
    gd[:, 0] += gdens.double()[:, 0] * (d[:, 0] > 0)
    gW2, gb2 = b(gd).T @ b(h1), gd.sum(0)
    gz1 = (b(gd) @ b(W2)) * (z1 > 0)
    gW1, gb1 = b(gz1).T @ b(X), gz1.sum(0)
    gX = b(gz1) @ b(W1)
    return density, rgb, gX, [gW1, gb1, gW2, gb2, gW3, gb3, gW4, gb4, gW5, gb5]


def rel(a, ref):
    ref = ref.double()
    return float((a.double() - ref).norm() / ref.norm().clamp_min(1e-30))


def run(heads, feats, vemb, ridx, gdens, grgb):
    for p in heads.parameters():
        p.grad = None
    x = feats.clone().requires_grad_(True)
    density, rgb = heads(x, vemb, ridx)
    torch.autograd.backward([density, rgb], [gdens, grgb])
    return density.detach(), rgb.detach(), x.grad, [p.grad.clone() for p in heads.parameters()]


@pytest.mark.parametrize("in_dim", [64, 96])
@pytest.mark.parametrize("S", [1, 127, 128, 129, 1 << 19])
def test_heads_match_the_bf16_rounding_oracle(lib, in_dim, S):
    from shacira_b200.nerf_heads import NerfHeads
    heads = NerfHeads(*make_heads(in_dim))
    feats, vemb, ridx, gd, grgb = make_inputs(S, in_dim)
    got = run(heads, feats, vemb, ridx, gd, grgb)
    want = oracle(heads.parameters(), feats, vemb, ridx, gd, grgb)
    unrounded = oracle(heads.parameters(), feats, vemb, ridx, gd, grgb, rounded=False)
    errs = {"density": rel(got[0], want[0]), "rgb": rel(got[1], want[1]), "g_X": rel(got[2], want[2])}
    errs.update({n: rel(g, w) for n, g, w in zip(NAMES, got[3], want[3])})
    far = {"density": rel(got[0], unrounded[0]), "rgb": rel(got[1], unrounded[1]), "g_X": rel(got[2], unrounded[2])}
    far.update({n: rel(g, w) for n, g, w in zip(NAMES, got[3], unrounded[3])})
    worst = max(errs, key=errs.get)
    print("in_dim %d S %d: worst %s %.2e against the bf16 oracle; against the unrounded fp64 oracle %.2e .. %.2e"
          % (in_dim, S, worst, errs[worst], min(far.values()), max(far.values())))
    for k, e in errs.items():
        assert e <= GATE, (k, e, errs)


def test_out_of_range_ridx_takes_a_zero_embedding(lib):
    from shacira_b200.nerf_heads import NerfHeads
    heads = NerfHeads(*make_heads(64))
    feats, vemb, ridx, gd, grgb = make_inputs(300, 64, bad_ridx=False)
    bad = ridx.clone()
    bad[::7] = -3
    bad[1::7] = vemb.shape[0]
    bad[2::7] = 2 ** 31 - 1
    zero_row = torch.cat([vemb, torch.zeros(1, vemb.shape[1], device=DEV)])
    moved = torch.where((bad >= 0) & (bad < vemb.shape[0]), bad, torch.full_like(bad, vemb.shape[0]))
    a = run(heads, feats, vemb, bad, gd, grgb)
    b = run(heads, feats, zero_row, moved, gd, grgb)
    for x, y in zip(a[:3] + tuple(a[3]), b[:3] + tuple(b[3])):
        assert torch.equal(x, y)


def test_backward_is_bit_identical_across_launches(lib):
    from shacira_b200.nerf_heads import NerfHeads
    heads = NerfHeads(*make_heads(96))
    inp = make_inputs(100_000, 96)
    a, b = run(heads, *inp), run(heads, *inp)
    for x, y in zip(a[:3] + tuple(a[3]), b[:3] + tuple(b[3])):
        assert torch.equal(x, y)


def test_nan_row_poisons_only_its_own_sample(lib):
    """density and rgb of the NaN sample are NaN (relu keeps NaN, as torch.relu); its g_X row is zero, as torch's
    autograd gives (the ReLU masks of a NaN pre-activation are off); every other sample stays finite."""
    from shacira_b200.nerf_heads import NerfHeads
    heads = NerfHeads(*make_heads(64))
    feats, vemb, ridx, gd, grgb = make_inputs(1000, 64)
    feats[300, 5] = float("nan")
    density, rgb, gX, _ = run(heads, feats, vemb, ridx, gd, grgb)
    others = torch.ones(1000, dtype=torch.bool, device=DEV)
    others[300] = False
    assert torch.isnan(density[300]).all() and torch.isnan(rgb[300]).all()
    assert torch.equal(gX[300], torch.zeros_like(gX[300]))
    assert torch.isfinite(density[others]).all() and torch.isfinite(rgb[others]).all()
    assert torch.isfinite(gX[others]).all()


@pytest.mark.parametrize("in_dim", [64, 96])
def test_density_only_equals_the_full_forward(lib, in_dim):
    from shacira_b200.nerf_heads import NerfHeads
    heads = NerfHeads(*make_heads(in_dim))
    feats, vemb, ridx, _, _ = make_inputs(5000, in_dim)
    with torch.no_grad():
        density, _ = heads(feats, vemb, ridx)
    assert torch.equal(heads.density(feats), density)
    assert heads.density(feats[:0]).shape == (0, 1)


def test_empty_input_is_a_no_op(lib):
    from shacira_b200.nerf_heads import NerfHeads
    heads = NerfHeads(*make_heads(64))
    feats, vemb, ridx, gd, grgb = make_inputs(0, 64)
    density, rgb, gX, grads = run(heads, feats, vemb, ridx, gd, grgb)
    assert density.shape == (0, 1) and rgb.shape == (0, 3) and gX.shape == (0, 64)
    assert all(float(g.abs().sum()) == 0.0 for g in grads)


def test_cuda_graph_capture_matches_eager(lib):
    from shacira_b200.nerf_heads import NerfHeads
    heads = NerfHeads(*make_heads(96))
    feats, vemb, ridx, gd, grgb = make_inputs(20_000, 96)
    x = feats.clone().requires_grad_(True)
    eager = run(heads, feats, vemb, ridx, gd, grgb)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):          # warm-up on the capture stream
            for p in heads.parameters():
                p.grad = None
            x.grad = None
            density, rgb = heads(x, vemb, ridx)
            torch.autograd.backward([density, rgb], [gd, grgb])
    torch.cuda.current_stream().wait_stream(s)
    for p in heads.parameters():
        p.grad = None
    x.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        density, rgb = heads(x, vemb, ridx)
        torch.autograd.backward([density, rgb], [gd, grgb])
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(density, eager[0]) and torch.equal(rgb, eager[1]) and torch.equal(x.grad, eager[2])
    for p, g in zip(heads.parameters(), eager[3]):
        assert torch.equal(p.grad, g)


# ---- NeRF-shape fit: the synthetic scene of benchmarks/fit_nerf.py with the reference's head shapes -----------------

def view_embedding(d):
    """The reference's view_embedder (4 frequencies, input included): 3 + 3 * 2 * 4 = 27 columns."""
    out = [d]
    for k in range(4):
        out += [torch.sin(d * 2.0 ** k), torch.cos(d * 2.0 ** k)]
    return torch.cat(out, 1)


def nerf_fit(impl, seed, steps):
    import fit_nerf as fn
    from shacira_b200.grids import LatentGrid
    from shacira_b200.nerf_heads import NerfHeads
    torch.manual_seed(seed)
    grid = LatentGrid.from_geometric(feature_dim=fn.F, num_lods=fn.L, latent_dim=fn.C, multiscale_type="cat",
                                     resolution_dim=3, feature_std=0.1, codebook_bitwidth=fn.BW, min_grid_res=16,
                                     max_grid_res=2048, init_grid="uniform", conf_latent_decoder=dict(fn.DEC),
                                     conf_entropy_reg=dict(fn.ENT))
    dd = nn.Sequential(nn.Linear(fn.L * fn.F, 128), nn.ReLU(), nn.Linear(128, 16))
    dc = nn.Sequential(nn.Linear(16 + 27, 128), nn.ReLU(), nn.Linear(128, 128), nn.ReLU(), nn.Linear(128, 3))
    with torch.no_grad():
        grid.codebook.mul_(fn.LATENT_SCALE)
        grid.latent_dec.layers[0].scale.mul_(0.1)
    grid, dd, dc = grid.to(DEV), dd.to(DEV), dc.to(DEV)
    native = NerfHeads(dd, dc) if impl == "kernel" else None

    def heads(feats, vemb, ridx):
        if native is not None:
            return native(feats, vemb, ridx)
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=impl == "autocast"):
            d = dd(feats)
            rgb = torch.sigmoid(dc(torch.cat([d, vemb[ridx]], 1)))
        return torch.relu(d[:, :1]).float(), rgb.float()

    params = [dict(params=list(dd.parameters()) + list(dc.parameters()), lr=1e-3),
              dict(params=[grid.codebook], lr=1e-2),
              dict(params=[p for p in grid.latent_dec.parameters() if p.requires_grad], lr=1e-3),
              dict(params=list(grid.prob_model.parameters()), lr=1e-4)]
    opt = torch.optim.RMSprop(params)
    gen = torch.Generator().manual_seed(1000 + seed)
    test_gen = torch.Generator().manual_seed(77)
    to, td, ttn, ttf = fn.make_rays(fn.RAYS, test_gen, DEV)
    test_px = fn.target_pixels(to, td, ttn, ttf, test_gen)
    ridx = torch.arange(fn.RAYS, device=DEV, dtype=torch.int32).repeat_interleave(fn.K)

    def render(o, d, tn, tf, g):
        pts, delta = fn.sample(o, d, tn, tf, g)
        density, rgb = heads(grid.interpolate(pts, 0), view_embedding(-d), ridx)
        return fn.integrate(rgb, density[:, 0] * delta, o.shape[0])

    for it in range(steps):
        o, d, tn, tf = fn.make_rays(fn.RAYS, gen, DEV)
        gt = fn.target_pixels(o, d, tn, tf, gen)
        opt.zero_grad(set_to_none=True)
        pred = render(o, d, tn, tf, gen)
        avg_bits, _ = grid.ent_loss(it, is_val=True)
        loss = torch.abs(pred - gt).mean() + 1e-4 * avg_bits
        loss.backward()
        opt.step()
    with torch.no_grad():
        pred = render(to, td, ttn, ttf, torch.Generator().manual_seed(78))
    return fn.psnr(pred, test_px)


def test_nerf_shape_fit_with_kernel_heads_matches_autocast_heads(lib):
    """300 steps, 16 levels, the reference's head shapes. Gate: |PSNR(kernel) - mean PSNR(autocast bf16)| within
    0.05 dB plus the spread of two autocast runs, floored at 0.15 dB as in test_nerf_shape_fit_matches_reference_kernels
    (the grid's float atomics make two runs of one seed differ)."""
    steps = 300
    kern = nerf_fit("kernel", 0, steps)
    a1, a2 = nerf_fit("autocast", 0, steps), nerf_fit("autocast", 0, steps)
    fp32 = nerf_fit("fp32", 0, steps)
    spread = max(abs(a1 - a2), 0.15)
    print("PSNR kernel %.3f  autocast-bf16 %.3f / %.3f  fp32 %.3f dB" % (kern, a1, a2, fp32))
    assert kern > 15.0
    assert abs(kern - 0.5 * (a1 + a2)) <= 0.05 + spread
