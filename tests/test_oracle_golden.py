"""The CPU oracle against the golden vectors produced by the reference's own Python modules
(tests/golden/make_golden.py). CPU only."""
import os

import numpy as np
import pytest
import torch

import oracle
from oracle import latent_oracle as lo
from helpers import REF_KERNEL_CASES, affine_from_case, case_from_golden, prob_params_from_case, ref_kernel_case, rel_err

CASES = ["img_c1f1", "img_c2f4_h", "nerf_c1f4", "nerf_c4f4_dft"]


def _decode(c, codebook):
    w_hat = lo.ste_round(codebook)
    def one(i):
        scale = torch.from_numpy(c["scale%d" % i])
        if c["dft"]:
            return torch.from_numpy(c["div%d" % i]), scale, torch.from_numpy(c["dft%d" % i])
        return torch.from_numpy(c["div%d" % i]), scale, None
    if c["hier"]:
        outs = torch.empty((c["T"], c["F"]))
        bounds = c["first_idx"] + [c["T"]]
        for l in range(c["L"]):
            div, scale, dft = one(l)
            a, b = bounds[l], bounds[l + 1]
            outs[a:b] = lo.decode_single(w_hat[a:b], div, scale, torch.from_numpy(c["shift%d" % l]))
        return outs
    div, scale, dft = one(0)
    if dft is not None:  # DecoderLayer dft branch: matmul(x, dft) * scale + shift
        return torch.matmul(w_hat / div, dft) * scale + torch.from_numpy(c["shift0"])
    return lo.decode_single(w_hat, div, scale, torch.from_numpy(c["shift0"]))


@pytest.mark.parametrize("name", CASES)
def test_decode_table_bit_exact(golden, name):
    c = case_from_golden(golden, name)
    table = _decode(c, torch.from_numpy(c["codebook"]))
    # same torch ops on the same machine: identical bits
    assert np.array_equal(table.numpy(), c["table"])


@pytest.mark.parametrize("name", CASES)
def test_quantized_latents_are_integers(golden, name):
    c = case_from_golden(golden, name)
    q = lo.ste_round(torch.from_numpy(c["codebook"])).numpy()
    assert np.array_equal(q, np.rint(c["codebook"]))  # half-to-even both
    assert np.abs(q).max() < 2 ** 15


@pytest.mark.parametrize("name", CASES)
def test_composed_interpolate_matches_reference(golden, name):
    c = case_from_golden(golden, name)
    feats = lo.latent_interpolate(c["coords"], torch.from_numpy(c["codebook"]), c["first_idx"], c["resolutions"],
                                  c["bw"], lambda cb: _decode(c, cb))
    assert np.array_equal(feats, c["feats"])


@pytest.mark.parametrize("name", CASES)
def test_fused_formulation_within_tolerance(golden, name):
    """interp(round(w)) @ A + shift (what the CUDA kernel computes) vs the reference's
    decode-then-interpolate: <= 1e-5 relative."""
    c = case_from_golden(golden, name)
    A, S = affine_from_case(c)
    q = np.rint(c["codebook"]).astype(np.float32)
    z = oracle.forward(c["coords"], q, c["first_idx"], c["resolutions"], c["bw"]).reshape(-1, c["L"], c["C"])
    nA = A.shape[0]
    feats = np.stack([z[:, l] @ A[l if nA > 1 else 0] + S[l if nA > 1 else 0] for l in range(c["L"])], 1)
    assert rel_err(feats.reshape(c["feats"].shape), c["feats"]) <= 1e-5


@pytest.mark.parametrize("name", CASES)
@pytest.mark.parametrize("mode", ["train", "val"])
def test_ent_loss_matches_reference(golden, name, mode):
    c = case_from_golden(golden, name)
    _, params = prob_params_from_case(c)
    avg, tot = lo.ent_loss(torch.from_numpy(c["codebook"]), torch.from_numpy(c["noise"]), params, c["layers"],
                           is_val=(mode == "val"))
    ref_tot, ref_avg = c["ent_%s_total" % mode]
    assert tot.item() == ref_tot and avg.item() == ref_avg


@pytest.mark.parametrize("name", CASES)
def test_size_bits_matches_reference(golden, name):
    c = case_from_golden(golden, name)
    assert lo.size_bits(torch.from_numpy(c["codebook"])) == c["size"][1]
    C, F, nA = c["C"], c["F"], (c["L"] if c["hier"] else 1)
    n_params = nA * (C + (F if c["dft"] else C * F) + F + (C * F if c["dft"] else 0))
    assert c["size"][0] == 32 * n_params  # latent_dec.size(): every Parameter, fp32


def test_symbol_stream_round_trip(golden):
    c = case_from_golden(golden, "img_c2f4_h")
    col = torch.from_numpy(c["codebook"][:, 0])
    sym, cdf, uniq, counts = lo.symbol_stream(col)
    assert sym.dtype == torch.int16 and sym.min() == 0 and sym.max() == uniq.numel() - 1
    assert cdf[0] == 0 and cdf[-1] == 1 and bool((cdf[1:] > cdf[:-1]).all())
    back = uniq[sym.long()] + torch.round(col).long().min()
    assert torch.equal(back, torch.round(col).long())


def test_oracle_hash_known_answers():
    """Hand-computed corner indices: dense level and hashed level, 2D and 3D."""
    # 2D, res 17, bw 14: dense (17 < 2^14, 289 < 2^14). coord (0,0) -> x = 8.5 -> cell 8, frac .5
    idx, w = oracle.corners(np.array([[0.0, 0.0]], np.float32), [17], 14)
    assert idx[0, 0].tolist() == [8 + 8 * 17, 8 + 9 * 17, 9 + 8 * 17, 9 + 9 * 17]
    assert np.allclose(w[0, 0], 0.25)
    # 2D, res 513, bw 16: hashed. coord (-1,-1) -> cell (0,0)
    idx, _ = oracle.corners(np.array([[-1.0, -1.0]], np.float32), [513], 16)
    P = 2654435761
    assert idx[0, 0].tolist() == [0, P % 65536, 1, (1 ^ P) % 65536]
    # 3D hashed, res 2049, bw 19, coord (1,1,1): clamp bound is exactly res-1 = 2048 (SURVEY Q4)
    idx, w = oracle.corners(np.array([[1.0, 1.0, 1.0]], np.float32), [2049], 19)
    Q = 805459861
    x = 2048
    want = [((x + ((j >> 2) & 1)) ^ (((x + ((j >> 1) & 1)) * P) & 0xFFFFFFFF) ^ (((x + (j & 1)) * Q) & 0xFFFFFFFF)) % (1 << 19)
            for j in range(8)]
    assert idx[0, 0].tolist() == want
    assert w[0, 0, 0] == 1.0 and np.all(w[0, 0, 1:] == 0.0)


def test_oracle_backward_is_adjoint_of_forward():
    rng = np.random.default_rng(3)
    res = oracle.geometric_resolutions(4, 40, 5)
    sizes, first, T = oracle.level_layout(res, 8, 3)
    coords = (rng.random((300, 3), dtype=np.float32) * 2 - 1)
    table = rng.standard_normal((T, 2)).astype(np.float32)
    g = rng.standard_normal((300, 10)).astype(np.float32)
    f = oracle.forward(coords, table, first, res, 8)
    gt = oracle.backward(coords, g, T, first, res, 8, 2)
    assert abs(float((f.astype(np.float64) * g).sum()) - float((gt.astype(np.float64) * table).sum())) < 1e-3


def test_oracle_empty_input():
    res = [17, 33]
    sizes, first, T = oracle.level_layout(res, 10, 2)
    f = oracle.forward(np.zeros((0, 2), np.float32), np.zeros((T, 2), np.float32), first, res, 10)
    assert f.shape == (0, 4)
    g = oracle.backward(np.zeros((0, 2), np.float32), np.zeros((0, 4), np.float32), T, first, res, 10, 2)
    assert g.shape == (T, 2) and not g.any()


# ---- the C oracle against the reference's OWN CUDA kernels (captured on a B200) --------------------------
def _ref_kernel_cases():
    import os
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "hashgrid_ref_kernels.npz")
    return np.load(path)


@pytest.mark.parametrize("name", list(REF_KERNEL_CASES))
def test_oracle_matches_reference_cuda_kernels(name):
    """tests/golden/make_golden_gpu.py ran oracle/_ref (the reference's .cu files, unmodified, sm_100a) on a B200.
    Forward: the oracle reproduces the kernel's floats bit for bit. Backward: atomics are order dependent -> 1e-5."""
    c = ref_kernel_case(_ref_kernel_cases(), name)
    feats = oracle.forward(c["coords"], c["table"], c["first_idx"], c["resolutions"], c["bw"])
    assert np.array_equal(feats.view(np.uint32), c["feats"].view(np.uint32))
    grad = oracle.backward(c["coords"], c["grad_out"], c["T"], c["first_idx"], c["resolutions"], c["bw"], c["F"])
    assert rel_err(grad[c["grad_rows"]], c["grad_vals"]) <= 1e-5
    assert int((np.abs(grad).sum(1) != 0).sum()) == c["grad_nonzero_rows"]
    assert rel_err(grad.astype(np.float64).sum(0), c["grad_total"]) <= 1e-5


def test_render_oracle_closed_forms():
    """oracle/render_oracle.py (restated kaolin exponential integration, parity with kaolin unpinned): closed forms.
    A ray of equal samples tau: w_i = e^{-i tau}(1 - e^{-tau}), alpha = 1 - e^{-n tau}; rays are independent."""
    import numpy as np
    from oracle import render_oracle as ro
    n, tau = 9, 0.37
    feats = np.ones((2 * n, 2))
    feats[:, 1] = np.arange(2 * n)
    taus = np.full(2 * n, tau)
    boundary = np.zeros(2 * n, dtype=bool)
    boundary[[0, n]] = True
    ray, w = ro.exponential_integration(feats, taus, boundary)
    want_w = np.exp(-tau * np.arange(n)) * (1 - np.exp(-tau))
    assert np.allclose(w[:n], want_w, rtol=1e-12) and np.allclose(w[n:], want_w, rtol=1e-12)
    assert np.allclose(ray[:, 0], 1 - np.exp(-n * tau), rtol=1e-12)
    assert np.allclose(ray[1, 1] - ray[0, 1], n * (1 - np.exp(-n * tau)), rtol=1e-12)
    import torch
    r2, w2 = ro.exponential_integration_torch(torch.from_numpy(feats), torch.from_numpy(taus), torch.from_numpy(boundary))
    assert np.allclose(r2.numpy(), ray) and np.allclose(w2.numpy(), w)


def test_voxel_sample_oracle_matches_the_reference_sampling_helpers():
    """oracle.render_oracle.voxel_samples against tests/golden/sampling_ref.npz = outputs of the reference's OWN
    wisp/ops/spc/sampling.py (sample_from_depth_intervals, expand_pack_boundary) on seeded inputs: bit-exact."""
    import os
    import numpy as np
    from oracle import render_oracle as ro
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sampling_ref.npz"))
    for name in ("a", "b", "c", "d"):
        depth, jitter, ridx = g[name + "/depth"], g[name + "/jitter"], g[name + "/ridx"]
        K = int(g[name + "/K"])
        R = int(ridx.max()) + 1
        rng = np.random.default_rng(0)
        o, d = rng.standard_normal((R, 3)).astype(np.float32), rng.standard_normal((R, 3)).astype(np.float32)
        ridx_out, samples, ds, deltas, boundary = ro.voxel_samples(o, d, ridx, depth, jitter)
        assert np.array_equal(ds.reshape(-1, K).view(np.uint32), g[name + "/depth_samples"].view(np.uint32)), name
        assert np.array_equal(boundary.astype(np.uint8), g[name + "/boundary"]), name
        assert np.array_equal(ridx_out, np.repeat(ridx.astype(np.int64), K))
        # deltas telescope back to the depths; samples lie on their rays
        assert np.allclose(depth[:, 0] + deltas.reshape(-1, K).sum(1), ds.reshape(-1, K)[:, -1], rtol=1e-5)
        assert np.allclose(samples, o[ridx_out] + d[ridx_out] * ds[:, None], rtol=1e-6, atol=1e-6)


def _sga_golden():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sga_ref.npz"))


@pytest.mark.parametrize("name", ["t1.0_diff", "t0.37_diff_c2", "t0.1_diff", "t0.5_nodiff", "t0.05_diff_c4"])
def test_sga_oracle_matches_the_reference_decoder(name):
    """oracle.sga_quantize on the recorded uniform draws == the reference's LatentDecoder.forward(use_sga) output and
    its autograd gradient (same torch CPU ops in the same order: bit for bit)."""
    g = _sga_golden()
    p = "dec/" + name + "/"
    T, C, diff = [int(v) for v in g[p + "meta"]]
    w = torch.from_numpy(g[p + "w"]).clone().requires_grad_(True)
    w_hat = lo.sga_quantize(w, torch.from_numpy(g[p + "u"]), float(g[p + "tau"][0]), bool(diff))
    assert np.array_equal(w_hat.detach().numpy(), g[p + "w_hat"])
    (w_hat * torch.from_numpy(g[p + "gout"])).sum().backward()
    assert np.allclose(w.grad.numpy(), g[p + "grad_w"], rtol=1e-6, atol=1e-7 * np.abs(g[p + "grad_w"]).max())
