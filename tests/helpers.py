"""Shared helpers for the parity tests (CPU + GPU)."""
import numpy as np
import torch

import oracle


def case_from_golden(golden, name):
    p = name + "/"
    dim, L, bw, C, F, layers, hier, dft = [int(v) for v in golden[p + "meta"]]
    d = dict(name=name, dim=dim, L=L, bw=bw, C=C, F=F, layers=layers, hier=bool(hier), dft=bool(dft))
    for k in golden:
        if k.startswith(p):
            d[k[len(p):]] = golden[k]
    d["resolutions"] = [int(v) for v in d["resolutions"]]
    sizes, first, T = oracle.level_layout(d["resolutions"], bw, dim)
    d["first_idx"], d["sizes"], d["T"] = first, sizes, T
    return d


def affine_from_case(c):
    """A [nA, C, F] and shift [nA, F] (float32 numpy) exactly as LatentDecoder.affine_map builds them."""
    nA = c["L"] if c["hier"] else 1
    As, Ss = [], []
    for i in range(nA):
        scale = torch.from_numpy(c["scale%d" % i])
        if c["dft"]:
            scale = torch.from_numpy(c["dft%d" % i]) * scale
        div = torch.from_numpy(c["div%d" % i])
        As.append((scale / div.unsqueeze(1)).numpy())
        Ss.append(c["shift%d" % i].reshape(-1))
    return np.stack(As).astype(np.float32), np.stack(Ss).astype(np.float32)


def prob_params_from_case(c):
    """[4, 3, C] packed like BitEstimator.packed_params and the dict form for the oracle."""
    C = c["C"]
    packed = np.zeros((4, 3, C), dtype=np.float32)
    d = {}
    for fi in range(4):
        h, b = c["prob_h%d" % fi], c["prob_b%d" % fi]
        a = c.get("prob_a%d" % fi)
        packed[fi, 0], packed[fi, 1] = h.reshape(-1), b.reshape(-1)
        if a is not None:
            packed[fi, 2] = a.reshape(-1)
        d["f%d" % (fi + 1)] = (torch.from_numpy(h), torch.from_numpy(b), torch.from_numpy(a) if a is not None else None)
    return packed, d


REF_KERNEL_CASES = {"2d_cfg1": "uniform", "2d_cfg2_arbitrary": "arbitrary", "2d_q4_dense": "uniform",
                    "3d_cfg4": "arbitrary", "3d_lego24_f4": "uniform"}


def ref_kernel_case(g, name):
    """One case of tests/golden/hashgrid_ref_kernels.npz (outputs of the reference's own CUDA kernels, captured by
    make_golden_gpu.py) with its seeded table / upstream gradient regenerated: the same draws as make_case(seed=...)
    there (the coordinate kind decides the first draw; the stored coordinates carry the edge rows)."""
    p = name + "/"
    dim, L, bw, F = [int(v) for v in g[p + "meta"]]
    res = [int(v) for v in g[p + "resolutions"]]
    coords = g[p + "coords"]
    n = coords.shape[0]
    rng = np.random.default_rng(int(g[p + "seed"][0]))
    if REF_KERNEL_CASES[name] == "uniform":
        rng.random((n, dim), dtype=np.float32)
    else:
        rng.standard_normal((n, dim))
    sizes, first, T = oracle.level_layout(res, bw, dim)
    table = rng.standard_normal((T, F)).astype(np.float32)
    gout = rng.standard_normal((n, L * F)).astype(np.float32)
    assert np.array_equal(table[:16], g[p + "table_seed_check"])
    return dict(dim=dim, L=L, bw=bw, F=F, resolutions=res, first_idx=first, T=T, coords=coords, table=table,
                grad_out=gout, feats=g[p + "feats"], grad_rows=g[p + "grad_rows"], grad_vals=g[p + "grad_vals"],
                grad_nonzero_rows=int(g[p + "grad_nonzero_rows"][0]), grad_total=g[p + "grad_total"])


def rel_err(a, b):
    """max |a-b| / max |b| -- the relative error the north_star tolerances are stated in."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(float(np.max(np.abs(b))), 1e-30))


def make_case(dim, L, bw, rmin, rmax, n, F, seed, coord_kind="uniform"):
    rng = np.random.default_rng(seed)
    res = oracle.geometric_resolutions(rmin, rmax, L) if L > 1 else [rmin]
    sizes, first, T = oracle.level_layout(res, bw, dim)
    if coord_kind == "uniform":
        coords = (rng.random((n, dim), dtype=np.float32) * 2 - 1).astype(np.float32)
    elif coord_kind == "arbitrary":  # full-mantissa coords, like NeRF o + t*d samples
        coords = np.clip(rng.standard_normal((n, dim)) * 0.6, -1, 1).astype(np.float32)
    elif coord_kind == "pixels":
        h = int(np.sqrt(n))
        ys, xs = np.meshgrid(np.arange(h), np.arange(h), indexing="ij")
        coords = np.stack([(ys.reshape(-1) / h - 0.5) * 2, (xs.reshape(-1) / h - 0.5) * 2], 1).astype(np.float32)
        coords = coords[rng.permutation(coords.shape[0])]
    else:
        raise ValueError(coord_kind)
    table = rng.standard_normal((T, F)).astype(np.float32)
    gout = rng.standard_normal((coords.shape[0], L * F)).astype(np.float32)
    return dict(dim=dim, L=L, bw=bw, resolutions=res, first_idx=first, sizes=sizes, T=T, coords=coords, table=table,
                grad_out=gout, F=F)


def level_rel_err(a, b, first_idx, sizes):
    """max over levels of (max |a-b| over the level's rows) / (max |b| over the level's rows): a small gradient on a
    fine level is not allowed to hide behind a large one on a coarse level."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    worst = 0.0
    for f, s in zip(first_idx, sizes):
        da, db = a[f:f + s], b[f:f + s]
        worst = max(worst, float(np.max(np.abs(da - db)) / max(float(np.max(np.abs(db))), 1e-30)))
    return worst


def level_rms_err(a, b, first_idx, sizes):
    """max over levels of rms(a-b) / rms(b)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    worst = 0.0
    for f, s in zip(first_idx, sizes):
        da, db = a[f:f + s], b[f:f + s]
        worst = max(worst, float(np.sqrt(np.mean((da - db) ** 2)) / max(float(np.sqrt(np.mean(db ** 2))), 1e-30)))
    return worst
