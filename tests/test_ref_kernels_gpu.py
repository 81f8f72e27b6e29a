"""The reference's OWN CUDA kernels (oracle/_ref, compiled for sm_100a from the files under
/root/reference by oracle/build_ref.py) against the C oracle and against this package.
This is what pins the oracle: the reference ships no CPU path, tests or golden vectors."""
import os

import numpy as np
import pytest
import torch

import oracle
from helpers import REF_KERNEL_CASES, make_case, ref_kernel_case, rel_err

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ref():
    from oracle import build_ref
    build_ref.build()            # no-op on the GPU box (no /root/reference there): uses the shipped .so
    mod = build_ref.load()
    if mod is None:
        pytest.skip("oracle/_ref/wisp_ref_ops.so not present")
    return mod


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


REF_CASES = [(2, 16, 14, 16, 512, 5000, 2, "uniform"), (2, 16, 16, 16, 512, 5000, 2, "pixels"),
             (2, 16, 16, 16, 512, 3000, 4, "arbitrary"), (3, 16, 19, 16, 2048, 5000, 2, "arbitrary"),
             (3, 16, 19, 16, 2048, 2000, 4, "uniform"), (3, 24, 19, 16, 512, 2000, 2, "arbitrary")]


@pytest.mark.parametrize("dim,L,bw,rmin,rmax,n,F,kind", REF_CASES)
def test_reference_kernels_vs_oracle_and_ours(lib, ref, dim, L, bw, rmin, rmax, n, F, kind):
    c = make_case(dim, L, bw, rmin, rmax, n, F, seed=31 + dim + F, coord_kind=kind)
    coords, table, gout = _dev(c["coords"]), _dev(c["table"]), _dev(c["grad_out"])
    first_dev = torch.tensor(c["first_idx"], dtype=torch.int32, device="cuda")
    fwd = ref.hashgrid_interpolate2d_cuda if dim == 2 else ref.hashgrid_interpolate_cuda
    bwd = ref.hashgrid_interpolate2d_backward_cuda if dim == 2 else ref.hashgrid_interpolate_backward_cuda
    f_ref = fwd(coords, table, first_dev, c["resolutions"], bw).cpu().numpy()
    f_orc = oracle.forward(c["coords"], c["table"], c["first_idx"], c["resolutions"], bw)
    f_our = lib.hashgrid_forward(coords, table, c["first_idx"], c["resolutions"], bw).cpu().numpy()
    # the oracle restates the reference kernel's arithmetic, FMA order included: identical bits expected
    exact = np.array_equal(f_ref.view(np.uint32), f_orc.view(np.uint32))
    print("ref-vs-oracle forward bit-exact:", exact, "max rel", rel_err(f_orc, f_ref))
    assert rel_err(f_orc, f_ref) <= 1e-6
    assert rel_err(f_our, f_ref) <= 1e-5
    g_ref = bwd(coords, gout, table, first_dev, c["resolutions"], bw, F, False).cpu().numpy()
    g_orc = oracle.backward(c["coords"], c["grad_out"], c["T"], c["first_idx"], c["resolutions"], bw, F)
    g_our = lib.hashgrid_backward(coords, gout, c["first_idx"], c["resolutions"], bw, F, c["T"]).cpu().numpy()
    assert rel_err(g_orc, g_ref) <= 1e-4
    assert rel_err(g_our, g_ref) <= 1e-4


def test_reference_forward_bit_exact_with_oracle(lib):
    """This package's forward and backward kernels against the reference kernels' own outputs, stored in
    tests/golden/hashgrid_ref_kernels.npz (make_golden_gpu.py; domain edges and points outside the domain included),
    so the comparison needs no build of the reference: forward to 1e-5, backward rows, touched-row count and column
    totals to 1e-4. The oracle's bit-exactness on the same vectors is re-asserted alongside (the CPU suite's
    test_oracle_matches_reference_cuda_kernels is its primary check)."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "hashgrid_ref_kernels.npz"))
    bad = 0
    for name in REF_KERNEL_CASES:
        c = ref_kernel_case(g, name)
        f_orc = oracle.forward(c["coords"], c["table"], c["first_idx"], c["resolutions"], c["bw"])
        bad += int((c["feats"].view(np.uint32) != f_orc.view(np.uint32)).sum())
        coords = _dev(c["coords"])
        f_our = lib.hashgrid_forward(coords, _dev(c["table"]), c["first_idx"], c["resolutions"], c["bw"]).cpu().numpy()
        assert rel_err(f_our, c["feats"]) <= 1e-5, name
        g_our = lib.hashgrid_backward(coords, _dev(c["grad_out"]), c["first_idx"], c["resolutions"], c["bw"], c["F"],
                                      c["T"]).cpu().numpy()
        assert rel_err(g_our[c["grad_rows"]], c["grad_vals"]) <= 1e-4, name
        assert int((np.abs(g_our).sum(1) != 0).sum()) == c["grad_nonzero_rows"], name
        assert rel_err(g_our.astype(np.float64).sum(0), c["grad_total"]) <= 1e-4, name
    assert bad == 0, "%d elements differ in their bits" % bad
