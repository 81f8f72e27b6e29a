"""The drop-in boundary as the reference drives it: the four `wisp._C.ops` names called the way
wisp/ops/grid.py:69-196 calls them (custom_fwd(cast_inputs=half) under autocast -- AMP is the default of app/nerf,
main_nerf.py:246-249,603) and the way LatentGrid.interpolate feeds them a decoded one-channel table
(latent_grid.py:359-370: repeat(1, 2) in, [:, ::2] out). /root/reference is absent on the GPU box, so the two
autograd Functions are restated here from the cited lines; everything below them is this package."""
import numpy as np
import pytest
import torch

import oracle
from helpers import affine_from_case, case_from_golden, make_case, rel_err

pytestmark = pytest.mark.gpu


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _reference_functions(C_ops):
    """wisp/ops/grid.py:69-111 (3D) and :135-176 (2D), line for line in behaviour, bound to `C_ops`."""

    def make(fwd_name, bwd_name):
        class Fn(torch.autograd.Function):
            @staticmethod
            @torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.half)     # grid.py:73,138
            def forward(ctx, coords, resolutions, codebook_bitwidth, lod_idx, codebook, codebook_sizes, codebook_first_idx):
                if codebook[0].shape[-1] % 2 == 1:                                    # grid.py:75,140
                    raise Exception("The codebook feature dimension needs to be a multiple of 2.")
                feats_out = getattr(C_ops, fwd_name)(coords.float().contiguous(), codebook, codebook_first_idx,
                                                     resolutions, codebook_bitwidth).contiguous()
                ctx.save_for_backward(coords, codebook, codebook_first_idx)
                ctx.resolutions, ctx.codebook_bitwidth, ctx.feature_dim = resolutions, codebook_bitwidth, codebook.shape[-1]
                return feats_out

            @staticmethod
            @torch.amp.custom_bwd(device_type="cuda")                                # grid.py:95,160
            def backward(ctx, grad_output):
                coords, codebook, first_idx = ctx.saved_tensors
                grad_codebook = getattr(C_ops, bwd_name)(coords.float().contiguous(), grad_output.contiguous(), codebook,
                                                         first_idx, ctx.resolutions, ctx.codebook_bitwidth,
                                                         ctx.feature_dim, ctx.needs_input_grad[0])
                return (None, None, None, None, grad_codebook, None, None)
        return Fn

    return (make("hashgrid_interpolate_cuda", "hashgrid_interpolate_backward_cuda"),
            make("hashgrid_interpolate2d_cuda", "hashgrid_interpolate2d_backward_cuda"))


@pytest.mark.parametrize("dim", [2, 3])
def test_reference_autograd_functions_over_the_shim_fp32_and_autocast(lib, dim):
    from shacira_b200 import compat
    C = compat.install_as_wisp_C()
    Fn3, Fn2 = _reference_functions(C.ops)
    Fn = Fn2 if dim == 2 else Fn3
    c = make_case(dim, 16, 16 if dim == 2 else 19, 16, 512 if dim == 2 else 2048, 30000, 2, seed=40 + dim)
    coords, g = _dev(c["coords"]), _dev(c["grad_out"])
    first = torch.tensor(c["first_idx"], dtype=torch.int32, device="cuda")           # a DEVICE tensor, as the reference passes
    want = oracle.forward(c["coords"], c["table"], c["first_idx"], c["resolutions"], c["bw"])
    want_g = oracle.backward(c["coords"], c["grad_out"], c["T"], c["first_idx"], c["resolutions"], c["bw"], 2)
    # fp32, no autocast (kodak.yaml disables AMP)
    table = _dev(c["table"]).requires_grad_(True)
    feats = Fn.apply(coords, c["resolutions"], c["bw"], 0, table, None, first)
    assert feats.dtype == torch.float32 and rel_err(feats.detach().cpu().numpy(), want) <= 1e-5
    feats.backward(g)
    assert rel_err(table.grad.cpu().numpy(), want_g) <= 1e-4
    # autocast: inputs arrive as half, the result and the gradient come back as half (the reference's dtypes)
    table_h = _dev(c["table"]).requires_grad_(True)
    with torch.autocast("cuda", dtype=torch.float16):
        feats_h = Fn.apply(coords, c["resolutions"], c["bw"], 0, table_h, None, first)
    assert feats_h.dtype == torch.float16
    # what the kernel saw: half-rounded coordinates and table, evaluated in fp32
    ch = c["coords"].astype(np.float16).astype(np.float32)
    th = c["table"].astype(np.float16).astype(np.float32)
    want_h = oracle.forward(ch, th, c["first_idx"], c["resolutions"], c["bw"])
    assert rel_err(feats_h.detach().float().cpu().numpy(), want_h) <= 2e-3                  # one rounding to half on the way out
    feats_h.float().backward(g)
    assert table_h.grad is not None and table_h.grad.dtype == torch.float32        # autograd casts back to the leaf
    want_gh = oracle.backward(ch, c["grad_out"].astype(np.float16).astype(np.float32), c["T"], c["first_idx"],
                              c["resolutions"], c["bw"], 2)
    assert rel_err(table_h.grad.cpu().numpy(), want_gh) <= 3e-3
    # double tables are served too (AT_DISPATCH_FLOATING_TYPES_AND_HALF)
    fwd = C.ops.hashgrid_interpolate2d_cuda if dim == 2 else C.ops.hashgrid_interpolate_cuda
    feats_d = fwd(coords, _dev(c["table"]).double(), first, c["resolutions"], c["bw"])
    assert feats_d.dtype == torch.float64 and rel_err(feats_d.cpu().numpy(), want) <= 1e-5


@pytest.mark.parametrize("name", ["img_c1f1", "nerf_c1f4"])
def test_latent_call_pattern_of_the_reference_grid(lib, golden, name):
    """LatentGrid.interpolate of the reference (latent_grid.py:359-370) on top of the shim: decode the table with torch,
    pad a one-channel table to two (repeat(1, 2)), interpolate, take every other column -- against the features and
    table gradients the reference produced (tests/golden/latent_ref_<case>.npz)."""
    from shacira_b200 import compat
    C = compat.install_as_wisp_C()
    Fn3, Fn2 = _reference_functions(C.ops)
    c = case_from_golden(golden, name)
    A, S = affine_from_case(c)
    first = torch.tensor(c["first_idx"], dtype=torch.int32, device="cuda")
    cb = _dev(c["codebook"]).requires_grad_(True)
    q = cb + (torch.round(cb) - cb).detach()                       # StraightThrough
    table = q @ _dev(A[0]) + _dev(S[0])                            # decode: (w / div) @ scale + shift
    pad = table.shape[1] == 1
    if pad:
        table = table.repeat(1, 2)
    Fn = Fn2 if c["dim"] == 2 else Fn3
    feats = Fn.apply(_dev(c["coords"]), c["resolutions"], c["bw"], 0, table, None, first)
    if pad:
        feats = feats[:, ::2]
    assert rel_err(feats.detach().cpu().numpy(), c["feats"]) <= 1e-5
    feats.backward(_dev(c["grad_out"]))
    assert rel_err(cb.grad.cpu().numpy(), c["grad_codebook"]) <= 1e-4
