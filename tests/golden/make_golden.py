"""Generate tests/golden/latent_ref_<case>.npz (one file per case) by running the REFERENCE's own Python modules
(imported from /root/reference with its missing third-party deps stubbed) on seeded inputs.

Run in the build container only (`python tests/golden/make_golden.py`); the fixture is
committed, /root/reference does not exist on the GPU box. What runs is the reference's code:
  wisp.models.latent_decoders.{LatentDecoder, HierarchicalLatentDecoder}
  wisp.models.prob_models.BitEstimator
  wisp.models.grids.LatentGrid.{ent_loss, size, interpolate}  (+ wisp.ops.grid autograd Functions)
with `wisp._C.ops` served by the C oracle (oracle/hashgrid_oracle.c) since the reference's kernels
are CUDA-only; the kernels themselves are pinned separately on the GPU (make_golden_gpu.py).
"""
import os
import sys
import types
from unittest.mock import MagicMock

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import oracle  # noqa: E402

REF = "/root/reference"


def import_reference():
    sys.path.insert(0, REF)
    for name in ["kaolin", "kaolin.ops", "kaolin.ops.spc", "kaolin.render", "kaolin.render.spc", "kaolin.render.camera",
                 "kaolin.rep", "kaolin.rep.spc", "kaolin.ops.mesh", "kaolin.io", "kaolin.ops.batch", "polyscope",
                 "tinyobjloader", "skimage", "skimage.metrics", "lpips", "torchac", "pydispatch", "attrdict",
                 "kaolin.render.camera.intrinsics", "kaolin.visualize", "kaolin.utils", "kaolin.utils.testing",
                 "kaolin.ops.conversions", "cv2", "glumpy", "OpenEXR", "Imath", "pycuda"]:
        if name not in sys.modules:
            sys.modules[name] = MagicMock()
    # wisp._C.ops backed by the CPU oracle
    ops = types.ModuleType("wisp._C.ops")

    def _fwd(coords, codebook, first_idx, resolution, bitwidth):
        f = oracle.forward(coords.detach().numpy(), codebook.detach().numpy(), first_idx.numpy(), list(resolution), bitwidth)
        return torch.from_numpy(f)

    def _bwd(coords, grad_output, codebook, first_idx, resolution, bitwidth, feature_dim, req):
        g = oracle.backward(coords.detach().numpy(), grad_output.detach().numpy(), codebook.shape[0], first_idx.numpy(),
                            list(resolution), bitwidth, feature_dim)
        return torch.from_numpy(g)

    ops.hashgrid_interpolate_cuda = _fwd
    ops.hashgrid_interpolate2d_cuda = _fwd
    ops.hashgrid_interpolate_backward_cuda = _bwd
    ops.hashgrid_interpolate2d_backward_cuda = _bwd
    C = types.ModuleType("wisp._C")
    C.ops = ops
    sys.modules["wisp._C"] = C
    sys.modules["wisp._C.ops"] = ops
    import wisp  # noqa: F401
    wisp._C = C
    import wisp.accelstructs as acc
    acc.OctreeAS.make_dense = classmethod(lambda cls, level: MagicMock())
    import wisp.models.grids.latent_grid as lg
    import wisp.models.grids.hash_grid as hg
    lg.spc_ops.unbatched_get_level_points = lambda *a, **k: torch.zeros(1, 3)
    hg.spc_ops.unbatched_get_level_points = lambda *a, **k: torch.zeros(1, 3)
    return lg, hg


def dec_cfg(kind="single", C=1, use_shift=True, matrix="sq", std=0.1):
    return dict(ldecode_enabled=True, ldecode_type=kind, use_sga=False, diff_sampling=True, use_shift=use_shift,
                ldecode_matrix=matrix, latent_dim=C, norm="max", norm_every=10, ldec_std=std, decay_period=0.9,
                temperature=0.1)


def ent_cfg(layers):
    return dict(num_prob_layers=layers, entropy_reg=1e-3, entropy_reg_end=1e-4, entropy_reg_sched="cosine",
                noise_freq=2)


def main():
    lg, hg = import_reference()
    out = {}
    cases = []
    # (name, dim, L, bw, min, max, C, F, decoder kind, matrix, prob layers)
    specs = [
        ("img_c1f1", 2, 8, 10, 16, 128, 1, 1, "single", "sq", 2),
        ("img_c2f4_h", 2, 6, 9, 8, 96, 2, 4, "hierarchical", "sq", 4),
        ("nerf_c1f4", 3, 6, 12, 8, 64, 1, 4, "single", "sq", 1),
        ("nerf_c4f4_dft", 3, 4, 11, 8, 40, 4, 4, "single", "dft", 3),
    ]
    for si, (name, dim, L, bw, rmin, rmax, C, F, kind, matrix, layers) in enumerate(specs):
        torch.manual_seed(100 + si)
        grid = lg.LatentGrid.from_geometric(feature_dim=F, num_lods=L, latent_dim=C, multiscale_type="cat",
                                            resolution_dim=dim, feature_std=0.1, codebook_bitwidth=bw,
                                            min_grid_res=rmin, max_grid_res=rmax, init_grid="uniform",
                                            conf_latent_decoder=dec_cfg(kind, C, True, matrix),
                                            conf_entropy_reg=ent_cfg(layers))
        with torch.no_grad():
            grid.codebook.mul_(60.0)  # +-6: rounding is non-trivial
            decs = grid.latent_dec.decoders if kind == "hierarchical" else [grid.latent_dec]
            for d in decs:
                d.div.data = torch.rand(C) * 2 + 0.5
                for layer in d.layers:
                    if hasattr(layer, "shift") and layer.shift is not None:
                        layer.shift.normal_(0, 0.05)
            for f in (grid.prob_model.f1, grid.prob_model.f2, grid.prob_model.f3, grid.prob_model.f4):
                f.h.normal_(0, 0.3)
                f.b.normal_(0, 0.3)
                if f.a is not None:
                    f.a.normal_(0, 0.3)
            if kind == "hierarchical":
                # the reference leaves the last level undecoded (torch.empty garbage, SURVEY Q5):
                # repair its offsets so the fixture is well defined; this is the documented deviation.
                grid.latent_dec.offsets = torch.cat((grid.codebook_lod_first_idx,
                                                     torch.tensor([grid.codebook.shape[0]], dtype=torch.int32)))
        N = 1500
        coords = torch.rand(N, dim) * 2 - 1
        coords[:8] = torch.tensor([[-1.0] * dim, [1.0] * dim, [0.0] * dim, [-1.0, 1.0, 0.5][:dim], [0.999999] * dim,
                                   [-0.999999] * dim, [1.5] * dim, [-1.5] * dim])
        gout = torch.randn(N, L * F)
        # decode (table side)
        table = grid.latent_dec(grid.codebook)
        # interpolate + backward through the reference's own autograd graph
        feats = grid.interpolate(coords, 0)
        grid.zero_grad()
        feats.backward(gout)
        p = name + "/"
        out[p + "resolutions"] = np.array(grid.resolutions, dtype=np.int32)
        out[p + "meta"] = np.array([dim, L, bw, C, F, layers, 1 if kind == "hierarchical" else 0,
                                    1 if matrix == "dft" else 0], dtype=np.int32)
        out[p + "codebook"] = grid.codebook.detach().numpy().copy()
        out[p + "coords"] = coords.numpy()
        out[p + "grad_out"] = gout.numpy()
        out[p + "table"] = table.detach().numpy()
        out[p + "feats"] = feats.detach().numpy()
        out[p + "grad_codebook"] = grid.codebook.grad.numpy().copy()
        for di, d in enumerate(decs):
            out[p + "div%d" % di] = d.div.detach().numpy().copy()
            out[p + "scale%d" % di] = d.layers[0].scale.detach().numpy().copy()
            out[p + "shift%d" % di] = d.layers[0].shift.detach().numpy().copy()
            out[p + "grad_scale%d" % di] = d.layers[0].scale.grad.numpy().copy()
            out[p + "grad_shift%d" % di] = d.layers[0].shift.grad.numpy().copy()
            if matrix == "dft":
                out[p + "dft%d" % di] = d.layers[0].dft.detach().numpy().copy()
        # entropy loss with a fixed noise tensor (noise_freq=2, odd idx -> uses grid.noise)
        grid.noise = torch.rand(grid.codebook.shape) - 0.5
        out[p + "noise"] = grid.noise.numpy().copy()
        for fi, f in enumerate((grid.prob_model.f1, grid.prob_model.f2, grid.prob_model.f3, grid.prob_model.f4)):
            out[p + "prob_h%d" % fi] = f.h.detach().numpy().copy()
            out[p + "prob_b%d" % fi] = f.b.detach().numpy().copy()
            if f.a is not None:
                out[p + "prob_a%d" % fi] = f.a.detach().numpy().copy()
        for tag, is_val in (("train", False), ("val", True)):
            grid.zero_grad()
            avg, tot = grid.ent_loss(1, is_val=is_val)
            tot.backward()
            out[p + "ent_%s_total" % tag] = np.array([tot.item(), avg.item()], dtype=np.float64)
            g = grid.codebook.grad
            out[p + "ent_%s_grad_codebook" % tag] = (g.numpy().copy() if g is not None
                                                    else np.zeros(grid.codebook.shape, np.float32))
            for fi, f in enumerate((grid.prob_model.f1, grid.prob_model.f2, grid.prob_model.f3, grid.prob_model.f4)):
                for pn in ("h", "b", "a"):
                    prm = getattr(f, pn)
                    if prm is not None:
                        out[p + "ent_%s_grad_%s%d" % (tag, pn, fi)] = (prm.grad.numpy().copy() if prm.grad is not None
                                                                      else np.zeros(prm.shape, np.float32))
        # storage size (empirical entropy branch) and the probability-model variant
        ld, cb = grid.size(use_torchac=False)
        ld2, cb2 = grid.size(use_torchac=False, use_prob_model=True)
        out[p + "size"] = np.array([ld, cb, ld2, cb2], dtype=np.float64)
        cases.append(name)
    for name in cases:  # one file per case: each stays under 1 MB
        path = os.path.join(ROOT, "tests", "golden", "latent_ref_%s.npz" % name)
        np.savez_compressed(path, **{k: v for k, v in out.items() if k.startswith(name + "/")})
        print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
