"""The NeRF decoder heads of `NeuralRadianceField.rgba` (wisp/models/nefs/nerf.py:218-233) on the tensor cores.

    heads = NerfHeads(nef.decoder_density, nef.decoder_color)
    density, rgb = heads(feats, vemb, ridx)        # [S, 1], [S, 3]; differentiable in feats and the ten parameters

`feats` [S, IN] is the grid's output (IN = 64 or 96), `vemb` [R, E] one view embedding per ray (the reference's
`view_embedder(-ray_d)`, E <= 32) and `ridx` [S] the sample -> ray map. Operands are rounded to bf16, products and
biases accumulate in fp32 (DESIGN section 9). The modules keep their fp32 parameters; the kernels read them on every
call, so an optimizer step needs no synchronisation with this object. There is no PyTorch fallback.
"""
import ctypes

import torch
import torch.nn as nn

from . import _lib
from ._lib import ERR_INVALID_ARGUMENT, ERR_UNSUPPORTED, ShaciraError

IN_DIMS = (64, 96)
HIDDEN = 128
DENSITY_OUT = 16
MAX_EMB = 32


def _linears(seq, n, what):
    """The Linear layers of a (Linear, ReLU, Linear[, ReLU, Linear]) Sequential with n Linear layers."""
    mods = list(seq) if isinstance(seq, nn.Sequential) else None
    want = 2 * n - 1
    if mods is None or len(mods) != want or any(
            not isinstance(m, nn.Linear if i % 2 == 0 else nn.ReLU) for i, m in enumerate(mods)):
        raise ShaciraError(ERR_UNSUPPORTED, "%s must be nn.Sequential(%s)" % (
            what, ", ".join(["Linear", "ReLU"] * (n - 1) + ["Linear"])))
    lins = mods[0::2]
    for lin in lins:
        if lin.bias is None:
            raise ShaciraError(ERR_UNSUPPORTED, "%s: every Linear needs a bias" % what)
    return lins


def _cuda_i32(t, name):
    if not t.is_cuda:
        raise ShaciraError(ERR_INVALID_ARGUMENT, "%s must be a CUDA tensor (no CPU fallback)" % name)
    if t.dtype not in (torch.int32, torch.int64):
        raise ShaciraError(ERR_INVALID_ARGUMENT, "%s must be an integer tensor, got %s" % (name, t.dtype))
    return t.to(torch.int32).contiguous()


def _param_array(tensors):
    arr = (ctypes.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])
    return arr


class _HeadsFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, heads, feats, vemb, ridx, *params):
        density, rgb = heads._forward(feats, vemb, ridx, params, density_only=False)
        ctx.heads = heads
        ctx.save_for_backward(feats, vemb, ridx, *params)
        return density, rgb

    @staticmethod
    def backward(ctx, g_density, g_rgb):
        feats, vemb, ridx, *params = ctx.saved_tensors
        g_feats, g_params = ctx.heads._backward(feats, vemb, ridx, params, g_density, g_rgb)
        return (None, g_feats, None, None, *g_params)


class NerfHeads:
    """decoder_density: Sequential(Linear(IN, 128), ReLU, Linear(128, 16));
    decoder_color: Sequential(Linear(16 + E, 128), ReLU, Linear(128, 128), ReLU, Linear(128, 3))."""

    def __init__(self, decoder_density, decoder_color):
        d1, d2 = _linears(decoder_density, 2, "decoder_density")
        c1, c2, c3 = _linears(decoder_color, 3, "decoder_color")
        in_dim = d1.in_features
        if in_dim not in IN_DIMS:
            raise ShaciraError(ERR_UNSUPPORTED, "decoder_density input width %d has no kernel (%s)" % (in_dim, IN_DIMS))
        if d1.out_features != HIDDEN or d2.in_features != HIDDEN or d2.out_features != DENSITY_OUT:
            raise ShaciraError(ERR_UNSUPPORTED, "decoder_density must be %d -> %d -> %d, got %d -> %d -> %d" % (
                in_dim, HIDDEN, DENSITY_OUT, in_dim, d1.out_features, d2.out_features))
        emb = c1.in_features - DENSITY_OUT
        if not 0 <= emb <= MAX_EMB:
            raise ShaciraError(ERR_UNSUPPORTED, "decoder_color input width %d: 16 + E with E <= %d" % (
                c1.in_features, MAX_EMB))
        if (c1.out_features, c2.in_features, c2.out_features, c3.in_features, c3.out_features) != (
                HIDDEN, HIDDEN, HIDDEN, HIDDEN, 3):
            raise ShaciraError(ERR_UNSUPPORTED, "decoder_color must be %d -> %d -> %d -> 3" % (
                c1.in_features, HIDDEN, HIDDEN))
        self.linears = (d1, d2, c1, c2, c3)
        self.in_dim, self.emb_dim = in_dim, emb

    def parameters(self):
        return [t for lin in self.linears for t in (lin.weight, lin.bias)]

    def _params(self):
        ps = self.parameters()
        for i, p in enumerate(ps):
            _lib._f32c(p, "parameter %d" % i)
            if not p.is_contiguous():
                raise ShaciraError(ERR_INVALID_ARGUMENT, "parameter %d is not contiguous" % i)
        return ps

    def _check_feats(self, feats):
        feats = _lib._f32c(feats, "feats")
        if feats.dim() != 2 or feats.shape[1] != self.in_dim:
            raise ShaciraError(ERR_INVALID_ARGUMENT, "feats must be [S, %d], got %s" % (self.in_dim, tuple(feats.shape)))
        if feats.data_ptr() % 16:
            feats = feats.clone()
        return feats

    def __call__(self, feats, vemb, ridx):
        """(density [S, 1], rgb [S, 3]); backward through the native kernel."""
        feats = self._check_feats(feats)
        vemb = _lib._f32c(vemb, "vemb")
        if vemb.dim() != 2 or vemb.shape[1] != self.emb_dim:
            raise ShaciraError(ERR_INVALID_ARGUMENT, "vemb must be [R, %d], got %s" % (self.emb_dim, tuple(vemb.shape)))
        ridx = _cuda_i32(ridx, "ridx")
        if ridx.shape != (feats.shape[0],):
            raise ShaciraError(ERR_INVALID_ARGUMENT, "ridx must be [%d], got %s" % (feats.shape[0], tuple(ridx.shape)))
        if feats.device != vemb.device or feats.device != ridx.device:
            raise ShaciraError(ERR_INVALID_ARGUMENT, "feats, vemb and ridx must be on one device")
        return _HeadsFn.apply(self, feats, vemb, ridx, *self._params())

    def density(self, feats):
        """density [S, 1] from the density head alone (no autograd): `render.prune_dense`'s density_fn composed with
        the grid, e.g. `lambda x: heads.density(grid.interpolate(x, 0))`."""
        feats = self._check_feats(feats)
        density, _ = self._forward(feats, None, None, self._params(), density_only=True)
        return density

    def _forward(self, feats, vemb, ridx, params, density_only):
        lib = _lib.load()
        S, dev = feats.shape[0], feats.device
        density = torch.empty((S, 1), dtype=torch.float32, device=dev)
        rgb = None if density_only else torch.empty((S, 3), dtype=torch.float32, device=dev)
        R = 0 if vemb is None else vemb.shape[0]
        pa = _param_array(params)
        with torch.cuda.device(dev):
            _lib._check(lib.shacira_nerf_heads_forward(
                _lib._ptr(feats), S, self.in_dim, HIDDEN, _lib._ptr(vemb), R, self.emb_dim, _lib._ptr(ridx), pa,
                1 if density_only else 0, _lib._ptr(density), _lib._ptr(rgb), _lib._stream()))
        return density, rgb

    def _backward(self, feats, vemb, ridx, params, g_density, g_rgb):
        lib = _lib.load()
        S, dev = feats.shape[0], feats.device
        g_density = torch.zeros((S, 1), dtype=torch.float32, device=dev) if g_density is None else g_density
        g_rgb = torch.zeros((S, 3), dtype=torch.float32, device=dev) if g_rgb is None else g_rgb
        g_density = _lib._f32c(g_density, "grad_density")
        g_rgb = _lib._f32c(g_rgb, "grad_rgb")
        g_feats = torch.empty_like(feats)
        alloc = torch.zeros if S == 0 else torch.empty
        g_params = [alloc(p.shape, dtype=torch.float32, device=dev) for p in params]
        with torch.cuda.device(dev):
            ws_bytes = int(lib.shacira_nerf_heads_workspace_bytes(self.in_dim))
            if ws_bytes < 0:
                _lib._check(_lib.ERR_UNSUPPORTED)
            ws = torch.empty((max(ws_bytes, 1),), dtype=torch.uint8, device=dev)
            _lib._check(lib.shacira_nerf_heads_backward(
                _lib._ptr(feats), S, self.in_dim, HIDDEN, _lib._ptr(vemb), vemb.shape[0], self.emb_dim,
                _lib._ptr(ridx), _param_array(params), _lib._ptr(g_density), _lib._ptr(g_rgb), _lib._ptr(g_feats),
                _param_array(g_params), _lib._ptr(ws), ws_bytes, _lib._stream()))
        return g_feats, g_params
