"""One training step of the image INR fit, natively fused (SURVEY section 8 rows f-1 and f-4).

Mirrors `ImageTrainer.step` (wisp/trainers/image_trainer.py:269-359) for the static-coordinate image fit:

    feats = grid.interpolate(coords)            latent_grid.py:340-382   -> tiled forward kernel
    rgb   = decoder_color(feats)                nefs/image.py:109-120,152 \\  fused MLP + MSE kernel
    rgb_loss = ((rgb - gt) ** 2).mean()         image_trainer.py:298-300  /  (value + every gradient)
    ent   = grid.ent_loss(it)[0]                latent_grid.py:122-136   -> fused bit-rate kernel
    loss  = rgb_loss + lambda * ent             image_trainer.py:314-319
    loss.backward(); optimizer.step()           :321-359, parameter groups base_trainer.py:206-266

In PyTorch terms that step is ~50 kernels (autograd glue, gradient scaling passes over the table, one multi-tensor
Adam per group). Here it is TWO launches (+ one 2.4 KB memset) and no autograd:
  * shacira_fit_tile_step -- grid forward + decoder MLP + MSE + grid backward in one tile-resident kernel
    (csrc/fit_kernels.cuh): the [N, 16] feature rows and their gradient never leave the SM;
  * shacira_fit_optimizer_step -- everything table-side in one launch (csrc/optimizer_kernels.cuh): the bit-rate loss of
    the latents (value + gradients; the latents' bit-rate gradient goes straight into the table's Adam, lambda is a device
    scalar), Adam over the table and over all ~20 small tensors with their chain rules, and the NEXT step's SGA sample of
    the freshly updated latents.
Shapes outside the fused kernels' (latent_dim / feature_dim != 1, levels that do not fit a tile, injected SGA draws) keep
the separate launches: tiled forward -> tensor-core MLP -> tiled backward, bit-rate kernel on a forked stream, SGA kernel.
Grid and MLP exchange rows in the plan's tile order (sorted-I/O plan, targets permuted once), and with device_noise=True
the bit-rate noise is drawn in the kernel. The whole step is CUDA-graph capturable; `set_lambda` / `set_temperature` /
`set_sga` / `draw_noise` / `update_div` are the host-side schedule hooks of the trainer (image_trainer.py:131-137,284-296).

The module parameters stay the single source of truth: the kernels read and update the storage of
`grid.codebook`, `grid.latent_dec.layers[0].{scale,shift}`, `grid.prob_model.f*.{h,b,a}` and the MLP in place, so
`grid.interpolate`, `grid.size()`, `state_dict()` etc. see the trained values at any time.

The trainer's schedules can run on the device too (image_trainer.py:113-193): after `set_schedule(recipe)` the optimizer
launch writes the next step's lambda and SGA temperature itself and appends every step's rgb_loss / bits / lambda /
temperature to a device log (`history`), so a CUDA graph of K captured steps is K schedule steps with no host work.
`fit_image` / `fit_images` run the reference's whole recipe (`ImageRecipe`, kodak.yaml) that way.

Model selection and evaluation stay on the device as well (image_trainer.py:173-178,305-310,471-502): with
track_best=True the optimizer launch keeps the parameters of the lowest rgb_loss seen so far (`best_loss`, `best_step`,
`restore_best`), and `render` / `render_image` turn a model of the fused kernel's shape into pixels and its clamped
PSNR in one forward-only kernel (shacira_fit_render).
"""
import ctypes
import dataclasses
import math
import os

import torch

from . import _lib, grid_ops

_LAMBDA_KINDS = {"cosine": _lib.LAMBDA_COSINE, "fix": _lib.LAMBDA_FIX}


def lambda_at(it, num_epochs, start=1e-3, end=1e-4, kind="cosine"):
    """Bit-rate weight lambda before step `it` (0-based) of a `num_epochs` fit (utils/schedulers.py, 'cosine' or 'fix').
    The optimizer launch of a scheduled ImageFitStep evaluates the same expression on the device."""
    if kind == "fix":
        return start
    if kind != "cosine":
        raise _lib.ShaciraError(_lib.ERR_UNSUPPORTED, "unknown lambda schedule %r" % (kind,))
    return end + 0.5 * (start - end) * (1 + math.cos(math.pi * it / num_epochs))


def temperature_at(it, num_epochs, end=0.1, decay_period=0.9):
    """SGA temperature before step `it` (0-based): the reference's DecayScheduler('exp', start 1.0, end) at epoch it + 1
    (utils/schedulers.py:21-23, base_trainer.py:155-157)."""
    return max(end, math.exp(-math.log(1.0 / end) * (it + 1) / num_epochs / decay_period))


@dataclasses.dataclass(frozen=True)
class ImageRecipe:
    """The reference's Kodak training recipe (app/image/configs/kodak.yaml; Adam groups of base_trainer.py:219-239):
    `epochs` full-image steps; lambda from `lambda_start` to `lambda_end` ('cosine') or fixed at `lambda_start` ('fix');
    SGA with temperature 1 -> `temperature_end` while epoch / epochs <= `decay_period`, straight-through rounding after;
    norm='max' div updates before the steps of `div_epochs` (1-based); bit-rate noise drawn on the device."""
    epochs: int = 60_000
    lr: float = 1e-3
    grid_lr: float = 2e-2
    ldec_lr: float = 1e-2
    prob_lr: float = 1e-4
    weight_decay: float = 0.0
    weight_decay_decoder: float = 1e-2
    betas: tuple = (0.9, 0.999)
    eps: float = 1e-8
    lambda_start: float = 1e-3
    lambda_end: float = 1e-4
    lambda_kind: str = "cosine"
    temperature_end: float = 0.1
    decay_period: float = 0.9
    div_epochs: tuple = (1, 2, 5, 10)
    device_noise: bool = True

    def __post_init__(self):
        bad = lambda msg: _lib.ShaciraError(_lib.ERR_INVALID_ARGUMENT, "ImageRecipe: " + msg)
        if int(self.epochs) < 1 or (self.div_epochs and int(self.epochs) < max(self.div_epochs)):
            raise bad("epochs %r: at least 1 and at least the last div epoch %r" % (self.epochs, self.div_epochs))
        if any(int(e) < 1 for e in self.div_epochs):
            raise bad("div epochs count from 1")
        if not 0.0 < float(self.decay_period) <= 1.0:
            raise bad("decay_period %r outside (0, 1]" % (self.decay_period,))
        if not float(self.temperature_end) > 0.0:
            raise bad("temperature_end %r must be > 0" % (self.temperature_end,))
        if self.lambda_kind not in _LAMBDA_KINDS:
            raise _lib.ShaciraError(_lib.ERR_UNSUPPORTED, "ImageRecipe: unknown lambda kind %r" % (self.lambda_kind,))

    @property
    def switch(self):
        """The first straight-through step: SGA while epoch / epochs <= decay_period (image_trainer.py:136-137)."""
        return int(math.floor(self.decay_period * self.epochs))

    def lambda_at(self, it):
        return lambda_at(it, self.epochs, self.lambda_start, self.lambda_end, self.lambda_kind)

    def temperature_at(self, it):
        return temperature_at(it, self.epochs, self.temperature_end, self.decay_period)

    def step_kwargs(self):
        """The ImageFitStep arguments of this recipe."""
        return dict(lr=self.lr, grid_lr=self.grid_lr, ldec_lr=self.ldec_lr, prob_lr=self.prob_lr,
                    weight_decay=self.weight_decay, weight_decay_decoder=self.weight_decay_decoder, betas=self.betas,
                    eps=self.eps, device_noise=self.device_noise)


class ImageFitStep:
    def __init__(self, grid, mlp, coords, target, lr=1e-3, grid_lr=2e-2, ldec_lr=1e-2, prob_lr=1e-4,
                 weight_decay=0.0, weight_decay_decoder=1e-2, betas=(0.9, 0.999), eps=1e-8, device_noise=False,
                 noise_seed=0, track_best=False):
        """`grid`: shacira_b200.grids.LatentGrid (2D, single affine decoder; SGA sampling or STE rounding as the decoder's
        `use_sga` says -- see set_sga / set_temperature); `mlp`:
        nn.Sequential(Linear(L*F,16), ReLU, Linear(16,16), ReLU, Linear(16,3)); coords [N,2], target [N,3].
        Learning rates / weight decays: the reference's parameter groups (base_trainer.py:219-239; kodak.yaml:61-70).
        device_noise=True draws the bit-rate noise inside the kernel (fresh on every step, also under graph replay:
        `draw_noise` is then unnecessary); False reads `self.noise`, which `draw_noise` fills (parity runs).
        track_best=True keeps the state of the lowest rgb_loss inside the optimizer launch (see best_loss / restore_best);
        it needs the one-launch optimizer (not SHACIRA_FIT_OPT_FUSED=0)."""
        dec = grid.latent_dec
        amap = dec.affine_map() if hasattr(dec, "affine_map") else None
        if amap is None or amap[0].shape[0] != 1 or "dft" in dec.layers[0].ldecode_matrix:
            raise _lib.ShaciraError(_lib.ERR_UNSUPPORTED, "ImageFitStep: needs ONE affine 'sq' latent decoder")
        if grid.prob_model is None:
            raise _lib.ShaciraError(_lib.ERR_UNSUPPORTED, "ImageFitStep: needs the bit-rate model (entropy_reg > 0)")
        self.grid, self.mlp = grid, mlp
        self.coords = _lib._f32c(coords, "coords")
        self.target = _lib._f32c(target, "target")
        dev = self.coords.device
        self.dev = dev
        self.n = self.coords.shape[0]
        self.T, self.C = grid.codebook.shape
        self.L = grid.num_lods
        layer = dec.layers[0]
        self.F = layer.scale.shape[1]
        self.fi, _ = _lib._i32_array(grid._first_idx())
        self.rs, _ = _lib._i32_array(grid.resolutions)
        self.bw = int(grid.codebook_bitwidth)
        self.betas, self.eps = betas, float(eps)
        self.grid_lr, self.weight_decay = float(grid_lr), float(weight_decay)
        self.lin = [mlp[0], mlp[2], mlp[4]]
        self.IN, self.H, self.OUT = self.lin[0].in_features, self.lin[0].out_features, self.lin[2].out_features
        if self.IN != self.L * self.F:
            raise _lib.ShaciraError(_lib.ERR_INVALID_ARGUMENT, "MLP input width must be num_lods * feature_dim")
        if self.n < 4096 or self.L % 4:
            raise _lib.ShaciraError(_lib.ERR_UNSUPPORTED, "ImageFitStep: coordinate set / level count outside the tiled path")
        # A plan of its own, in sorted-I/O mode: the step's consumers of the feature rows (per-point MLP, mean loss)
        # do not care about the order of the points, so grid and MLP exchange rows in the plan's tile order (targets
        # permuted once here) and the grid kernels lose their perm -> row dependent loads.
        self.plan = _lib.Plan(self.coords).set_sorted_io(True)
        self.perm = self.plan.perm_tensor()
        self.target = self.target[self.perm].contiguous()
        f32 = dict(dtype=torch.float32, device=dev)
        # density-model parameters live in ONE [4, 3, C] buffer (the kernel's layout); the module's h / b / a become
        # views of it, so nothing is packed per step
        pm = grid.prob_model
        self.prob = torch.zeros((4, 3, self.C), **f32)
        for i, f in enumerate((pm.f1, pm.f2, pm.f3, pm.f4)):
            for k, name in enumerate(("h", "b", "a")):
                p = getattr(f, name, None)
                if p is None:
                    continue
                self.prob[i, k].copy_(p.detach().reshape(-1))
                p.data = self.prob[i, k].view(1, self.C)
        self.num_prob_layers = int(pm.num_layers)
        # step buffers
        self.A = torch.empty((1, self.C, self.F), **f32)
        self.feats = torch.empty((self.n, self.L * self.F), **f32)
        self.gfeat = torch.empty_like(self.feats)
        self.use_bound = self.IN == 16   # the tensor-core kernel
        # one tile-resident kernel for grid forward + MLP / MSE + grid backward where its shapes apply (SHACIRA_FIT_FUSED=0:
        # the three-kernel path, kept for every other shape and as the parity reference of the fused kernel)
        self.opt_fused = os.environ.get("SHACIRA_FIT_OPT_FUSED", "1") != "0"   # one optimizer launch (incl. next SGA sample)
        if track_best and not self.opt_fused:
            raise _lib.ShaciraError(_lib.ERR_UNSUPPORTED, "ImageFitStep: track_best needs the one-launch optimizer "
                                                          "(SHACIRA_FIT_OPT_FUSED=0 is set)")
        self._what_valid = False
        # the bit-rate loss evaluated inside the optimizer launch's table pass (latent_dim 1): no bit-rate launch, no
        # forked stream, the latents' bit-rate gradient never goes through memory
        self.ent_in_opt = self.opt_fused and self.C == 1 and os.environ.get("SHACIRA_FIT_ENT_FUSED", "1") != "0"
        self.fused = (os.environ.get("SHACIRA_FIT_FUSED", "1") != "0" and self.use_bound and self.H == 16 and
                      self.OUT == 3 and self.C == 1 and self.F == 1 and self.L == 16 and amap[0].shape[0] == 1)
        n_par = self.H * self.IN + self.H + self.H * self.H + self.H + self.OUT * self.H + self.OUT
        # double SSE | packed MLP gradients | max |feature gradient| per column (reduced by the MLP kernel; kept behind
        # the gradients so that the call clears everything with one memset)
        self.mlp_out = torch.zeros(2 + n_par + 16, **f32)
        self.gfeat_max = self.mlp_out[2 + n_par:]
        # accumulated into by the backward, cleared by the table's Adam kernel after use: no memset per step
        self.g_grid = torch.zeros((self.T, self.C), **f32)
        self.g_ent = torch.empty((self.T, self.C), **f32)
        self.g_prob = torch.zeros((4, 3, self.C), **f32)
        self.g_dec = torch.zeros((self.L * self.C * self.F + self.L * self.F,), **f32)   # dA rows | dshift rows
        self.bits = torch.zeros((1 + self.L,), dtype=torch.float64, device=dev)
        self.noise = torch.zeros((self.T, self.C), **f32)
        self.lam = torch.zeros((), **f32)
        self.device_noise, self.noise_seed = bool(device_noise), int(noise_seed)
        self.rng_step = torch.zeros((), dtype=torch.int64, device=dev)
        # SGA (basic_latent_decoder.py:183-191): the reference's quantiser until epoch / max_epochs > decay_period
        # (image_trainer.py:136-137). One table-side kernel per step writes w_hat (what the grid kernels interpolate,
        # rounding off) and d w_hat / d w (multiplied into the grid gradient inside the table's Adam kernel).
        self.sga = bool(getattr(dec, "use_sga", False))
        self.diff_sampling = bool(getattr(dec, "diff_sampling", True))
        self.temperature = torch.full((), float(getattr(dec, "temperature", 1.0)), **f32)
        self.w_hat = torch.empty((self.T, self.C), **f32)
        self.dw = torch.empty((self.T, self.C), **f32)
        self.sga_uniforms = None     # [T, C, 2]: injected draws (parity runs); None = drawn in the kernel
        self.sga_rng_step = torch.zeros((), dtype=torch.int64, device=dev)
        self.ent_scratch = torch.zeros(int(_lib.load().shacira_entropy_scratch_bytes(self.C, self.L)),
                                       dtype=torch.uint8, device=dev)
        # Adam state
        self.m_table, self.v_table = torch.zeros_like(grid.codebook.data), torch.zeros_like(grid.codebook.data)
        self.step_table = torch.zeros((), **f32)
        self.step_small = torch.zeros((), **f32)
        self.adam_ticket = torch.zeros((), dtype=torch.int32, device=dev)   # arrival counter of the per-tensor CTAs
        self._keep = []
        self._seg_params = []   # the tensor each Adam segment updates, in segment order (best-state snapshot)
        # the bit-rate kernel depends on nothing but the table: it runs on a forked stream beside the grid / MLP
        # kernels (it is latency bound: 17 us alone) and joins before the optimizer kernels
        self.side = torch.cuda.Stream(device=dev)
        self._forked = torch.cuda.Event()
        segs = []

        def seg(param, grad, n, lr, wd, rows=1, stride=0, scale=None, mul=1.0, div=None, group=1, zero=False):
            m, v = torch.zeros(n, **f32), torch.zeros(n, **f32)
            self._keep += [m, v]
            s = _lib.AdamSeg()
            s.param, s.grad = param.data_ptr(), grad.data_ptr()
            s.exp_avg, s.exp_avg_sq = m.data_ptr(), v.data_ptr()
            s.grad_scale = scale.data_ptr() if scale is not None else None
            s.grad_div = div.data_ptr() if div is not None else None
            s.n, s.grad_rows, s.grad_row_stride, s.div_group = n, rows, stride, group
            s.lr, s.weight_decay, s.grad_mul, s.zero_grad = lr, wd, mul, 1.0 if zero else 0.0
            segs.append(s)
            self._seg_params.append(param)

        packed = self.mlp_out[2:2 + n_par]
        off = 0
        for lin in self.lin:                       # decoder group: lr, weight decay 0 (base_trainer.py:222-224)
            for p in (lin.weight, lin.bias):
                seg(p.data, packed[off:], p.numel(), float(lr), 0.0)
                off += p.numel()
        CF = self.C * self.F
        # latent_dec group (base_trainer.py:225-229): scale = A * div  =>  dscale = (sum_l dA_l) / div
        seg(layer.scale.data, self.g_dec, CF, float(ldec_lr), float(weight_decay_decoder), rows=self.L, stride=CF,
            div=dec.div.data, group=self.F, zero=True)
        self.has_shift = layer.shift is not None
        if self.has_shift:
            seg(layer.shift.data, self.g_dec[self.L * CF:], self.F, float(ldec_lr), float(weight_decay_decoder),
                rows=self.L, stride=self.F, zero=True)
        # prob_model group: lr fixed 1e-4 (base_trainer.py:230-234); gradient = lambda / rows * d(bits)
        used = [0] if self.num_prob_layers > 1 else []
        if self.num_prob_layers > 2:
            used.append(1)
        if self.num_prob_layers > 3:
            used.append(2)
        used.append(3)
        for i, f in zip(range(4), (pm.f1, pm.f2, pm.f3, pm.f4)):
            if i not in used:
                continue                            # never receives a gradient: torch.optim.Adam skips it too
            for k, name in enumerate(("h", "b", "a")):
                p = getattr(f, name, None)
                if p is None or not p.requires_grad:
                    continue
                seg(self.prob[i, k], self.g_prob[i, k], self.C, float(prob_lr), float(weight_decay_decoder),
                    scale=self.lam, mul=1.0 / self.T)
        if len(segs) > _lib.MAX_ADAM_SEGS:
            raise _lib.ShaciraError(_lib.ERR_UNSUPPORTED, "too many small tensors")
        self.segs = (_lib.AdamSeg * len(segs))(*segs)
        self.nseg = len(segs)
        self.layer = layer
        self.refresh_A()
        self.track_best = bool(track_best)
        if self.track_best:
            # best-state snapshot, written by the optimizer launch on improving steps (shacira_fit_snapshot_t)
            self.best_loss_t = torch.full((), float("inf"), **f32)
            self.best_step_t = torch.full((), -1, dtype=torch.int64, device=dev)
            self.best_table = torch.empty_like(grid.codebook.data)
            self.best_segs = [torch.empty_like(p) for p in self._seg_params]
            self.best_div = torch.empty_like(dec.div.data)
            self.best_A = torch.empty_like(self.A)
            snap = _lib.FitSnapshot()
            snap.sse, snap.count = self.mlp_out.data_ptr(), self.n * self.OUT
            snap.best_loss, snap.best_step = self.best_loss_t.data_ptr(), self.best_step_t.data_ptr()
            snap.table, snap.div, snap.A = self.best_table.data_ptr(), self.best_div.data_ptr(), self.best_A.data_ptr()
            for i, b in enumerate(self.best_segs):
                snap.seg_param[i] = b.data_ptr()
            self.snap = snap
        self.sse_u8 = torch.zeros((), dtype=torch.int64, device=dev)
        self.sched = None

    # ---- device-side schedule ---------------------------------------------------------------------
    def set_schedule(self, recipe, log_capacity=None):
        """From the next step on, the optimizer launch advances lambda and the SGA temperature itself (the values of
        recipe.lambda_at / recipe.temperature_at at the step counter) and logs every step (`history`) at its index, for
        the first `log_capacity` steps (default recipe.epochs). set_lambda / set_temperature still overwrite the device
        scalars; the launch replaces them after the next step. Needs the one-launch optimizer. A CUDA graph captured
        before this call keeps the previous schedule and log (kept alive here): re-capture after calling it."""
        if not self.opt_fused:
            raise _lib.ShaciraError(_lib.ERR_UNSUPPORTED, "ImageFitStep: a device-side schedule needs the one-launch "
                                                          "optimizer (SHACIRA_FIT_OPT_FUSED=0 is set)")
        cap = int(recipe.epochs if log_capacity is None else log_capacity)
        if cap < 0:
            raise _lib.ShaciraError(_lib.ERR_INVALID_ARGUMENT, "ImageFitStep.set_schedule: log_capacity < 0")
        if self.sched is not None:
            self._keep.append(self.log)   # a graph captured earlier still writes into the previous log
        self.log = torch.full((max(cap, 1), 4), float("nan"), dtype=torch.float32, device=self.dev)
        sc = _lib.FitSchedule()
        sc.num_epochs, sc.lambda_kind = int(recipe.epochs), _LAMBDA_KINDS[recipe.lambda_kind]
        sc.lambda_start, sc.lambda_end = float(recipe.lambda_start), float(recipe.lambda_end)
        sc.temperature_end, sc.decay_period = float(recipe.temperature_end), float(recipe.decay_period)
        sc.sse, sc.count = self.mlp_out.data_ptr(), self.n * self.OUT
        sc.log, sc.log_capacity = self.log.data_ptr(), cap
        self.sched, self.recipe = sc, recipe
        it = int(self.step_small)
        self.set_lambda(recipe.lambda_at(it))
        self.set_temperature(recipe.temperature_at(it))

    def history(self):
        """The step log of the scheduled steps as float32 device tensors, one entry per step taken (up to the log's
        capacity): rgb_loss (bit for bit rgb_loss()), bits (total_bits()), and the lambda and temperature the step used.
        Reads the step counter on the host."""
        if self.sched is None:
            raise _lib.ShaciraError(_lib.ERR_INVALID_ARGUMENT, "ImageFitStep.history: no schedule (set_schedule)")
        k = min(int(self.step_small), int(self.sched.log_capacity))
        log = self.log[:k]
        return dict(rgb_loss=log[:, 0], bits=log[:, 1], lam=log[:, 2], temperature=log[:, 3])

    # ---- host-side schedule hooks ------------------------------------------------------------
    def refresh_A(self):
        """A = scale / div (latent_decoders.affine_map); call after changing scale or div outside step()."""
        with torch.no_grad():
            self.A.copy_((self.layer.scale.data / self.grid.latent_dec.div.data.unsqueeze(1)).unsqueeze(0))

    def set_lambda(self, value):
        self.lam.fill_(float(value))

    def set_temperature(self, value, refresh=False):
        """SGA temperature of this epoch (image_trainer.py:131-133; base_trainer.py:155-157 builds the schedule). The
        sample of the NEXT step has already been drawn by the previous optimizer launch with the temperature of that
        moment: refresh=True discards it, so the new value applies from the very next step (an epoch-boundary caller);
        without it the new value applies one step later (a per-step schedule under CUDA-graph replay)."""
        self.temperature.fill_(float(value))
        self.grid.latent_dec.temperature = float(value)
        if refresh:
            self._what_valid = False

    def set_sga(self, flag):
        """Switch between SGA and straight-through rounding (the trainer turns SGA off once epoch / max_epochs >
        decay_period). A captured CUDA graph holds the mode it was captured with: re-capture after switching."""
        self.sga = bool(flag)
        self.grid.latent_dec.use_sga = bool(flag)
        self._what_valid = False

    def draw_noise(self, generator=None):
        """U(-0.5, 0.5) per latent (latent_grid.py:128); with a CPU generator the reference's stream."""
        if generator is not None:
            self.noise.copy_(torch.rand((self.T, self.C), generator=generator) - 0.5)
        else:
            self.noise.uniform_(-0.5, 0.5)

    def update_div(self):
        """norm='max' (image_trainer.py:284-296): div = max(|min|, |max|) per latent channel."""
        with torch.no_grad():
            w = self.grid.codebook.data
            self.grid.latent_dec.div.data.copy_(torch.max(torch.abs(w.min(dim=0)[0]), torch.abs(w.max(dim=0)[0])))
        self.refresh_A()

    # ---- the step --------------------------------------------------------------------------------
    def step(self):
        lib, P, chk = _lib.load(), _lib._ptr, _lib._check
        g, dec = self.grid, self.grid.latent_dec
        lat = g.codebook.data
        shift = self.layer.shift.data if self.has_shift else None
        lin = self.lin
        with torch.cuda.device(self.dev):
            st = _lib._stream()
            cur = torch.cuda.current_stream(self.dev)
            self._forked.record(cur)   # the table as the previous optimizer launch left it
            q_lat, rflag, gmul = lat, 1, None
            # SGA sample of this step: normally already there -- the previous step's optimizer launch sampled the latents it
            # had just updated (shacira_fit_optimizer_step); drawn here on the first step, after set_sga / a refreshing
            # set_temperature, and whenever the draws are injected (parity runs)
            prefetch = self.sga and self.opt_fused and self.sga_uniforms is None
            if self.sga:
                if not (prefetch and self._what_valid):
                    chk(lib.shacira_sga_quantize(P(lat), P(self.sga_uniforms), self.T * self.C, P(self.temperature),
                                                 1 if self.diff_sampling else 0, self.noise_seed + 0x5A17,
                                                 P(self.sga_rng_step), P(self.w_hat), P(self.dw), st))
                q_lat, rflag, gmul = self.w_hat, 0, self.dw
            CF = self.C * self.F
            if not self.has_shift:
                self.g_dec[self.L * CF:].zero_()   # no segment consumes (and clears) the shift rows
            fused_done = False
            if self.fused:
                # grid forward + MLP / MSE + grid backward as ONE tile-resident kernel (csrc/fit_kernels.cuh): the feature
                # rows and their gradient never leave the SM
                rc = lib.shacira_fit_tile_step(self.plan.handle, P(q_lat), self.fi, self.rs, self.L, self.bw, rflag,
                                               P(self.A), P(shift), P(self.target), P(lin[0].weight.data),
                                               P(lin[0].bias.data), P(lin[1].weight.data), P(lin[1].bias.data),
                                               P(lin[2].weight.data), P(lin[2].bias.data), self.T, P(self.g_grid),
                                               P(self.g_dec), P(self.g_dec[self.L * CF:]), P(self.mlp_out), st)
                if rc == _lib.ERR_UNSUPPORTED:
                    self.fused = False     # e.g. a level whose node box does not fit a tile: the three-kernel path
                else:
                    chk(rc)
                    fused_done = True
            if not fused_done:
                chk(lib.shacira_latent_forward_planned(self.plan.handle, P(q_lat), self.fi, self.rs, self.L, self.bw, self.C,
                                                       self.F, rflag, P(self.A), P(shift), 0, P(self.feats), st))
                # the MLP kernel reduces max |feature gradient| per column on the way; the tiled backward takes its
                # fixed-point scales from that bound and skips its own pass over the gradient rows
                bound = P(self.gfeat_max) if self.use_bound else None
                chk(lib.shacira_mlp_mse_step_bounded(P(self.feats), P(self.target), self.n, self.IN, self.H, self.OUT,
                                                     P(lin[0].weight.data), P(lin[0].bias.data), P(lin[1].weight.data),
                                                     P(lin[1].bias.data), P(lin[2].weight.data), P(lin[2].bias.data),
                                                     P(self.gfeat), None, P(self.mlp_out), bound, st))
                chk(lib.shacira_latent_backward_planned_bounded(self.plan.handle, P(self.gfeat), P(q_lat), self.fi, self.rs,
                                                                self.L, self.bw, self.C, self.F, rflag, P(self.A), 0, self.T, 0,
                                                                P(self.g_grid), P(self.g_dec), P(self.g_dec[self.L * CF:]),
                                                                bound, st))
            # The bit-rate loss: normally evaluated inside the optimizer launch's table pass (ent_in_opt). Otherwise its own
            # kernel on a forked stream, launched AFTER the tile kernel (it only depends on the table).
            ent_folded = self.ent_in_opt and self.opt_fused
            if not ent_folded:
                self.side.wait_event(self._forked)
                with torch.cuda.stream(self.side):
                    if self.device_noise:
                        chk(lib.shacira_entropy_bits_rng(P(lat), self.noise_seed, P(self.rng_step), self.T, self.C,
                                                         P(self.prob), self.num_prob_layers, self.fi, self.L, P(self.bits),
                                                         P(self.g_ent), P(self.g_prob), P(self.ent_scratch),
                                                         self.ent_scratch.numel(), _lib._stream()))
                    else:
                        chk(lib.shacira_entropy_bits(P(lat), P(self.noise), self.T, self.C, P(self.prob),
                                                     self.num_prob_layers, self.fi, self.L, P(self.bits), P(self.g_ent),
                                                     P(self.g_prob), P(self.ent_scratch), self.ent_scratch.numel(),
                                                     _lib._stream()))
                cur.wait_stream(self.side)
            self._optimize(prefetch, gmul, ent_folded, st)

    def _optimize(self, prefetch, gmul, ent_folded, st):
        """The optimizer side of the step (one launch unless SHACIRA_FIT_OPT_FUSED=0)."""
        lib, P, chk = _lib.load(), _lib._ptr, _lib._check
        dec, lat = self.grid.latent_dec, self.grid.codebook.data
        if self.opt_fused:
            # ONE optimizer launch: small tensors + table Adam + the next step's SGA sample (csrc/optimizer_kernels.cuh)
            args = [ctypes.cast(self.segs, ctypes.c_void_p), self.nseg, P(lat), P(self.g_grid),
                    P(gmul), None if ent_folded else P(self.g_ent), P(self.lam),
                    1.0 / self.T, P(self.m_table),
                    P(self.v_table), self.T * self.C, self.grid_lr, self.weight_decay,
                    self.betas[0], self.betas[1], self.eps, P(self.step_small),
                    P(self.step_table), P(self.layer.scale.data), P(dec.div.data), P(self.A),
                    self.C, self.F, P(self.temperature), 1 if self.diff_sampling else 0,
                    self.noise_seed + 0x5A17, P(self.sga_rng_step),
                    P(self.w_hat) if prefetch else None, P(self.dw) if prefetch else None,
                    P(self.prob) if ent_folded else None, self.num_prob_layers,
                    None if self.device_noise else P(self.noise), self.noise_seed,
                    P(self.rng_step), P(self.bits), P(self.g_prob), P(self.ent_scratch),
                    self.ent_scratch.numel(), P(self.adam_ticket)]
            if self.sched is not None:   # the same launch, advancing lambda / temperature and logging the step
                chk(lib.shacira_fit_optimizer_step_sched(*args, ctypes.byref(self.snap) if self.track_best else None,
                                                         ctypes.byref(self.sched), st))
            elif self.track_best:   # the same launch, snapshotting the parameters of an improving step
                chk(lib.shacira_fit_optimizer_step_best(*args, ctypes.byref(self.snap), st))
            else:
                chk(lib.shacira_fit_optimizer_step(*args, st))
            self._what_valid = prefetch
        else:
            chk(lib.shacira_adam_step_sum_mul(P(lat), P(self.g_grid), P(gmul), P(self.g_ent), P(self.lam), 1.0 / self.T,
                                              P(self.m_table), P(self.v_table), self.T * self.C, self.grid_lr,
                                              self.betas[0], self.betas[1], self.eps, self.weight_decay,
                                              P(self.step_table), 0, 1, st))
            chk(lib.shacira_multi_adam_step(ctypes.cast(self.segs, ctypes.c_void_p), self.nseg, self.betas[0],
                                            self.betas[1], self.eps, P(self.step_small), P(self.step_table),
                                            P(self.layer.scale.data), P(dec.div.data), P(self.A), self.C, self.F,
                                            P(self.adam_ticket), st))
            self._what_valid = False

    # ---- results of the last step (device tensors; reading them synchronises) -------------------
    def rgb_loss(self):
        return (self.mlp_out[:2].view(torch.float64)[0] / (self.n * self.OUT)).to(torch.float32)

    def total_bits(self):
        return self.bits[0].to(torch.float32)

    # ---- best state (track_best=True) --------------------------------------------------------------
    def _need_best(self):
        if not self.track_best:
            raise _lib.ShaciraError(_lib.ERR_INVALID_ARGUMENT, "ImageFitStep: constructed without track_best=True")

    def best_loss(self):
        """Lowest rgb_loss() over the steps so far (+inf before the first step): float32 device scalar."""
        self._need_best()
        return self.best_loss_t.clone()

    def best_step(self):
        """0-based index of the step (call of step()) that produced best_loss(); -1 before the first step."""
        self._need_best()
        return self.best_step_t.clone()

    def restore_best(self):
        """Copy the best state into the module parameters in place: latent table, MLP, latent decoder, density model,
        div and A, as they were when that step's forward ran (the reference reloads its best model, not the optimizer
        state: the Adam moments stay as they are). Reads best_step() on the host."""
        self._need_best()
        if int(self.best_step_t) < 0:
            raise _lib.ShaciraError(_lib.ERR_INVALID_ARGUMENT, "ImageFitStep.restore_best: no step has been taken")
        with torch.no_grad():
            self.grid.codebook.data.copy_(self.best_table)
            for p, b in zip(self._seg_params, self.best_segs):
                p.copy_(b)
            self.grid.latent_dec.div.data.copy_(self.best_div)
            self.A.copy_(self.best_A)
        self._what_valid = False   # the prefetched SGA sample belongs to the replaced latents

    # ---- evaluation ------------------------------------------------------------------------------------
    def render(self, target=True):
        """(rgb [N, 3] in the caller's coordinate order, clamped PSNR as a float64 device scalar or None) of the current
        parameters, rounding the latents (the stored model is integers): one kernel over the step's own plan."""
        rgb = torch.empty((self.n, self.OUT), dtype=torch.float32, device=self.dev)
        with torch.cuda.device(self.dev):
            _render(self.plan, self.grid.codebook.data, self.fi, self.rs, self.L, self.bw, self.A,
                    self.layer.shift.data if self.has_shift else None, self.lin, rgb,
                    self.target if target else None, self.sse_u8)
            out = torch.empty_like(rgb)
            out[self.perm] = rgb       # tile order -> original order
        return out, (_psnr(self.sse_u8, self.n * self.OUT) if target else None)

    def close(self):
        if self.plan is not None:
            self.plan.close()
            self.plan = None


def _render(plan, latents, fi, rs, L, bw, A, shift, lin, rgb, target, sse):
    P = _lib._ptr
    _lib._check(_lib.load().shacira_fit_render(plan.handle, P(latents), fi, rs, L, bw, P(A), P(shift),
                                               P(lin[0].weight.data), P(lin[0].bias.data), P(lin[1].weight.data),
                                               P(lin[1].bias.data), P(lin[2].weight.data), P(lin[2].bias.data), P(rgb),
                                               P(target), P(sse) if target is not None else None, _lib._stream()))


def _psnr(sse, count):
    """clamped_psnr of wisp/ops/image/metrics.py:39-57 from the integer uint8 SSE (device float64 scalar)."""
    mse = torch.clamp(sse.to(torch.float64) / count, min=1e-12)
    return 20.0 * math.log10(255.0) - 10.0 * torch.log10(mse)


def _renders(grid, mlp):
    """True for a model of the fused fit kernel's shape (what render_image / shacira_fit_render take)."""
    dec = grid.latent_dec
    amap = dec.affine_map() if hasattr(dec, "affine_map") else None
    lin = [mlp[0], mlp[2], mlp[4]] if len(mlp) == 5 else None
    return not (amap is None or amap[0].shape[0] != 1 or "dft" in getattr(dec.layers[0], "ldecode_matrix", "") or
                grid.resolution_dim != 2 or grid.num_lods != 16 or tuple(grid.codebook.shape[1:]) != (1,) or
                tuple(amap[0].shape) != (1, 1, 1) or lin is None or
                [(l.in_features, l.out_features) for l in lin] != [(16, 16), (16, 16), (16, 3)])


def render_image(grid, mlp, coords, target=None):
    """mlp(grid.interpolate(coords)) for a model of the fused fit kernel's shape -- 2D LatentGrid with 16 levels,
    latent_dim = feature_dim = 1, one affine 'sq' latent decoder, MLP 16 -> 16 -> 16 -> 3 -- in one forward-only kernel
    with the latents rounded: a trained or a decoded codec model, on any coordinate set (e.g. a 2x upsampled pixel
    grid). Returns (rgb [N, 3] in the order of `coords`, clamped PSNR against `target` [N, 3] as a float64 device
    scalar, or None without a target). Other shapes raise ShaciraError (use mlp(grid.interpolate(coords)))."""
    if not _renders(grid, mlp):
        raise _lib.ShaciraError(_lib.ERR_UNSUPPORTED, "render_image: needs the fused fit kernel's model shape")
    lin = [mlp[0], mlp[2], mlp[4]]
    coords = _lib._f32c(coords, "coords")
    n = coords.shape[0]
    if coords.dim() != 2 or coords.shape[1] != 2:
        raise _lib.ShaciraError(_lib.ERR_INVALID_ARGUMENT, "render_image: coords must be [N, 2]")
    if target is not None:
        target = _lib._f32c(target, "target")
        if tuple(target.shape) != (n, 3):
            raise _lib.ShaciraError(_lib.ERR_INVALID_ARGUMENT, "render_image: target must be [N, 3]")
    # the cached plan of these coordinates; small sets get a plan of their own with small tiles, so that every level's
    # node box fits a tile's shared memory
    plan = grid_ops.plan_for(coords) if coords.shape[0] >= grid_ops.PLAN_MIN_POINTS else None
    if plan is None:
        plan = _lib.Plan(coords, tile_points=32)
    fi, _ = _lib._i32_array(grid._first_idx())
    rs, L = _lib._i32_array(grid.resolutions)
    A, shift = grid.latent_dec.affine_map()
    with torch.no_grad():
        A = A.detach().contiguous()
        shift = shift.detach().contiguous() if shift is not None else None
    rgb = torch.empty((n, 3), dtype=torch.float32, device=coords.device)
    sse = torch.zeros((), dtype=torch.int64, device=coords.device) if target is not None else None
    with torch.cuda.device(coords.device):
        _render(plan, _lib._f32c(grid.codebook.data, "codebook"), fi, rs, L, int(grid.codebook_bitwidth), A, shift, lin,
                rgb, target, sse)
    return rgb, (_psnr(sse, n * 3) if target is not None else None)


def _clamped_psnr(pred, target):
    """clamped_psnr (wisp/ops/image/metrics.py:39-57) of a prediction against its target: float64 device scalar."""
    q = lambda v: (torch.clamp(v, 0, 1) * 255).to(torch.uint8).to(torch.int64)
    return _psnr(((q(pred) - q(target)) ** 2).sum(), pred.numel())


def fit_image(grid, mlp, coords, target, recipe=ImageRecipe(), chunk=100, noise_seed=0):
    """Fit one image with the reference's training recipe (ImageTrainer, image_trainer.py:113-193,269-359,471-514):
    fit_images with one fit in flight. Returns its result dict (see fit_images)."""
    return fit_images([(grid, mlp, coords, target)], recipe, in_flight=1, chunk=chunk, noise_seeds=[noise_seed])[0]


def fit_images(fits, recipe=ImageRecipe(), in_flight=3, chunk=100, noise_seeds=None):
    """Independent fits [(grid, mlp, coords, target), ...] with `recipe`, `in_flight` at a time on one stream and one set
    of CUDA graphs each (independent fits overlap each other's latency). Every model ImageFitStep takes is accepted.

    Each fit runs an ImageFitStep with track_best and the recipe's device-side schedule: the first max(div_epochs) steps
    (at least one) eagerly, with update_div before the steps of div_epochs; then the SGA phase and, from step floor(decay_period x
    epochs), the straight-through phase, each as replays of one captured graph of `chunk` steps plus one of the
    remainder. The best state is restored into the modules at the end.

    Returns one dict per fit: best_step, best_loss (lowest rgb_loss and its 0-based step), psnr (clamped PSNR of the best
    state: render_image where the model has the fused shape, mlp(grid.interpolate(coords)) otherwise), blob
    (codec.encode_model), size (codec.size_report: reference-formula and file bpp), history (ImageFitStep.history,
    device tensors), steps and device_ms per phase ('eager', 'sga', 'ste': CUDA-event time on the fit's stream)."""
    from . import codec
    if int(chunk) < 1:
        raise _lib.ShaciraError(_lib.ERR_INVALID_ARGUMENT, "fit_images: chunk %r < 1" % (chunk,))
    if int(in_flight) < 1:
        raise _lib.ShaciraError(_lib.ERR_INVALID_ARGUMENT, "fit_images: in_flight %r < 1" % (in_flight,))
    fits = list(fits)
    seeds = list(noise_seeds) if noise_seeds is not None else list(range(len(fits)))
    if len(seeds) != len(fits):
        raise _lib.ShaciraError(_lib.ERR_INVALID_ARGUMENT, "fit_images: one noise seed per fit")
    out = []
    for g0 in range(0, len(fits), int(in_flight)):
        runs = []
        try:
            for f, s in zip(fits[g0:g0 + int(in_flight)], seeds[g0:g0 + int(in_flight)]):
                runs.append(_RecipeFit(*f, recipe, s))
            _run_recipe(runs, recipe, int(chunk))
            out += [r.result(codec) for r in runs]
        finally:
            for r in runs:
                r.fs.close()
    return out


class _RecipeFit:
    """One fit of fit_images: its ImageFitStep, stream, and per-phase events."""

    def __init__(self, grid, mlp, coords, target, recipe, noise_seed):
        self.grid, self.mlp, self.coords, self.target = grid, mlp, coords, target
        self.fs = ImageFitStep(grid, mlp, coords, target, noise_seed=noise_seed, track_best=True, **recipe.step_kwargs())
        self.fs.set_sga(recipe.switch > 0)
        self.fs.set_schedule(recipe)
        self.stream = torch.cuda.Stream(device=self.fs.dev)
        self.events = {}
        self.steps = {}

    def mark(self, phase, end):
        ev = torch.cuda.Event(enable_timing=True)
        ev.record(self.stream)
        self.events.setdefault(phase, [None, None])[1 if end else 0] = ev

    def capture(self, k):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=self.stream):
            for _ in range(k):
                self.fs.step()
        return g

    def result(self, codec):
        fs = self.fs
        if fs.sga:
            fs.set_sga(False)   # evaluate the rounded model (decay_period = 1 never reaches the STE phase)
        fs.restore_best()
        with torch.no_grad():
            if _renders(self.grid, self.mlp):
                psnr = render_image(self.grid, self.mlp, self.coords, self.target)[1]
            else:
                psnr = _clamped_psnr(self.mlp(self.grid.interpolate(self.coords, 0)), self.target)
        blob = codec.encode_model(self.grid, self.mlp)
        return dict(best_step=int(fs.best_step()), best_loss=float(fs.best_loss()), psnr=float(psnr), blob=blob,
                    size=codec.size_report(self.grid, self.mlp, blob, self.coords.shape[0]),
                    history={k: v.clone() for k, v in fs.history().items()}, steps=dict(self.steps),
                    device_ms={p: e[0].elapsed_time(e[1]) for p, e in self.events.items()})


def _run_recipe(runs, recipe, chunk):
    epochs, switch = recipe.epochs, recipe.switch
    # at least one eager step: it draws the first SGA sample, so that every captured step takes the one the previous
    # optimizer launch drew (as the host-driven loop does) instead of redrawing it
    eager = max(1, min(max(recipe.div_epochs, default=0), epochs))
    torch.cuda.synchronize()
    for r in runs:
        r.mark("eager", False)
    for it in range(eager):
        for r in runs:
            with torch.cuda.stream(r.stream):
                if it == switch:
                    r.fs.set_sga(False)
                if it + 1 in recipe.div_epochs:
                    r.fs.update_div()
                r.fs.step()
    for r in runs:
        r.mark("eager", True)
        r.steps["eager"] = eager
    for phase, a, b in (("sga", eager, switch), ("ste", max(eager, switch), epochs)):
        if b <= a:
            continue
        full, rem = divmod(b - a, chunk)
        for r in runs:
            if phase == "ste" and r.fs.sga:
                r.fs.set_sga(False)   # a captured graph holds its quantiser
        # capture synchronises the device; it records the steps without running them
        graphs = [(r.capture(chunk) if full else None, r.capture(rem) if rem else None) for r in runs]
        for r in runs:
            r.mark(phase, False)
        for _ in range(full):
            for r, (g, _g) in zip(runs, graphs):
                with torch.cuda.stream(r.stream):
                    g.replay()
        for r, (_g, g) in zip(runs, graphs):
            if g is not None:
                with torch.cuda.stream(r.stream):
                    g.replay()
        for r in runs:
            r.mark(phase, True)
            r.steps[phase] = b - a
    torch.cuda.synchronize()
