"""CPU restatement (PyTorch-on-CPU / numpy, float32) of the table-side half of the path:
quantise + decode, the factorized-density bit-rate loss and the storage-size estimate.
TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

Restates, operation by operation and in the reference's order:
  ste_round / decode_single      wisp/models/latent_decoders/basic_latent_decoder.py:28-36,85-90,192-198
  decode_hierarchical            wisp/models/latent_decoders/hierarchical_latent_decoder.py:10-15
                                 (with the last level decoded -- SURVEY Q5 is fenced, not reproduced)
  bitparm / bit_estimator        wisp/models/prob_models/bit_estimator.py:27-44,58-65
  ent_loss                       wisp/models/grids/latent_grid.py:122-136
  size_bits                      wisp/models/grids/latent_grid.py:138-153 (use_torchac=False branch)
  symbol_stream / float_cdf      wisp/models/grids/latent_grid.py:160-169 (what is handed to torchac)
  latent_interpolate             wisp/models/grids/latent_grid.py:355-370 (decode -> repeat -> hashgrid -> [::2])
  sga_quantize                   wisp/models/latent_decoders/basic_latent_decoder.py:183-191 with torch's
                                 RelaxedOneHotCategorical written out (ExpRelaxedCategorical.rsample + exp), the
                                 uniform draws passed in; pinned by tests/golden/sga_ref.npz (make_golden_sga.py)

Pinned against the reference's own Python modules imported under stubs: tests/golden/make_golden.py
writes tests/golden/latent_ref_<case>.npz, tests/test_oracle_golden.py compares.
"""
import numpy as np
import torch
import torch.nn.functional as F

import oracle as _o


def ste_round(w):
    return torch.round(w)


def sga_quantize(w, u, temperature, diff_sampling=True):
    """w [T, C] (requires_grad for the derivative), u [T, C, 2] uniform draws in [0, 1). Returns w_hat [T, C];
    autograd through it gives the reference's gradient (rsample when diff_sampling, else straight-through floor)."""
    eps6 = 1e-6
    wf = torch.floor(w) if diff_sampling else (w + (torch.floor(w) - w).detach())
    wc = wf + 1
    lf = -torch.tanh(torch.clamp(w - wf, min=-1 + eps6, max=1 - eps6)).unsqueeze(-1) / temperature
    lc = -torch.tanh(torch.clamp(wc - w, min=-1 + eps6, max=1 - eps6)).unsqueeze(-1) / temperature
    logits = torch.cat((lf, lc), dim=-1)
    logits = logits - logits.logsumexp(dim=-1, keepdim=True)          # Categorical(logits=...) normalises
    fe = torch.finfo(u.dtype).eps
    uni = u.clamp(min=fe, max=1 - fe)                                  # clamp_probs
    gumbels = -((-(uni.log())).log())
    scores = (logits + gumbels) / temperature
    sample = (scores - scores.logsumexp(dim=-1, keepdim=True)).exp()   # ExpTransform of the log-sample
    if not diff_sampling:
        sample = sample.detach()
    return wf * sample[..., 0] + wc * sample[..., 1]


def decode_single(w_hat, div, scale, shift):
    """(w_hat / div) @ scale + shift, all float32 torch ops on CPU."""
    out = torch.matmul(w_hat / div, scale)
    return out + shift if shift is not None else out


def decode_hierarchical(w_hat, first_idx, divs, scales, shifts):
    T = w_hat.shape[0]
    bounds = list(first_idx) + [T]
    out = torch.empty((T, scales[0].shape[1]), dtype=w_hat.dtype)
    for l in range(len(first_idx)):
        a, b = bounds[l], bounds[l + 1]
        out[a:b] = decode_single(w_hat[a:b], divs[l], scales[l], shifts[l] if shifts is not None else None)
    return out


def bitparm(x, h, b, a, final):
    x = x * F.softplus(h) + b
    if final:
        return torch.sigmoid(x)
    return x + torch.tanh(x) * torch.tanh(a)


def bit_estimator(x, params, num_layers):
    """params: dict f1..f4 -> (h, b, a) tensors of shape [1, C] (a None for f4)."""
    if num_layers > 1:
        x = bitparm(x, *params["f1"], final=False)
    if num_layers > 2:
        x = bitparm(x, *params["f2"], final=False)
    if num_layers > 3:
        x = bitparm(x, *params["f3"], final=False)
    h, b, _ = params["f4"]
    return bitparm(x, h, b, None, final=True)


def ent_loss(codebook, noise, params, num_layers, is_val=False):
    weight = (codebook + noise) if not is_val else torch.round(codebook)
    prob = bit_estimator(weight + 0.5, params, num_layers) - bit_estimator(weight - 0.5, params, num_layers)
    total_bits = torch.sum(torch.clamp(-1.0 * torch.log(prob + 1e-10) / np.log(2.0), 0, 50))
    return total_bits / codebook.shape[0], total_bits


def size_bits(codebook):
    bits = 0
    for dim in range(codebook.size(1)):
        weight = torch.round(codebook[:, dim]).long()
        _, counts = torch.unique(weight, return_counts=True)
        probs = counts / torch.sum(counts)
        info = torch.clamp(-1.0 * torch.log(probs + 1e-10) / np.log(2.0), 0, 1000)
        bits += torch.sum(info * counts).item()
    return bits


def symbol_stream(column):
    """int16 dense ranks and the float32 CDF row the reference feeds torchac."""
    weight = torch.round(column).long()
    weight = weight - weight.min()
    unique_vals, counts = torch.unique(weight, return_counts=True)
    mapping = torch.zeros((weight.max().item() + 1))
    mapping[unique_vals] = torch.arange(unique_vals.size(0)).to(mapping)
    sym = mapping[weight].to(torch.int16)
    cdf = torch.cumsum(counts / counts.sum(), dim=0)
    cdf = torch.cat((torch.Tensor([0.0]), cdf))
    cdf = cdf / cdf[-1:]
    return sym, cdf, unique_vals, counts


def latent_interpolate(coords, codebook, first_idx, resolutions, bitwidth, decode):
    """Decode the whole table, then interpolate with the C oracle (the reference's order).
    `decode` maps the [T, C] latents to the [T, F] table; F == 1 is padded to 2 and strided back."""
    table = decode(codebook).detach()
    rep = table.shape[1] == 1
    if rep:
        table = table.repeat(1, 2)
    feats = _o.forward(np.asarray(coords), table.numpy(), first_idx, resolutions, bitwidth)
    return feats[:, ::2] if rep else feats
