"""NerfHeads layout checks and the C entries' argument errors. CPU only: every check runs before any CUDA call."""
import ctypes

import pytest
import torch
import torch.nn as nn


def _heads(in_dim=64, emb=27, hidden=128, dout=16):
    dd = nn.Sequential(nn.Linear(in_dim, hidden), nn.ReLU(), nn.Linear(hidden, dout))
    dc = nn.Sequential(nn.Linear(16 + emb, hidden), nn.ReLU(), nn.Linear(hidden, hidden), nn.ReLU(),
                       nn.Linear(hidden, 3))
    return dd, dc


def test_supported_layouts_are_accepted(lib):
    from shacira_b200.nerf_heads import NerfHeads
    for in_dim in (64, 96):
        for emb in (0, 27, 32):
            h = NerfHeads(*_heads(in_dim, emb))
            assert (h.in_dim, h.emb_dim) == (in_dim, emb)
            assert len(h.parameters()) == 10


@pytest.mark.parametrize("kw", [dict(in_dim=32), dict(in_dim=128), dict(emb=33), dict(hidden=64), dict(dout=8)])
def test_unsupported_widths_raise(lib, kw):
    from shacira_b200.nerf_heads import NerfHeads
    with pytest.raises(lib.ShaciraError) as e:
        NerfHeads(*_heads(**kw))
    assert e.value.code == lib.ERR_UNSUPPORTED


def test_other_layouts_raise(lib):
    from shacira_b200.nerf_heads import NerfHeads
    dd, dc = _heads()
    bad = [
        (nn.Sequential(nn.Linear(64, 128), nn.Tanh(), nn.Linear(128, 16)), dc),
        (nn.Sequential(nn.Linear(64, 128), nn.ReLU(), nn.Linear(128, 128), nn.ReLU(), nn.Linear(128, 16)), dc),
        (dd, nn.Sequential(nn.Linear(43, 128), nn.ReLU(), nn.Linear(128, 3))),
        (dd, nn.Sequential(nn.Linear(43, 128), nn.ReLU(), nn.Linear(128, 128, bias=False), nn.ReLU(),
                           nn.Linear(128, 3))),
        ([dd[0], dd[1], dd[2]], dc),
    ]
    for a, b in bad:
        with pytest.raises(lib.ShaciraError):
            NerfHeads(a, b)


def test_cpu_and_non_fp32_inputs_raise(lib):
    from shacira_b200.nerf_heads import NerfHeads
    h = NerfHeads(*_heads())
    with pytest.raises(lib.ShaciraError, match="CUDA tensor"):
        h(torch.zeros(4, 64), torch.zeros(1, 27), torch.zeros(4, dtype=torch.int32))
    with pytest.raises(lib.ShaciraError, match="CUDA tensor"):
        h.density(torch.zeros(4, 64))
    with pytest.raises(lib.ShaciraError, match="CUDA tensor"):
        h.density(torch.zeros(4, 64, dtype=torch.float16))


P = ctypes.c_void_p


def _params(n=10, null_at=None):
    return (P * n)(*[None if i == null_at else 16 * (i + 1) for i in range(n)])


def test_forward_argument_errors_return_codes(lib):
    L = lib.load()
    ok = dict(feats=P(256), n=1000, in_dim=64, hidden=128, vemb=P(256), R=10, E=27, ridx=P(256), params=_params(),
              donly=0, density=P(256), rgb=P(256))

    def call(**kw):
        a = dict(ok, **kw)
        return L.shacira_nerf_heads_forward(a["feats"], a["n"], a["in_dim"], a["hidden"], a["vemb"], a["R"], a["E"],
                                            a["ridx"], a["params"], a["donly"], a["density"], a["rgb"], None)

    assert call(n=-1) == lib.ERR_INVALID_ARGUMENT
    assert call(in_dim=48) == lib.ERR_UNSUPPORTED and b"in_dim" in L.shacira_last_error()
    assert call(hidden=64) == lib.ERR_UNSUPPORTED and b"hidden_dim" in L.shacira_last_error()
    assert call(E=33) == lib.ERR_UNSUPPORTED and b"emb_dim" in L.shacira_last_error()
    assert call(E=-1) == lib.ERR_UNSUPPORTED
    assert call(R=-1) == lib.ERR_INVALID_ARGUMENT
    assert call(params=None) == lib.ERR_INVALID_ARGUMENT
    assert call(params=_params(null_at=7)) == lib.ERR_INVALID_ARGUMENT and b"params[7]" in L.shacira_last_error()
    assert call(feats=None) == lib.ERR_INVALID_ARGUMENT
    assert call(density=None) == lib.ERR_INVALID_ARGUMENT
    assert call(rgb=None) == lib.ERR_INVALID_ARGUMENT
    assert call(ridx=None) == lib.ERR_INVALID_ARGUMENT
    assert call(vemb=None) == lib.ERR_INVALID_ARGUMENT
    assert call(feats=P(260)) == lib.ERR_INVALID_ARGUMENT and b"aligned" in L.shacira_last_error()
    # the density head alone reads none of the colour head's arguments
    assert call(donly=1, params=_params(4), rgb=None, ridx=None, vemb=None, n=0, E=99) == lib.OK
    # empty input is a successful no-op
    assert call(n=0, feats=None, density=None, rgb=None) == lib.OK


def test_backward_argument_errors_return_codes(lib):
    L = lib.load()
    ws = int(L.shacira_nerf_heads_workspace_bytes(96))
    assert ws > 0 and ws % 4 == 0
    assert L.shacira_nerf_heads_workspace_bytes(80) < 0
    ok = dict(feats=P(256), n=1 << 19, in_dim=96, hidden=128, vemb=P(256), R=10, E=27, ridx=P(256), params=_params(),
              gd=P(256), grgb=P(256), gfeats=P(256), gparams=_params(), ws=P(256), ws_bytes=ws)

    def call(**kw):
        a = dict(ok, **kw)
        return L.shacira_nerf_heads_backward(a["feats"], a["n"], a["in_dim"], a["hidden"], a["vemb"], a["R"], a["E"],
                                             a["ridx"], a["params"], a["gd"], a["grgb"], a["gfeats"], a["gparams"],
                                             a["ws"], a["ws_bytes"], None)

    assert call(in_dim=100) == lib.ERR_UNSUPPORTED
    assert call(hidden=256) == lib.ERR_UNSUPPORTED
    assert call(E=40) == lib.ERR_UNSUPPORTED
    assert call(n=-5) == lib.ERR_INVALID_ARGUMENT
    assert call(gparams=_params(null_at=9)) == lib.ERR_INVALID_ARGUMENT and b"grad_params[9]" in L.shacira_last_error()
    assert call(gparams=None) == lib.ERR_INVALID_ARGUMENT
    for k in ("feats", "ridx", "gd", "grgb", "gfeats", "vemb"):
        assert call(**{k: None}) == lib.ERR_INVALID_ARGUMENT, k
    assert call(gfeats=P(264)) == lib.ERR_INVALID_ARGUMENT
    assert call(ws=None) == lib.ERR_INVALID_ARGUMENT and b"workspace" in L.shacira_last_error()
    assert call(ws_bytes=ws - 4) == lib.ERR_INVALID_ARGUMENT and b"workspace" in L.shacira_last_error()
    assert call(n=0, feats=None, gd=None, grgb=None, gfeats=None, ws=None, ws_bytes=0) == lib.OK
