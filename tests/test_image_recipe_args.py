"""The image-fit recipe's host side: ImageRecipe validation, the schedule formulas, and the argument checks of the
scheduled optimizer launch (shacira_fit_optimizer_step_sched). CPU only: validation runs before any CUDA call."""
import ctypes
import math

import pytest


def test_recipe_defaults_are_kodak_yaml():
    from shacira_b200.image_fit import ImageRecipe
    r = ImageRecipe()
    assert (r.epochs, r.lambda_start, r.lambda_end, r.lambda_kind) == (60_000, 1e-3, 1e-4, "cosine")
    assert (r.temperature_end, r.decay_period, r.div_epochs, r.device_noise) == (0.1, 0.9, (1, 2, 5, 10), True)
    assert (r.lr, r.grid_lr, r.ldec_lr, r.prob_lr, r.weight_decay, r.weight_decay_decoder) == \
        (1e-3, 2e-2, 1e-2, 1e-4, 0.0, 1e-2)
    assert r.switch == 54_000


@pytest.mark.parametrize("kw, code", [
    (dict(epochs=9), "ERR_INVALID_ARGUMENT"),             # fewer epochs than the last div epoch
    (dict(epochs=0, div_epochs=()), "ERR_INVALID_ARGUMENT"),
    (dict(decay_period=0.0), "ERR_INVALID_ARGUMENT"),
    (dict(decay_period=1.5), "ERR_INVALID_ARGUMENT"),
    (dict(temperature_end=0.0), "ERR_INVALID_ARGUMENT"),
    (dict(lambda_kind="linear"), "ERR_UNSUPPORTED"),
])
def test_recipe_validation(lib, kw, code):
    from shacira_b200.image_fit import ImageRecipe
    with pytest.raises(lib.ShaciraError) as e:
        ImageRecipe(**kw)
    assert e.value.code == getattr(lib, code)


def test_recipe_accepts_edge_values():
    from shacira_b200.image_fit import ImageRecipe
    assert ImageRecipe(epochs=10, decay_period=1.0).switch == 10
    assert ImageRecipe(epochs=1, div_epochs=(), lambda_kind="fix").lambda_at(0) == 1e-3


def test_fit_images_rejects_bad_chunk_before_any_work(lib):
    from shacira_b200.image_fit import ImageRecipe, fit_image, fit_images
    with pytest.raises(lib.ShaciraError, match="chunk"):
        fit_image(None, None, None, None, ImageRecipe(epochs=20), chunk=0)
    with pytest.raises(lib.ShaciraError, match="in_flight"):
        fit_images([], ImageRecipe(epochs=20), in_flight=0)


def test_schedule_formulas():
    from shacira_b200.image_fit import ImageRecipe, lambda_at, temperature_at
    n = 60_000
    for it in (0, 1, 2, 17, 29_999, 30_000, 53_999, 54_000, 59_999):
        assert lambda_at(it, n) == 1e-4 + 0.5 * (1e-3 - 1e-4) * (1 + math.cos(math.pi * it / n))
        assert temperature_at(it, n) == max(0.1, math.exp(-math.log(1.0 / 0.1) * (it + 1) / n / 0.9))
    assert lambda_at(0, n) == pytest.approx(1e-3, rel=1e-15)
    assert lambda_at(n, n) == pytest.approx(1e-4, rel=1e-12)
    assert temperature_at(0, n) == pytest.approx(math.exp(-math.log(10.0) / n / 0.9))
    assert temperature_at(54_000, n) == 0.1 and temperature_at(53_998, n) > 0.1   # reaches T_end at decay_period
    assert lambda_at(123, n, start=5e-4, kind="fix") == 5e-4
    r = ImageRecipe(epochs=400, lambda_start=2e-3, temperature_end=0.2, decay_period=0.5)
    assert r.lambda_at(7) == lambda_at(7, 400, 2e-3, 1e-4) and r.temperature_at(7) == temperature_at(7, 400, 0.2, 0.5)


def test_schedule_struct_matches_the_header(lib):
    # 2 x int32 + 4 doubles + pointer + int64 + pointer + int64 on LP64
    assert ctypes.sizeof(lib.FitSchedule) == 8 + 4 * 8 + 4 * 8


FAKE = 256   # never dereferenced: every case fails validation first


def _opt_sched(lib, sched, scale2=FAKE, temperature=FAKE):
    L = lib.load()
    f = ctypes.c_float
    seg = lib.AdamSeg()
    seg.param = seg.grad = seg.exp_avg = seg.exp_avg_sq = FAKE
    seg.n, seg.grad_rows, seg.div_group = 1, 1, 1
    return L.shacira_fit_optimizer_step_sched(
        ctypes.byref(seg), 1, FAKE, FAKE, None, None, scale2, f(1.0), FAKE, FAKE, 1024, f(1e-2), f(0.0), f(0.9), f(0.999),
        f(1e-8), FAKE, FAKE, FAKE, FAKE, None, 1, 1, temperature, 0, 0, None, None, None, None, 0, None, 0, None, None,
        None, None, 0, FAKE, None, sched, None)


def _sched(lib, **kw):
    s = lib.FitSchedule()
    s.num_epochs, s.lambda_kind, s.lambda_start, s.lambda_end = 100, lib.LAMBDA_COSINE, 1e-3, 1e-4
    s.temperature_end, s.decay_period, s.sse, s.count, s.log, s.log_capacity = 0.1, 0.9, FAKE, 3 * 4096, FAKE, 100
    for k, v in kw.items():
        setattr(s, k, v)
    return ctypes.byref(s)


@pytest.mark.parametrize("kw, code, msg", [
    (None, "ERR_INVALID_ARGUMENT", b"descriptor is NULL"),
    (dict(log=None), "ERR_INVALID_ARGUMENT", b"log is NULL"),
    (dict(log_capacity=-1), "ERR_INVALID_ARGUMENT", b"log_capacity -1 < 0"),
    (dict(sse=None), "ERR_INVALID_ARGUMENT", b"sse / count"),
    (dict(num_epochs=0), "ERR_INVALID_ARGUMENT", b"num_epochs"),
    (dict(decay_period=0.0), "ERR_INVALID_ARGUMENT", b"decay_period"),
    (dict(decay_period=1.0 + 1e-12), "ERR_INVALID_ARGUMENT", b"decay_period"),
    (dict(decay_period=float("nan")), "ERR_INVALID_ARGUMENT", b"decay_period"),
    (dict(temperature_end=0.0), "ERR_INVALID_ARGUMENT", b"temperature_end"),
    (dict(temperature_end=-0.1), "ERR_INVALID_ARGUMENT", b"temperature_end"),
    (dict(lambda_kind=7), "ERR_UNSUPPORTED", b"lambda kind"),
    (dict(log=FAKE + 4), "ERR_INVALID_ARGUMENT", b"16-byte aligned"),
])
def test_fit_optimizer_step_sched_validates_the_descriptor(lib, kw, code, msg):
    L = lib.load()
    assert _opt_sched(lib, None if kw is None else _sched(lib, **kw)) == getattr(lib, code)
    assert msg in L.shacira_last_error()


def test_fit_optimizer_step_sched_needs_the_scalars_it_writes(lib):
    L = lib.load()
    assert _opt_sched(lib, _sched(lib), scale2=None) == lib.ERR_INVALID_ARGUMENT
    assert b"scale2" in L.shacira_last_error()
    assert _opt_sched(lib, _sched(lib), temperature=None) == lib.ERR_INVALID_ARGUMENT
