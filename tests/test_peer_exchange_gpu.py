"""The peer-memory exchange (csrc/peer_kernels.cuh, peer_allreduce_kernel<N, ADAM>) at every compiled world size
N in {2, 4, 8}, plain and Adam-fused, with N ranks driven from one process.

On one device the N ranks are N arenas on cuda:0 whose kernels are launched on N streams and meet at the barriers.
Their grids are sized as launch_peer sizes them, and every case asserts that all N grids fit on the device at once:
the barriers spin (bounded at about 4 s), so a rank whose kernel could not start would stall the others.
With two GPUs that have peer access, the NeRF-scale arena runs once across the two devices.

The plain exchange adds in rank order, ((x0 + x1) + x2) + ..., and stores the same sum into every arena: the result
is compared bit for bit with the same fp32 sum formed by torch on the device.

The Adam-fused pass is compared with a float64 Adam run on the host and fed the same fp32 gradient sum. The oracle
uses the fp32-rounded hyperparameters, float(np.float32(0.999)) and so on: every Adam kernel of this library takes
its betas, lr, eps and weight decay as `float` and forms 1 - powf(beta, t) in fp32. 0.999f is off from 0.999 by
about 1.3e-5 relative in 1 - beta2 at t = 1, so an oracle with the double literals would differ by about 6e-6
relative in the step size. That is a convention, not a kernel error. The per-element tolerances are derived from
the kernel's operations (see _AdamOracle), not tuned; every case prints its worst error-to-bound ratio.

The argument checks of shacira_peer_allreduce_adam at the end need no GPU: validation rejects those calls before
any CUDA call or launch.
"""
import ctypes
import math

import numpy as np
import pytest
import torch

U = 2.0 ** -24                   # unit roundoff of fp32 (round to nearest)
PEER_THREADS = 512               # kPeerThreads (peer_kernels.cuh): float4 pieces per CTA-stride
PEER_CTAS_PER_SM = 2             # kPeerBlocksPerSm (peer_capi.cu): the grid's cap
SMALL = [(16, 1, 4), (16, 4), (4, 3, 1), (1,)]   # the NeRF path's decoder / density-model gradients
NERF_ROWS = 6098925              # the NeRF latent table (benchmarks/peer_check.py)
FAKE = ctypes.c_void_p(256)      # never dereferenced: every argument case fails validation first


def _pieces(shape):
    """float4 pieces a tensor takes in an arena (PeerArena pads every tensor to a multiple of 4 floats)."""
    return (math.prod(shape) + 3) // 4


def _per(n4, world):
    """float4 pieces of one rank's slice: the exchange gives rank r the pieces [r * per, (r + 1) * per)."""
    return -(-n4 // world)


def _grid(numel, world, sms):
    """CTAs of one rank's kernel, exactly as launch_peer sizes them."""
    blocks = -(-_per(numel // 4, world) // PEER_THREADS)
    return max(1, min(blocks, PEER_CTAS_PER_SM * sms))


def _locate(j, per):
    return "element %d (piece %d, in the slice of rank %d)" % (j, j // 4, (j // 4) // per)


def _bits(t):
    """An fp32 tensor's bit patterns: equality on them also tells -0.0 from 0.0 and compares NaNs."""
    return t.view(torch.int32)


def _rank_sum(xs):
    """((x0 + x1) + x2) + ... in fp32 on the device: the exchange adds in this order, so the comparison is exact."""
    s = xs[0].clone()
    for x in xs[1:]:
        s = s + x.to(s.device)
    return s


def _wide_values(rng, n):
    """n fp32 values whose magnitudes span 1e-6 .. 1e6, with random signs, exact zeros and -0.0 among them."""
    x = rng.choice([-1.0, 1.0], n) * 10.0 ** rng.uniform(-6.0, 6.0, n)
    k = rng.random(n)
    x[k < 0.05] = 0.0
    x[(k >= 0.05) & (k < 0.1)] = -0.0
    return torch.from_numpy(x.astype(np.float32))


def _first_diff(got, want):
    return int(np.flatnonzero(got.view(np.int32) != want.view(np.int32))[0])


class _Ranks:
    """`world` ranks of the exchange in this process: rank r lives on devices[r] and launches on a stream of its own."""

    def __init__(self, lib, devices):
        self.lib = lib
        self.devices = [torch.device(d) for d in devices]
        self.world = len(self.devices)
        self.streams = [torch.cuda.Stream(device=d) for d in self.devices]
        # ranks sharing a stream would queue behind each other's kernel and never meet at the barrier
        assert len({s.cuda_stream for s in self.streams}) == self.world

    def check_coresident(self, numel):
        """Every rank's grid on a device must be resident at once, or a spinning rank would keep another one out."""
        for d in set(self.devices):
            here = sum(1 for x in self.devices if x == d)
            if here > 1:
                sms = torch.cuda.get_device_properties(d).multi_processor_count
                g = _grid(numel, self.world, sms)
                assert here * g <= sms, "%d ranks x %d CTAs do not fit on %d SMs: the case is sized wrongly" % (
                    here, g, sms)

    def run(self, call, bufs):
        """call(r) for every rank on its own stream, then wait; checks one launch per rank and that no barrier gave up."""
        for d in set(self.devices):
            torch.cuda.synchronize(d)           # the inputs, written on the default streams, are in place
        before = self.lib.launch_count()
        for r in range(self.world):
            with torch.cuda.device(self.devices[r]), torch.cuda.stream(self.streams[r]):
                call(r)
        for d in set(self.devices):
            torch.cuda.synchronize(d)
        assert self.lib.launch_count() - before == self.world
        for r, b in enumerate(bufs):
            assert not b.timed_out(), "rank %d: a barrier of the exchange gave up" % r


# ---- plain exchange: peer_allreduce_kernel<N, false> ------------------------------------------------------------------

PLAIN_SIZES = ["one_piece", "kN+1", "kN-1", "cta_edge-1", "cta_edge", "cta_edge+1", "most_ctas"]


def _plain_pieces(kind, world, sms):
    """float4 pieces of a plain-exchange arena."""
    k = 5
    return {
        "one_piece": 1,                                  # rank 0 owns everything, every other rank nothing
        "kN+1": k * world + 1,                           # the last rank's slice is short
        "kN-1": k * world - 1,
        "cta_edge-1": PEER_THREADS * world - 1,          # per = 512: one full CTA-stride per rank, the last one short
        "cta_edge": PEER_THREADS * world,
        "cta_edge+1": PEER_THREADS * world + 1,          # per = 513: a second CTA that holds a single piece
        "most_ctas": PEER_THREADS * world * (sms // world) - 3,   # as many CTAs per rank as fit beside the others
    }[kind]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", PLAIN_SIZES)
@pytest.mark.parametrize("world", [2, 4, 8])
def test_exchange_stores_the_rank_ordered_sum_on_every_rank(lib, world, kind):
    from shacira_b200 import peer
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    numel = 4 * _plain_pieces(kind, world, sms)
    ranks = _Ranks(lib, ["cuda:0"] * world)
    ranks.check_coresident(numel)
    bufs = [peer.PeerBuffer(numel, "cuda:0") for _ in range(world)]
    for r, b in enumerate(bufs):
        b.connect_local(bufs, r)
    per = _per(numel // 4, world)
    rng = np.random.default_rng(100 * world + PLAIN_SIZES.index(kind))
    try:
        for call in range(3):                    # the flag block's epoch and ticket are reused by every call
            xs = [_wide_values(rng, numel).cuda() for _ in range(world)]
            for b, x in zip(bufs, xs):
                b.flat.copy_(x)
            ranks.run(lambda r: lib._check(bufs[r].lib.shacira_peer_allreduce(
                bufs[r].ptr_array(), bufs[r].flags_offset, r, world, numel, lib._stream())), bufs)
            want = _rank_sum(xs).cpu().numpy()
            for r, b in enumerate(bufs):
                got = b.flat.cpu().numpy()
                assert np.array_equal(got.view(np.int32), want.view(np.int32)), "call %d, rank %d: %s is %r, want %r" % (
                    call, r, _locate(_first_diff(got, want), per), got[_first_diff(got, want)],
                    want[_first_diff(got, want)])
        print("plain <%d>: %s, %d floats, %d CTAs per rank" % (world, kind, numel, _grid(numel, world, sms)))
    finally:
        for b in bufs:
            b.close()


# ---- Adam-fused exchange: peer_allreduce_kernel<N, true> --------------------------------------------------------------

ADAM_CASES = ["ends_in_rank0", "ends_on_rank_boundary", "ends_in_last_rank", "whole_arena"]


def _adam_layout(case, world):
    """(table rows, small tensor shapes) of an Adam-fused arena: [table gradient, then the small tensors]."""
    s4 = sum(_pieces(s) for s in SMALL)
    if case == "ends_in_rank0":
        return 4 * (s4 // world) - 1, SMALL              # 1 padding float
    if case == "ends_on_rank_boundary":
        return 4 * s4 * (world - 1), SMALL               # per = s4: the small tensors are exactly the last slice
    if case == "ends_in_last_rank":
        return 4 * (64 * (world - 1) + 20) - 3, SMALL    # 3 padding floats
    if case == "whole_arena":
        return 4 * 1100 * world - 2, []                  # 3 CTAs per rank, 2 padding floats
    if case == "nerf":
        return NERF_ROWS, SMALL
    raise ValueError(case)


def _check_layout(case, t4, n4, per, world):
    holds = {
        "ends_in_rank0": 0 < t4 < per,
        "ends_on_rank_boundary": t4 % per == 0 and t4 < n4,
        "ends_in_last_rank": (world - 1) * per < t4 < n4,
        "whole_arena": t4 == n4,
        "nerf": t4 < n4,
    }[case]
    assert holds, "case %s: the table's %d pieces do not end where the case says (arena %d, slice %d)" % (
        case, t4, n4, per)


def _ulp32(x):
    return np.spacing(np.float32(x)).astype(np.float64)


class _AdamOracle:
    """torch.optim.Adam in float64 over the padded table, fed the fp32 gradient sum, with per-element bounds on how
    far the fp32 kernel may be from it.

    Derivation, u = 2^-24, t = step, g = G + wd * p, per element. The kernel does (peer_kernels.cuh)
        gk = fmaf(wd, P, G)                    1 rounding, and P itself is off by at most ep_{t-1}
        M  = fmaf(b1, M, (1 - b1) * gk)        1 rounding of the product, 1 of the fma   (1 - b1 is exact: Sterbenz)
        V  = fmaf(b2, V, (1 - b2) * gk * gk)   2 roundings of the products, 1 of the fma
    With M_abs = b1 M_abs + (1 - b1)|g|, V_abs = b2 V_abs + (1 - b2) g^2 and B = b2 B + (1 - b2)|g|, summing the
    per-step errors through the recurrences (sum_s b^(t-s) M_abs_s <= t M_abs_t) gives
        |dm| <= (t + 2) u M_abs + wd ep_{t-1},     |dv| <= (t + 4) u V_abs + 2 wd ep_{t-1} B
    to first order; one more u M_abs (u V_abs) covers the O(t^2 u^2) terms. The update
        P -= (lr / bc1) * M / (sqrtf(V) * bc2s + eps),   bc1 = 1 - powf(b1, t),  bc2s = rsqrtf(1 - powf(b2, t))
    is bounded as an interval: powf within 4 ulp and rsqrtf within 2 ulp (CUDA's documented maximum errors), one
    rounding for the subtraction from 1, the divide and the multiply, sqrtf correctly rounded, two roundings for the
    denominator (fused or not), M and V within the bounds above. Then |dp_t| <= |dp_{t-1}| + the update's error +
    one fp32 rounding of p."""

    def __init__(self, p0, lr, betas, eps, weight_decay):
        f = lambda x: float(np.float32(x))              # what the kernel receives as `float`
        self.lr, self.b1, self.b2, self.eps, self.wd = f(lr), f(betas[0]), f(betas[1]), f(eps), f(weight_decay)
        self.p = p0.astype(np.float64)
        z = np.zeros_like(self.p)
        self.m, self.v, self.ep, self.m_abs, self.v_abs, self.b_abs = z, z, z, z, z, z
        self.em, self.ev = z, z
        self.t = 0

    @np.errstate(invalid="ignore")          # a NaN gradient makes that element's bounds NaN; _within masks it
    def step(self, G):
        t = self.t = self.t + 1
        lr, b1, b2, eps, wd = self.lr, self.b1, self.b2, self.eps, self.wd
        c1, c2 = 1.0 - b1, 1.0 - b2
        ep0 = self.ep
        g = G + wd * self.p
        a = np.abs(g)
        self.m = b1 * self.m + c1 * g
        self.v = b2 * self.v + c2 * g * g
        self.m_abs = b1 * self.m_abs + c1 * a
        self.v_abs = b2 * self.v_abs + c2 * a * a
        self.b_abs = b2 * self.b_abs + c2 * a
        self.em = (t + 3) * U * self.m_abs + wd * ep0
        self.ev = (t + 5) * U * self.v_abs + 2.0 * wd * ep0 * self.b_abs
        bc1, bc2 = 1.0 - b1 ** t, 1.0 - b2 ** t
        d1 = 4.0 * _ulp32(b1 ** t) + U * bc1            # |bc1 - kernel's bc1|
        d2 = 4.0 * _ulp32(b2 ** t) + U * bc2
        alpha = lr / bc1
        den = np.sqrt(self.v) / math.sqrt(bc2) + eps
        upd = alpha * self.m / den
        a_lo, a_hi = lr / (bc1 + d1) * (1 - U), lr / (bc1 - d1) * (1 + U)
        s_lo, s_hi = (1 - 4 * U) / math.sqrt(bc2 + d2), (1 + 4 * U) / math.sqrt(bc2 - d2)
        ma = np.abs(self.m)
        den_lo = (np.sqrt(np.maximum(self.v - self.ev, 0.0)) * (1 - U) * s_lo + eps) * (1 - U) ** 2
        den_hi = (np.sqrt(self.v + self.ev) * (1 + U) * s_hi + eps) * (1 + U) ** 2
        u_lo = a_lo * np.maximum(ma - self.em, 0.0) * (1 - U) ** 2 / den_hi
        u_hi = a_hi * (ma + self.em) * (1 + U) ** 2 / den_lo
        ua = np.abs(upd)
        eu = np.where(self.em < ma, np.maximum(u_hi - ua, ua - u_lo), u_hi + ua)   # M's sign may flip: either side
        self.p = self.p - upd
        self.ep = ep0 + eu + U * (np.abs(self.p) + ep0 + eu)


def _within(what, got, want, bound, per, offset=0):
    """|got - want| <= bound elementwise, NaN exactly where the oracle has NaN; returns the worst err / bound."""
    got = got.astype(np.float64)
    gn, wn = np.isnan(got), np.isnan(want)
    if not np.array_equal(gn, wn):
        j = int(np.flatnonzero(gn != wn)[0])
        raise AssertionError("%s: %s is %r, the oracle %r" % (what, _locate(offset + j, per), got[j], want[j]))
    ok = ~wn
    err = np.abs(got[ok] - want[ok])
    b = bound[ok]
    bad = err > b
    if bad.any():
        k = int(np.flatnonzero(bad)[0])
        j = int(np.flatnonzero(ok)[k])
        raise AssertionError("%s: %s is %r, the oracle %r: error %.3g over the bound %.3g" % (
            what, _locate(offset + j, per), got[j], want[j], err[k], b[k]))
    pos = b > 0
    return float(np.max(err[pos] / b[pos])) if pos.any() else 0.0


def _run_adam(lib, devices, case, weight_decay, seed, nan_at=None):
    """Adam-fused steps on N ranks, with plain exchanges on the same arenas between them; every step is checked
    against _AdamOracle. nan_at = (adam step, rank, element): one NaN in that rank's table gradient."""
    from shacira_b200 import peer
    world = len(devices)
    rows, small = _adam_layout(case, world)
    ranks = _Ranks(lib, devices)
    rng = np.random.default_rng(seed)
    w0 = rng.standard_normal(rows).astype(np.float32)
    arenas, tables = [], []
    try:
        for d in ranks.devices:
            params = [torch.nn.Parameter(torch.zeros(rows, 1, device=d))]
            params += [torch.nn.Parameter(torch.zeros(s, device=d)) for s in small]
            arenas.append(peer.PeerArena(params, connect=False))
            tables.append(peer.PeerTable(torch.from_numpy(w0).view(rows, 1).to(d), arenas[-1].buf.numel, connect=False))
        for r in range(world):
            arenas[r].buf.connect_local([a.buf for a in arenas], r)
            tables[r].buf.connect_local([t.buf for t in tables], r)
            tables[r].init_state(arenas[r].buf.numel)
        numel, tnumel = arenas[0].buf.numel, tables[0].buf.numel
        t4, n4 = tnumel // 4, numel // 4
        per = _per(n4, world)
        _check_layout(case, t4, n4, per, world)
        assert tnumel == 4 * _pieces((rows,)) and numel == tnumel + 4 * sum(_pieces(s) for s in small)
        for r, t in enumerate(tables):           # PeerTable's slice of the Adam state is the kernel's slice
            assert t.slice == (min(4 * per * r, tnumel), min(4 * per * (r + 1), tnumel))
        ranks.check_coresident(numel)
        bufs = [a.buf for a in arenas]

        hp = dict(lr=2e-2, betas=(0.9, 0.999), eps=1e-8, weight_decay=weight_decay)
        oracle = _AdamOracle(np.pad(w0, (0, tnumel - rows)), **hp)
        mag = 10.0 ** rng.uniform(-3.0, 2.0, rows)      # each element's gradient magnitude, fixed over the steps
        mag[np.arange(rows) % 7 == 3] = 0.0             # these elements' gradient stays exactly 0 on every rank
        worst = dict(p=0.0, m=0.0, v=0.0)
        plan = ["adam", "adam", "plain", "adam", "adam", "plain", "adam", "adam", "adam", "adam"]
        adam_steps = 0
        for call, kind in enumerate(plan):
            if kind == "plain":
                state = [(t.buf.flat.clone(), t.m.clone(), t.v.clone(), t.step.clone()) for t in tables]
                xs = [_wide_values(rng, numel).to(d) for d in ranks.devices]
                for a, x in zip(arenas, xs):
                    a.flat.copy_(x)
                ranks.run(lambda r: arenas[r].allreduce(), bufs)
                want = _rank_sum(xs).cpu().numpy()
                for r, a in enumerate(arenas):
                    got = a.flat.cpu().numpy()
                    assert np.array_equal(got.view(np.int32), want.view(np.int32)), "call %d (plain), rank %d: %s" % (
                        call, r, _locate(_first_diff(got, want), per))
                for r, (t, s) in enumerate(zip(tables, state)):   # the plain pass leaves the table and its state alone
                    for now, then in zip((t.buf.flat, t.m, t.v, t.step), s):
                        assert torch.equal(_bits(now), _bits(then)), "call %d (plain) changed rank %d's table" % (call, r)
                continue

            scale = 10.0 ** (adam_steps % 4 - 2)        # the gradient's scale changes by decades from step to step
            gt = [(rng.standard_normal(rows) * mag * scale).astype(np.float32) for _ in range(world)]
            if nan_at is not None and nan_at[0] == adam_steps:
                gt[nan_at[1]][nan_at[2]] = np.nan
            gs = [[_wide_values(rng, math.prod(s)).view(s) for s in small] for _ in range(world)]
            for r, a in enumerate(arenas):
                a.zero_()
                a.params[0].grad.copy_(torch.from_numpy(gt[r]).view(rows, 1))
                for p, g in zip(a.params[1:], gs[r]):
                    p.grad.copy_(g)
            G = _rank_sum([torch.from_numpy(g).to(ranks.devices[0]) for g in gt]).cpu().numpy().astype(np.float64)
            small_want = _rank_sum([a.flat[tnumel:] for a in arenas]).cpu().numpy()
            ranks.run(lambda r: arenas[r].allreduce_adam(tables[r], **hp), bufs)
            oracle.step(np.pad(G, (0, tnumel - rows)))
            adam_steps += 1
            what = "world %d, %s, wd %g, adam step %d (call %d)" % (world, case, weight_decay, adam_steps, call)

            p0 = tables[0].buf.flat.cpu().numpy()
            for r, (t, a) in enumerate(zip(tables, arenas)):
                p = t.buf.flat.cpu().numpy()
                assert np.array_equal(p.view(np.int32), p0.view(np.int32)), (
                    "%s: rank %d's table differs from rank 0's at %s" % (what, r, _locate(_first_diff(p, p0), per)))
                assert float(t.step) == adam_steps
                arena = a.flat.cpu().numpy()
                assert not arena[:tnumel].view(np.int32).any(), "%s: rank %d's table gradient not cleared at %s" % (
                    what, r, _locate(int(np.flatnonzero(arena[:tnumel].view(np.int32))[0]), per))
                assert np.array_equal(arena[tnumel:].view(np.int32), small_want.view(np.int32)), (
                    "%s: rank %d's small gradients at %s" % (what, r, _locate(
                        tnumel + _first_diff(arena[tnumel:], small_want), per)))
            worst["p"] = max(worst["p"], _within(what + ", table", p0, oracle.p, oracle.ep, per))
            for r, t in enumerate(tables):
                begin, end = t.slice
                for name, buf, want, bound in (("m", t.m, oracle.m, oracle.em), ("v", t.v, oracle.v, oracle.ev)):
                    got = buf.cpu().numpy()
                    worst[name] = max(worst[name], _within("%s, rank %d's %s" % (what, r, name), got[:end - begin],
                                                           want[begin:end], bound[begin:end], per, begin))
                    assert not got[end - begin:].view(np.int32).any(), "%s: rank %d's %s past its slice" % (what, r, name)
        print("adam <%d>: %s, %d rows + %d small, wd %g%s: worst err/bound p %.3g m %.3g v %.3g" % (
            world, case, rows, len(small), weight_decay, ", NaN" if nan_at else "", worst["p"], worst["m"], worst["v"]))
        return oracle
    finally:
        for t in tables:
            t.close()
        for a in arenas:
            a.close()


@pytest.mark.gpu
@pytest.mark.parametrize("weight_decay", [0.0, 0.01])
@pytest.mark.parametrize("case", ADAM_CASES)
@pytest.mark.parametrize("world", [2, 4, 8])
def test_adam_exchange_matches_a_float64_adam_on_every_rank(lib, world, case, weight_decay):
    _run_adam(lib, ["cuda:0"] * world, case, weight_decay, seed=1000 * world + 10 * ADAM_CASES.index(case)
              + int(weight_decay > 0))


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 4, 8])
def test_adam_exchange_nan_gradient_poisons_only_its_own_parameter(lib, world):
    """One NaN in the last rank's gradient of an element that rank 0 owns: that parameter and its m and v become NaN
    on every rank (as torch.optim.Adam does), every other element still follows the oracle."""
    rows, _ = _adam_layout("ends_in_last_rank", world)
    j = 4 * 3 + 1                                       # rank 0's slice; j % 7 != 3, so its gradient is not held at 0
    oracle = _run_adam(lib, ["cuda:0"] * world, "ends_in_last_rank", 0.01, seed=7 + world,
                          nan_at=(2, world - 1, j))
    assert j < rows and np.flatnonzero(np.isnan(oracle.p)).tolist() == [j]


@pytest.mark.gpu
def test_adam_exchange_across_two_gpus_at_nerf_scale(lib):
    if torch.cuda.device_count() < 2 or not torch.cuda.can_device_access_peer(0, 1):
        pytest.skip("needs two GPUs with peer access")
    _run_adam(lib, ["cuda:0", "cuda:1"], "nerf", 0.01, seed=2)


# ---- argument checks of shacira_peer_allreduce_adam (no GPU) ---------------------------------------------------------

def _adam_call(lib, world=2, rank=0, numel=16, flags_offset=4096, params="all", null_param=None, table_numel=8,
               exp_avg=FAKE, exp_avg_sq=FAKE, step=FAKE):
    arr = lambda n: (ctypes.c_void_p * n)(*([FAKE.value] * n))
    bufs = arr(world)
    if params == "all":
        params = arr(world)
        if null_param is not None:
            params[null_param] = None
    f = ctypes.c_float
    return lib.load().shacira_peer_allreduce_adam(bufs, flags_offset, rank, world, numel, params, table_numel, exp_avg,
                                                  exp_avg_sq, step, f(1e-2), f(0.9), f(0.999), f(1e-8), f(0.0), None)


@pytest.mark.parametrize("bad, code, msg", [
    (dict(table_numel=0), "invalid", b"table_numel"),
    (dict(table_numel=-4), "invalid", b"table_numel"),
    (dict(table_numel=6), "invalid", b"table_numel"),
    (dict(table_numel=20), "invalid", b"table_numel"),             # larger than numel
    (dict(numel=6), "invalid", b"numel"),
    (dict(numel=16, flags_offset=32), "invalid", b"exceeds the arena"),
    (dict(params=None), "invalid", b"NULL"),
    (dict(null_param=1), "invalid", b"table of rank 1 is NULL"),
    (dict(exp_avg=None), "invalid", b"NULL"),
    (dict(exp_avg_sq=None), "invalid", b"NULL"),
    (dict(step=None), "invalid", b"NULL"),
    (dict(world=1), "unsupported", b"world size 1"),
    (dict(world=3), "unsupported", b"world size 3"),
    (dict(world=16), "unsupported", b"world size 16"),
    (dict(rank=2), "invalid", b"bad rank"),
    (dict(rank=-1), "invalid", b"bad rank"),
])
def test_peer_allreduce_adam_rejects_bad_arguments_before_any_launch(lib, bad, code, msg):
    before = lib.launch_count()
    want = lib.ERR_INVALID_ARGUMENT if code == "invalid" else lib.ERR_UNSUPPORTED
    assert _adam_call(lib, **bad) == want
    assert msg in lib.load().shacira_last_error()
    assert lib.launch_count() == before
