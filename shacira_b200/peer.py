"""Exchange step of the ray-batch data-parallel path over NVLink / NVSwitch peer memory (SURVEY section 8e).

`PeerArena` is `dp.GradArena` with the flat gradient buffer living in CUDA-IPC shared device memory: every rank maps
every other rank's arena, and `allreduce()` is ONE kernel per rank (csrc/peer_kernels.cuh: cross-GPU barrier, rank r
reduces slice r from all arenas in rank order and stores the sum into all arenas, cross-GPU barrier) instead of an
NCCL collective. torch.distributed is only used once, to exchange the 64-byte IPC handles. The result is bit-identical
on all ranks. `PeerTable` puts the latent table itself in such memory so that `allreduce_adam()` can also run the
table's Adam step on the owner's slice and broadcast the updated parameters in the same pass.

The reference is single-GPU; BASELINE.json's north_star asks for the NVLink gradient exchange.
"""
import ctypes

import torch
import torch.distributed as dist

from . import _lib


class _Raw:
    """__cuda_array_interface__ holder: a float32 vector over raw device memory."""

    def __init__(self, ptr, numel):
        self.__cuda_array_interface__ = {"shape": (int(numel),), "typestr": "<f4", "data": (int(ptr), False), "version": 2}


def _as_tensor(ptr, numel, device):
    return torch.as_tensor(_Raw(ptr, numel), device=device)


class PeerBuffer:
    """`numel` float32 (rounded up to a multiple of 4) in peer-mappable device memory + the 256-byte flag block; after
    `connect()` `self.ptrs[p]` is rank p's buffer as mapped into this process."""

    def __init__(self, numel, device):
        self.lib = _lib.load()
        self.device = torch.device(device)
        self.numel = (int(numel) + 3) & ~3
        self.bytes = self.numel * 4
        p = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            _lib._check(self.lib.shacira_peer_alloc(self.bytes, ctypes.byref(p)))
        self.ptr = p.value
        self.flags_offset = int(self.lib.shacira_peer_flags_offset(self.bytes))
        self.flat = _as_tensor(self.ptr, self.numel, self.device)
        self.ptrs, self._opened, self.rank, self.world = None, [], 0, 1

    def connect(self, group=None):
        """Exchange the IPC handles over torch.distributed and map every peer's buffer. Collective."""
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        h = ctypes.create_string_buffer(64)
        with torch.cuda.device(self.device):
            _lib._check(self.lib.shacira_peer_export(ctypes.c_void_p(self.ptr), h))
        handles = [None] * self.world
        dist.all_gather_object(handles, bytes(h.raw), group=group)
        self.ptrs = []
        with torch.cuda.device(self.device):
            for r, hb in enumerate(handles):
                if r == self.rank:
                    self.ptrs.append(self.ptr)
                    continue
                q = ctypes.c_void_p()
                _lib._check(self.lib.shacira_peer_open(ctypes.create_string_buffer(hb, 64), ctypes.byref(q)))
                self._opened.append(q.value)
                self.ptrs.append(q.value)
        torch.cuda.synchronize(self.device)
        dist.barrier(group=group)     # nobody launches an exchange before every mapping exists
        return self

    def connect_local(self, buffers, rank):
        """Single process, several GPUs: `buffers` = the PeerBuffers of all ranks in rank order (peer access enabled)."""
        self.rank, self.world = int(rank), len(buffers)
        for b in buffers:
            if b is not self and b.device != self.device:
                _lib._check(self.lib.shacira_peer_enable_access(self.device.index, b.device.index))
        self.ptrs = [b.ptr for b in buffers]
        return self

    def ptr_array(self):
        return (ctypes.c_void_p * self.world)(*self.ptrs)

    def timed_out(self):
        """True if a cross-GPU barrier of an exchange on this buffer gave up (a peer never arrived). Synchronises."""
        v = ctypes.c_int32(0)
        with torch.cuda.device(self.device):
            _lib._check(self.lib.shacira_peer_status(ctypes.c_void_p(self.ptr), self.flags_offset, ctypes.byref(v)))
        return bool(v.value)

    def close(self):
        with torch.cuda.device(self.device):
            for q in self._opened:
                self.lib.shacira_peer_close(ctypes.c_void_p(q))
            self._opened = []
            if self.ptr:
                torch.cuda.synchronize(self.device)
                self.flat = None
                self.lib.shacira_peer_free(ctypes.c_void_p(self.ptr))
                self.ptr = 0


def _agreed_create(cls, params, group):
    """cls(params, connect=False) then .connect(group) on every rank; None on EVERY rank if any step failed anywhere."""
    params = list(params)
    dev = params[0].device
    ok = torch.ones(1, dtype=torch.int32, device=dev)
    arena = None
    try:
        arena = cls(params, group=group, connect=False)
    except Exception:
        ok.zero_()
    dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
    if int(ok.item()) == 0:
        if arena is not None:
            arena.close()
        return None
    try:
        arena.connect(group)
    except Exception:
        ok.zero_()
    dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
    if int(ok.item()) == 0:
        arena.close()
        return None
    return arena


class PeerArena:
    """One flat float32 gradient buffer for a set of parameters (every `.grad` is a view into it, as dp.GradArena), in
    peer-mapped memory. `allreduce()` = shacira_peer_allreduce on the current stream."""

    def __init__(self, params, group=None, connect=True):
        self.params = list(params)
        dev = self.params[0].device
        offs, total = [], 0
        for p in self.params:
            offs.append(total)
            total += (p.numel() + 3) & ~3        # every tensor starts on a 16-byte boundary
        self.buf = PeerBuffer(total, dev)
        self.flat = self.buf.flat
        for p, off in zip(self.params, offs):
            p.grad = self.flat[off:off + p.numel()].view_as(p)
        self.offsets = offs
        if connect:
            self.connect(group)

    def connect(self, group=None):
        self.buf.connect(group)
        return self

    @classmethod
    def try_create(cls, params, group=None):
        """PeerArena on every rank, or None on every rank (the ranks agree: CUDA IPC can be unavailable, e.g. across
        containers or without peer access) -- the caller then keeps the NCCL form (dp.GradArena). Collective."""
        return _agreed_create(cls, params, group)

    def zero_(self):
        self.flat.zero_()

    def allreduce(self):
        """SUM over ranks, in place, one kernel. Returns the number of exchange launches (1)."""
        b = self.buf
        with torch.cuda.device(b.device):
            _lib._check(b.lib.shacira_peer_allreduce(b.ptr_array(), b.flags_offset, b.rank, b.world, b.numel,
                                                     _lib._stream()))
        return 1

    def timed_out(self):
        return self.buf.timed_out()

    def allreduce_adam(self, table, lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        """The same pass with the Adam step of `table` (a PeerTable whose gradient is the FIRST tensor of this arena)
        on the owner's slice; the updated table is broadcast, its gradient slots come back zeroed."""
        b = self.buf
        with torch.cuda.device(b.device):
            _lib._check(b.lib.shacira_peer_allreduce_adam(
                b.ptr_array(), b.flags_offset, b.rank, b.world, b.numel, table.buf.ptr_array(), table.buf.numel,
                ctypes.c_void_p(table.m_base), ctypes.c_void_p(table.v_base), _lib._ptr(table.step), float(lr),
                float(betas[0]), float(betas[1]), float(eps), float(weight_decay), _lib._stream()))
            table.step += 1.0
        return 1

    def close(self):
        for p in self.params:
            p.grad = None
        self.flat = None
        self.buf.close()


class McArena:
    """The gradient arena bound to an NVSwitch multicast object (NVLS): `allreduce()` = shacira_peer_allreduce_multimem,
    the sum is formed inside the switch. The multicast mapping (cuMulticastCreate / bind over the ranks) is plumbing:
    torch's symmetric-memory allocator does it; the cross-GPU barrier flags live in a small PeerBuffer of our own."""

    def __init__(self, params, group=None, connect=True):
        import torch.distributed._symmetric_memory as symm
        self.params = list(params)
        dev = self.params[0].device
        offs, total = [], 0
        for p in self.params:
            offs.append(total)
            total += (p.numel() + 3) & ~3
        self.numel = total
        self.flat = symm.empty(total, dtype=torch.float32, device=dev)
        self.flat.zero_()
        for p, off in zip(self.params, offs):
            p.grad = self.flat[off:off + p.numel()].view_as(p)
        self.flags = PeerBuffer(4, dev)
        self.hdl = None
        if connect:
            self.connect(group)

    def connect(self, group=None):
        import torch.distributed._symmetric_memory as symm
        self.hdl = symm.rendezvous(self.flat, group if group is not None else dist.group.WORLD)
        if not int(getattr(self.hdl, "multicast_ptr", 0) or 0):
            raise RuntimeError("no multicast support on this fabric")
        self.flags.connect(group)
        return self

    @classmethod
    def try_create(cls, params, group=None):
        return _agreed_create(cls, params, group)

    def zero_(self):
        self.flat.zero_()

    def allreduce(self):
        f = self.flags
        with torch.cuda.device(f.device):
            _lib._check(f.lib.shacira_peer_allreduce_multimem(ctypes.c_void_p(int(self.hdl.multicast_ptr)), f.ptr_array(),
                                                              f.flags_offset, f.rank, f.world, self.numel, _lib._stream()))
        return 1

    def timed_out(self):
        return self.flags.timed_out()

    def close(self):
        for p in self.params:
            p.grad = None
        self.flags.close()
        self.hdl = None
        self.flat = None


class PeerTable:
    """The latent table [T, C] in peer-mapped memory (every rank holds the full, replicated table; rank r owns the Adam
    state of slice r only: 1/world of exp_avg / exp_avg_sq per GPU)."""

    def __init__(self, init, arena_numel, group=None, connect=True):
        init = init.detach()
        self.shape = tuple(init.shape)
        dev = init.device
        self.buf = PeerBuffer(init.numel(), dev)
        self.buf.flat[:init.numel()].copy_(init.reshape(-1))
        self.data = self.buf.flat[:init.numel()].view(self.shape)
        self.m = self.v = self.step = None
        if connect:
            self.buf.connect(group)
            self.init_state(arena_numel)

    def init_state(self, arena_numel):
        """Allocate this rank's slice of the Adam state. Called by the constructor after connect(); a single-process
        caller (connect=False, then buf.connect_local) calls it once the world size is known."""
        # the exchange kernel splits the ARENA (table gradient + small gradients) into `world` slices of float4 pieces
        w, r = self.buf.world, self.buf.rank
        n4 = ((int(arena_numel) + 3) & ~3) // 4
        per = (n4 + w - 1) // w
        begin, end = min(per * r * 4, self.buf.numel), min(per * (r + 1) * 4, self.buf.numel)
        dev = self.buf.device
        self.m = torch.zeros(max(end - begin, 4), dtype=torch.float32, device=dev)
        self.v = torch.zeros_like(self.m)
        # pointers offset so that element i of the table is m_base[i]
        self.m_base = self.m.data_ptr() - 4 * begin
        self.v_base = self.v.data_ptr() - 4 * begin
        self.step = torch.zeros((), dtype=torch.float32, device=dev)
        # allreduce_adam() advances `step` right behind this rank's exchange kernel. The first launch of that add can
        # load its kernel, and loading can wait for the device to go idle: in a process that launches several ranks,
        # that would wait on an exchange that waits for the next rank's launch until the barriers give up. Load it here.
        self.step += 0.0
        self.slice = (begin, end)

    def close(self):
        self.data = None
        self.buf.close()
