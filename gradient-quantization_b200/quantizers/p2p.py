"""Peer-to-peer exchange of packed records (ps topology, one user per GPU, one NVSwitch node).

Each rank owns one cudaMalloc'ed, IPC-exported buffer
    [parity 0: U records | parity 1: U records | flags]
and maps every peer's buffer.  A step encodes the local record straight into row `rank` of the
current parity, then either
  push   : stores it into row `rank` of every peer's buffer (posted NVLink writes), runs the
           barrier kernel (gq_peer_barrier) and decodes its own, now complete, [U, record] block;
  gather : runs the barrier, pulls every peer's row into the local block (wide loads), decodes;
  direct : runs the barrier and lets the decode kernel pull the peers' rows itself.
Double buffering makes one barrier per step sufficient: a row of parity p is overwritten two steps
later, after every rank has passed the next barrier, i.e. finished reading that parity.
"""
import ctypes

import torch
import torch.distributed as dist

from .. import _lib


class _CudaBuffer:
    """Exposes a raw device pointer to torch (zero copy)."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (int(ptr), False),
                                         "version": 2}


class PeerRecords:
    FLAG_BYTES = 256
    COUNTER_OFFSET = 64   # in the local flag area: the arrival counter of the delivering sign / QSGD encodes

    def __init__(self, record_bytes, rank, world, device):
        assert world <= 8
        self.record_bytes, self.rank, self.world, self.device = record_bytes, rank, world, device
        total = 2 * world * record_bytes + self.FLAG_BYTES
        self.mc_base = 0            # multicast (NVLS) address of the buffer, 0 = none
        self._opened = []
        self._symm = None
        self.local_ptr = None
        import os
        how = os.environ.get("GQ_P2P_ALLOC", "symm")
        if how == "symm" and not self._alloc_symmetric(total):
            how = "ipc"
        if how != "symm":
            self._alloc_ipc(total)
        self.alloc = how
        self._flag_ptrs = (ctypes.c_void_p * world)(*[b + 2 * world * record_bytes for b in self.base])
        self.epoch = 0
        self.step = 0
        dist.barrier()   # every rank has mapped every buffer before anyone writes flags

    def _alloc_symmetric(self, total):
        """torch symmetric memory (CUDA VMM): peer mappings plus, on NVSwitch, a multicast mapping.
        Returns False (on every rank alike) when it is not available."""
        ok, t, hdl = 1, None, None
        try:
            import torch.distributed._symmetric_memory as symm
            t = symm.empty(total, dtype=torch.uint8, device=self.device)
        except Exception:  # noqa: BLE001
            ok = 0
        flags = [None] * self.world
        dist.all_gather_object(flags, ok)
        if not all(flags):
            return False
        try:
            hdl = symm.rendezvous(t, dist.group.WORLD)
            t.zero_()
            torch.cuda.synchronize()
            base = [int(p) for p in hdl.buffer_ptrs]
            mc = int(hdl.multicast_ptr) if hdl.has_multicast_support else 0
        except Exception:  # noqa: BLE001
            ok = 0
        dist.all_gather_object(flags, ok)
        if not all(flags):
            return False
        self._symm = (t, hdl)
        self.base = base
        import os
        # multicast pays when there are several receivers (N = 2: 15 us vs 9.5 us for plain stores)
        want_mc = os.environ.get("GQ_P2P_MULTICAST", "1" if self.world > 2 else "0") != "0"
        self.mc_base = mc if want_mc else 0
        self.local_ptr = base[self.rank]
        # [2 * U, record_bytes] uint8 view of the local buffer: row parity * U + user
        self.records = t[:2 * self.world * self.record_bytes].view(2 * self.world, self.record_bytes)
        return True

    def _alloc_ipc(self, total):
        """cudaMalloc + CUDA IPC handles exchanged through the process group."""
        rank, world = self.rank, self.world
        ptr = ctypes.c_void_p()
        handle = (ctypes.c_char * 64)()
        _lib.call("gq_ipc_alloc", total, ctypes.byref(ptr), ctypes.cast(handle, ctypes.c_void_p))
        self.local_ptr = ptr.value
        handles = [None] * world
        dist.all_gather_object(handles, bytes(handle.raw))
        self.base = []
        for r in range(world):
            if r == rank:
                self.base.append(self.local_ptr)
            else:
                pp = ctypes.c_void_p()
                hbuf = (ctypes.c_char * 64).from_buffer_copy(handles[r])
                _lib.call("gq_ipc_open", ctypes.cast(hbuf, ctypes.c_void_p), ctypes.byref(pp))
                self.base.append(pp.value)
                self._opened.append(pp.value)
        self._holder = _CudaBuffer(self.local_ptr, 2 * world * self.record_bytes)
        # [2 * U, record_bytes] uint8 view of the local buffer: row parity * U + user
        self.records = torch.as_tensor(self._holder, device=self.device).view(2 * world, self.record_bytes)

    @property
    def parity(self):
        return self.step & 1

    def _delivery(self, plan, deltas, mc, flag_ranks, epoch, with_ident):
        """Attach a delivery now and return a function that attaches it again: deliver(announce, ident)
        before every launch of an encode made of several calls (FusedPlan.encode), so that each launch
        delivers its own sections and only the last one announces `epoch`."""
        local = self._addr(self.rank, self.rank)
        g_id = next((g for g in plan.groups if g.kind == "identity" and g.n), None) if with_ident else None
        delta_arr = (ctypes.c_int64 * len(deltas))(*deltas)
        flags = (ctypes.c_void_p * len(flag_ranks))(*[int(self._flag_ptrs[r]) + 4 * self.rank for r in flag_ranks])
        counter = int(self._flag_ptrs[self.rank]) + self.COUNTER_OFFSET

        def deliver(announce=True, ident=True):
            g = g_id if ident else None
            _lib.call("gq_attach_remote_record", len(deltas), mc, delta_arr, local + g.raw_off if g is not None else None,
                      (g.n * 4 + 15) // 16 * 16 if g is not None else 0, ctypes.cast(flags, ctypes.c_void_p),
                      len(flag_ranks) if announce else 0, int(epoch))
            _lib.call("gq_attach_delivery_counter", counter)

        deliver()
        return deliver

    def attach_delivery(self, plan):
        """Fused push: the next encode of `plan` into row `row()` also stores the record into the same
        row of every peer's block (or once through the multicast mapping) and then announces the new
        epoch in every rank's flag array (its own included).  Returns the function that re-attaches the
        delivery for each launch of a multi-launch encode (FusedPlan.encode(delivery=...))."""
        self.epoch += 1
        local = self._addr(self.rank, self.rank)
        if self.mc_base:
            deltas = [self.mc_base + self.row() * self.record_bytes - local]
            mc = 1
        else:
            deltas = [self._addr(r, self.rank) - local for r in range(self.world) if r != self.rank]
            mc = 0
        return self._delivery(plan, deltas, mc, list(range(self.world)), self.epoch, True)

    def attach_delivery_to(self, plan, targets, epoch, with_ident=True):
        """Ring hop: the next encode of `plan` into row `row()` also stores what it writes into the same
        row of the blocks of `targets` (all other ranks: once through the multicast mapping when there
        is one) and then writes `epoch` into this rank's word of those ranks' flag arrays.  Returns the
        re-attaching function, as attach_delivery does."""
        local = self._addr(self.rank, self.rank)
        everyone = len(targets) == self.world - 1
        if everyone and self.mc_base and self.world > 2:
            deltas = [self.mc_base + self.row() * self.record_bytes - local]
            mc = 1
            flag_ranks = list(range(self.world))
        else:
            deltas = [self._addr(r, self.rank) - local for r in targets]
            mc = 0
            flag_ranks = list(targets)
        return self._delivery(plan, deltas, mc, flag_ranks, epoch, with_ident)

    @staticmethod
    def _wait(flags, n, epoch):
        """Attach a wait now and return the function that attaches it again before each decode launch
        (FusedPlan.decode(wait=...))."""
        def wait():
            _lib.call("gq_attach_peer_wait", flags, n, epoch)

        wait()
        return wait

    def attach_wait_for(self, src_rank, epoch):
        """Ring hop, receiving side: the next decode waits until `src_rank` has announced `epoch` here."""
        return self._wait(int(self._flag_ptrs[self.rank]) + 4 * src_rank, 1, int(epoch))

    def attach_wait(self):
        """Fused push, receiving side: the next decode waits for every rank's flag of this epoch."""
        return self._wait(int(self._flag_ptrs[self.rank]), self.world, self.epoch)

    def barrier(self):
        self.epoch += 1
        _lib.call("gq_peer_barrier", ctypes.cast(self._flag_ptrs, ctypes.c_void_p), self.rank, self.world,
                  self.epoch, _lib.stream())

    def row(self, user=None):
        """Row of `records` holding `user`'s (default: this rank's) record of the current parity."""
        return self.parity * self.world + (self.rank if user is None else user)

    def _addr(self, owner, user):
        return self.base[owner] + self.row(user) * self.record_bytes

    def push(self):
        """Store the local record into row `rank` of every peer's block (call before barrier())."""
        if self.world == 1:
            return
        if self.mc_base:   # one multimem store stream, replicated by the switch to every rank
            _lib.call("gq_peer_push_multicast", self._addr(self.rank, self.rank),
                      self.mc_base + self.row() * self.record_bytes, self.record_bytes, _lib.stream())
            return
        dsts = (ctypes.c_void_p * (self.world - 1))(*[self._addr(r, self.rank) for r in range(self.world)
                                                       if r != self.rank])
        _lib.call("gq_peer_push", self._addr(self.rank, self.rank), ctypes.cast(dsts, ctypes.c_void_p),
                  self.record_bytes, self.world - 1, _lib.stream())

    def gather(self):
        """Pull every user's record of the current parity into the local block (after barrier());
        one launch -- the own row is copied onto itself."""
        srcs = (ctypes.c_void_p * self.world)(*[self._addr(r, r) for r in range(self.world)])
        _lib.call("gq_peer_gather", self._addr(self.rank, 0), ctypes.cast(srcs, ctypes.c_void_p),
                  self.record_bytes, self.record_bytes, self.world, _lib.stream())

    def user0_record_ptr(self):
        """direct mode: address of user 0's record in ITS OWNER's buffer."""
        return self._addr(0, 0)

    def user_offsets(self):
        """host int64 array: byte distance of user u's record (in u's buffer) from user 0's."""
        a0 = self._addr(0, 0)
        return (ctypes.c_int64 * self.world)(*[self._addr(u, u) - a0 for u in range(self.world)])

    def advance(self):
        self.step += 1

    def close(self):
        try:
            torch.cuda.synchronize()
            for p in self._opened:
                _lib.call("gq_ipc_close", p)
            if self._symm is None and self.local_ptr:
                _lib.call("gq_ipc_free", self.local_ptr)
            self.local_ptr = None
        except Exception:  # noqa: BLE001 - best effort at interpreter shutdown
            pass
        self._opened = []
