"""Whole-model fused codec plan: the engine under PSQuantizer / RingQuantizer.

The reference loops over parameters and calls compress()/decompress() per tensor
(quantizers/ps_quantizer.py:33-44); on a B200 that is ~160 tiny launches per
user.  Here the parameters are grouped by codec shape once, their gradients are
staged in one flat fp32 *arena* (group by group, tensors end to end), and each
user's compressed form is one contiguous *packed record*:

    record = [ per HSQ group : codes | l (or fp32 norms) | lb/ub table ]
             [ per QSGD group: chunk norms | packed sign+level          ]
             [ sign group    : 2-bit packed signs (or base-3, 5 per byte)   ]
             [ top-k group   : int32 indices | fp32 values              ]
             [ identity      : raw fp32 (tensors with <= 1000 elements) ]

records is a [U, record_bytes] uint8 buffer -- exactly the receive buffer of an
NCCL all-gather with one user per rank -- and decode is one fused
decode-and-reduce launch per group over all U records, in user order.
Every section starts on a 256-byte boundary.
"""
import os

import torch

from .. import _lib
from ..compressors import (IdenticalCompressor, NearestNeighborCompressor, QSGDCompressor,
                           SignSGDCompressor, TopKSparsificationCompressor)
from ..compressors._common import chunk_dim, load_codebook

_ALIGN = 256


def _up(x, a=_ALIGN):
    return (x + a - 1) // a * a


class _Group:
    """A set of tensors sharing one codec configuration, contiguous in the arena."""

    def __init__(self, kind, key):
        self.kind, self.key = kind, key
        self.tensors = []      # indices into plan.shapes
        self.sizes = []
        self.arena_off = 0     # element offset of the group in the arena
        self.n = 0             # elements

    def add(self, idx, size):
        self.tensors.append(idx)
        self.sizes.append(size)
        self.n += size


class FusedPlan:
    SUPPORTED = (NearestNeighborCompressor, QSGDCompressor, SignSGDCompressor,
                 TopKSparsificationCompressor, IdenticalCompressor)

    @classmethod
    def supports(cls, Compressor):
        return Compressor in cls.SUPPORTED

    def __init__(self, Compressor, shapes, args, device, n_users):
        self.Compressor = Compressor
        self.shapes = [tuple(s) for s in shapes]
        self.sizes = [int(torch.Size(s).numel()) for s in self.shapes]
        self.args = args
        self.device = device
        self.n_users = n_users
        self.random = 1 if getattr(args, "random", True) else 0
        self.algo = getattr(args, "hsq_algo", _lib.ALGO_AUTO)
        self.groups = []
        self._classify()
        self._layout()
        self.arena = torch.zeros(self.arena_elems, dtype=torch.float32, device=device)
        self._records = torch.zeros(n_users, self.record_bytes, dtype=torch.uint8, device=device)
        self._pending = None   # deferred levels: (row, group, seed, offset, uniforms) of the last encode
        self.workspace = torch.empty(max(self.workspace_bytes, _ALIGN), dtype=torch.uint8, device=device)
        self.u_scratch = torch.empty(max(self.max_chunks, 1), dtype=torch.float32, device=device)

    @property
    def records(self):
        """[rows, record_bytes] uint8: the packed records.  Reading it completes a record whose levels
        an encode(defer_levels=True) left to the next decode."""
        self._complete()
        return self._records

    @records.setter
    def records(self, buf):
        self._complete()
        self._records = buf

    # ------------------------------------------------------------ planning ---
    def _classify(self):
        a = self.args
        by_key = {}
        order = []

        def group(kind, key):
            if (kind, key) not in by_key:
                by_key[(kind, key)] = _Group(kind, key)
                order.append((kind, key))
            return by_key[(kind, key)]

        self.tensor_group = []
        for i, size in enumerate(self.sizes):
            # the reference compresses only tensors with more than 1000 elements
            # (ps_quantizer.py:15-20)
            if size <= 1000 or self.Compressor is IdenticalCompressor:
                g = group("identity", None)
            elif self.Compressor is NearestNeighborCompressor:
                assert a.c_dim > 0 and a.k_bit >= 0 and a.n_bit > 0
                dim = chunk_dim(size, a.c_dim)
                assert size % dim == 0, "not divisible size {} c_dim {} dim {}".format(size, a.c_dim, dim)
                K = dim if a.k_bit <= 0 else 2 ** a.k_bit
                if K == dim:
                    raise _lib.GQError("fused plan: random orthogonal codebooks (K == dim) are per-tensor; "
                                       "use the per-parameter path")
                g = group("hsq", (dim, K))
            elif self.Compressor is QSGDCompressor:
                dim = chunk_dim(size, a.c_dim)
                assert dim != 0 and size % dim == 0
                g = group("qsgd", "tensor" if (a.c_dim == 0 or size < a.c_dim) else dim)
            elif self.Compressor is SignSGDCompressor:
                g = group("sign", None)
            elif self.Compressor is TopKSparsificationCompressor:
                g = group("topk", None)
            else:
                raise _lib.GQError("fused plan does not support %r" % (self.Compressor,))
            g.add(i, size)
            self.tensor_group.append(g)
        # HSQ groups: tensors whose chunk count is a multiple of 16 first (model order otherwise), so that
        # every tensor boundary among them is a 16-byte boundary of the code / level sections and the ring's
        # stages (make_parts) can be cut there -- ResNet-50's first convolution (108 chunks) would otherwise
        # misalign every later boundary
        for (kind, key), g in by_key.items():
            if kind == "hsq":
                pairs = sorted(zip(g.tensors, g.sizes), key=lambda p: (p[1] // key[0]) % 16 != 0)
                g.tensors, g.sizes = [p[0] for p in pairs], [p[1] for p in pairs]
        # identity last, compressed groups in first-appearance order
        self.groups = [by_key[k] for k in order if k[0] != "identity"]
        self.groups += [by_key[k] for k in order if k[0] == "identity"]

    def _layout(self):
        a = self.args
        dev = self.device
        off_el = 0
        rec = 0
        ws = 0
        self.max_chunks = 0
        self.tensor_off = [0] * len(self.sizes)
        for g in self.groups:
            off_el = _up(off_el * 4) // 4
            g.arena_off = off_el
            t_off = off_el
            for idx, size in zip(g.tensors, g.sizes):
                self.tensor_off[idx] = t_off
                t_off += size
            off_el += g.n
            if g.kind == "hsq":
                dim, K = g.key
                g.dim, g.K = dim, K
                g.n_chunks = g.n // dim
                g.n_seg = len(g.tensors)
                starts = [0]
                for size in g.sizes:
                    starts.append(starts[-1] + size // dim)
                g.seg_start = torch.tensor(starts, dtype=torch.int64, device=dev)
                g.seg_start_host = starts
                g.codebook = torch.from_numpy(load_codebook(dim, K)).to(dev)
                g.code_bytes = 1 if a.k_bit <= 8 else 4
                g.n_bit = a.n_bit
                g.l_bytes = 1 if a.n_bit <= 7 else 4
                g.codes_off = rec
                rec += _up(g.n_chunks * g.code_bytes)
                g.l_off = rec                       # l codes, or fp32 norms when n_bit == 32
                rec += _up(g.n_chunks * (4 if a.n_bit == 32 else g.l_bytes))
                g.lbub_off = rec
                rec += _up(g.n_seg * 8)
                ws = max(ws, _lib.value("gq_hsq_encode_workspace_bytes", g.n_chunks, dim, K, g.n_seg))
                self.max_chunks = max(self.max_chunks, g.n_chunks)
            elif g.kind == "qsgd":
                g.n_bit = a.n_bit
                g.bits = _lib.value("gq_qsgd_wire_bits", a.n_bit)
                if g.key == "tensor":       # one chunk per tensor (TernGrad, c_dim == 0)
                    g.dim = 0
                    g.n_chunks = len(g.tensors)
                    starts = [0]
                    for size in g.sizes:
                        starts.append(starts[-1] + size)
                    g.chunk_start = torch.tensor(starts, dtype=torch.int64, device=dev)
                else:
                    g.dim = g.key
                    g.n_chunks = g.n // g.dim
                    g.chunk_start = None
                g.norm_off = rec
                rec += _up(g.n_chunks * 4)
                g.packed_off = rec
                rec += _up((g.n + 3) // 4 * 4 * g.bits // 8)
            elif g.kind == "sign":
                # wire container: 2 bits per element (default) or the base-3 form, five elements per byte
                # (args.sign_wire = "t5", SURVEY 8f-4); the decoded values are the same
                g.t5 = getattr(a, "sign_wire", "2bit") == "t5"
                g.wire_bytes = int(_lib.value("gq_sign_t5_bytes", g.n)) if g.t5 else (g.n + 3) // 4
                g.packed_off = rec
                rec += _up(g.wire_bytes)
            elif g.kind == "topk":
                g.n_seg = len(g.tensors)
                starts, ks, kp = [0], [], [0]
                for size in g.sizes:
                    starts.append(starts[-1] + size)
                    ks.append(size // a.cr)
                    kp.append(kp[-1] + ks[-1])
                g.k_total = kp[-1]
                g.seg_start = torch.tensor(starts, dtype=torch.int64, device=dev)
                g.k = torch.tensor(ks, dtype=torch.int64, device=dev)
                g.k_prefix = torch.tensor(kp[:-1], dtype=torch.int64, device=dev)
                g.idx_off = rec
                rec += _up(g.k_total * 4)
                g.val_off = rec
                rec += _up(g.k_total * 4)
                ws = max(ws, _lib.value("gq_topk_workspace_bytes", g.n, g.n_seg))
            elif g.kind == "identity":
                g.raw_off = rec
                rec += _up(g.n * 4)
        self.arena_elems = _up(off_el * 4) // 4
        self.record_bytes = _up(rec)
        self.workspace_bytes = ws

    # --------------------------------------------------------------- parts ---
    def make_parts(self, n_parts):
        """Cut the plan into n_parts stages for the pipelined ring (SURVEY 8e: the chain is per tensor, so
        rank r can work on one group of tensors while rank r + 1 works on the previous one).  Every HSQ
        group is cut at tensor boundaries into contiguous sub-ranges of about equal chunk counts (cuts
        only where the chunk offset is a multiple of 16, so that every section of a part stays 16-byte
        aligned); all other groups (and the identity tensors) belong to part 0.  Returns the number of
        parts actually made.  encode(part=p) / decode(part=p) / part_byte_ranges(p) then address one part."""
        n_parts = max(1, int(n_parts))
        for g in self.groups:
            g.part_cuts = None
            if g.kind != "hsq" or n_parts == 1 or g.n_bit == 32:
                continue
            starts = g.seg_start_host
            cuts = [0]
            for k in range(1, n_parts):
                target = g.n_chunks * k // n_parts
                # first tensor boundary at or after the target whose chunk offset is 16-aligned
                t = next((i for i in range(cuts[-1] + 1, g.n_seg) if starts[i] >= target and starts[i] % 16 == 0), None)
                if t is None:
                    break
                cuts.append(t)
            cuts.append(g.n_seg)
            if len(cuts) > 2:
                g.part_cuts = cuts
                g.part_seg = [torch.tensor([x - starts[cuts[k]] for x in starts[cuts[k]:cuts[k + 1] + 1]],
                                           dtype=torch.int64, device=self.device) for k in range(len(cuts) - 1)]
        self.n_parts = max([len(g.part_cuts) - 1 for g in self.groups if getattr(g, "part_cuts", None)] or [1])
        return self.n_parts

    def _part_range(self, g, part):
        """(first tensor, last tensor + 1, first chunk, last chunk + 1) of HSQ group g in `part`, or None."""
        cuts = getattr(g, "part_cuts", None)
        if cuts is None:
            return (0, g.n_seg, 0, g.n_chunks) if part == 0 else None
        if part >= len(cuts) - 1:
            return None
        ta, tb = cuts[part], cuts[part + 1]
        return ta, tb, g.seg_start_host[ta], g.seg_start_host[tb]

    def part_byte_ranges(self, part):
        """Byte ranges [(begin, end)] of one packed record that `part` produces (what travels per hop)."""
        out = []
        for g in self.groups:
            if g.kind == "hsq" and getattr(g, "part_cuts", None) is not None:
                r = self._part_range(g, part)
                if r is None:
                    continue
                ta, tb, ca, cb = r
                out.append((g.codes_off + ca * g.code_bytes, g.codes_off + cb * g.code_bytes))
                out.append((g.l_off + ca * g.l_bytes, g.l_off + cb * g.l_bytes))
                out.append((g.lbub_off + 8 * ta, g.lbub_off + 8 * tb))
            elif part == 0:
                if g.kind == "hsq":
                    out.append((g.codes_off, g.lbub_off + _up(g.n_seg * 8)))
                elif g.kind == "qsgd":
                    out.append((g.norm_off, g.packed_off + _up((g.n + 3) // 4 * 4 * g.bits // 8)))
                elif g.kind == "sign":
                    out.append((g.packed_off, g.packed_off + _up(g.wire_bytes)))
                elif g.kind == "topk":
                    out.append((g.idx_off, g.val_off + _up(g.k_total * 4)))
                elif g.kind == "identity" and g.n:
                    out.append((g.raw_off, g.raw_off + _up(g.n * 4)))
        return out

    # --------------------------------------------------------------- views ---
    def view(self, i, buf=None):
        """View of tensor i inside the arena (or another buffer laid out like it)."""
        buf = self.arena if buf is None else buf
        o = self.tensor_off[i]
        return buf[o:o + self.sizes[i]].view(self.shapes[i])

    def views(self, buf=None):
        return [self.view(i, buf) for i in range(len(self.sizes))]

    def locate(self, tensors):
        """If the tensors are views of ONE buffer laid out like the arena (e.g. made with views(buf)),
        return that buffer's base address (encode can read it in place); else None."""
        if len(tensors) != len(self.sizes) or not tensors:
            return None
        base = tensors[0].data_ptr() - self.tensor_off[0] * 4
        for t, o in zip(tensors, self.tensor_off):
            if t.data_ptr() != base + o * 4 or t.dtype != torch.float32 or not t.is_contiguous():
                return None
        return base if base % 256 == 0 else None

    def gather(self, tensors, buf=None, feedback=0, scale=0.0):
        """Copy per-parameter gradients into the arena (skips views already in it): one
        multi-tensor kernel (gq_gather_f32), the pointer table travels as its parameter.
        feedback = 1 / 2: `buf` holds the user's error state and becomes grad + scale * error
        (2: written back into the gradient tensors too) -- every tensor is then processed."""
        import ctypes
        buf = self.arena if buf is None else buf
        base = buf.data_ptr()
        ptrs, offs, sizes, keep = [], [], [], []
        for i, t in enumerate(tensors):
            if t.data_ptr() == base + self.tensor_off[i] * 4 and not feedback:
                continue
            if t.dtype != torch.float32 or not t.is_contiguous():
                t = _lib.f32c(t.detach())
                keep.append(t)            # alive until the launch below is queued (stream-ordered free)
            _lib.require_cuda(t, "gradient")
            ptrs.append(t.data_ptr())
            offs.append(self.tensor_off[i])
            sizes.append(self.sizes[i])
        n = len(ptrs)
        if n:
            _lib.call("gq_gather_f32", (ctypes.c_void_p * n)(*ptrs), (ctypes.c_int64 * n)(*offs),
                      (ctypes.c_int64 * n)(*sizes), n, base, int(feedback), float(scale), _lib.stream())

    def compressed_elems(self):
        return sum(g.n for g in self.groups if g.kind != "identity")

    def total_elems(self):
        return sum(self.sizes)

    def wire_bytes(self):
        """Useful (unpadded) bytes of one packed record."""
        b = 0
        for g in self.groups:
            if g.kind == "hsq":
                b += g.n_chunks * g.code_bytes + g.n_chunks * (4 if g.n_bit == 32 else g.l_bytes) + g.n_seg * 8
            elif g.kind == "qsgd":
                b += g.n_chunks * 4 + (g.n * g.bits + 7) // 8
            elif g.kind == "sign":
                b += g.wire_bytes
            elif g.kind == "topk":
                b += g.k_total * 8
            else:
                b += g.n * 4
        return b

    # ------------------------------------------------------------- uniforms ---
    def split_uniform_stream(self, stream, skip=()):
        """Cut a flat uniform stream drawn in the reference's call order (tensor by
        tensor: rand(N/d) per HSQ tensor, rand(size) per QSGD tensor; tensors in
        `skip` consume nothing) into one device array per group."""
        per_group = {id(g): {} for g in self.groups}
        pos = 0
        for i, g in enumerate(self.tensor_group):
            if g.kind == "hsq":
                n = self.sizes[i] // g.dim
            elif g.kind == "qsgd":
                n = self.sizes[i]
            else:
                continue
            if i in skip:
                chunk = torch.zeros(n, dtype=torch.float32)
            else:
                chunk = torch.as_tensor(stream[pos:pos + n], dtype=torch.float32)
                assert chunk.numel() == n, "uniform stream exhausted"
                pos += n
            per_group[id(g)][i] = chunk
        out = {}
        for g in self.groups:
            if per_group[id(g)]:       # in the group's own tensor order (HSQ groups are not in model order)
                out[id(g)] = torch.cat([per_group[id(g)][i] for i in g.tensors]).to(self.device)
        return out, pos

    # --------------------------------------------------------------- encode ---
    def encode(self, user, src=None, uniforms=None, rng_user=None, shared_rng=False, part=None, defer_levels=False):
        """Compress the arena (or `src`, laid out like it) into records[user].
        rng_user: logical user whose Philox stream the stochastic rounding draws from (default: the
        record row); shared_rng: the rank-independent stream instead (second phase of --two-phase).
        defer_levels: on a plan that can_defer_levels(), launch only the search and leave the norm
        quantization to the next decode of this one record, which then computes the levels itself
        (gq_hsq_decode_quantize): the encode loses its grid barrier and tail, the step one kernel
        phase.  Any other use of the record -- reading `records`, another decode, an encode of another
        row -- completes it first with the stand-alone quantizer.  The bytes are the same either way.
        Launches: HSQ 2 per group on the tcgen05 path (search, quantize; 3 with the separate init
        kernel of the exact path), QSGD 1 (chunked) or 3, sign 1, top-k 10; the copy of the identity tensors rides
        in the first HSQ group's first kernel (1 launch of its own when there is no HSQ group)."""
        src = self.arena if src is None else src
        src_ptr = src if isinstance(src, int) else src.data_ptr()   # tensor or raw device address
        rng_user = user if rng_user is None else rng_user
        take = _lib.PHILOX.take_shared if shared_rng else (lambda n: _lib.PHILOX.take(n, rng_user))
        if self._pending is not None:
            if part is None and self._pending[0] == user:
                self._pending = None        # codes, u and keys of that row are about to be overwritten
            else:
                self._complete()            # u_scratch and the keys are shared by every row
        rec = self._records[user]
        st = _lib.stream()
        base = rec.data_ptr()
        ident, carrier = self._rider_pair()
        if part is not None and not hasattr(self, "n_parts"):
            raise _lib.GQError("encode(part=...) needs make_parts() first")
        for g in self.groups:
            gp = src_ptr + g.arena_off * 4
            r = None if uniforms is None else uniforms.get(id(g))
            if part is not None:
                if g.kind == "hsq" and getattr(g, "part_cuts", None) is not None:
                    pr = self._part_range(g, part)
                    if pr is None:
                        continue
                    ta, tb, ca, cb = pr
                    if g is carrier and part == 0:
                        _lib.call("gq_attach_f32_reduce", src_ptr + ident.arena_off * 4, 0, None, 1, ident.n, 0, 0,
                                  base + ident.raw_off)
                    # the same Philox indices as the whole-group call: chunk i of the group draws element offset + i
                    if part == 0:
                        n_rand = g.n_chunks if self.random else 0
                        g._part_rng = take(n_rand) if (n_rand and r is None) else (0, 0)
                    seed, off = g._part_rng
                    _lib.call("gq_hsq_encode", gp + ca * g.dim * 4, cb - ca, g.dim, _lib.ptr(g.codebook), g.K,
                              _lib.ptr(g.part_seg[part]), tb - ta, g.n_bit, self.random,
                              None if r is None else r.data_ptr() + ca * 4, seed, off + (ca if r is None else 0),
                              base + g.codes_off + ca * g.code_bytes, g.code_bytes, base + g.l_off + ca * g.l_bytes,
                              g.l_bytes, base + g.lbub_off + 8 * ta, self.u_scratch.data_ptr() + ca * 4,
                              _lib.ptr(self.workspace), self.workspace.numel(), self.algo, st)
                    continue
                if part != 0:
                    continue
            if g is carrier:   # out = the raw fp32 tensors, copied into the record by the next call
                _lib.call("gq_attach_f32_reduce", src_ptr + ident.arena_off * 4, 0, None, 1, ident.n, 0, 0,
                          base + ident.raw_off)
            if g.kind == "hsq":
                n_rand = g.n_chunks if (self.random and g.n_bit != 32) else 0
                seed, off = take(n_rand) if (n_rand and r is None) else (0, 0)
                if defer_levels and part is None and self.can_defer_levels():
                    _lib.call("gq_hsq_encode_search", gp, g.n_chunks, g.dim, _lib.ptr(g.codebook), g.K,
                              _lib.ptr(g.seg_start), g.n_seg, base + g.codes_off, g.code_bytes,
                              _lib.ptr(self.u_scratch), _lib.ptr(self.workspace), self.workspace.numel(), st)
                    self._pending = (user, g, seed, off, r)
                elif g.n_bit == 32:
                    _lib.call("gq_hsq_encode", gp, g.n_chunks, g.dim, _lib.ptr(g.codebook), g.K,
                              _lib.ptr(g.seg_start), g.n_seg, 32, 0, None, 0, 0, base + g.codes_off,
                              g.code_bytes, None, 4, None, base + g.l_off, _lib.ptr(self.workspace),
                              self.workspace.numel(), self.algo, st)
                else:
                    _lib.call("gq_hsq_encode", gp, g.n_chunks, g.dim, _lib.ptr(g.codebook), g.K,
                              _lib.ptr(g.seg_start), g.n_seg, g.n_bit, self.random, _lib.ptr(r), seed, off,
                              base + g.codes_off, g.code_bytes, base + g.l_off, g.l_bytes,
                              base + g.lbub_off, _lib.ptr(self.u_scratch), _lib.ptr(self.workspace),
                              self.workspace.numel(), self.algo, st)
            elif g.kind == "qsgd":
                seed, off = take(g.n) if (self.random and r is None) else (0, 0)
                _lib.call("gq_qsgd_encode", gp, g.n, _lib.ptr(g.chunk_start), g.n_chunks, g.dim, g.n_bit,
                          self.random, _lib.ptr(r), seed, off, base + g.norm_off, None, None,
                          base + g.packed_off, st)
            elif g.kind == "sign":
                if g.t5:
                    _lib.call("gq_sign_encode_t5", gp, g.n, base + g.packed_off, st)
                else:
                    _lib.call("gq_sign_encode", gp, g.n, None, base + g.packed_off, st)
            elif g.kind == "topk":
                _lib.call("gq_topk_select", gp, g.n, _lib.ptr(g.seg_start), _lib.ptr(g.k),
                          _lib.ptr(g.k_prefix), g.n_seg, None, base + g.idx_off, base + g.val_off,
                          _lib.ptr(self.workspace), self.workspace.numel(), st)
            elif g.kind == "identity":
                if g.n and carrier is None:   # a plain copy of the raw fp32 tensors into the record
                    _lib.call("gq_f32_reduce_users", gp, 0, 1, g.n, 0, 0, base + g.raw_off, st)

    def _rider_pair(self, n_users=1):
        """(identity group, group whose first kernel carries the identity tensors' copy / reduction) or
        (None, None).  Carriers: HSQ, the one-launch sign / QSGD kernels, top-k's setup / fill kernels (their C entry points consume
        a pending gq_attach_f32_reduce; a path without a carrier kernel launches it on its own)."""
        ident = next((g for g in self.groups if g.kind == "identity" and g.n), None)
        # (the largest group: its kernel has the threads to spare -- riding in a group of a few chunks made
        #  that 6 us launch a 60 us one)
        carrier = max((g for g in self.groups if g.kind in ("hsq", "sign", "qsgd", "topk")), key=lambda g: g.n, default=None)
        if ident is None or carrier is None or n_users > 8:
            return None, None
        return ident, carrier

    # --------------------------------------------------------------- decode ---
    def supports_scattered(self):
        """Peer-to-peer decode handles HSQ groups with chunk dim 4/8/16, a codebook of at most
        64 KB and quantized norms, plus the identity tensors."""
        for g in self.groups:
            if g.kind == "identity":
                continue
            if g.kind != "hsq" or g.dim not in (4, 8, 16) or g.K * g.dim * 4 > 65536 or g.n_bit == 32:
                return False
        return True

    def supports_fused_delivery(self):
        """The one-launch tcgen05 encode can deliver the record to the peers itself when the plan is a
        single HSQ group of the headline shape (d = 16, K = 256, uint8 codes and levels) plus identity."""
        import os
        if os.environ.get("GQ_TC_V", "2") == "1" or self.algo == _lib.ALGO_EXACT:
            return False
        hsq = [g for g in self.groups if g.kind != "identity"]
        if len(hsq) != 1 or hsq[0].kind != "hsq":
            return False
        g = hsq[0]
        return (g.dim in (8, 16, 32) and g.K == 256 and g.code_bytes == 1 and g.n_bit <= 7 and g.l_bytes == 1
                and g.n_seg <= 1024 and g.n_chunks > 0)

    def can_defer_levels(self):
        """encode(defer_levels=True) defers the norm quantization on this plan: a single HSQ group of the
        headline shape on the second-generation tcgen05 path (d = 16, K = 256, uint8 codes and levels,
        n_bit <= 7, at most 1024 tensors), not cut into ring parts.  GQ_DEFER_LEVELS=0 turns it off
        (read at every call, so one process can A/B the two)."""
        if os.environ.get("GQ_DEFER_LEVELS", "1") == "0":
            return False
        if os.environ.get("GQ_TC_V", "2") == "1" or self.algo == _lib.ALGO_EXACT:
            return False
        hsq = [g for g in self.groups if g.kind != "identity"]
        if len(hsq) != 1 or hsq[0].kind != "hsq":
            return False
        g = hsq[0]
        return (g.dim == 16 and g.K == 256 and g.code_bytes == 1 and g.l_bytes == 1 and 1 <= g.n_bit <= 7
                and g.n_seg <= 1024 and g.n_chunks > 0 and getattr(g, "part_cuts", None) is None)

    def _complete(self):
        """Write the levels and lb/ub of the record an encode(defer_levels=True) left pending (one
        launch of the stand-alone quantizer over the search's u and min/max keys)."""
        if self._pending is None:
            return
        row, g, seed, off, r = self._pending
        self._pending = None
        base = self._records.data_ptr() + row * self.record_bytes
        _lib.call("gq_norm_quantize", _lib.ptr(self.u_scratch), g.n_chunks, _lib.ptr(g.seg_start), g.n_seg, g.n_bit,
                  self.random, _lib.ptr(r), seed, off, base + g.l_off, g.l_bytes, base + g.lbub_off,
                  _lib.ptr(self.workspace), 1, _lib.stream())

    def supports_inplace_feedback(self):
        """Error feedback without extra sweeps needs decode kernels with the subtract mode
        (accumulate = 2): everything but the top-k scatter."""
        return all(g.kind != "topk" for g in self.groups)

    def decode(self, first_user=0, n_users=None, mean=True, accumulate=False, out=None,
               base_ptr=None, user_offsets=None, part=None):
        """out (arena layout) = [out +] reduce over records[first_user : first_user+n_users].
        base_ptr / user_offsets (ctypes int64 array): user 0's record address and every user's byte
        offset from it, for records that live in different buffers (peer-to-peer exchange)."""
        out = self.arena if out is None else out
        n_users = self.n_users if n_users is None else n_users
        st = _lib.stream()
        mean = 1 if mean else 0
        acc = int(accumulate)            # 0 store, 1 out += decoded, 2 out -= decoded (error feedback)
        ident, carrier = self._rider_pair(n_users)
        pending = self._pending
        if pending is not None and not (user_offsets is None and part is None and n_users == 1
                                        and first_user == pending[0]):
            self._complete()
            pending = None
        if user_offsets is not None:
            for g in self.groups:
                op = out.data_ptr() + g.arena_off * 4
                if g is carrier:
                    _lib.call("gq_attach_f32_reduce", base_ptr + ident.raw_off, 0, user_offsets, n_users, ident.n,
                              mean, acc, out.data_ptr() + ident.arena_off * 4)
                if g.kind == "hsq":
                    _lib.call("gq_hsq_decode_reduce_scattered", base_ptr + g.codes_off, g.code_bytes,
                              base_ptr + g.l_off, g.l_bytes, base_ptr + g.lbub_off, user_offsets, n_users,
                              g.n_chunks, g.dim, _lib.ptr(g.codebook), g.K, _lib.ptr(g.seg_start), g.n_seg,
                              g.n_bit, mean, acc, op, st)
                elif carrier is None:
                    _lib.call("gq_f32_reduce_users_scattered", base_ptr + g.raw_off, user_offsets, n_users, g.n,
                              mean, acc, op, st)
            return out
        base = self._records.data_ptr() + first_user * self.record_bytes
        stride = self.record_bytes
        for g in self.groups:
            op = out.data_ptr() + g.arena_off * 4
            if part is not None:
                if g.kind == "hsq" and getattr(g, "part_cuts", None) is not None:
                    pr = self._part_range(g, part)
                    if pr is None:
                        continue
                    ta, tb, ca, cb = pr
                    if g is carrier and part == 0:
                        _lib.call("gq_attach_f32_reduce", base + ident.raw_off, stride, None, n_users, ident.n, mean, acc,
                                  out.data_ptr() + ident.arena_off * 4)
                    _lib.call("gq_hsq_decode_reduce", base + g.codes_off + ca * g.code_bytes, g.code_bytes,
                              base + g.l_off + ca * g.l_bytes, g.l_bytes, base + g.lbub_off + 8 * ta, None, stride,
                              n_users, cb - ca, g.dim, _lib.ptr(g.codebook), g.K, _lib.ptr(g.part_seg[part]), tb - ta,
                              g.n_bit, mean, acc, op + ca * g.dim * 4, st)
                    continue
                if part != 0:
                    continue
            if g is carrier:
                _lib.call("gq_attach_f32_reduce", base + ident.raw_off, stride, None, n_users, ident.n, mean, acc,
                          out.data_ptr() + ident.arena_off * 4)
            if g.kind == "hsq":
                if pending is not None:
                    _, _, seed, off, r = pending
                    self._pending = None
                    _lib.call("gq_hsq_decode_quantize", base + g.codes_off, base + g.l_off, base + g.lbub_off,
                              _lib.ptr(self.u_scratch), _lib.ptr(self.workspace), g.n_chunks, g.dim,
                              _lib.ptr(g.codebook), g.K, _lib.ptr(g.seg_start), g.n_seg, g.n_bit, self.random,
                              _lib.ptr(r), seed, off, acc, op, st)
                elif g.n_bit == 32:
                    _lib.call("gq_hsq_decode_reduce", base + g.codes_off, g.code_bytes, None, 1, None,
                              base + g.l_off, stride, n_users, g.n_chunks, g.dim, _lib.ptr(g.codebook), g.K,
                              _lib.ptr(g.seg_start), g.n_seg, 32, mean, acc, op, st)
                else:
                    _lib.call("gq_hsq_decode_reduce", base + g.codes_off, g.code_bytes, base + g.l_off,
                              g.l_bytes, base + g.lbub_off, None, stride, n_users, g.n_chunks, g.dim,
                              _lib.ptr(g.codebook), g.K, _lib.ptr(g.seg_start), g.n_seg, g.n_bit, mean,
                              acc, op, st)
            elif g.kind == "qsgd":
                _lib.call("gq_qsgd_decode_reduce", base + g.norm_off, base + g.packed_off, stride, n_users,
                          g.n, _lib.ptr(g.chunk_start), g.n_chunks, g.dim, g.n_bit, mean, acc, op, st)
            elif g.kind == "sign":
                _lib.call("gq_sign_decode_reduce_t5" if g.t5 else "gq_sign_decode_reduce", base + g.packed_off, stride,
                          n_users, g.n, mean, acc, op, st)
            elif g.kind == "topk":
                _lib.call("gq_topk_scatter_reduce", base + g.idx_off, base + g.val_off, stride, n_users,
                          g.k_total, g.n, mean, acc, op, st)
            elif g.kind == "identity" and carrier is None:
                _lib.call("gq_f32_reduce_users", base + g.raw_off, stride, n_users, g.n, mean, acc, op, st)
        return out

    def launches_per_encode(self):
        per = {"hsq": 3, "qsgd": 3, "sign": 1, "topk": 10, "identity": 1}
        n = 0
        for g in self.groups:
            k = per[g.kind]
            if g.kind == "hsq" and g.n_bit == 32:
                k -= 2          # search only
            elif (g.kind == "hsq" and g.dim in (8, 16, 32) and g.K == 256 and g.code_bytes == 1
                  and self.algo != _lib.ALGO_EXACT):
                # tcgen05: the search kernel resets the min/max keys itself; second generation: the norm
                # quantization is its fused tail as well (one launch)
                import os
                v1 = os.environ.get("GQ_TC_V", "2") == "1"
                k -= 1 if (v1 or g.n_seg > 1024 or g.n_bit > 7) else 2
            n += k
        ident, carrier = self._rider_pair()
        if carrier is not None and (carrier.kind != "hsq" or carrier.n_bit != 32):   # the copy rides in the carrier's kernel
            n -= 1
        return n

    def launches_per_decode(self, n_users):
        n = 0
        for g in self.groups:
            n += (2 + n_users) if g.kind == "topk" else 1
        ident, carrier = self._rider_pair(n_users)
        if carrier is not None and (carrier.kind != "hsq" or (
                carrier.dim == 16 and carrier.K == 256 and carrier.code_bytes == 1
                and carrier.l_bytes == 1 and carrier.n_bit != 32)):   # rides in the (staged) decode kernel
            n -= 1
        return n
