import os
import sys

import torch

from .. import _lib
from . import exchange as xch
from ._shared import QuantizerBase, feedback_scale


class PSQuantizer(QuantizerBase):
    """Parameter-server exchange (reference quantizers/ps_quantizer.py:6-65).

    record(user, epoch): compress that user's gradients (after adding
    scale * error[user] under --ef, and storing the new error).
    apply(): average the users' decompressed gradients, optionally compress the
    average once more (--two-phase), and put the result in param.grad.data.

    Fused path (HSQ, QSGD, sign, top-k, identity): record() packs the whole model
    into records[user]; apply() is one decode-and-average pass over all users.
    With torch.distributed initialised (one user per rank), record(rank) packs the
    local gradient and apply() all-gathers the packed records over NCCL first --
    the packed codes, never fp32 gradients, cross NVLink.
    """

    def __init__(self, Compressor, parameters, args):
        super().__init__(Compressor, parameters, args)
        self.two_phase = self.args.two_phase
        if self.error_feedback and self.two_phase:
            for param in self.parameters:
                param.server_error = torch.zeros_like(param)
        if self.plan is not None and self.two_phase:
            self._phase2_plan = None  # built lazily (a 1-user plan for the averaged gradient)
        self.p2p = None
        self.fused_push = False
        if self.distributed and self.plan is not None:
            self._setup_p2p()
        if self.distributed and self.two_phase:
            # the second compression must give the same result on every rank: one shared Philox seed
            # (rank 0's generator seed), a stream of its own (DESIGN.md section 7)
            import torch.distributed as dist
            box = [_lib.PHILOX.share_seed() if self.rank == 0 else None]
            dist.broadcast_object_list(box, src=0)
            _lib.PHILOX.share_seed(box[0])

    def _setup_p2p(self):
        """Peer-to-peer exchange instead of an NCCL all-gather when every rank can do it
        (args.p2p = False or GQ_P2P=0 turns it off)."""
        import torch.distributed as dist
        want = getattr(self.args, "p2p", True) and os.environ.get("GQ_P2P", "1") != "0"
        ok = 1 if (want and self.world <= 8 and self.plan.supports_scattered()) else 0
        p2p = None
        err = None
        if ok:
            try:
                from .p2p import PeerRecords
                p2p = PeerRecords(self.plan.record_bytes, self.rank, self.world, self.device)
            except Exception as e:  # noqa: BLE001
                err = e
                ok = 0
        flag = torch.tensor([ok], device=self.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if want and err is not None and os.environ.get("GQ_P2P_FALLBACK", "0") != "1":
            # a silent fall-back to NCCL is a 2-3x slower exchange nobody notices: fail loudly unless
            # the caller opted in (GQ_P2P_FALLBACK=1) or turned peer-to-peer off (GQ_P2P=0 / args.p2p=False)
            raise _lib.GQError("peer-to-peer exchange could not be set up on rank %d: %r (set GQ_P2P=0 to use "
                               "the NCCL all-gather, or GQ_P2P_FALLBACK=1 to fall back automatically)" % (self.rank, err))
        if int(flag.item()) == 1:
            self.p2p = p2p
            # "push" (default): store the local record into every peer's block before the barrier
            # (posted NVLink writes), decode locally.  "gather": pull the peers' records after the
            # barrier with a wide-load copy kernel (reads pay a round trip: 15 vs 5 us at N = 2).
            # "direct": the decode kernel pulls the peers' records itself through its cp.async stage.
            self.p2p_mode = os.environ.get("GQ_P2P_MODE", getattr(self.args, "p2p_mode", "push"))
            if self.p2p_mode not in ("push", "gather", "direct"):
                raise _lib.GQError("unknown peer-to-peer mode %r" % (self.p2p_mode,))
            self.plan.records = p2p.records          # [2 * U, record_bytes]: row = parity * U + user
            # push + barrier launches disappear when the encode kernel delivers the record itself
            self.fused_push = (self.p2p_mode == "push" and os.environ.get("GQ_P2P_FUSED", "1") != "0"
                               and self.plan.supports_fused_delivery())
        elif p2p is not None:
            p2p.close()
        if self.rank == 0:
            print("gq_b200: ps exchange = %s" % self.exchange_name(), file=sys.stderr, flush=True)   # stdout stays clean for callers that parse it

    def exchange_name(self):
        if self.p2p is None:
            return "NCCL all-gather"
        if self.p2p_mode == "push":
            how = "NVLS multicast stores" if self.p2p.mc_base else "peer stores"
            return ("push fused into the encode kernel, %s, flags instead of a barrier launch" % how
                    if self.fused_push else "push kernel (%s) + barrier kernel" % how)
        return self.p2p_mode

    def launches_per_step(self):
        """My kernel launches in one encode -> exchange -> decode step (bench.py's gpu_launches)."""
        n = self.plan.launches_per_encode() + self.plan.launches_per_decode(self.world if self.distributed else self.args.num_users)
        if self.p2p is not None:
            n += {"push": 0 if self.fused_push else 2, "gather": 2, "direct": 1}[self.p2p_mode]
        return n

    # ------------------------------------------------------------------ record
    def record(self, user, epoch, uniforms=None):
        scale = feedback_scale(self.args, epoch)
        if self.plan is None:
            return self._record_per_parameter(user, scale)
        plan = self.plan
        if self.distributed and user != self.rank:
            raise _lib.GQError("distributed mode: rank %d records user %d only" % (self.rank, self.rank))
        slot = self.p2p.row() if self.p2p is not None else user   # row of plan.records to write
        grads = self._grads()
        if not self.error_feedback:
            flat = plan.locate(grads)
            if flat is not None:          # gradients already form one arena-shaped buffer: read in place
                self._encode(slot, user, src=flat, uniforms=uniforms)
                return
        if self.error_feedback and plan.supports_inplace_feedback():
            # The user's error state E_u (arena layout) becomes g + scale * E_u inside the gather kernel
            # (ps_quantizer.py:35; written back into param.grad too, which the reference mutates in
            # place), is encoded in place, and the decode of the fresh record subtracts itself from
            # it: E_u = g' - decompress(compress(g'))  (:36-39).  No axpy / sub sweeps, no scratch arena.
            err = self._ef_buffers(user)
            plan.gather(grads, buf=err, feedback=2, scale=scale)
            self._encode(slot, user, src=err, uniforms=uniforms)
            plan.decode(first_user=slot, n_users=1, mean=False, accumulate=2, out=err)
            return
        plan.gather(grads)
        if self.error_feedback:
            err = self._ef_buffers(user)
            n = plan.arena.numel()
            # grad += scale * error[user]   (ps_quantizer.py:35)
            _lib.call("gq_axpy", _lib.ptr(plan.arena), _lib.ptr(err), float(scale), n,
                      _lib.ptr(plan.arena), _lib.stream())
            for p, v in zip(self.parameters, plan.views()):
                p.grad.data = v               # the reference mutates param.grad in place
            self._encode(slot, user, uniforms=uniforms)
            # error[user] = grad - decompress(compress(grad))   (:36-39)
            dec = plan.decode(first_user=slot, n_users=1, mean=False, out=self._scratch())
            _lib.call("gq_sub", _lib.ptr(plan.arena), _lib.ptr(dec), n, _lib.ptr(err), _lib.stream())
        else:
            self._encode(slot, user, uniforms=uniforms)

    def _encode(self, slot, user, src=None, uniforms=None):
        """Fused encode of `user`'s gradient into row `slot`; with the fused peer-to-peer push the same
        launch also delivers the record to every rank and announces the step epoch.  With one user in
        one process the record is decoded right after it is made (apply(), or the error feedback's
        decode), so the norm quantization moves into that decode (FusedPlan.encode(defer_levels=True));
        across processes the levels must exist before the record leaves the GPU."""
        if self.fused_push:
            self.p2p.attach_delivery(self.plan)
        defer = not self.distributed and self.plan.n_users == 1 and self.p2p is None
        self.plan.encode(slot, src=src, uniforms=uniforms, rng_user=user, defer_levels=defer)

    def _scratch(self):
        if not hasattr(self, "_scratch_buf"):
            self._scratch_buf = torch.empty_like(self.plan.arena)
        return self._scratch_buf

    def _record_per_parameter(self, user, scale):
        for i, param in enumerate(self.parameters):
            if self.error_feedback:
                param.grad.data.add_(scale * param.error[user])
                decompressed_g = self.compressors[i].decompress(
                    self.compressors[i].compress(param.grad.data))
                param.error[user].data = param.grad.data - decompressed_g
            else:
                decompressed_g = self.compressors[i].decompress(
                    self.compressors[i].compress(param.grad.data))
            self.compressed_gradients[i].append(decompressed_g)

    # ----------------------------------------------- fused building blocks
    def encode_local(self, user, src=None, uniforms=None):
        """Pack one user's gradient (the arena, or `src` laid out like it) into its record.
        Returns the row of plan.records that was written."""
        slot = self.p2p.row() if self.p2p is not None else user
        self._encode(slot, user, src=src, uniforms=uniforms)
        return slot

    def exchange_and_decode(self, out=None):
        """Make every user's record available and decode-and-average them into `out`
        (default: the arena).  Peer-to-peer: one barrier kernel, the decode kernel reads the
        peers' records over NVLink.  Otherwise: NCCL all-gather (or nothing in one process)."""
        plan = self.plan
        out = plan.arena if out is None else out
        if self.p2p is not None:
            if self.fused_push:
                self.p2p.attach_wait()       # the decode kernel waits for every rank's delivery flag itself
            else:
                if self.p2p_mode == "push":
                    self.p2p.push()
                self.p2p.barrier()
                if self.p2p_mode == "gather":
                    self.p2p.gather()
            g = self.decode_exchanged(out)
            self.p2p.advance()
            return g
        self.exchange()
        return plan.decode(mean=True, out=out)

    def decode_exchanged(self, out=None):
        """Decode-and-average all users' records of the current step (after the exchange)."""
        plan = self.plan
        out = plan.arena if out is None else out
        if self.p2p is None:
            return plan.decode(mean=True, out=out)
        if self.p2p_mode == "direct":
            return plan.decode(n_users=self.world, mean=True, out=out, base_ptr=self.p2p.user0_record_ptr(),
                               user_offsets=self.p2p.user_offsets())
        return plan.decode(first_user=self.p2p.row(0), n_users=self.world, mean=True, out=out)

    # ------------------------------------------------------------------- apply
    def exchange(self):
        """All-gather the packed records: rank r's record is already in slot r."""
        if self.distributed:
            xch.ps_all_gather(self.plan.records, self.rank)

    def apply(self, uniforms=None):
        if self.plan is None:
            return self._apply_per_parameter()
        g = self.exchange_and_decode()
        if self.two_phase:
            g = self._second_phase(g, uniforms)
        self._set_grads_from(g)

    def phase2_plan(self):
        """The 1-user plan that compresses the averaged gradient once more (--two-phase); built lazily."""
        from .fused import FusedPlan
        if self._phase2_plan is None:
            self._phase2_plan = FusedPlan(self.plan.Compressor, self.plan.shapes, self.args, self.device, 1)
        return self._phase2_plan

    def _second_phase(self, g, uniforms):
        """Compress the averaged gradient once more (ps_quantizer.py:52-61).  Every rank
        holds the same average; with identical uniforms (or the shared Philox state)
        every rank computes the same result."""
        p2 = self.phase2_plan()
        n = g.numel()
        if self.error_feedback and p2.supports_inplace_feedback():
            # server_error S becomes g + S (ps_quantizer.py:54), is compressed, and the decode of that
            # record is both stored as the new gradient and subtracted from S (S = g' - D, :57)
            if not hasattr(self, "_server_err"):
                self._server_err = torch.zeros_like(g)
                for p, v in zip(self.parameters, self.plan.views(self._server_err)):
                    p.server_error = v
            p2.gather(self.plan.views(g), buf=self._server_err, feedback=1, scale=1.0)
            p2.encode(0, src=self._server_err, uniforms=uniforms, shared_rng=True, defer_levels=True)
            p2.decode(mean=False, out=g)
            p2.decode(mean=False, accumulate=2, out=self._server_err)
            return g
        if self.error_feedback:
            if not hasattr(self, "_server_err"):
                self._server_err = torch.zeros_like(g)
                for p, v in zip(self.parameters, self.plan.views(self._server_err)):
                    p.server_error = v
            _lib.call("gq_axpy", _lib.ptr(g), _lib.ptr(self._server_err), 1.0, n, _lib.ptr(g), _lib.stream())
        p2.encode(0, src=g, uniforms=uniforms, shared_rng=True, defer_levels=True)
        dec = p2.decode(mean=False, out=self._scratch())
        if self.error_feedback:
            _lib.call("gq_sub", _lib.ptr(g), _lib.ptr(dec), n, _lib.ptr(self._server_err), _lib.stream())
        g.copy_(dec)
        return g

    def _apply_per_parameter(self):
        for i, param in enumerate(self.parameters):
            # stack(...).mean(0) with the reference's CPU semantics: sum in user order,
            # then a true division (torch's CUDA mean multiplies by 1/U instead)
            stacked = torch.stack([_lib.f32c(t) for t in self.compressed_gradients[i]], dim=0)
            g = torch.empty_like(stacked[0])
            _lib.call("gq_f32_reduce_users", _lib.ptr(stacked), g.numel() * 4, stacked.shape[0],
                      g.numel(), 1, 0, _lib.ptr(g), _lib.stream())
            if self.two_phase:
                if self.error_feedback:
                    g.add_(param.server_error)
                    decompressed_g = self.compressors[i].decompress(self.compressors[i].compress(g))
                    param.server_error = g - decompressed_g
                    g = decompressed_g
                else:
                    g = self.compressors[i].decompress(self.compressors[i].compress(g))
            param.grad.data = g
        for compressed in self.compressed_gradients:
            compressed.clear()
