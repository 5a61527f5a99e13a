import torch

from .. import _lib
from . import exchange as xch
from ._shared import QuantizerBase, feedback_scale


class RingQuantizer(QuantizerBase):
    """Ring exchange (reference quantizers/ring_quantizer.py:7-49): a lossy running
    SUM passed from user to user, acc_r = D(C(g_r + acc_{r-1})); apply() hands the
    last user's decompressed sum (not divided by the number of users) to every
    parameter.

    Fused path: record(user) decodes records[user-1] straight into the gradient
    arena (decode-accumulate), then packs the sum into records[user].  With one
    user per rank the packed record travels rank r -> r+1 with NCCL send/recv and
    the last rank broadcasts its record; fp32 never crosses NVLink.
    """

    def __init__(self, Compressor, parameters, args):
        super().__init__(Compressor, parameters, args)
        # Pipelined chain (SURVEY 8e): the chain is per tensor, so the plan is cut into stages and rank r
        # works on stage s while rank r + 1 works on stage s - 1: all ranks are busy after U - 1 stages.
        # args.ring_parts / GQ_RING_PARTS; default 4 stages from three ranks on, 2 for two ranks.
        import os
        self.parts = 1
        self.p2p = None
        self._step = 0
        if self.distributed and self.plan is not None and not self.error_feedback:
            self._setup_p2p()
        if self.plan is not None and not self.error_feedback:
            want = getattr(args, "ring_parts", None)
            if want is None:
                want = os.environ.get("GQ_RING_PARTS")
            if want is None:
                # stages pay when a hop costs microseconds (peer-to-peer stores + flags); over NCCL send/recv
                # a hop costs ~50 us and more stages only add hops (measured: 594 / 600 / 606 us per step at
                # 4 ranks with 4 / 1 / 8 stages)
                want = (4 if self.world >= 3 else 2) if self.p2p is not None else 1
            self.parts = self.plan.make_parts(int(want))
        if self.distributed and self.rank == 0:
            import sys
            print("gq_b200: ring exchange = %s" % self.exchange_name(), file=sys.stderr, flush=True)

    def _setup_p2p(self):
        """Hops through peer-mapped memory: the encode kernel of rank r stores each stage of its record
        straight into rank r + 1's receive block and raises a flag the decode-accumulate kernel there
        waits on (the last rank: into every rank's block) -- the ps exchange's machinery, one target per
        hop.  Needs a delivering encode and a plan the peer-to-peer exchange handles (FusedPlan.supports_p2p and
        supports_fused_delivery: HSQ d = 8 / 16 / 32 with K = 256, sign, QSGD / TernGrad) on every rank."""
        import os
        import torch.distributed as dist
        want = getattr(self.args, "p2p", True) and os.environ.get("GQ_P2P", "1") != "0"
        ok = 1 if (want and self.world <= 8 and self.plan.supports_p2p() and self.plan.supports_fused_delivery()) else 0
        p2p, err = None, None
        if ok:
            try:
                from .p2p import PeerRecords
                p2p = PeerRecords(self.plan.record_bytes, self.rank, self.world, self.device)
            except Exception as e:  # noqa: BLE001
                err, ok = e, 0
        flag = torch.tensor([ok], device=self.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if want and err is not None and os.environ.get("GQ_P2P_FALLBACK", "0") != "1":
            raise _lib.GQError("peer-to-peer ring could not be set up on rank %d: %r (GQ_P2P=0: NCCL send/recv, "
                               "GQ_P2P_FALLBACK=1: fall back automatically)" % (self.rank, err))
        if int(flag.item()) == 1:
            self.p2p = p2p
            self.plan.records = p2p.records
        elif p2p is not None:
            p2p.close()

    def _epoch(self, part):
        return self._step * self.parts + part + 1

    def record(self, user, epoch, uniforms=None):
        scale = feedback_scale(self.args, epoch)
        if self.plan is None:
            return self._record_per_parameter(user, scale)
        plan = self.plan
        if self.distributed and user != self.rank:
            raise _lib.GQError("distributed mode: rank %d records user %d only" % (self.rank, self.rank))
        plan.gather(self._grads())
        if self.parts > 1 or self.p2p is not None:
            return self._chain_parts(user, plan.arena, uniforms)
        if user != 0:
            if self.distributed:
                xch.ring_receive_previous(plan.records, user)
            # grad += previous hop's decompressed running sum   (ring_quantizer.py:31-32)
            plan.decode(first_user=user - 1, n_users=1, mean=False, accumulate=True, out=plan.arena)
        n = plan.arena.numel()
        if self.error_feedback and plan.supports_inplace_feedback():
            # E_u = (grad + previous) + scale * E_u in one multi-tensor pass over the arena's views
            # (same order of additions as ring_quantizer.py:32-34), encoded in place, and the decode of
            # the fresh record subtracts itself: E_u = grad' - decompress(compress(grad'))  (:36-38)
            err = self._ef_buffers(user)
            plan.gather(plan.views(), buf=err, feedback=1, scale=scale)
            plan.encode(user, src=err, uniforms=uniforms, rng_user=user)
            plan.decode(first_user=user, n_users=1, mean=False, accumulate=2, out=err)
        elif self.error_feedback:
            err = self._ef_buffers(user)
            _lib.call("gq_axpy", _lib.ptr(plan.arena), _lib.ptr(err), float(scale), n,
                      _lib.ptr(plan.arena), _lib.stream())
            plan.encode(user, uniforms=uniforms, rng_user=user)
            if not hasattr(self, "_scratch_buf"):
                self._scratch_buf = torch.empty_like(plan.arena)
            dec = plan.decode(first_user=user, n_users=1, mean=False, out=self._scratch_buf)
            _lib.call("gq_sub", _lib.ptr(plan.arena), _lib.ptr(dec), n, _lib.ptr(err), _lib.stream())
        else:
            plan.encode(user, uniforms=uniforms, rng_user=user)
        if self.distributed:
            xch.ring_send_next(plan.records, user, self.world)

    def _chain_parts(self, user, buf, uniforms=None):
        """This user's hop of the chain, stage by stage: receive the stage of the previous hop's record,
        add its decode to the local gradient, encode the sum, send the stage on."""
        plan = self.plan
        last = self.args.num_users - 1
        for p in range(self.parts):
            if self.p2p is not None:
                # peer-to-peer hop: wait for the previous rank's flag inside the decode kernel, deliver this
                # stage from inside the encode kernel (to the next rank; the last rank: to everybody)
                if user != 0:
                    wait = self.p2p.attach_wait_for(user - 1, self._epoch(p))
                    plan.decode(first_user=self.p2p.row(user - 1), n_users=1, mean=False, accumulate=True, out=buf, part=p,
                                wait=wait)
                targets = [user + 1] if user < last else [r for r in range(self.world) if r != user]
                delivery = self.p2p.attach_delivery_to(plan, targets, self._epoch(p), with_ident=(p == 0))
                plan.encode(self.p2p.row(), src=buf, uniforms=uniforms, rng_user=user, part=p, delivery=delivery)
                continue
            ranges = plan.part_byte_ranges(p)
            if user != 0:
                if self.distributed:
                    xch.ring_receive_previous_part(plan.records, user, ranges)
                plan.decode(first_user=user - 1, n_users=1, mean=False, accumulate=True, out=buf, part=p)
            plan.encode(user, src=buf, uniforms=uniforms, rng_user=user, part=p)
            if self.distributed:
                xch.ring_send_next_part(plan.records, user, self.world, ranges)

    def step_buffers(self, src, out):
        """One ring step on raw arena-shaped device buffers (bench.py): this rank's hop -- receive the
        previous hop's record, add its decode to the local gradient IN PLACE (ring_quantizer.py:31-32
        mutates param.grad), encode the sum, send it on -- then the broadcast of the last hop and the
        final decode into `out`.  Single process: all users' hops one after the other on `src`."""
        plan = self.plan
        users = [self.rank] if self.distributed else range(self.args.num_users)
        for user in users:
            if self.parts > 1 or self.p2p is not None:
                self._chain_parts(user, src)
                continue
            if user != 0:
                if self.distributed:
                    xch.ring_receive_previous(plan.records, user)
                plan.decode(first_user=user - 1, n_users=1, mean=False, accumulate=True, out=src)
            plan.encode(user, src=src)
            if self.distributed:
                xch.ring_send_next(plan.records, user, self.world)
        return self._final_decode(out)

    def _final_decode(self, out):
        """The last hop's record is what every rank decodes (ring_quantizer.py:45-49)."""
        plan = self.plan
        last = self.args.num_users - 1
        if self.p2p is not None:
            wait = self.p2p.attach_wait_for(last, self._epoch(self.parts - 1)) if self.rank != last else None
            g = plan.decode(first_user=self.p2p.row(last), n_users=1, mean=False, out=out, wait=wait)
            self.p2p.advance()
            self._step += 1
            return g
        if self.distributed:
            xch.ring_broadcast_last(plan.records, self.world)
        return plan.decode(first_user=last, n_users=1, mean=False, out=out)

    def launches_per_step(self):
        """My kernel launches per rank and step: (decode-accumulate +) encode + final decode."""
        # every extra stage of the pipelined chain adds one encode (and one decode-accumulate) launch per
        # partitioned group
        extra = (self.parts - 1) * sum(1 for g in self.plan.groups if getattr(g, "part_cuts", None))
        enc = self.plan.launches_per_encode() + extra
        dec = self.plan.launches_per_decode(1)
        if self.distributed:
            return enc + dec + ((dec + extra) if self.rank > 0 else 0)
        u = self.args.num_users
        return u * enc + (u - 1) * (dec + extra) + dec

    def exchange_name(self):
        if not self.distributed:
            return "none"
        if self.p2p is not None:
            return ("peer-to-peer chain pipelined over %d stage%s of tensors: every stage delivered into the next "
                    "rank's memory by the encode kernel, flags instead of send/recv, the last hop to every rank%s"
                    % (self.parts, "" if self.parts == 1 else "s", " (NVLS multicast)" if self.p2p.mc_base and self.world > 2 else ""))
        if self.parts > 1:
            return "NCCL batched send/recv chain pipelined over %d stages of tensors + broadcast" % self.parts
        return "NCCL send/recv chain + broadcast"

    def _record_per_parameter(self, user, scale):
        for i, param in enumerate(self.parameters):
            if user != 0:
                param.grad.data.add_(self.compressed_gradients[i][-1])
            if self.error_feedback:
                param.grad.data.add_(scale * param.error[user])
                decompressed_g = self.compressors[i].decompress(
                    self.compressors[i].compress(param.grad.data))
                param.error[user].data = param.grad.data - decompressed_g
            else:
                decompressed_g = self.compressors[i].decompress(
                    self.compressors[i].compress(param.grad.data))
            self.compressed_gradients[i].append(decompressed_g)

    def apply(self):
        if self.plan is None:
            for i, param in enumerate(self.parameters):
                param.grad.data = self.compressed_gradients[i][-1]
            for compressed in self.compressed_gradients:
                compressed.clear()
            return
        self._set_grads_from(self._final_decode(self.plan.arena))
