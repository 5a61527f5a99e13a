"""Peer-to-peer exchange for SignSGD, QSGD and TernGrad: the encode kernel delivers the packed record to
the peers' copies and raises the flag, the decode kernel waits for it.

CPU: which plans take the peer-to-peer exchange and the fused delivery, and the launch counts.
GPU, one process: a delivery whose remote copy is a second buffer on the same GPU, for every delivering
kernel instantiation; refusals; decodes behind a satisfied wait.
GPU, two processes on one GPU (gloo + CUDA IPC, as tests/test_gpu_p2p.py): ps and ring steps against the
oracle, bit for bit."""
import ctypes
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import gq_b200  # noqa: E402
from gq_b200 import _lib  # noqa: E402
from gq_b200.quantizers.fused import FusedPlan  # noqa: E402
from gq_b200.quantizers.ps_quantizer import PSQuantizer  # noqa: E402
from oracle import gq_oracle as O  # noqa: E402
from util import FCN_SHAPES, gen_input, make_args, resnet50_shapes, torch_uniform_stream  # noqa: E402

CPU = torch.device("cpu")
QSGD_SHAPES = FCN_SHAPES + [(64, 3, 3, 3)]      # chunk dims 128 and 192 at c_dim = 128: two QSGD groups


def _plan(Comp, shapes, users=2, **kw):
    return FusedPlan(Comp, shapes, make_args(**kw), CPU, users)


# ------------------------------------------------------------------------------------ CPU: plans ---
def test_plan_predicates_sign_qsgd_terngrad():
    for wire in ("2bit", "t5"):
        p = _plan(gq_b200.SignSGDCompressor, resnet50_shapes(), sign_wire=wire)
        assert p.supports_p2p() and p.supports_fused_delivery() and not p.supports_scattered()
    q = _plan(gq_b200.QSGDCompressor, resnet50_shapes(), c_dim=128, n_bit=2)
    assert sorted(g.dim for g in q.groups if g.kind == "qsgd") == [128, 192]
    assert q.supports_p2p() and q.supports_fused_delivery() and not q.supports_scattered()
    t = _plan(gq_b200.QSGDCompressor, resnet50_shapes(), c_dim=0, n_bit=1)
    assert [g.dim for g in t.groups if g.kind == "qsgd"] == [0]
    assert t.supports_p2p() and t.supports_fused_delivery()


def test_plan_predicates_reject_topk_and_generic_qsgd():
    k = _plan(gq_b200.TopKSparsificationCompressor, resnet50_shapes())
    assert not k.supports_p2p() and not k.supports_fused_delivery()
    # chunk dim 4096 > 2048: the generic QSGD kernels, exchanged by the push / barrier kernels
    g = _plan(gq_b200.QSGDCompressor, [(4096, 4)], c_dim=4096, n_bit=2)
    assert g.supports_p2p() and not g.supports_fused_delivery()
    # chunk dim 6 (dim % 4 != 0): generic as well
    g6 = _plan(gq_b200.QSGDCompressor, [(600, 6)], c_dim=6, n_bit=2)
    assert g6.supports_p2p() and not g6.supports_fused_delivery()


def test_plan_predicates_hsq_unchanged():
    for kw in (dict(), dict(c_dim=8), dict(c_dim=32)):
        p = _plan(gq_b200.NearestNeighborCompressor, resnet50_shapes(), **kw)
        assert p.supports_p2p() == p.supports_scattered()
        assert p.supports_fused_delivery()
    exact = _plan(gq_b200.NearestNeighborCompressor, resnet50_shapes(), hsq_algo=_lib.ALGO_EXACT)
    assert not exact.supports_fused_delivery() and exact.supports_p2p()


def _ps(plan, mode, fused):
    q = object.__new__(PSQuantizer)
    q.plan, q.distributed, q.world, q.args = plan, True, 2, make_args(num_users=2)
    q.p2p, q.p2p_mode, q.fused_push = object(), mode, fused
    return q


@pytest.mark.parametrize("codec", ["sign", "qsgd", "terngrad"])
def test_launches_per_step_by_exchange_mode(codec):
    Comp, kw = {"sign": (gq_b200.SignSGDCompressor, {}), "qsgd": (gq_b200.QSGDCompressor, dict(c_dim=128, n_bit=2)),
                "terngrad": (gq_b200.QSGDCompressor, dict(c_dim=0, n_bit=1))}[codec]
    plan = _plan(Comp, resnet50_shapes(), **kw)
    local = plan.launches_per_encode() + plan.launches_per_decode(2)
    if codec == "sign":
        assert local == 2                     # one encode launch and one decode launch, as on one GPU
    assert _ps(plan, "push", True).launches_per_step() == local
    assert _ps(plan, "push", False).launches_per_step() == local + 2     # push kernel + barrier kernel
    assert _ps(plan, "gather", False).launches_per_step() == local + 2   # barrier kernel + gather kernel


# ------------------------------------------------------------------ GPU: delivery on one GPU ---
def _up(x, a=256):
    return (x + a - 1) // a * a


def _attach(delta, flag_ptr, epoch, counter, ident_ptr=None, ident_bytes=0, announce=True):
    d = (ctypes.c_int64 * 1)(delta)
    f = (ctypes.c_void_p * 1)(flag_ptr)
    _lib.call("gq_attach_remote_record", 1, 0, d, ident_ptr, ident_bytes, ctypes.cast(f, ctypes.c_void_p),
              1 if announce else 0, epoch)
    _lib.call("gq_attach_delivery_counter", counter)


def _deliver_and_compare(encode, body_bytes, n_ident, seed):
    """encode(grad_step, record_ptr) writes a record of body_bytes (+ identity section): run it without and
    with a delivery into a second buffer on the same GPU, twice (both runs reuse the counter)."""
    dev = torch.device("cuda")
    ident_off = _up(body_bytes)
    S = _up(ident_off + n_ident * 4)
    ident_bytes = _up(n_ident * 4, 16)
    buf = torch.zeros(2, S, dtype=torch.uint8, device=dev)     # row 0: local record, row 1: the "peer's" copy
    ref = torch.zeros(S, dtype=torch.uint8, device=dev)
    fl = torch.zeros(64, dtype=torch.int32, device=dev)        # flag word 0, arrival counter word 16
    idv = torch.randn(max(n_ident, 1), device=dev)
    for step, epoch in enumerate((7, 8)):
        for rec, deliver in ((ref, False), (buf[0], True)):
            if n_ident:
                _lib.call("gq_attach_f32_reduce", idv.data_ptr(), 0, None, 1, n_ident, 0, 0, rec.data_ptr() + ident_off)
            if deliver:
                _attach(S, fl.data_ptr(), epoch, fl.data_ptr() + 64, rec.data_ptr() + ident_off if n_ident else None,
                        ident_bytes if n_ident else 0)
            encode(step, rec.data_ptr())
        torch.cuda.synchronize()
        assert torch.equal(buf[0], ref), "step %d: the local record differs from a run without delivery" % step
        assert torch.equal(buf[1], buf[0]), "step %d: the remote copy differs from the local record" % step
        assert int(fl[0]) == epoch and int(fl[16]) == 0, (step, int(fl[0]), int(fl[16]))


def _grad(n, seed):
    g = torch.from_numpy(gen_input(seed, n)).cuda()
    g[::37] = 0.0                                              # zeros: sign 0, QSGD level 0
    return g


@pytest.mark.gpu
@pytest.mark.parametrize("n", [15, 16, 1000003, 3 * 2 ** 20 + 7])
@pytest.mark.parametrize("n_ident", [0, 22410])
def test_sign_2bit_delivery(n, n_ident):
    grads = [_grad(n, 10 + s) for s in range(2)]
    wire = (n + 3) // 4

    def enc(step, rec):
        _lib.call("gq_sign_encode", grads[step].data_ptr(), n, None, rec, _lib.stream())
    _deliver_and_compare(enc, wire, n_ident, n)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [19, 1000003, 3 * 2 ** 20 + 11])
@pytest.mark.parametrize("n_ident", [0, 22410])
def test_sign_t5_delivery(n, n_ident):
    grads = [_grad(n, 20 + s) for s in range(2)]

    def enc(step, rec):
        _lib.call("gq_sign_encode_t5", grads[step].data_ptr(), n, rec, _lib.stream())
    _deliver_and_compare(enc, int(_lib.value("gq_sign_t5_bytes", n)), n_ident, n)


# every lanes-per-chunk / float4-per-lane variant: dim / 4 <= 8 (8 lanes), <= 32, 64, 128, 256, 512 (32 lanes
# with 1, 2, 4, 8, 16 float4 each), and odd dim / 4 in both lane widths (12: 3, 36: 9, 100: 25)
QSGD_DIMS = [(12, 3001), (32, 2999), (36, 1001), (100, 777), (128, 3001), (192, 1501), (512, 401), (1024, 203),
             (2048, 101)]


@pytest.mark.gpu
@pytest.mark.parametrize("n_bit", [2, 4, 8])          # wire widths 4, 8 and 16 bits
@pytest.mark.parametrize("dim,n_chunks", QSGD_DIMS)
def test_qsgd_chunked_delivery(dim, n_chunks, n_bit):
    n = dim * n_chunks
    bits = _lib.value("gq_qsgd_wire_bits", n_bit)
    grads = [_grad(n, 30 + s) for s in range(2)]
    norm_b = _up(n_chunks * 4)
    packed_b = (n + 3) // 4 * 4 * bits // 8

    def enc(step, rec):
        _lib.call("gq_qsgd_encode", grads[step].data_ptr(), n, None, n_chunks, dim, n_bit, 1, None, 1234 + step, 8,
                  rec, None, None, rec + norm_b, _lib.stream())
    _deliver_and_compare(enc, norm_b + packed_b, 22410 if dim == 128 else 0, n)


@pytest.mark.gpu
@pytest.mark.parametrize("n_ident", [0, 22410])
def test_terngrad_delivery(n_ident):
    # tensor boundaries inside warp spans (512 elements) and CTA ranges, and a section ending mid-word
    sizes = [1001, 5000, 777, 300001, 33, 4096, 1500000, 2049]
    n = sum(sizes)
    starts = torch.tensor(np.concatenate([[0], np.cumsum(sizes)]), dtype=torch.int64, device="cuda")
    grads = [_grad(n, 40 + s) for s in range(2)]
    norm_b = _up(len(sizes) * 4)
    packed_b = (n + 3) // 4 * 2

    def enc(step, rec):
        _lib.call("gq_qsgd_encode", grads[step].data_ptr(), n, starts.data_ptr(), len(sizes), 0, 1, 1, None, 99 + step,
                  3, rec, None, None, rec + norm_b, _lib.stream())
    _deliver_and_compare(enc, norm_b + packed_b, n_ident, n)


@pytest.mark.gpu
def test_delivery_refused_by_generic_qsgd_and_topk():
    dev = torch.device("cuda")
    S = 1 << 16
    buf = torch.zeros(2, S, dtype=torch.uint8, device=dev)
    fl = torch.zeros(64, dtype=torch.int32, device=dev)
    g = _grad(600, 5)
    for call in (
        # dim % 4 != 0: the generic QSGD kernels
        lambda: _lib.call("gq_qsgd_encode", g.data_ptr(), 600, None, 100, 6, 2, 0, None, 0, 0, buf[0].data_ptr(), None,
                          None, buf[0].data_ptr() + 1024, _lib.stream()),
        # unpacked outputs
        lambda: _lib.call("gq_qsgd_encode", g.data_ptr(), 512, None, 4, 128, 2, 0, None, 0, 0, buf[0].data_ptr(),
                          buf[0].data_ptr() + 1024, buf[0].data_ptr() + 4096, None, _lib.stream()),
        # fp32 sign output
        lambda: _lib.call("gq_sign_encode", g.data_ptr(), 600, buf[0].data_ptr(), None, _lib.stream()),
        # top-k has no delivering encode
        lambda: _lib.call("gq_topk_select", g.data_ptr(), 600, None, None, None, 1, None, None, None, None, 0,
                          _lib.stream()),
    ):
        _attach(S, fl.data_ptr(), 3, fl.data_ptr() + 64)
        with pytest.raises(_lib.GQError, match=r"failed \(3\)"):
            call()
        # the pending delivery is gone: the next plain encode runs as without one
        _lib.call("gq_sign_encode", g.data_ptr(), 600, None, buf[0].data_ptr(), _lib.stream())
        torch.cuda.synchronize()
        assert int(buf[1].count_nonzero()) == 0 and int(fl[0]) == 0
    # a sign / QSGD delivery without an arrival counter is a caller error
    d = (ctypes.c_int64 * 1)(S)
    f = (ctypes.c_void_p * 1)(fl.data_ptr())
    _lib.call("gq_attach_remote_record", 1, 0, d, None, 0, ctypes.cast(f, ctypes.c_void_p), 1, 3)
    with pytest.raises(_lib.GQError, match="counter"):
        _lib.call("gq_sign_encode", g.data_ptr(), 600, None, buf[0].data_ptr(), _lib.stream())
    with pytest.raises(_lib.GQError):
        _lib.call("gq_attach_delivery_counter", fl.data_ptr() + 64)      # nothing attached


def _gpu_plan(kind, users):
    Comp, kw = {"sign": (gq_b200.SignSGDCompressor, {}), "t5": (gq_b200.SignSGDCompressor, dict(sign_wire="t5")),
                "qsgd": (gq_b200.QSGDCompressor, dict(c_dim=128, n_bit=2)),
                "qsgd8": (gq_b200.QSGDCompressor, dict(c_dim=128, n_bit=4)),
                "terngrad": (gq_b200.QSGDCompressor, dict(c_dim=0, n_bit=1))}[kind]
    plan = FusedPlan(Comp, QSGD_SHAPES, make_args(num_users=users, **kw), torch.device("cuda"), users)
    for u in range(users):
        for i, v in enumerate(plan.views()):
            v.copy_(torch.from_numpy(gen_input(300 + 10 * u + i, v.numel())).view_as(v))
        plan.encode(u)
    return plan


def _satisfied_wait():
    fl = torch.full((8,), 5, dtype=torch.int32, device="cuda")

    def wait():
        _lib.call("gq_attach_peer_wait", fl.data_ptr(), 2, 5)
    return wait, fl


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["sign", "t5", "qsgd", "qsgd8", "terngrad"])
@pytest.mark.parametrize("users", [1, 2, 3])
def test_decode_behind_satisfied_wait_is_bit_identical(kind, users):
    plan = _gpu_plan(kind, users)
    wait, fl = _satisfied_wait()
    for acc in (0, 1):
        base = torch.randn_like(plan.arena)
        a = plan.decode(mean=True, accumulate=acc, out=base.clone())
        b = plan.decode(mean=True, accumulate=acc, out=base.clone(), wait=wait)
        torch.cuda.synchronize()
        assert torch.equal(a, b), (kind, users, acc)
    # a generic QSGD decode (16-byte misaligned output) waits in a one-warp kernel of its own
    g = next(g for g in plan.groups if g.kind in ("sign", "qsgd"))
    if g.kind == "qsgd":
        out = torch.zeros(g.n + 1, device="cuda")
        res = []
        for w in (False, True):
            if w:
                wait()
            _lib.call("gq_qsgd_decode_reduce", plan.records.data_ptr() + g.norm_off, plan.records.data_ptr() + g.packed_off,
                      plan.record_bytes, users, g.n, _lib.ptr(g.chunk_start), g.n_chunks, g.dim, g.n_bit, 1, 0,
                      out.data_ptr() + 4, _lib.stream())
            res.append(out.clone())
        torch.cuda.synchronize()
        assert torch.equal(res[0], res[1])


def _launch_worker(rank, out_dir):
    import json
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    torch.cuda.set_device(0)
    from torch.profiler import ProfilerActivity, profile
    res = {}
    for kind in ("sign", "t5", "qsgd", "terngrad"):
        plan = _gpu_plan(kind, 2)
        wait, fl = _satisfied_wait()
        out = torch.empty_like(plan.arena)
        plan.decode(mean=True, out=out, wait=wait)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            plan.decode(mean=True, out=out, wait=wait)
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        res[kind] = dict(names=names, expected=plan.launches_per_decode(2))
    with open(os.path.join(out_dir, "launches.json"), "w") as fh:
        json.dump(res, fh)


@pytest.mark.gpu
def test_waiting_decode_adds_no_launch(tmp_path):
    """A decode behind a wait launches exactly launches_per_decode(U) kernels: the wait is in the decode
    kernels' prologue, not a kernel of its own (profiled in a child process of its own)."""
    import json
    mp.start_processes(_launch_worker, args=(str(tmp_path),), nprocs=1, join=True, start_method="spawn")
    res = json.load(open(tmp_path / "launches.json"))
    for kind, r in res.items():
        assert len(r["names"]) == r["expected"], (kind, r)
        assert not any("peer_wait" in n for n in r["names"]), (kind, r)


# ----------------------------------------------------------- GPU: two processes on one GPU ---
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


CODECS = {
    "sign": (dict(), lambda n, s: O.Sign(n, s)),
    "t5": (dict(sign_wire="t5"), lambda n, s: O.Sign(n, s)),
    "qsgd": (dict(c_dim=128, n_bit=2), lambda n, s: O.QSGD(n, s, 128, 2, True)),
    "terngrad": (dict(c_dim=0, n_bit=1), lambda n, s: O.QSGD(n, s, 0, 1, True)),
}


def _worker(rank, world, port, out_dir, topology, codec, mode, fused, ef):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ["GQ_P2P_MODE"] = mode
    os.environ["GQ_P2P_FUSED"] = "1" if fused else "0"
    os.environ["GQ_P2P_ALLOC"] = "ipc"     # two ranks on ONE device: CUDA IPC
    import torch.distributed as dist
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    dev = torch.device("cuda", 0)
    kw, oracle = CODECS[codec]
    Comp = gq_b200.SignSGDCompressor if codec in ("sign", "t5") else gq_b200.QSGDCompressor
    sizes = [int(np.prod(s)) for s in QSGD_SHAPES]
    a = make_args(mode=topology, num_users=world, ef=ef, **kw)
    params = [torch.nn.Parameter(torch.zeros(s, device=dev)) for s in QSGD_SHAPES]
    msg = []
    try:
        q = gq_b200.Quantizer(Comp, params, a)
    except _lib.GQError as e:
        with open(os.path.join(out_dir, "rank%d.txt" % rank), "w") as fh:
            fh.write("GQError: %s" % e)
        dist.destroy_process_group()
        return
    if q.p2p is None:
        msg.append("peer-to-peer not active")
    if topology == "ps" and mode == "push" and q.fused_push != fused:
        msg.append("fused_push is %s" % q.fused_push)
    per_user = sum(n for n in sizes if n > 1000) if Comp is gq_b200.QSGDCompressor else 0
    codecs = [oracle(n, s) if n > 1000 else O.Identity() for n, s in zip(sizes, QSGD_SHAPES)]
    errs = [[np.zeros(s, dtype=np.float32) for s in QSGD_SHAPES] for _ in range(world)] if ef else None
    for it in range(3):     # three steps: both record parities and their reuse
        grads = [[gen_input(9300 + 100 * it + 10 * u + i, n).reshape(s) for i, (n, s) in enumerate(zip(sizes, QSGD_SHAPES))]
                 for u in range(world)]
        stream = torch_uniform_stream(700 + it, per_user * world)
        for p, g in zip(params, grads[rank]):
            p.grad = torch.from_numpy(g).to(dev)
        parts, _ = q.plan.split_uniform_stream(stream[rank * per_user:(rank + 1) * per_user])
        q.record(rank, epoch=1, uniforms=parts)
        q.apply()
        torch.cuda.synchronize()
        if topology == "ps":
            ref = O.ps_step(codecs, grads, O.UniformStream(stream), ef_errors=errs, scale=O.ps_scale(1) if ef else 0.0)
        else:
            ref = O.ring_step(codecs, grads, O.UniformStream(stream))
        for i, (p, r) in enumerate(zip(params, ref)):
            got = p.grad.data.cpu().numpy()
            if not np.array_equal(got, r.reshape(got.shape)):
                msg.append("step %d tensor %d differs from the oracle" % (it, i))
    with open(os.path.join(out_dir, "rank%d.txt" % rank), "w") as fh:
        fh.write("; ".join(msg) or "ok")
    dist.barrier()
    if q.p2p is not None:
        q.p2p.close()
    dist.destroy_process_group()


def _two_processes(tmp_path, topology, codec, mode="push", fused=True, ef=False):
    world = 2
    mp.start_processes(_worker, args=(world, _free_port(), str(tmp_path), topology, codec, mode, fused, ef),
                       nprocs=world, join=True, start_method="spawn")
    return [open(tmp_path / ("rank%d.txt" % r)).read() for r in range(world)]


@pytest.mark.gpu
@pytest.mark.parametrize("mode,fused", [("push", True), ("push", False), ("gather", False)])
@pytest.mark.parametrize("codec", ["sign", "t5", "qsgd", "terngrad"])
def test_ps_peer_to_peer_two_processes_one_gpu(tmp_path, codec, mode, fused):
    assert _two_processes(tmp_path, "ps", codec, mode, fused) == ["ok", "ok"]


@pytest.mark.gpu
@pytest.mark.parametrize("codec", ["sign", "qsgd"])
def test_ring_peer_to_peer_two_processes_one_gpu(tmp_path, codec):
    assert _two_processes(tmp_path, "ring", codec) == ["ok", "ok"]


@pytest.mark.gpu
def test_ps_qsgd_error_feedback_peer_to_peer(tmp_path):
    assert _two_processes(tmp_path, "ps", "qsgd", ef=True) == ["ok", "ok"]


@pytest.mark.gpu
def test_direct_mode_refused_for_sign(tmp_path):
    res = _two_processes(tmp_path, "ps", "sign", mode="direct")
    assert all(r.startswith("GQError") and "direct" in r for r in res), res
