"""HSQ at chunk dim 32 (the reference's default --c-dim) across users and GPUs.

CPU: a d = 32 plan with K = 256 and uint8 codes and levels takes the peer-to-peer decode and carries the
identity tensors in its decode kernel; other d = 32 shapes do not.

GPU: the staged decode-and-average at d = 32, every user count 1..8, against the CPU oracle bit for bit --
with the records equally spaced (gq_hsq_decode_reduce) and scattered at uneven offsets
(gq_hsq_decode_reduce_scattered) -- and against the plain d = 32 kernel (GQ_DECODE_STAGED=0); the launch
count of a fused decode (in a child process); and two processes on one GPU running the ps exchange (push, gather, direct) and
the peer-to-peer ring at c_dim = 32, every rank equal to the oracle's step.
"""
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
from oracle import gq_oracle as O  # noqa: E402
from util import FCN_SHAPES, codebook, gen_input, make_args, resnet50_shapes, torch_uniform_stream  # noqa: E402

D, K, NBIT = 32, 256, 6
P2P_SHAPES = FCN_SHAPES + [(64, 3, 3, 3)]


# ------------------------------------------------------------------------------------------------ CPU ---
def _cpu_plan(shapes, n_users=2, **kw):
    return FusedPlan(gq_b200.NearestNeighborCompressor, shapes, make_args(num_users=n_users, **kw),
                     torch.device("cpu"), n_users)


def test_resnet50_plan_at_d32():
    p = _cpu_plan(resnet50_shapes(), c_dim=32)
    g, ident = p.groups
    assert g.kind == "hsq" and g.key == (32, 256) and g.n_chunks == 734326 and ident.n == 22410
    assert p.record_bytes == 1559552
    assert p.supports_scattered() and p.supports_fused_delivery()
    assert p.launches_per_decode(1) == 1 and p.launches_per_decode(2) == 1


def test_fcn_plan_at_d32():
    p = _cpu_plan(P2P_SHAPES, c_dim=32)
    assert [g.key for g in p.groups if g.kind == "hsq"] == [(32, 256)]
    assert p.supports_scattered() and p.supports_fused_delivery()
    assert p.launches_per_decode(1) == 1 and p.launches_per_decode(2) == 1


@pytest.mark.parametrize("shapes,kw", [
    (resnet50_shapes(), dict(c_dim=32, n_bit=8)),            # int32 levels
    (resnet50_shapes(), dict(c_dim=32, k_bit=12)),           # K = 4096, int32 codes
    (P2P_SHAPES, dict(c_dim=32, n_bit=8)),
    ([(45, 24), (10,)], dict(c_dim=24)),                     # d = 24
    ([(64, 48), (10,)], dict(c_dim=48)),                     # d = 48
], ids=["resnet50-n8", "resnet50-k4096", "fcn-n8", "d24", "d48"])
def test_other_shapes_keep_the_nccl_exchange(shapes, kw):
    assert not _cpu_plan(shapes, **kw).supports_scattered()


# ------------------------------------------------------------------------------------ GPU: the kernel ---
DEV = torch.device("cuda", 0) if torch.cuda.is_available() else None
# chunk counts per tensor.  Group A: 5262 chunks (not a multiple of the 1024-chunk tile), tensor boundaries
# inside 32-chunk warp slots (3001, 3078, ...), a constant tensor (lb == ub) and a tensor with a NaN gradient
# element.  Group B: 511 chunks, shorter than one tile.
GROUP_A = [3001, 77, 2050, 5, 129]
GROUP_B = [300, 211]
CONST_T, NAN_T = 1, 3          # in group A


def _up(x, a=256):
    return (x + a - 1) // a * a


def _records(chunks, U, seed):
    """Oracle-compressed records of U users (codes | levels | lb/ub, sections 256-byte aligned), and
    each user's oracle decode.  Returns (records uint8 [U, stride], layout, decoded [U, n] float32)."""
    cb = codebook(D, K)
    n_chunks, n_seg = sum(chunks), len(chunks)
    l_off = _up(n_chunks)
    lbub_off = 2 * l_off
    stride = _up(lbub_off + 8 * n_seg)
    rec = np.zeros((U, stride), np.uint8)
    dec = np.zeros((U, n_chunks * D), np.float32)
    stream = O.UniformStream(np.random.RandomState(seed).random_sample(U * n_chunks).astype(np.float32))
    for u in range(U):
        c0 = 0
        lbub = np.zeros(2 * n_seg, np.float32)
        for s, n in enumerate(chunks):
            if s == CONST_T and len(chunks) == len(GROUP_A):
                x = np.tile(gen_input(seed + 100 * u + s, D), n)          # every chunk the same: lb == ub
            else:
                x = gen_input(seed + 100 * u + s, n * D)
            codec = O.HSQ(n * D, (n * D,), cb, NBIT, True)
            (lb, ub, lv), codes = codec.compress(x, stream)
            if s == NAN_T and len(chunks) == len(GROUP_A):
                # a NaN gradient element: torch.max propagates it, so the tensor's ub is NaN (so is the
                # encode's max key) and every element of the tensor decodes to NaN
                ub = np.float32(np.nan)
                lv = np.clip(lv, 0, 1 << NBIT)
            d = codec.decompress([(lb, ub, lv), codes]).reshape(-1)
            if s == NAN_T and len(chunks) == len(GROUP_A):
                assert np.isnan(d).all()
            if s == CONST_T and len(chunks) == len(GROUP_A):
                assert lb == ub
            rec[u, c0:c0 + n] = codes.astype(np.uint8)
            rec[u, l_off + c0:l_off + c0 + n] = lv.astype(np.uint8)
            lbub[2 * s], lbub[2 * s + 1] = lb, ub
            dec[u, c0 * D:(c0 + n) * D] = d
            c0 += n
        rec[u, lbub_off:lbub_off + 8 * n_seg] = lbub.view(np.uint8)
    starts = np.concatenate([[0], np.cumsum(chunks)]).astype(np.int64)
    return rec, dict(n_chunks=n_chunks, n_seg=n_seg, l_off=l_off, lbub_off=lbub_off, stride=stride,
                     seg=starts), dec


def _expected(dec, mean, accumulate, init):
    """The reference: the users' decodes summed in user order (then a true division by U), then out +/- r."""
    if mean:
        r = O.ps_mean(dec)
    else:
        r = dec[0].copy()
        for u in range(1, dec.shape[0]):
            r = r + dec[u]
    if accumulate == 1:
        return init + r
    if accumulate == 2:
        return init - r
    return r


def _same(a, b):
    return np.array_equal(a, b, equal_nan=True)


@pytest.fixture(scope="module")
def groups():
    out = {}
    for name, chunks, seed in (("A", GROUP_A, 11), ("B", GROUP_B, 23)):
        rec, lay, dec = _records(chunks, 8, seed)
        out[name] = (torch.from_numpy(rec).to(DEV), lay, dec, torch.from_numpy(lay["seg"]).to(DEV))
    out["cb"] = torch.from_numpy(codebook(D, K)).to(DEV)
    return out


def _call(groups, name, U, mean, accumulate, out, scattered=None):
    """One gq_hsq_decode_reduce (records equally spaced) or, with scattered = (buffer, byte offset of every
    user's record), one gq_hsq_decode_reduce_scattered call into the device tensor `out`."""
    recs, lay, _, seg = groups[name]
    if scattered is None:
        base, tail = recs.data_ptr(), (None, lay["stride"], U)
        fn = "gq_hsq_decode_reduce"
    else:
        buf, offs = scattered
        base = buf.data_ptr() + offs[0]
        tail = ((ctypes.c_int64 * U)(*[o - offs[0] for o in offs[:U]]), U)
        fn = "gq_hsq_decode_reduce_scattered"
    _lib.call(fn, base, 1, base + lay["l_off"], 1, base + lay["lbub_off"], *tail, lay["n_chunks"], D,
              groups["cb"].data_ptr(), K, seg.data_ptr(), lay["n_seg"], NBIT, mean, accumulate, out.data_ptr(),
              _lib.stream())


def _decode(groups, name, U, mean, accumulate, init, scattered=None):
    out = torch.from_numpy(init).to(DEV)
    _call(groups, name, U, mean, accumulate, out, scattered)
    torch.cuda.synchronize()
    return out.cpu().numpy()


def _kernel_names(fn):
    """Names of the kernels (and copies) one call of fn puts on the GPU."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["A", "B"])
@pytest.mark.parametrize("U", [1, 2, 3, 4, 5, 6, 7, 8])
def test_strided_decode_equals_oracle_and_plain_kernel(groups, name, U, monkeypatch):
    _, lay, dec, _ = groups[name]
    init = gen_input(77 + U, lay["n_chunks"] * D)
    for mean in (0, 1):
        for acc in (0, 1, 2):
            got = _decode(groups, name, U, mean, acc, init)
            assert _same(got, _expected(dec[:U], mean, acc, init)), (mean, acc)
            monkeypatch.setenv("GQ_DECODE_STAGED", "0")
            plain = _decode(groups, name, U, mean, acc, init)
            monkeypatch.delenv("GQ_DECODE_STAGED")
            assert _same(got, plain), (mean, acc)
    if name == "A":
        seg = lay["seg"]
        out = _decode(groups, name, U, 1, 0, init).reshape(-1, D)
        assert np.isnan(out[seg[NAN_T]:seg[NAN_T + 1]]).all()
        assert not np.isnan(np.delete(out, np.s_[seg[NAN_T]:seg[NAN_T + 1]], axis=0)).any()


def _uneven(recs, seed):
    """The records (rows of recs) copied into one buffer at uneven, 16-byte aligned offsets, user 0 in the
    middle (distances from it are negative and positive, and not multiples of one another).
    Returns (buffer, byte offset of every user's record)."""
    n, stride = recs.shape
    rs = np.random.RandomState(seed)
    order = list(range(1, n))
    order.insert(len(order) // 2, 0)             # order[i]: the user at position i of the buffer
    offs, pos = [0] * n, 48
    for u in order:
        offs[u] = pos
        pos += stride + 16 * int(rs.randint(1, 40))
    buf = torch.zeros(pos, dtype=recs.dtype, device=recs.device)
    for u in range(n):
        buf[offs[u]:offs[u] + stride].copy_(recs[u])
    return buf, offs


def _scatter(groups, name, seed):
    return _uneven(groups[name][0], seed)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["A", "B"])
def test_scattered_decode_equals_strided(groups, name):
    _, lay, _, _ = groups[name]
    buf, offs = _scatter(groups, name, 5)
    assert min(o - offs[0] for o in offs) < 0 < max(o - offs[0] for o in offs)
    init = gen_input(5, lay["n_chunks"] * D)
    for U in range(1, 9):
        for mean in (0, 1):
            for acc in (0, 1, 2):
                got = _decode(groups, name, U, mean, acc, init, scattered=(buf, offs))
                assert _same(got, _decode(groups, name, U, mean, acc, init)), (U, mean, acc)


@pytest.mark.gpu
def test_scattered_decode_outside_the_staged_conditions_is_refused(groups, monkeypatch):
    _, lay, _, _ = groups["A"]
    buf, offs = _scatter(groups, "A", 6)
    init = np.zeros(lay["n_chunks"] * D, np.float32)
    bad = list(offs)
    bad[1] += 4                                  # user 1's record 4 bytes off a 16-byte boundary
    with pytest.raises(_lib.GQError, match="chunk dim 32 with K = 256"):
        _decode(groups, "A", 2, 1, 0, init, scattered=(buf, bad))
    monkeypatch.setenv("GQ_DECODE_STAGED", "0")
    with pytest.raises(_lib.GQError, match="chunk dim 32 with K = 256"):
        _decode(groups, "A", 2, 1, 0, init, scattered=(buf, offs))


def _encoded_plan(U, seed):
    plan = FusedPlan(gq_b200.NearestNeighborCompressor, P2P_SHAPES, make_args(c_dim=32, num_users=U), DEV, U)
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    for u in range(U):
        plan.encode(u, src=torch.randn(plan.arena_elems, device=DEV, generator=g) * 0.01)
    return plan


@pytest.mark.gpu
@pytest.mark.parametrize("U", [1, 2, 3, 8])
def test_fused_decode_with_the_identity_tensors_equals_plain_kernel(U, monkeypatch):
    """plan.decode at d = 32, the identity tensors' reduction riding in the staged kernel, equals the plain
    kernel followed by a launch of its own for the identity tensors."""
    plan = _encoded_plan(U, 3)
    got = plan.decode(mean=True, out=torch.zeros_like(plan.arena)).clone()
    monkeypatch.setenv("GQ_DECODE_STAGED", "0")
    ref = plan.decode(mean=True, out=torch.zeros_like(plan.arena))
    torch.cuda.synchronize()
    for i, (a, b) in enumerate(zip(plan.views(got), plan.views(ref))):
        assert torch.equal(a, b), i


def _launch_worker(rank, out_dir):
    """Kernel names of one fused decode (records equally spaced, and scattered at uneven offsets) for
    U = 1..8 users, profiled in a fresh process."""
    import json
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    torch.cuda.set_device(0)
    res = {}
    for U in range(1, 9):
        plan = _encoded_plan(U, 10 + U)
        out = torch.empty_like(plan.arena)
        buf, offs = _uneven(plan.records, U)
        rel = (ctypes.c_int64 * U)(*[o - offs[0] for o in offs])
        res[U] = dict(
            strided=_kernel_names(lambda: plan.decode(mean=True, out=out)),
            scattered=_kernel_names(lambda: plan.decode(n_users=U, mean=True, out=out,
                                                        base_ptr=buf.data_ptr() + offs[0], user_offsets=rel)),
            expected=plan.launches_per_decode(U))
    with open(os.path.join(out_dir, "launches.json"), "w") as fh:
        json.dump(res, fh)


@pytest.mark.gpu
def test_fused_decode_is_one_launch_of_the_staged_kernel(tmp_path):
    """One fused decode at d = 32, strided or scattered, is exactly launches_per_decode(U) == 1 kernel: the
    staged one, carrying the identity tensors.  (Profiled in a child process of its own: in a long-running
    test process a later torch.profiler session can come back without CUDA events.)"""
    import json
    mp.start_processes(_launch_worker, args=(str(tmp_path),), nprocs=1, join=True, start_method="spawn")
    res = json.load(open(tmp_path / "launches.json"))
    for U in range(1, 9):
        r = res[str(U)]
        assert r["expected"] == 1, U
        for how in ("strided", "scattered"):
            names = r[how]
            assert len(names) == 1 and "hsq_decode_reduce_staged_d32_kernel<%d>" % U in names[0], (U, how, names)


# ------------------------------------------------------------------------ GPU: two processes, one GPU ---
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out_dir, topology, p2p_mode):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ["GQ_P2P_MODE"] = p2p_mode
    os.environ["GQ_P2P_ALLOC"] = "ipc"     # two ranks on ONE device: CUDA IPC (symmetric memory / NVLS need one GPU per rank)
    import torch.distributed as dist
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    dev = torch.device("cuda", 0)
    sizes = [int(np.prod(s)) for s in P2P_SHAPES]
    a = make_args(mode=topology, num_users=world, c_dim=D, n_bit=NBIT)
    params = [torch.nn.Parameter(torch.zeros(s, device=dev)) for s in P2P_SHAPES]
    q = gq_b200.Quantizer(gq_b200.NearestNeighborCompressor, params, a)
    msg = []
    if q.p2p is None:
        msg.append("peer-to-peer not active")
    if topology == "ps" and p2p_mode == "push" and not q.fused_push:
        msg.append("push not fused into the encode")
    if topology == "ring" and q.parts != 2:
        msg.append("ring stages: %d" % q.parts)
    per_user = sum(n // D for n in sizes if n > 1000)
    codecs = [O.HSQ(n, s, codebook(D, K), NBIT, True) if n > 1000 else O.Identity() for n, s in zip(sizes, P2P_SHAPES)]
    for it in range(3):     # three steps: both record parities and their reuse
        grads = [[gen_input(9100 + 100 * it + 10 * u + i, n).reshape(s) for i, (n, s) in enumerate(zip(sizes, P2P_SHAPES))]
                 for u in range(world)]
        stream = torch_uniform_stream(600 + it, per_user * world)
        for p, g in zip(params, grads[rank]):
            p.grad = torch.from_numpy(g).to(dev)
        parts, _ = q.plan.split_uniform_stream(stream[rank * per_user:(rank + 1) * per_user])
        q.record(rank, epoch=1, uniforms=parts)
        q.apply()
        torch.cuda.synchronize()
        step = O.ps_step if topology == "ps" else O.ring_step
        ref = step(codecs, grads, O.UniformStream(stream))
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


def _two_processes(tmp_path, topology, p2p_mode):
    world = 2
    mp.start_processes(_worker, args=(world, _free_port(), str(tmp_path), topology, p2p_mode), nprocs=world,
                       join=True, start_method="spawn")
    for r in range(world):
        assert open(tmp_path / ("rank%d.txt" % r)).read() == "ok", "rank %d" % r


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["push", "gather", "direct"])
def test_ps_peer_to_peer_d32_two_processes_one_gpu(tmp_path, mode):
    _two_processes(tmp_path, "ps", mode)


@pytest.mark.gpu
def test_ring_peer_to_peer_d32_two_processes_one_gpu(tmp_path):
    _two_processes(tmp_path, "ring", "push")
