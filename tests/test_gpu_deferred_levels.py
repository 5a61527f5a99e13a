"""GPU: deferred levels (FusedPlan.encode(defer_levels=True) + gq_hsq_decode_quantize).

With one user in one process the HSQ encode launches only the search and the decode of the record computes
the levels itself.  Every case here runs the same work with GQ_DEFER_LEVELS=0 (the one-launch encode with
its fused tail, then the plain decode) and with deferral, and requires the same bytes: the whole record
(codes, levels, lb/ub, identity section) and the decoded output -- and, where the draws are known, the
levels of the CPU oracle.
"""
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import gq_b200  # noqa: E402
from gq_b200 import _lib  # noqa: E402
from gq_b200.quantizers.fused import FusedPlan  # noqa: E402
from oracle import gq_oracle as O  # noqa: E402
from philox_ref import philox_uniforms  # noqa: E402
from util import make_args, resnet50_shapes  # noqa: E402

DEV = torch.device("cuda", 0)
SEED = 0x5DEECE66D
OFFSETS = [0, 1, 2, 3, (1 << 34) + 1]
# 5257 chunks: the last 1024-chunk tile is partly filled and n_chunks % 4 == 1; one constant tensor and one
# all-zero tensor (lb == ub); two identity tensors ride along
SMALL_SHAPES = [(3001, 16), (10,), (77, 16), (2050, 16), (300,), (129, 16)]


def _plan(shapes, n_users=1, **kw):
    return FusedPlan(gq_b200.NearestNeighborCompressor, shapes, make_args(num_users=n_users, **kw), DEV, n_users)


def _input(plan, seed, special=False):
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    x = torch.randn(plan.arena_elems, device=DEV, generator=g) * 0.01
    if special:
        views = plan.views(x)
        views[0].copy_(views[0][:1].expand_as(views[0]))   # every chunk the same: one u value, lb == ub
        views[2].zero_()                                    # u == 0 throughout: lb == ub == 0
    return x


def _fixed_stream(monkeypatch, off):
    monkeypatch.setattr(_lib.PHILOX, "take", lambda n, user=0: (SEED, off))


def _run(plan, monkeypatch, defer, fn):
    monkeypatch.setenv("GQ_DEFER_LEVELS", "1" if defer else "0")
    out = fn()
    torch.cuda.synchronize()
    return out


def _encode_decode(plan, x, uniforms=None, accumulate=0, init=None, defer=True):
    out = torch.zeros_like(plan.arena) if init is None else init.clone()
    plan.encode(0, src=x, uniforms=uniforms, defer_levels=defer)
    assert (plan._pending is not None) == (defer and plan.can_defer_levels())
    plan.decode(first_user=0, n_users=1, mean=False, accumulate=accumulate, out=out)
    assert plan._pending is None
    return plan.records[0].clone(), out


def _both(plan, monkeypatch, *args, **kw):
    ref = _run(plan, monkeypatch, False, lambda: _encode_decode(plan, *args, **kw))
    got = _run(plan, monkeypatch, True, lambda: _encode_decode(plan, *args, **kw))
    assert torch.equal(got[0], ref[0]), "record differs from the one-launch encode"
    assert torch.equal(got[1], ref[1]), "decoded output differs from the one-launch encode"
    return got


def _check_oracle(plan, rec, r_all):
    """levels and lb/ub of every tensor against O.psc_compress on the search's u."""
    g = plan.groups[0]
    u = plan.u_scratch[:g.n_chunks].cpu().numpy()
    rec = rec.cpu().numpy()
    l = rec[g.l_off:g.l_off + g.n_chunks].astype(np.int32)
    lbub = rec[g.lbub_off:g.lbub_off + 8 * g.n_seg].view(np.float32)
    starts = g.seg_start_host
    for s in range(g.n_seg):
        a, b = starts[s], starts[s + 1]
        olb, oub, ol, _ = O.psc_compress(u[a:b], g.n_bit, True, r_all[a:b])
        assert lbub[2 * s] == olb and lbub[2 * s + 1] == oub, s
        assert np.array_equal(l[a:b], ol), s


@pytest.fixture(scope="module")
def resnet():
    plan = _plan(resnet50_shapes())
    return plan, _input(plan, 3)


@pytest.mark.parametrize("off", OFFSETS)
def test_resnet50_philox(resnet, off, monkeypatch):
    plan, x = resnet
    _fixed_stream(monkeypatch, off)
    rec, _ = _both(plan, monkeypatch, x)
    _check_oracle(plan, rec, philox_uniforms(SEED, off, plan.groups[0].n_chunks))


def test_resnet50_external_uniforms(resnet, monkeypatch):
    plan, x = resnet
    g = plan.groups[0]
    r = np.random.RandomState(5).random_sample(g.n_chunks).astype(np.float32)
    rec, _ = _both(plan, monkeypatch, x, uniforms={id(g): torch.from_numpy(r).to(DEV)})
    _check_oracle(plan, rec, r)


@pytest.mark.parametrize("accumulate", [0, 1, 2])
def test_resnet50_accumulate(resnet, accumulate, monkeypatch):
    plan, x = resnet
    _fixed_stream(monkeypatch, 2)
    _both(plan, monkeypatch, x, accumulate=accumulate, init=_input(plan, 9))


@pytest.mark.parametrize("n_bit", [1, 2, 3, 4, 5, 6, 7])
@pytest.mark.parametrize("off", [0, 3])
def test_small_partial_tile_constant_tensors(n_bit, off, monkeypatch):
    plan = _plan(SMALL_SHAPES, n_bit=n_bit)
    g = plan.groups[0]
    assert g.n_chunks % 1024 != 0 and g.n_chunks % 4 == 1 and plan.can_defer_levels()
    _fixed_stream(monkeypatch, off)
    rec, _ = _both(plan, monkeypatch, _input(plan, 4, special=True))
    _check_oracle(plan, rec, philox_uniforms(SEED, off, g.n_chunks))


def test_small_external_uniforms_partial_tile(monkeypatch):
    plan = _plan(SMALL_SHAPES)
    g = plan.groups[0]
    r = np.random.RandomState(6).random_sample(g.n_chunks).astype(np.float32)
    rec, _ = _both(plan, monkeypatch, _input(plan, 4, special=True), uniforms={id(g): torch.from_numpy(r).to(DEV)})
    _check_oracle(plan, rec, r)


def test_reading_records_completes_the_record(monkeypatch):
    plan = _plan(SMALL_SHAPES)
    x = _input(plan, 7)
    _fixed_stream(monkeypatch, 1)
    plan.records.fill_(0xEE)                   # (the padding between sections keeps this in both runs)
    ref_rec, ref_out = _run(plan, monkeypatch, False, lambda: _encode_decode(plan, x, defer=False))
    monkeypatch.setenv("GQ_DEFER_LEVELS", "1")
    plan.records.fill_(0xEE)
    plan.encode(0, src=x, defer_levels=True)
    assert plan._pending is not None
    mid = plan.records[0].clone()              # completes the record (stand-alone quantizer)
    assert plan._pending is None
    out = torch.zeros_like(plan.arena)
    plan.decode(first_user=0, n_users=1, mean=False, out=out)
    torch.cuda.synchronize()
    assert torch.equal(mid, ref_rec) and torch.equal(plan.records[0], ref_rec) and torch.equal(out, ref_out)


def test_two_encodes_without_a_decode(monkeypatch):
    plan = _plan(SMALL_SHAPES, n_users=2)
    x1, x2, x3 = _input(plan, 11), _input(plan, 12), _input(plan, 13)

    def seq(defer):
        plan.records.zero_()
        plan.encode(0, src=x1, defer_levels=defer)     # overwritten before anyone decodes it
        plan.encode(0, src=x2, defer_levels=defer)
        plan.encode(1, src=x3, defer_levels=defer)     # another row: completes row 0 first
        out = torch.zeros_like(plan.arena)
        plan.decode(first_user=1, n_users=1, mean=False, out=out)
        return plan.records.clone(), out

    _fixed_stream(monkeypatch, 0)
    ref = _run(plan, monkeypatch, False, lambda: seq(False))
    got = _run(plan, monkeypatch, True, lambda: seq(True))
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])


# ------------------------------------------------------------------------------------- through the quantizer ---
def _quantizer_step(shapes, defer, monkeypatch, **kw):
    monkeypatch.setenv("GQ_DEFER_LEVELS", "1" if defer else "0")
    torch.manual_seed(1)
    _lib.PHILOX.share_seed()          # the --two-phase stream restarts at offset 0 in both runs
    params = [torch.nn.Parameter(torch.zeros(s, device=DEV)) for s in shapes]
    q = gq_b200.Quantizer(gq_b200.NearestNeighborCompressor, params, make_args(num_users=1, **kw))
    g = torch.Generator(device=DEV)
    g.manual_seed(21)
    res = []
    for epoch in (1, 2):
        for p in params:
            p.grad = torch.randn(p.shape, device=DEV, generator=g) * 0.01
        q.record(0, epoch=epoch)
        if defer:   # error feedback: record() has decoded the fresh record already (accumulate = 2)
            assert (q.plan._pending is None) == bool(kw.get("ef"))
        q.apply()
        res += [p.grad.detach().clone() for p in params]
        if kw.get("ef"):
            res += [p.error[0].detach().clone() for p in params]
        if kw.get("ef") and kw.get("two_phase"):
            res += [p.server_error.detach().clone() for p in params]
    torch.cuda.synchronize()
    return res


@pytest.mark.parametrize("ef,two_phase", [(False, False), (True, False), (False, True), (True, True)])
def test_quantizer_error_feedback_and_two_phase(ef, two_phase, monkeypatch):
    """record() / apply(): error feedback (decode with accumulate = 2 right after the encode) and the
    second compression of --two-phase (phase-2 plan), deferred and not."""
    shapes = resnet50_shapes()
    ref = _quantizer_step(shapes, False, monkeypatch, ef=ef, two_phase=two_phase)
    got = _quantizer_step(shapes, True, monkeypatch, ef=ef, two_phase=two_phase)
    assert len(got) == len(ref)
    for i, (a, b) in enumerate(zip(got, ref)):
        assert torch.equal(a, b), i


def test_quantizer_step_launches(monkeypatch):
    """encode_local + exchange_and_decode (what bench.py times) issues launches_per_step() kernels: 1 + 1."""
    monkeypatch.setenv("GQ_DEFER_LEVELS", "1")
    shapes = resnet50_shapes()
    params = [torch.nn.Parameter(torch.zeros(s, device=DEV)) for s in shapes]
    q = gq_b200.Quantizer(gq_b200.NearestNeighborCompressor, params, make_args(num_users=1))
    x = _input(q.plan, 8)
    out = torch.empty_like(x)
    for _ in range(2):
        q.encode_local(0, src=x)
        q.exchange_and_decode(out=out)
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        q.encode_local(0, src=x)
        assert q.plan._pending is not None
        q.exchange_and_decode(out=out)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert len(names) == q.launches_per_step() == 2, names
    assert any("hsq_decode_reduce_staged_kernel<1, true>" in n for n in names), names


def test_eligibility(monkeypatch):
    monkeypatch.setenv("GQ_DEFER_LEVELS", "1")
    assert _plan(SMALL_SHAPES).can_defer_levels()
    assert not _plan([(3001, 32), (64, 32)], c_dim=32).can_defer_levels()           # d = 32
    p = _plan([(1024, 16), (2048, 16), (1024, 16)])
    assert p.can_defer_levels() and p.make_parts(2) == 2
    assert not p.can_defer_levels()                                                 # cut into ring parts
    p.encode(0, src=_input(p, 1), part=0, defer_levels=True)
    assert p._pending is None
    monkeypatch.setenv("GQ_TC_V", "1")
    assert not _plan(SMALL_SHAPES).can_defer_levels()
    monkeypatch.delenv("GQ_TC_V")
    monkeypatch.setenv("GQ_DEFER_LEVELS", "0")
    assert not _plan(SMALL_SHAPES).can_defer_levels()
    monkeypatch.setenv("GQ_DEFER_LEVELS", "1")
    # several users in one process: the quantizer does not defer
    params = [torch.nn.Parameter(torch.zeros(s, device=DEV)) for s in SMALL_SHAPES]
    q = gq_b200.Quantizer(gq_b200.NearestNeighborCompressor, params, make_args(num_users=2))
    for p in params:
        p.grad = torch.randn(p.shape, device=DEV) * 0.01
    q.record(0, epoch=1)
    assert q.plan._pending is None
    q.record(1, epoch=1)
    q.apply()
