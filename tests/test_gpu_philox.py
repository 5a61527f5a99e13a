"""The built-in Philox stream, bit for bit.

When no uniforms are passed (random = 1, uniforms == NULL), every stochastic rounding draws from the
in-kernel Philox4x32-10 stream of include/gqb200.h: draw i of a call is word (offset + i) & 3 of the
block at counter (offset + i) >> 2, key = philox_seed.  Training and the benchmark run on this stream.
Each kernel that draws is run here on it and compared with the CPU oracle fed with the draws of the
host reference (tests/philox_ref.py), at offsets that take both the aligned (offset % 4 == 0) and the
unaligned draw branches, and one whose block counter needs its high word (2^34 + 1).  The second half
checks the seeding contract of DESIGN.md section 7 through the Python surface: which key and offset
each record() / phase-2 compression draws from, and that rng = "torch" replays the CPU generator.
"""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for _p in (ROOT, HERE):          # also run as a script (the GQ_TC_FUSED=1 child process below)
    if _p not in sys.path:
        sys.path.insert(0, _p)

import gq_b200  # noqa: E402
from gq_b200 import _lib  # noqa: E402
from oracle import gq_oracle as O  # noqa: E402
from philox_ref import ceil4, mix64, philox_uniforms  # noqa: E402
from util import codebook, gen_input, make_args, torch_uniform_stream  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda"
SEED = 0x5DEECE66D1234567        # both 32-bit halves non-zero
SEED2 = 0x0123456789ABCDEF
OFFSETS = [0, 1, 2, 3, (1 << 34) + 1]
INT32_MIN = np.int32(-2 ** 31)


def _t(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


def _first_diff(a, b):
    d = np.flatnonzero(np.asarray(a) != np.asarray(b))
    return None if d.size == 0 else (int(d[0]), a[d[0]], b[d[0]], int(d.size))


def _check_levels(u, starts, n_bit, seed, off, lbub, l):
    """lb/ub and l of every segment s against O.psc_compress fed with philox_uniforms(seed, off + start_s, len_s)
    (a slice of the draws of the whole range: the same numbers, see test_philox_ref.py)."""
    r_all = philox_uniforms(seed, off, u.size)
    for s in range(len(starts) - 1):
        a, b = int(starts[s]), int(starts[s + 1])
        olb, oub, ol, _ = O.psc_compress(u[a:b], n_bit, True, r_all[a:b])
        assert lbub[2 * s] == olb and lbub[2 * s + 1] == oub, (s, lbub[2 * s:2 * s + 2], olb, oub)
        got = l[a:b].astype(np.int32)
        assert np.array_equal(got, ol), ("segment", s, "first mismatch", _first_diff(got, ol))


# ------------------------------------------------------------------------------------ norm quantizer ---
def _starts_with_edges(rs, n, n_seg):
    """n_seg segments over n items: random cuts plus two segments of length 1."""
    cuts = set(rs.choice(np.arange(20, n), n_seg - 3, replace=False).tolist()) | {10, 11, 12}
    while len(cuts) < n_seg - 1:
        cuts.add(int(rs.randint(20, n)))
    return np.array([0] + sorted(cuts)[:n_seg - 1] + [n], dtype=np.int64)


def _norm_quantize(u, starts, n_bit, l_bytes, seed, off, shift=0):
    """gq_norm_quantize on u (optionally at u / l pointers moved by 4 bytes): (lbub, l as int32)."""
    n, n_seg = u.size, len(starts) - 1
    ubuf = torch.zeros(n + 8, device=DEV)
    ubuf[shift:shift + n] = _t(u)
    if l_bytes == 1:
        lbuf = torch.full((n + 32,), 0xEE, dtype=torch.uint8, device=DEV)
        lview = lbuf[4 * shift:4 * shift + n]
    else:
        lbuf = torch.full((n + 8,), -7, dtype=torch.int32, device=DEV)
        lview = lbuf[shift:shift + n]
    seg = torch.from_numpy(starts).to(DEV)
    lbub = torch.full((2 * n_seg,), float("nan"), device=DEV)
    keys = torch.empty(2 * n_seg, dtype=torch.int32, device=DEV)
    _lib.call("gq_norm_quantize", ubuf.data_ptr() + 4 * shift, n, seg.data_ptr(), n_seg, n_bit, 1, None, seed, off,
              lbuf.data_ptr() + 4 * shift, l_bytes, lbub.data_ptr(), keys.data_ptr(), 0, _lib.stream())
    return lbub.cpu().numpy(), lview.cpu().numpy().astype(np.int32)


NORM_LEVELS = [(1, 1), (1, 6), (1, 7), (4, 8), (4, 12), (4, 24)]   # (l_bytes, n_bit)


@pytest.mark.parametrize("n_mod4", [0, 1, 2, 3])
@pytest.mark.parametrize("layout", ["smem", "many_segments", "misaligned"])
@pytest.mark.parametrize("off", OFFSETS)
def test_norm_quantize_philox(off, layout, n_mod4):
    """The shared-memory kernel (<= 1024 tensors, aligned pointers) and the grid-stride kernel (1100 tensors;
    u / l pointers 4 bytes off), every norm width, n % 4 in 0..3, length-1 and constant (lb == ub) tensors."""
    n = 9000 + n_mod4
    rs = np.random.RandomState(17 + n_mod4)
    starts = _starts_with_edges(rs, n, 1100 if layout == "many_segments" else 37)
    u = (rs.standard_normal(n) * 0.01).astype(np.float32)
    u[starts[5]:starts[6]] = np.float32(0.37)                   # a constant tensor: lb == ub, all levels 0
    for l_bytes, n_bit in NORM_LEVELS:
        lbub, l = _norm_quantize(u, starts, n_bit, l_bytes, SEED, off, shift=1 if layout == "misaligned" else 0)
        _check_levels(u, starts, n_bit, SEED, off, lbub, l)


@pytest.mark.parametrize("l_bytes,n_bit", [(1, 6), (4, 12)])
@pytest.mark.parametrize("off", OFFSETS)
def test_norm_quantize_philox_several_items_per_thread(off, l_bytes, n_bit):
    """2 M chunks: the one-wave grid of the shared-memory kernel gives every thread more than one group
    of four (launch_norm_quantize's `items`)."""
    n = 2_000_003
    u = gen_input(23, n)
    starts = np.array([0, 700_001, 700_002, 1_500_000, n], dtype=np.int64)
    lbub, l = _norm_quantize(u, starts, n_bit, l_bytes, SEED2, off)
    _check_levels(u, starts, n_bit, SEED2, off, lbub, l)


# ------------------------------------------------------------------------------------------ HSQ encode ---
@functools.lru_cache(maxsize=None)
def _hsq_case(d, K, n_chunks, n_seg, seed):
    """Input, segment table and oracle search of one HSQ case (the search does not depend on the draws)."""
    rs = np.random.RandomState(seed)
    x = gen_input(seed, n_chunks * d).reshape(n_chunks, d)
    starts = _starts_with_edges(rs, n_chunks, n_seg)
    x[starts[4]:starts[5]] = 0.0                                 # all-zero chunks: u == 0, lb == ub
    cb = codebook(d, K)
    oc, ou = O.hsq_search(x, cb)
    return x, starts, cb, oc, ou


def _hsq_encode(x, cb, starts, n_bit, l_bytes, seed, off, algo=_lib.ALGO_AUTO):
    n_chunks, d = x.shape
    K, n_seg = cb.shape[0], len(starts) - 1
    code_bytes = 1 if K <= 256 else 4
    codes = torch.full((n_chunks,), 0xEE if code_bytes == 1 else -7,
                       dtype=torch.uint8 if code_bytes == 1 else torch.int32, device=DEV)
    l = torch.full((n_chunks,), 0xEE if l_bytes == 1 else -7,
                   dtype=torch.uint8 if l_bytes == 1 else torch.int32, device=DEV)
    lbub = torch.full((2 * n_seg,), float("nan"), device=DEV)
    u = torch.full((n_chunks,), float("nan"), device=DEV)
    ws = torch.empty(max(_lib.value("gq_hsq_encode_workspace_bytes", n_chunks, d, K, n_seg), 256),
                     dtype=torch.uint8, device=DEV)
    xt, cbt, seg = _t(x), _t(cb), torch.from_numpy(starts).to(DEV)
    _lib.call("gq_hsq_encode", xt.data_ptr(), n_chunks, d, cbt.data_ptr(), K, seg.data_ptr(), n_seg, n_bit, 1, None,
              seed, off, codes.data_ptr(), code_bytes, l.data_ptr(), l_bytes, lbub.data_ptr(), u.data_ptr(),
              ws.data_ptr(), ws.numel(), algo, _lib.stream())
    return dict(codes=codes.cpu().numpy().astype(np.int32), u=u.cpu().numpy(), lbub=lbub.cpu().numpy(),
                l=l.cpu().numpy().astype(np.int32))


def _check_hsq(got, case, n_bit, seed, off):
    x, starts, cb, oc, ou = case
    assert np.array_equal(got["codes"], oc), _first_diff(got["codes"], oc)
    assert np.array_equal(got["u"], ou), _first_diff(got["u"], ou)
    _check_levels(ou, starts, n_bit, seed, off, got["lbub"], got["l"])


# name: (d, K, n_chunks, n_seg, n_bit, l_bytes, algo, environment)
HSQ_PATHS = {
    # one-launch tcgen05 encode, norm quantization in its fused tail
    "tc2_tail_d8": (8, 256, 20011, 12, 6, 1, _lib.ALGO_AUTO, {}),
    "tc2_tail_d16": (16, 256, 20010, 12, 6, 1, _lib.ALGO_AUTO, {}),
    "tc2_tail_d32": (32, 256, 20009, 12, 6, 1, _lib.ALGO_AUTO, {}),
    # two CTAs: each CTA's tail walks its 10 000+ chunks in more than one pass of J float4 groups per thread
    "tc2_tail_multipass_d16": (16, 256, 30011, 9, 6, 1, _lib.ALGO_AUTO, {"GQ_TC_GRID": "2"}),
    "tc2_tail_multipass_d32": (32, 256, 30010, 9, 6, 1, _lib.ALGO_AUTO, {"GQ_TC_GRID": "2"}),
    # tcgen05 search, then the separate quantize launch: int32 levels / more tensors than the tail's table
    "tc2_then_quantize_l4": (16, 256, 20011, 12, 8, 4, _lib.ALGO_AUTO, {}),
    "tc2_then_quantize_1100_tensors": (16, 256, 20011, 1100, 6, 1, _lib.ALGO_AUTO, {}),
    "exact": (16, 256, 20011, 12, 6, 1, _lib.ALGO_EXACT, {}),
    "tck_k4096": (16, 4096, 6007, 7, 6, 1, _lib.ALGO_AUTO, {}),
    "tc_v1": (16, 256, 20011, 12, 6, 1, _lib.ALGO_AUTO, {"GQ_TC_V": "1"}),
}


@pytest.mark.parametrize("off", OFFSETS)
@pytest.mark.parametrize("path", sorted(HSQ_PATHS))
def test_hsq_encode_philox(path, off, monkeypatch):
    d, K, n_chunks, n_seg, n_bit, l_bytes, algo, env = HSQ_PATHS[path]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    case = _hsq_case(d, K, n_chunks, n_seg, 40 + d)
    got = _hsq_encode(case[0], case[2], case[1], n_bit, l_bytes, SEED, off, algo)
    _check_hsq(got, case, n_bit, SEED, off)


FUSED_CASE = (16, 256, 20011, 12, 56)


def _fused_child(out_path):
    """Runs in a child process with GQ_TC_FUSED=1 (read once per process): the opt-in single-launch
    encode of hsq_tc.cu, whose tail is quantize_range(), at every offset."""
    d, K, n_chunks, n_seg, seed = FUSED_CASE
    case = _hsq_case(d, K, n_chunks, n_seg, seed)
    res = {}
    for i, off in enumerate(OFFSETS):
        for k, v in _hsq_encode(case[0], case[2], case[1], 6, 1, SEED, off).items():
            res["%s_%d" % (k, i)] = v
    np.savez(out_path, **res)


def test_hsq_tc_fused_tail_in_child_process(tmp_path):
    out = str(tmp_path / "fused.npz")
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), out]
    r = subprocess.run(cmd, env=dict(os.environ, GQ_TC_FUSED="1"), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    res = np.load(out)
    d, K, n_chunks, n_seg, seed = FUSED_CASE
    case = _hsq_case(d, K, n_chunks, n_seg, seed)
    for i, off in enumerate(OFFSETS):
        _check_hsq({k: res["%s_%d" % (k, i)] for k in ("codes", "u", "lbub", "l")}, case, 6, SEED, off)


# ----------------------------------------------------------------------------------------------- QSGD ---
def _qsgd_encode(x, n_bit, seed, off, dim=0, starts=None, packed=True, unpacked=False):
    n = x.size
    n_chunks = len(starts) - 1 if starts is not None else n // dim
    bits = _lib.value("gq_qsgd_wire_bits", n_bit)
    norm = torch.full((n_chunks,), float("nan"), device=DEV)
    pk = torch.full(((n + 3) // 4 * 4 * bits // 8 + 16,), 0xEE, dtype=torch.uint8, device=DEV) if packed else None
    sg = torch.full((n,), 0xEE, dtype=torch.uint8, device=DEV) if unpacked else None
    l = torch.full((n,), -7, dtype=torch.int32, device=DEV) if unpacked else None
    cs = None if starts is None else torch.from_numpy(starts).to(DEV)
    xt = _t(x)
    _lib.call("gq_qsgd_encode", xt.data_ptr(), n, _lib.ptr(cs), n_chunks, dim, n_bit, 1, None, seed, off,
              norm.data_ptr(), _lib.ptr(sg), _lib.ptr(l), _lib.ptr(pk), _lib.stream())
    out = dict(norm=norm.cpu().numpy())
    if packed:
        out["wire"] = _unpack_wire(pk.cpu().numpy(), n, bits)
    if unpacked:
        out["signs"], out["l"] = sg.cpu().numpy(), l.cpu().numpy()
    return out


def _unpack_wire(packed, n, bits):
    """(sign, level) per element from the packed wire: element = (sign << (bits - 1)) | level,
    little-endian, element 0 in the low bits."""
    if bits == 4:
        w = np.stack([packed & 15, packed >> 4], axis=1).reshape(-1)
    elif bits == 8:
        w = packed
    else:
        w = packed.view("<u2")
    w = w[:n].astype(np.int64)
    return (w >> (bits - 1)).astype(np.uint8), (w & ((1 << (bits - 1)) - 1)).astype(np.int32)


def _qsgd_reference(x, n_bit, seed, off, dim=0, starts=None):
    """O.qsgd_compress chunk by chunk, fed with philox_uniforms(seed, off, n) (element i draws index off + i)."""
    r = philox_uniforms(seed, off, x.size)
    if starts is None:
        return O.qsgd_compress(x, dim, n_bit, True, r)
    parts = [O.qsgd_compress(x[a:b], int(b - a), n_bit, True, r[a:b]) for a, b in zip(starts[:-1], starts[1:])]
    return tuple(np.concatenate([p[k] for p in parts]) for k in range(3))


def _check_qsgd(got, ref):
    onorm, osigns, ol = ref
    assert np.array_equal(got["norm"], onorm)
    if "wire" in got:      # the wire has no INT32_MIN: a 0 / 0 element is level 0
        s, l = got["wire"]
        want = np.where(ol == INT32_MIN, 0, ol)
        assert np.array_equal(s, osigns), _first_diff(s, osigns)
        assert np.array_equal(l, want), _first_diff(l, want)
    if "l" in got:
        assert np.array_equal(got["signs"], osigns), _first_diff(got["signs"], osigns)
        assert np.array_equal(got["l"], ol), _first_diff(got["l"], ol)


@pytest.mark.parametrize("n_bit", [2, 6, 8])          # 4-, 8- and 16-bit wire
@pytest.mark.parametrize("dim", [8, 32, 128, 256, 512, 1024, 2048])   # every (NV, LPC) of the one-launch kernel
@pytest.mark.parametrize("off", OFFSETS)
def test_qsgd_chunks_kernel_philox(off, dim, n_bit):
    n_chunks = max(24, 65536 // dim) + 1
    x = gen_input(60 + dim, n_chunks * dim)
    x[3 * dim:4 * dim] = 0.0                                     # an all-zero chunk
    got = _qsgd_encode(x, n_bit, SEED, off, dim=dim)
    _check_qsgd(got, _qsgd_reference(x, n_bit, SEED, off, dim=dim))


def _var_chunks(n):
    sizes = [3000, 1, 7, 40000, 2, 12345, 50001]
    sizes.append(n - sum(sizes))
    assert sizes[-1] > 0
    return np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)


@pytest.mark.parametrize("n_mod4", [0, 1, 2, 3])
@pytest.mark.parametrize("off", OFFSETS)
def test_qsgd_ranges_kernel_philox(off, n_mod4):
    """Explicit chunk boundaries (one chunk per tensor, TernGrad's c_dim == 0) on the packed wire: the
    two-launch ranges kernels; n % 4 in 0..3, an all-zero chunk, chunks of 1 and 2 elements."""
    n = 120000 + n_mod4
    starts = _var_chunks(n)
    x = gen_input(61 + n_mod4, n)
    x[starts[5]:starts[6]] = 0.0
    for n_bit in (1, 6, 8):
        got = _qsgd_encode(x, n_bit, SEED2, off, starts=starts)
        _check_qsgd(got, _qsgd_reference(x, n_bit, SEED2, off, starts=starts))


@pytest.mark.parametrize("layout,wire", [("dim50", "unpacked"), ("dim50", "packed"), ("dim4096", "unpacked"),
                                         ("dim4096", "packed"), ("variable", "unpacked")])
@pytest.mark.parametrize("off", OFFSETS)
def test_qsgd_generic_kernel_philox(off, layout, wire):
    """The generic kernels: reference-dtype outputs (signs / int32 levels incl. INT32_MIN), chunk dims that
    are not a multiple of 4 or beyond 2048; n % 4 == 2 (dim 50) and 3 (variable chunks; packed variable
    chunks take the ranges kernel, test_qsgd_ranges_kernel_philox)."""
    if layout == "dim50":
        dim, starts, x = 50, None, gen_input(62, 50 * 101)
        x[150:200] = 0.0
    elif layout == "dim4096":
        dim, starts, x = 4096, None, gen_input(63, 4096 * 5)
        x[4096:8192] = 0.0
    else:
        dim, starts, x = 0, _var_chunks(120003), gen_input(64, 120003)
        x[starts[5]:starts[6]] = 0.0
    for n_bit in (2, 8):
        got = _qsgd_encode(x, n_bit, SEED, off, dim=dim, starts=starts,
                           packed=wire == "packed", unpacked=wire == "unpacked")
        _check_qsgd(got, _qsgd_reference(x, n_bit, SEED, off, dim=dim, starts=starts))


# ------------------------------------------------------------------------------------------------ PVC ---
@pytest.mark.parametrize("d", [8, 16])
@pytest.mark.parametrize("off", OFFSETS)
def test_pvc_search_philox(off, d):
    n_chunks, K = 3001, 256
    cb = codebook(d, K)
    dagger = np.linalg.pinv(cb.T).astype(np.float32)
    x = gen_input(70 + d, n_chunks * d).reshape(n_chunks, d)
    codes = torch.full((n_chunks,), 0xEE, dtype=torch.uint8, device=DEV)
    u = torch.full((n_chunks,), float("nan"), device=DEV)
    xt, dt = _t(x), _t(dagger)
    _lib.call("gq_pvc_search", xt.data_ptr(), n_chunks, d, dt.data_ptr(), K, None, SEED, off, codes.data_ptr(), 1,
              u.data_ptr(), _lib.stream())
    oc, ou = O.pvc_search(x, dagger, philox_uniforms(SEED, off, n_chunks))
    got = codes.cpu().numpy().astype(np.int32)
    assert np.array_equal(got, oc), _first_diff(got, oc)
    assert np.array_equal(u.cpu().numpy(), ou)


# ----------------------------------------------------------------------------------- seeding contract ---
def _gen():
    return torch.cuda.default_generators[torch.cuda.current_device()]


@pytest.fixture
def shared_stream():
    """PhiloxState is process-wide: start the shared (second-phase) stream unset, restore it afterwards."""
    st = _lib.PHILOX
    saved = (st.shared_seed, st.shared_offset)
    st.shared_seed, st.shared_offset = None, 0
    yield st
    st.shared_seed, st.shared_offset = saved


def test_take_key_is_mixed_from_seed_and_user_and_offsets_advance_by_blocks():
    torch.manual_seed(SEED)
    gen = _gen()
    assert gen.initial_seed() == SEED
    off0 = off = int(gen.get_offset())
    for n, user in [(1, 0), (4, 1), (5, 2), (7, 7), (1_000_001, 3), (922, 0)]:
        key, o = _lib.PHILOX.take(n, user)
        assert key == mix64(SEED, user) and o == off, (n, user)
        off += ceil4(n)
        assert int(gen.get_offset()) == off
    torch.manual_seed(SEED)
    assert _lib.PHILOX.take(5, 2) == (mix64(SEED, 2), off0)          # re-seeding replays
    torch.manual_seed(SEED2)
    assert _lib.PHILOX.take(5, 2)[0] == mix64(SEED2, 2)


def test_reseeding_replays_the_kernel_draws():
    """ProbabilisticScalarCompressor without uniforms draws philox_uniforms(mix64(seed, 0), generator offset, n);
    torch.rand on the device in between moves the offset, re-seeding replays the same levels."""
    psc = gq_b200.ProbabilisticScalarCompressor(6, make_args(n_bit=6))
    u = gen_input(31, 10007)
    ut = _t(u)
    gen = _gen()
    for seed in (SEED, SEED2):
        torch.manual_seed(seed)
        levels = []
        for _ in range(2):
            off = int(gen.get_offset())
            lb, ub, l = psc.compress(ut)
            assert int(gen.get_offset()) == off + ceil4(u.size)
            olb, oub, ol, _ = O.psc_compress(u, 6, True, philox_uniforms(mix64(seed, 0), off, u.size))
            got = l.cpu().numpy()
            assert np.float32(lb.item()) == olb and np.float32(ub.item()) == oub
            assert np.array_equal(got, ol), _first_diff(got, ol)
            levels.append(got)
            torch.rand(1000, device=DEV)
        torch.manual_seed(seed)
        assert np.array_equal(psc.compress(ut)[2].cpu().numpy(), levels[0])
        assert not np.array_equal(levels[0], levels[1])


def test_shared_stream_is_independent_of_the_generator(shared_stream):
    torch.manual_seed(SEED)
    gen = _gen()
    off = int(gen.get_offset())
    key, o = shared_stream.take_shared(10)
    assert (key, o) == (mix64(SEED, 1 << 32), 0)             # default shared seed: this process's generator seed
    assert int(gen.get_offset()) == off                      # the generator does not move
    torch.rand(1000, device=DEV)
    assert shared_stream.take_shared(3) == (key, 12)         # nor does the shared stream when the generator moves
    torch.manual_seed(SEED2)
    assert shared_stream.take_shared(1) == (key, 16)


# Model of the quantizer tests: tensors of 512, 128, 192 (all zero), 256 and 90 HSQ chunks (1178 in one group:
# not a multiple of 4) plus an identity tensor; QSGD c_dim 128: two groups (chunk dims 128 and 288).
SHAPES = [(64, 128), (100,), (32, 64), (24, 128), (16, 256), (40, 3, 3, 4)]
ZERO = 3


def _inputs(seed0, same_for_all, U):
    xs = []
    for u in range(U):
        base = seed0 if same_for_all else seed0 + 10 * u
        x = [gen_input(base + i, int(np.prod(s))).reshape(s) for i, s in enumerate(SHAPES)]
        x[ZERO][:] = 0.0
        xs.append(x)
    return xs


def _codec(codec):
    if codec == "hsq":
        return gq_b200.NearestNeighborCompressor, dict(c_dim=16, n_bit=6)
    return gq_b200.QSGDCompressor, dict(c_dim=128, n_bit=2)


def _oracle_codecs(codec):
    out = []
    for s in SHAPES:
        n = int(np.prod(s))
        if n <= 1000:
            out.append(O.Identity())
        elif codec == "hsq":
            out.append(O.HSQ(n, s, codebook(O.chunk_dim(n, 16), 256), 6, True))
        else:
            out.append(O.QSGD(n, s, 128, 2, True))
    return out


def _plan_draws(plan, key, off):
    """The documented rule of one fused encode: groups in plan order, one take of ceil4(the group's draws)
    each; chunk (HSQ) / element (QSGD) c of a group draws index offset + c.  -> ({tensor: draws}, next offset)."""
    draws = {}
    for g in plan.groups:
        if g.kind == "hsq":
            counts = [size // g.dim for size in g.sizes]
        elif g.kind == "qsgd":
            counts = list(g.sizes)
        else:
            continue
        pos = 0
        for i, m in zip(g.tensors, counts):
            draws[i] = philox_uniforms(key, off + pos, m)
            pos += m
        off += ceil4(pos)
    return draws, off


def _stream(per_user, codec, zero_in=(ZERO,)):
    """Flatten per-user draws into the oracle's call order (user-major, model order).  An HSQ tensor with
    lb == ub draws nothing in the reference: its index range is skipped, not its draws consumed."""
    parts = []
    for draws in per_user:
        for i in sorted(draws):
            if not (codec == "hsq" and i in zero_in):
                parts.append(draws[i])
    return np.concatenate(parts)


def _assert_grads(params, ref):
    for i, (p, r) in enumerate(zip(params, ref)):
        got = p.grad.data.cpu().numpy().reshape(-1)
        r = np.asarray(r).reshape(-1)
        if got.size > 1000:
            assert np.array_equal(got, r), (i, _first_diff(got, r))
        else:   # identity tensors: the device mean of a few users is not held to the last bit
            assert np.abs(got - r).max() <= 1e-6 * max(np.abs(r).max(), 1e-30), i


def _quantizer(codec, **kw):
    Comp, ca = _codec(codec)
    params = [torch.nn.Parameter(torch.zeros(s, device=DEV)) for s in SHAPES]
    a = make_args(**dict(ca, **kw))
    return gq_b200.Quantizer(Comp, params, a), params


@pytest.mark.parametrize("codec", ["hsq", "qsgd"])
def test_fused_ps_step_draws_from_per_user_keys(codec):
    """U = 3 users with the SAME gradient, no uniforms: user u draws from key mix64(seed, u), the offsets
    follow the CUDA generator, and the averaged step equals O.ps_step fed with those draws."""
    U = 3
    q, params = _quantizer(codec, num_users=U)
    assert q.plan is not None
    xs = _inputs(700, True, U)
    torch.manual_seed(SEED)
    gen = _gen()
    off = int(gen.get_offset())
    per_user = []
    for u in range(U):
        for p, x in zip(params, xs[u]):
            p.grad = _t(x)
        q.record(u, epoch=0)
        draws, off = _plan_draws(q.plan, mix64(SEED, u), off)
        per_user.append(draws)
    assert int(gen.get_offset()) == off
    rec = q.plan.records.cpu().numpy()
    q.apply()
    stream = O.UniformStream(_stream(per_user, codec))
    _assert_grads(params, O.ps_step(_oracle_codecs(codec), xs, stream))
    assert stream.pos == stream.draws.size
    assert not np.array_equal(rec[0], rec[1]) and not np.array_equal(rec[1], rec[2])   # decorrelated users


@pytest.mark.parametrize("codec", ["hsq", "qsgd"])
def test_per_parameter_ps_step_takes_once_per_tensor(codec):
    """fused = False: every compressed tensor's compress() takes its own draws (stream 0 -- the compressors do
    not know the user; the advancing offset keeps the users apart), in user-major, model order."""
    U = 3
    q, params = _quantizer(codec, num_users=U, fused=False)
    assert q.plan is None
    xs = _inputs(710, False, U)
    torch.manual_seed(SEED2)
    gen = _gen()
    off = int(gen.get_offset())
    per_user = []
    for u in range(U):
        for p, x in zip(params, xs[u]):
            p.grad = _t(x)
        q.record(u, epoch=0)
        draws = {}
        for i, s in enumerate(SHAPES):
            n = int(np.prod(s))
            if n > 1000:
                m = n // O.chunk_dim(n, 16) if codec == "hsq" else n
                draws[i] = philox_uniforms(mix64(SEED2, 0), off, m)
                off += ceil4(m)
        per_user.append(draws)
    assert int(gen.get_offset()) == off
    q.apply()
    stream = O.UniformStream(_stream(per_user, codec))
    _assert_grads(params, O.ps_step(_oracle_codecs(codec), xs, stream))
    assert stream.pos == stream.draws.size


def _ring_run(monkeypatch, parts):
    if parts is None:
        monkeypatch.delenv("GQ_RING_PARTS", raising=False)
    else:
        monkeypatch.setenv("GQ_RING_PARTS", str(parts))
    U = 3
    q, params = _quantizer("hsq", num_users=U, mode="ring")
    assert q.parts == (parts or 1)
    xs = _inputs(720, False, U)
    torch.manual_seed(SEED)
    gen = _gen()
    off = int(gen.get_offset())
    per_user = []
    for u in range(U):
        for p, x in zip(params, xs[u]):
            p.grad = _t(x)
        q.record(u, epoch=0)
        draws, off = _plan_draws(q.plan, mix64(SEED, u), off)
        per_user.append(draws)
    assert int(gen.get_offset()) == off
    q.apply()
    return params, xs, per_user


def test_ring_in_stages_draws_the_same_indices(monkeypatch):
    """The pipelined ring (3 stages of tensors) and the unstaged ring give the same result bit for bit, and
    both are O.ring_step fed with each user's Philox draws."""
    staged, xs, per_user = _ring_run(monkeypatch, 3)
    plain, _, _ = _ring_run(monkeypatch, None)
    for a, b in zip(staged, plain):
        assert torch.equal(a.grad, b.grad)
    stream = O.UniformStream(_stream(per_user, "hsq"))
    _assert_grads(plain, O.ring_step(_oracle_codecs("hsq"), xs, stream))
    assert stream.pos == stream.draws.size


def test_two_phase_second_compression_draws_from_the_shared_stream(shared_stream):
    """--two-phase without uniforms: phase 2 compresses the average with key mix64(shared seed, 2^32) from
    offset 0 of its own counter (the same on every rank), laid out like one user's fused encode."""
    U = 3
    q, params = _quantizer("hsq", num_users=U, two_phase=True)
    xs = _inputs(730, False, U)
    torch.manual_seed(SEED)
    gen = _gen()
    off = int(gen.get_offset())
    per_user = []
    for u in range(U):
        for p, x in zip(params, xs[u]):
            p.grad = _t(x)
        q.record(u, epoch=0)
        draws, off = _plan_draws(q.plan, mix64(SEED, u), off)
        per_user.append(draws)
    q.apply()
    assert int(gen.get_offset()) == off
    phase2, end = _plan_draws(q.phase2_plan(), mix64(SEED, 1 << 32), 0)
    assert shared_stream.shared_offset == end
    stream = O.UniformStream(_stream(per_user + [phase2], "hsq"))
    _assert_grads(params, O.ps_step(_oracle_codecs("hsq"), xs, stream, two_phase=True))
    assert stream.pos == stream.draws.size


def test_torch_rng_replays_the_reference_cpu_draws():
    """rng = "torch": the per-parameter compressors draw torch.rand on the CPU generator when the reference
    does -- one rand(N/d) per HSQ tensor with lb != ub, one rand(size) per QSGD tensor -- and never touch
    the Philox offset."""
    hsq = make_args(c_dim=16, n_bit=6, rng="torch")
    qsgd = make_args(c_dim=128, n_bit=2, rng="torch")
    shapes = [(64, 128), (24, 128), (40, 3, 3, 4), (32, 64)]
    kinds = ["hsq", "hsq", "hsq", "qsgd"]
    xs = [gen_input(740 + i, int(np.prod(s))).reshape(s) for i, s in enumerate(shapes)]
    xs[1][:] = 0.0                                             # lb == ub: draws nothing
    comps, ocs = [], []
    for s, k in zip(shapes, kinds):
        n = int(np.prod(s))
        if k == "hsq":
            comps.append(gq_b200.NearestNeighborCompressor(n, torch.Size(s), hsq))
            ocs.append(O.HSQ(n, s, codebook(16, 256), 6, True))
        else:
            comps.append(gq_b200.QSGDCompressor(n, torch.Size(s), qsgd))
            ocs.append(O.QSGD(n, s, 128, 2, True))
    torch.manual_seed(SEED)
    gen = _gen()
    off = int(gen.get_offset())
    sigs = [c.compress(_t(x)) for c, x in zip(comps, xs)]
    assert int(gen.get_offset()) == off
    n_draws = xs[0].size // 16 + xs[2].size // 16 + xs[3].size
    stream = O.UniformStream(torch_uniform_stream(SEED, n_draws))
    for i, (sig, oc, x, k) in enumerate(zip(sigs, ocs, xs, kinds)):
        osig = oc.compress(x, stream)
        if k == "hsq":
            (lb, ub, l), codes = sig
            (olb, oub, ol), ocodes = osig
            assert np.array_equal(codes.cpu().numpy().astype(np.int32), ocodes), i
            assert np.float32(lb.item()) == olb and np.float32(ub.item()) == oub, i
            assert np.array_equal(l.cpu().numpy(), ol), (i, _first_diff(l.cpu().numpy(), ol))
        else:
            norm, signs, l = sig
            assert np.array_equal(norm.cpu().numpy().reshape(-1), osig[0]), i
            assert np.array_equal(signs.cpu().numpy().reshape(-1).astype(np.uint8), osig[1]), i
            assert np.array_equal(l.cpu().numpy().reshape(-1), osig[2]), i
    assert stream.pos == n_draws


if __name__ == "__main__":
    _fused_child(sys.argv[1])
