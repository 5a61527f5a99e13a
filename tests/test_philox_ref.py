"""CPU checks of the host Philox / SplitMix64 reference (tests/philox_ref.py) that
test_gpu_philox.py pins the kernels against, and of the host half of the seeding contract."""
import numpy as np
import pytest

from philox_ref import ceil4, mix64, philox4x32_10, philox_uniforms, u01


@pytest.mark.parametrize("ctr,key,out", [
    # Random123 known-answer vectors of philox4x32_10 (kat_vectors)
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(ctr, key, out):
    """The reference's counter is (idx_lo, idx_hi, 0, 0): the vectors with non-zero high counter words
    go through a generalised copy of the same rounds, the all-zero one through philox4x32_10 itself."""
    seed = key[0] | (key[1] << 32)
    if ctr[2] == 0 and ctr[3] == 0:
        got = philox4x32_10(seed, [ctr[0] | (ctr[1] << 32)])[0]
    else:
        got = _philox_full_counter(ctr, key)
    assert tuple(int(w) for w in got) == out


def _philox_full_counter(ctr, key):
    """philox4x32_10 with all four counter words free (scalar, Python ints)."""
    c0, c1, c2, c3 = ctr
    k0, k1 = key
    for _ in range(10):
        p0, p1 = 0xD2511F53 * c0, 0xCD9E8D57 * c2
        c0, c1, c2, c3 = ((p1 >> 32) ^ c1 ^ k0) & 0xFFFFFFFF, p1 & 0xFFFFFFFF, ((p0 >> 32) ^ c3 ^ k1) & 0xFFFFFFFF, p0 & 0xFFFFFFFF
        k0, k1 = (k0 + 0x9E3779B9) & 0xFFFFFFFF, (k1 + 0xBB67AE85) & 0xFFFFFFFF
    return c0, c1, c2, c3


def test_full_counter_copy_agrees_with_the_reference():
    """The scalar copy above is the vectorised reference on counters (lo, hi, 0, 0)."""
    seed = 0x123456789ABCDEF0
    idx = [0, 1, 5, 1 << 33, (1 << 64) - 1]
    got = philox4x32_10(seed, idx)
    for i, x in enumerate(idx):
        want = _philox_full_counter((x & 0xFFFFFFFF, x >> 32, 0, 0), (seed & 0xFFFFFFFF, seed >> 32))
        assert tuple(int(w) for w in got[i]) == want


def test_u01_range_and_dtype():
    assert u01(np.uint32(0xFFFFFFFF)) < 1.0
    assert u01(np.uint32(0xFFFFFFFF)) == np.float32(1.0 - 2.0 ** -24)
    assert u01(np.uint32(0xFF)) == 0.0
    assert u01(np.uint32(0x100)) == np.float32(2.0 ** -24)
    r = philox_uniforms(0x0123456789ABCDEF, 3, 1001)
    assert r.dtype == np.float32 and r.shape == (1001,)
    assert r.min() >= 0.0 and r.max() < 1.0


def test_draws_index_words_of_blocks():
    """Draw i of offset off is word (off + i) & 3 of block (off + i) >> 2; offsets shift the stream."""
    seed = 0x5DEECE66D1234567
    blocks = philox4x32_10(seed, np.arange(8, dtype=np.uint64))
    flat = u01(blocks.reshape(-1))
    for off in (0, 1, 2, 3, 6):
        assert np.array_equal(philox_uniforms(seed, off, 20), flat[off:off + 20])
    base = philox_uniforms(seed, 1 << 34, 64)
    assert np.array_equal(philox_uniforms(seed, (1 << 34) + 5, 40), base[5:45])


def test_high_counter_and_key_words_matter():
    """Blocks at idx >= 2^32 are not the blocks at idx mod 2^32, and the key's high word changes them."""
    seed = 0x0123456789ABCDEF
    lo = np.arange(4, dtype=np.uint64)
    for hi in (1, 2, 0xFFFFFFFF):
        a = philox4x32_10(seed, lo)
        b = philox4x32_10(seed, lo + np.uint64(hi << 32))
        assert not np.any(np.all(a == b, axis=1))
    a = philox4x32_10(seed, lo)
    b = philox4x32_10(seed & 0xFFFFFFFF, lo)
    assert not np.any(np.all(a == b, axis=1))


def test_mix64_is_splitmix64():
    """SplitMix64 from state 0: the published first outputs of the generator."""
    assert [mix64(0, k) for k in range(3)] == [0xE220A8397B1DCDAF, 0x6E789E6AA1B965F4, 0x06C45D188009454F]
    keys = {mix64(0x5DEECE66D1234567, u) for u in list(range(64)) + [1 << 32]}
    assert len(keys) == 65
    assert ceil4(0) == 0 and ceil4(1) == 4 and ceil4(4) == 4 and ceil4(922) == 924


def test_shared_stream_bookkeeping():
    """PhiloxState.take_shared: key mix64(shared seed, 2^32), its own offset moving by ceil4(n) per take."""
    from gq_b200 import _lib
    st = _lib.PhiloxState()
    seed = 0x1F2E3D4C5B6A7988
    assert st.share_seed(seed) == seed
    offs = []
    for n in (5, 4, 1, 1000):
        key, off = st.take_shared(n)
        assert key == mix64(seed, 1 << 32)
        offs.append(off)
    assert offs == [0, 8, 12, 16] and st.shared_offset == 1016
    st.share_seed(seed + 1)
    assert st.take_shared(3) == (mix64(seed + 1, 1 << 32), 0)
