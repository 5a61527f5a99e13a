"""Host reference of the in-kernel random stream -- test infrastructure, independent of the package.

The stream the kernels draw from when no uniforms are passed (include/gqb200.h,
csrc/gq_common.cuh): Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy as
1, 2, 3", SC 2011) with counter = (idx_lo, idx_hi, 0, 0) and key = (seed_lo, seed_hi);
logical draw i of a call with offset `off` is word (off + i) & 3 of the block at
(off + i) >> 2, mapped to [0, 1) by its 24 high bits.  The per-user keys of the quantizers
come from SplitMix64 (DESIGN.md section 7).  Nothing here imports the package: a test
that compares the two compares two independent statements of the same stream.
"""
import numpy as np

_M32 = 0xFFFFFFFF
_M64 = 0xFFFFFFFFFFFFFFFF
_MUL0, _MUL1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = 0x9E3779B9, 0xBB67AE85


def philox4x32_10(seed, idx):
    """Blocks of Philox4x32-10 for key `seed` (64-bit int) at the 64-bit counters `idx`:
    uint32 array of shape idx.shape + (4,).  32x32 -> 64-bit products in uint64 are exact."""
    idx = np.asarray(idx, dtype=np.uint64)
    m32 = np.uint64(_M32)
    c0, c1 = idx & m32, idx >> np.uint64(32)
    c2, c3 = np.zeros_like(idx), np.zeros_like(idx)
    k0, k1 = int(seed) & _M32, (int(seed) >> 32) & _M32
    for _ in range(10):
        p0, p1 = _MUL0 * c0, _MUL1 * c2
        hi0, lo0 = p0 >> np.uint64(32), p0 & m32
        hi1, lo1 = p1 >> np.uint64(32), p1 & m32
        c0, c1, c2, c3 = hi1 ^ c1 ^ np.uint64(k0), lo1, hi0 ^ c3 ^ np.uint64(k1), lo0
        k0, k1 = (k0 + _W0) & _M32, (k1 + _W1) & _M32
    return np.stack([c0, c1, c2, c3], axis=-1).astype(np.uint32)


def u01(x):
    """24 high bits of a 32-bit word times 2^-24, in float32: [0, 1), like torch.rand."""
    return (np.asarray(x, dtype=np.uint32) >> np.uint32(8)).astype(np.float32) * np.float32(2.0 ** -24)


def philox_uniforms(seed, offset, n):
    """The n draws a kernel call with (philox_seed, philox_offset) = (seed, offset) uses for its
    logical indices 0 .. n-1: element i is u01 of word (offset + i) & 3 of block (offset + i) >> 2."""
    g = np.uint64(int(offset)) + np.arange(int(n), dtype=np.uint64)
    words = philox4x32_10(seed, g >> np.uint64(2))
    return u01(words[np.arange(int(n)), (g & np.uint64(3)).astype(np.intp)])


def mix64(seed, k):
    """SplitMix64 output number k + 1 from state `seed`: the Philox key of logical stream k
    (record(user): k = user; the shared second-phase stream: k = 2^32)."""
    z = (int(seed) + (int(k) + 1) * 0x9E3779B97F4A7C15) & _M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _M64
    return z ^ (z >> 31)


def ceil4(n):
    """How far one take of n draws moves a Philox offset: whole blocks of four."""
    return (int(n) + 3) // 4 * 4
