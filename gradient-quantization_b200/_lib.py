"""ctypes binding of libgqb200.so (include/gqb200.h) -- the only way the Python
classes reach the GPU.  There is no CPU fallback: if the library is missing or a
call fails, an exception is raised with the library's own error message.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgqb200.so")

c_void_p = ctypes.c_void_p
c_int = ctypes.c_int
c_i64 = ctypes.c_int64
c_u64 = ctypes.c_uint64
c_size = ctypes.c_size_t
c_float = ctypes.c_float

ALGO_AUTO, ALGO_EXACT, ALGO_TC = 0, 1, 2

_SIGNATURES = {
    "gq_abi_version": (c_int, []),
    "gq_device_info": (c_int, [ctypes.POINTER(c_int)] * 3 + [ctypes.POINTER(c_size)]),
    "gq_hsq_encode_workspace_bytes": (c_size, [c_i64, c_int, c_int, c_int]),
    "gq_hsq_encode": (c_int, [c_void_p, c_i64, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int,
                              c_void_p, c_u64, c_u64, c_void_p, c_int, c_void_p, c_int, c_void_p,
                              c_void_p, c_void_p, c_size, c_int, c_void_p]),
    "gq_hsq_search": (c_int, [c_void_p, c_i64, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p,
                              c_void_p, c_int, c_void_p, c_void_p, c_size, c_int, c_void_p]),
    "gq_norm_quantize": (c_int, [c_void_p, c_i64, c_void_p, c_int, c_int, c_int, c_void_p, c_u64, c_u64,
                                 c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p]),
    "gq_norm_dequantize": (c_int, [c_void_p, c_int, c_i64, c_void_p, c_int, c_int, c_void_p, c_void_p,
                                   c_void_p]),
    "gq_hsq_decode_reduce": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_i64, c_int,
                                     c_i64, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int,
                                     c_void_p, c_void_p]),
    "gq_hsq_encode_search": (c_int, [c_void_p, c_i64, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p, c_int,
                                     c_void_p, c_void_p, c_size, c_void_p]),
    "gq_hsq_decode_quantize": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_i64, c_int, c_void_p,
                                       c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_u64, c_u64, c_int,
                                       c_void_p, c_void_p]),
    "gq_hsq_decode_reduce_scattered": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int, c_i64,
                                               c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int,
                                               c_void_p, c_void_p]),
    "gq_f32_reduce_users_scattered": (c_int, [c_void_p, c_void_p, c_int, c_i64, c_int, c_int, c_void_p, c_void_p]),
    "gq_attach_f32_reduce": (c_int, [c_void_p, c_i64, c_void_p, c_int, c_i64, c_int, c_int, c_void_p]),
    "gq_ipc_alloc": (c_int, [c_size, ctypes.POINTER(c_void_p), c_void_p]),
    "gq_ipc_free": (c_int, [c_void_p]),
    "gq_ipc_open": (c_int, [c_void_p, ctypes.POINTER(c_void_p)]),
    "gq_ipc_close": (c_int, [c_void_p]),
    "gq_peer_barrier": (c_int, [c_void_p, c_int, c_int, ctypes.c_uint32, c_void_p]),
    "gq_peer_gather": (c_int, [c_void_p, c_void_p, c_size, c_size, c_int, c_void_p]),
    "gq_peer_push": (c_int, [c_void_p, c_void_p, c_size, c_int, c_void_p]),
    "gq_peer_push_multicast": (c_int, [c_void_p, c_void_p, c_size, c_void_p]),
    "gq_attach_remote_record": (c_int, [c_int, c_int, c_void_p, c_void_p, c_i64, c_void_p, c_int, ctypes.c_uint32]),
    "gq_attach_delivery_counter": (c_int, [c_void_p]),
    "gq_attach_peer_wait": (c_int, [c_void_p, c_int, ctypes.c_uint32]),
    "gq_f32_reduce_users": (c_int, [c_void_p, c_i64, c_int, c_i64, c_int, c_int, c_void_p, c_void_p]),
    "gq_qsgd_wire_bits": (c_int, [c_int]),
    "gq_qsgd_encode": (c_int, [c_void_p, c_i64, c_void_p, c_i64, c_int, c_int, c_int, c_void_p, c_u64,
                               c_u64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "gq_qsgd_decode_reduce": (c_int, [c_void_p, c_void_p, c_i64, c_int, c_i64, c_void_p, c_i64, c_int,
                                      c_int, c_int, c_int, c_void_p, c_void_p]),
    "gq_qsgd_decode_unpacked": (c_int, [c_void_p, c_void_p, c_void_p, c_i64, c_void_p, c_i64, c_int, c_int,
                                        c_void_p, c_void_p]),
    "gq_sign_encode": (c_int, [c_void_p, c_i64, c_void_p, c_void_p, c_void_p]),
    "gq_sign_decode_reduce": (c_int, [c_void_p, c_i64, c_int, c_i64, c_int, c_int, c_void_p, c_void_p]),
    "gq_sign_t5_bytes": (c_i64, [c_i64]),
    "gq_sign_encode_t5": (c_int, [c_void_p, c_i64, c_void_p, c_void_p]),
    "gq_sign_decode_reduce_t5": (c_int, [c_void_p, c_i64, c_int, c_i64, c_int, c_int, c_void_p, c_void_p]),
    "gq_topk_workspace_bytes": (c_size, [c_i64, c_int]),
    "gq_topk_select": (c_int, [c_void_p, c_i64, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p,
                               c_void_p, c_void_p, c_size, c_void_p]),
    "gq_topk_scatter_reduce": (c_int, [c_void_p, c_void_p, c_i64, c_int, c_i64, c_i64, c_int, c_int,
                                       c_void_p, c_void_p]),
    "gq_pvc_search": (c_int, [c_void_p, c_i64, c_int, c_void_p, c_int, c_void_p, c_u64, c_u64, c_void_p,
                              c_int, c_void_p, c_void_p]),
    "gq_hsq_tc_debug": (c_int, [c_void_p, c_i64, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p,
                                c_int, c_void_p]),
    "gq_hsq_tc2_trace": (c_int, [c_void_p, c_i64, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p,
                                 c_void_p, c_void_p]),
    "gq_gather_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_float, c_void_p]),
    "gq_axpy": (c_int, [c_void_p, c_void_p, c_float, c_i64, c_void_p, c_void_p]),
    "gq_sub": (c_int, [c_void_p, c_void_p, c_i64, c_void_p, c_void_p]),
    "gq_hsq_host_scratch_bytes": (c_size, [c_i64, c_int, c_int, c_int]),
    "gq_hsq_roundtrip_host": (c_int, [c_void_p, c_void_p, c_i64, c_int, c_void_p, c_int, c_void_p, c_int,
                                      c_int, c_int, c_u64, c_u64, c_void_p, c_size, c_int, c_void_p]),
}

EXPORTS = ["gq_last_error"] + sorted(_SIGNATURES)

_lib = None


class GQError(RuntimeError):
    pass


def load():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "libgqb200.so is missing (%s). Build it with `python gradient-quantization_b200/build.py` "
            "or __graft_entry__.build(); there is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    lib.gq_last_error.restype = ctypes.c_char_p
    lib.gq_last_error.argtypes = []
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def call(name, *args):
    """Call an int-returning entry point; raise GQError on a non-zero status."""
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise GQError("%s failed (%d): %s" % (name, rc, lib.gq_last_error().decode()))


def value(name, *args):
    return getattr(load(), name)(*args)


# ------------------------------------------------------------ torch glue ---
def require_cuda(t, what="tensor"):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise GQError("%s must be a CUDA tensor: this implementation has no CPU path" % what)
    return t


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


def f32c(t, what="tensor"):
    """fp32, contiguous, CUDA view of t (copies only when it must)."""
    require_cuda(t, what)
    if t.dtype != torch.float32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()


_M64 = 0xFFFFFFFFFFFFFFFF


def _mix64(seed, k):
    """SplitMix64 finaliser of (seed, k): statistically independent Philox keys per logical stream."""
    z = (seed + (k + 1) * 0x9E3779B97F4A7C15) & _M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _M64
    return z ^ (z >> 31)


class PhiloxState:
    """Seed/offset bookkeeping for the on-device Philox stream (DESIGN.md section 7).

    take(n, user): the stochastic-rounding draws of one simulated user's record().  The Philox key is
    mix(seed, user) -- with one user per rank and the usual identical torch.manual_seed on every rank
    (main.py:127) the users still draw INDEPENDENT uniforms, like the reference's single CPU stream
    does; the offset is read from and advanced on torch's CUDA generator of the current device, so
    torch.manual_seed(s) replays the same draws and interleaved torch.rand(device='cuda') calls never
    reuse them.

    take_shared(n): draws that every rank must reproduce identically (the second compression of
    --two-phase, ps_quantizer.py:52-61): key mix(shared seed, 2^32), own offset counter advanced only
    here, both independent of the rank's generator state.  The shared seed is the generator seed of
    rank 0 (share_seed(), broadcast once by the quantizer) or the local one in a single process."""

    SHARED_STREAM = 1 << 32

    def __init__(self):
        self.shared_seed = None
        self.shared_offset = 0

    def _gen(self):
        return torch.cuda.default_generators[torch.cuda.current_device()]

    def take(self, n, user=0):
        gen = self._gen()
        seed = gen.initial_seed() & _M64
        off = int(gen.get_offset())
        gen.set_offset(off + (int(n) + 3) // 4 * 4)
        return _mix64(seed, int(user)), off

    def share_seed(self, seed=None):
        """Fix the seed of the rank-independent stream (None: this process's generator seed)."""
        self.shared_seed = (self._gen().initial_seed() if seed is None else int(seed)) & _M64
        self.shared_offset = 0
        return self.shared_seed

    def take_shared(self, n):
        if self.shared_seed is None:
            self.share_seed()
        off = self.shared_offset
        self.shared_offset = off + (int(n) + 3) // 4 * 4
        return _mix64(self.shared_seed, self.SHARED_STREAM), off


PHILOX = PhiloxState()
