import torch

from .. import _lib
from ._common import single_segment, uniforms_arg


class ProbabilisticScalarCompressor(object):
    """n-bit affine stochastic quantizer of a whole tensor
    (reference compressors/probabilistic_scalar_compressor.py:4-33).

    compress(vec) -> (lower_bound, upper_bound, l) with l int32 in [0, 2^n];
    decompress((lb, ub, l)) -> l * (ub - lb) / 2^n + lb.  Unlike the reference
    there is no host synchronisation: the lb == ub case is handled on the device.
    """

    def __init__(self, n_bit, args):
        self.n_bit = n_bit
        self.s = 2 ** n_bit
        self.code_dtype = torch.int32
        self.random = args.random
        self.rng = getattr(args, "rng", "philox")

    def compress(self, vec, uniforms=None):
        v = _lib.f32c(vec, "vec").reshape(-1)
        n = v.numel()
        dev = v.device
        l = torch.empty(n, dtype=torch.int32, device=dev)
        lbub = torch.empty(2, dtype=torch.float32, device=dev)
        keys = torch.empty(2, dtype=torch.int32, device=dev)
        seg = single_segment(n, dev)
        random = 1 if self.random else 0
        r = uniforms_arg(uniforms, n, dev) if random else None
        torch_rng = random and r is None and self.rng == "torch"
        if torch_rng:
            # reference-faithful draw: CPU generator, skipped when lb == ub (:15-16, :23-25); the levels
            # are then all 0 whatever the draws, so the Philox stream is not touched either
            lo, hi = torch.aminmax(v)
            if (lo - hi).item() != 0.0:
                r = torch.rand(n).to(dev)
        seed, off = _lib.PHILOX.take(n) if (random and r is None and not torch_rng) else (0, 0)
        _lib.call("gq_norm_quantize", _lib.ptr(v), n, _lib.ptr(seg), 1, self.n_bit, random, _lib.ptr(r),
                  seed, off, _lib.ptr(l), 4, _lib.ptr(lbub), _lib.ptr(keys), 0, _lib.stream())
        return lbub[0], lbub[1], l.view(vec.shape)

    def decompress(self, signature):
        lower_bound, upper_bound, l = signature
        lc = _lib.require_cuda(l, "l").contiguous().view(-1)
        n = lc.numel()
        dev = lc.device
        lbub = torch.stack([lower_bound.reshape(()), upper_bound.reshape(())]).to(dev, torch.float32)
        out = torch.empty(n, dtype=torch.float32, device=dev)
        seg = single_segment(n, dev)
        if lc.dtype == torch.uint8:
            l_bytes = 1
        else:
            l_bytes = 4
            lc = lc.to(torch.int32)
        _lib.call("gq_norm_dequantize", _lib.ptr(lc), l_bytes, n, _lib.ptr(seg), 1, self.n_bit,
                  _lib.ptr(lbub), _lib.ptr(out), _lib.stream())
        return out.view(l.shape)
