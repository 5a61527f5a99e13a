#!/usr/bin/env python
"""Where the time of one HSQ step goes with and without deferred levels (one GPU, one user).

    python tools/defer_ab.py [--steps 200] [--rounds 5] [--workload resnet50|flat]

bench.py's headline workload (HSQ d=16, K=256, 6-bit norms, ps, one user) in one process:

  step       encode_local + exchange_and_decode (what bench.py times as ms_per_step), alternating
             GQ_DEFER_LEVELS=1 (search-only encode, levels computed by the decode) and =0 (one-launch
             encode with its grid barrier and quantization tail, plain decode) for --rounds rounds
  search     the search-only launch (gq_hsq_encode_search)
  dec_quant  the fused quantize-and-decode launch (gq_hsq_decode_quantize)
  encode     the one-launch encode (FusedPlan.encode without deferral)
  decode     the plain decode of a complete record

bench.py's per-kernel loops (roofline.encode_ms / decode_ms) time the last two, so with deferral
they no longer add up to ms_per_step; search + dec_quant is the split of the deferred step.
Inputs and outputs rotate over 4 buffers of the arena size (> 126 MB L2 in total), as in bench.py.
CUDA events on the launching stream; medians over the rounds.  Prints one JSON line.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--workload", default="resnet50", choices=["resnet50", "flat"])
    a = ap.parse_args()

    import torch

    import gq_b200
    from gq_b200 import _lib
    from util import make_args, resnet50_shapes

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    torch.manual_seed(1)
    shapes = resnet50_shapes() if a.workload == "resnet50" else [(25_600_000,)]
    params = [torch.nn.Parameter(torch.zeros(s, device=dev)) for s in shapes]
    q = gq_b200.Quantizer(gq_b200.NearestNeighborCompressor, params, make_args(num_users=1))
    plan = q.plan
    g = plan.groups[0]
    if not plan.can_defer_levels():
        raise SystemExit("this plan cannot defer its levels (GQ_DEFER_LEVELS / GQ_TC_V set?)")
    ROT = 4
    gen = torch.Generator(device=dev)
    gen.manual_seed(1)
    inputs = [torch.randn(plan.arena_elems, device=dev, generator=gen) * 0.01 for _ in range(ROT)]
    outputs = [torch.empty(plan.arena_elems, device=dev) for _ in range(ROT)]
    st = _lib.stream()

    def timed(fn, n):
        for i in range(3):
            fn(i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n * 1e3   # us

    def step(i):
        q.encode_local(0, src=inputs[i % ROT])
        q.exchange_and_decode(out=outputs[i % ROT])

    rec = plan.records[0].data_ptr()

    def search(i):
        _lib.call("gq_hsq_encode_search", inputs[i % ROT].data_ptr() + g.arena_off * 4, g.n_chunks, g.dim,
                  _lib.ptr(g.codebook), g.K, _lib.ptr(g.seg_start), g.n_seg, rec + g.codes_off, g.code_bytes,
                  _lib.ptr(plan.u_scratch), _lib.ptr(plan.workspace), plan.workspace.numel(), st)

    def dec_quant(i):   # u and the keys of the last search stay valid: the decode reads them only
        seed, off = _lib.PHILOX.take(g.n_chunks, 0)
        _lib.call("gq_hsq_decode_quantize", rec + g.codes_off, rec + g.l_off, rec + g.lbub_off,
                  _lib.ptr(plan.u_scratch), _lib.ptr(plan.workspace), g.n_chunks, g.dim, _lib.ptr(g.codebook), g.K,
                  _lib.ptr(g.seg_start), g.n_seg, g.n_bit, 1, None, seed, off, 0,
                  outputs[i % ROT].data_ptr() + g.arena_off * 4, st)

    def encode(i):
        plan.encode(0, src=inputs[i % ROT])

    def decode(i):
        plan.decode(first_user=0, n_users=1, mean=False, out=outputs[i % ROT])

    res = {k: [] for k in ("step_defer", "step_onelaunch", "search", "dec_quant", "encode", "decode")}
    for _ in range(a.rounds):
        for k, v in (("step_defer", "1"), ("step_onelaunch", "0")):
            os.environ["GQ_DEFER_LEVELS"] = v
            res[k].append(timed(step, a.steps))
        os.environ["GQ_DEFER_LEVELS"] = "1"
        res["search"].append(timed(search, a.steps))
        res["dec_quant"].append(timed(dec_quant, a.steps))
        plan.records   # noqa: B018  (no record left pending)
        res["encode"].append(timed(encode, a.steps))
        res["decode"].append(timed(decode, a.steps))
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        smi = "nvidia-smi unavailable: %r" % (e,)
    med = {k: statistics.median(v) for k, v in res.items()}
    print(json.dumps({"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi, "workload": a.workload,
                      "steps": a.steps, "rounds": a.rounds, "unit": "us",
                      "median": med, "all": res,
                      "step_defer_over_onelaunch": med["step_defer"] / med["step_onelaunch"]}), flush=True)


if __name__ == "__main__":
    main()
