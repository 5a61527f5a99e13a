#!/usr/bin/env python
"""bench.py -- benchmark of the gradient-compression hot path (BASELINE.json configs 2-5).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--codec hsq|qsgd|terngrad|sign|topk] [--k-bit 8|12] [--c-dim 8|16|32] [--n-bit n]
                    [--cr 100] [--mode ps|ring] [--workload resnet50|flat] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Default (the headline, BASELINE.json configs[1]): the 161 gradient tensors of the reference's CIFAR
ResNet-50 (23 520 842 elements; 76 tensors / 23 498 432 elements compressed, the rest identity), HSQ
d=16, K=256 learned codebook, 6-bit norms, one simulated user per GPU, ps exchange.
One step on every rank = fused encode of the local gradient into its packed record -> exchange of the
packed records (N > 1) -> fused decode-and-average (ps) or the chained decode-add-encode (ring).
Metric = gradient elements per second through the whole job (N * elements / step time).

Prints ONE JSON line (rank 0).  Timing: CUDA events on the launching stream, barrier + synchronize
on both sides, max over ranks; inputs rotate over buffers larger than L2.

--impl reference: the same workload through the reference's CPU path on the host cores (the
C/OpenMP oracle port with every host thread; rank 0 only), and -- when baseline/_ref is staged --
the UNMODIFIED Python reference (baseline/ref_runner.py) beside it as `reference_py_value`.

--dump-outputs DIR: after the timed steps, rank 0 writes the gradient its last timed step handed back
(every tensor flattened, concatenated in model order, float32) as DIR/gradient.npy.  Larger outputs are
cut to a fixed seeded sample of DUMP_MAX_ELEMS positions (see dump_outputs()).  The inputs depend only
on the arguments, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True          # the benchmark leaves the tree as it found it (it may be read-only)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

UNIT = "elements/s"
CODEC_DEFAULTS = {"hsq": dict(c_dim=16, n_bit=6), "qsgd": dict(c_dim=128, n_bit=2),
                  "terngrad": dict(c_dim=0, n_bit=1), "sign": dict(c_dim=16, n_bit=6),
                  "topk": dict(c_dim=16, n_bit=6)}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", type=str, default="b200", choices=["b200", "reference"])
    ap.add_argument("--algo", type=str, default="auto", choices=["auto", "exact", "tc"])
    ap.add_argument("--codec", type=str, default="hsq", choices=sorted(CODEC_DEFAULTS))
    ap.add_argument("--mode", type=str, default="ps", choices=["ps", "ring"])
    ap.add_argument("--workload", type=str, default="resnet50", choices=["resnet50", "flat"])
    ap.add_argument("--c-dim", type=int, default=None)
    ap.add_argument("--k-bit", type=int, default=8)
    ap.add_argument("--n-bit", type=int, default=None)
    ap.add_argument("--cr", type=int, default=100)
    ap.add_argument("--sign-wire", type=str, default="2bit", choices=["2bit", "t5"],
                    help="SignSGD wire container: 2 bits per element, or base 3 with five elements per byte")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", type=str, default=None, metavar="DIR",
                    help="write the gradient of the last timed step to DIR/gradient.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    d = CODEC_DEFAULTS[a.codec]
    if a.c_dim is None:
        a.c_dim = d["c_dim"]
    if a.n_bit is None:
        a.n_bit = d["n_bit"]
    return a


def workload_shapes(name):
    if name == "resnet50":
        from util import resnet50_shapes
        return resnet50_shapes()
    return [(25_600_000,)]       # BASELINE config 4: flat 25.6M-element gradient


def codec_label(a):
    if a.codec == "hsq":
        return "HSQ d=%d K=%d n=%d" % (a.c_dim, 2 ** a.k_bit, a.n_bit)
    if a.codec == "qsgd":
        return "QSGD d=%d %d-bit" % (a.c_dim, a.n_bit)
    if a.codec == "terngrad":
        return "TernGrad (c-dim 0, 1-bit)"
    if a.codec == "sign":
        return "SignSGD (ternary%s)" % (", base-3 wire" if getattr(a, "sign_wire", "2bit") == "t5" else "")
    return "top-k cr=%d" % a.cr


def metric_name(a):
    if a.codec == "hsq" and a.mode == "ps":
        return "HSQ gradient elems/s (encode+allgather+decode)"
    return "%s gradient elems/s (%s: encode+exchange+decode)" % (a.codec, a.mode)


def workload_label(a, users):
    """Identical in both arms (the driver compares `config.workload`)."""
    if a.workload == "resnet50":
        w = "ResNet-50 (reference CIFAR variant) 161 gradient tensors, 23520842 elements/user"
    else:
        w = "flat 25600000-element gradient/user"
    return "%s, %s, %d user%s (one per GPU), %s record/apply" % (w, codec_label(a), users, "" if users == 1 else "s", a.mode)


def make_args(a, num_users):
    from types import SimpleNamespace
    return SimpleNamespace(c_dim=a.c_dim, k_bit=a.k_bit, n_bit=a.n_bit, no_cuda=False, random=True, cr=a.cr,
                           ef=False, two_phase=False, mode=a.mode, scale="exp", num_users=num_users,
                           sign_wire=getattr(a, "sign_wire", "2bit"))


def algorithmic_bytes(a, n, users):
    """SURVEY 8(d) / BASELINE.md section 4 bytes per launch for n elements:
    (encode, decode-reduce over `users`, whole step per rank)."""
    if a.codec == "hsq":
        code = 1 if a.k_bit <= 8 else 2
        enc = n * (4 + (code + 1) / a.c_dim)
        dec = n * (4 + (code + 1) * users / a.c_dim)
    elif a.codec in ("qsgd", "terngrad"):
        # read 4 B, write (1 sign + level bits) and one fp32 norm per chunk
        bits = 4 if a.n_bit <= 2 else (8 if a.n_bit <= 6 else 16)
        per = bits / 8 + (4.0 / a.c_dim if a.c_dim else 0.0)
        enc = n * (4 + per)
        dec = n * (4 + per * users)
    elif a.codec == "sign":
        w = 0.2 if getattr(a, "sign_wire", "2bit") == "t5" else 0.25
        enc = n * (4 + w)
        dec = n * (4 + w * users)
    else:
        enc = n * (4 + 8.0 / a.cr)
        dec = n * (4 + 8.0 * users / a.cr)
    return enc, dec, enc + dec


def ncu_traffic_bytes(codec):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from the newest committed
    `ncu --set full` summary under profiles/ (per launch); None if there is none."""
    import csv
    import glob
    tag = {"hsq": "tc"}.get(codec, codec)
    best = None
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_prof_%s_*_summary.csv" % tag))):
        rd = wr = None
        with open(path) as fh:
            for row in csv.reader(fh):
                if len(row) >= 3 and row[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    v = float(row[2]) * {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0}.get(row[1], 1.0)
                    if row[0].endswith("read.sum"):
                        rd = v
                    else:
                        wr = v
        if rd is not None and wr is not None:
            best = (rd + wr, os.path.basename(path))
    return best


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return json.load(fh), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


DUMP_MAX_ELEMS = 8 * 1024 * 1024         # 32 MB of float32 per dump


def dump_outputs(out_dir, flat):
    """--dump-outputs: write `flat` (the step's gradient in model order) as out_dir/gradient.npy, float32.
    Above DUMP_MAX_ELEMS elements only a sample is written: the elements at the sorted positions
    np.random.RandomState(0).choice(n, DUMP_MAX_ELEMS, replace=False).  The sample depends on n alone,
    so it is the same in every build."""
    import numpy as np
    flat = np.asarray(flat, dtype=np.float32).reshape(-1)
    if flat.size > DUMP_MAX_ELEMS:
        flat = flat[np.sort(np.random.RandomState(0).choice(flat.size, DUMP_MAX_ELEMS, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "gradient.npy"), flat)


# ------------------------------------------------------------------ clocks ---
class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons with NVML while the timed loops run."""

    def __init__(self, index, period=0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(self.period)

    def finish(self):
        import numpy as np
        self._halt.set()
        self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


ORIG_AFFINITY = None


def bind_to_gpu_numa(index):
    """Place this rank's pinned host buffers on the NUMA node its GPU hangs off, BEFORE any of them is
    allocated: CPU affinity to that node's cores (first touch) and, where the kernel allows it, a
    preferred-node memory policy.  Round 1's end-to-end number did not scale (46 -> 8 GB/s per GPU from
    N = 1 to 8) because every rank's pinned buffers sat on node 0.  The node comes from sysfs, else from
    NVML's memory / CPU affinity of the device.  Returns a short description for the JSON line; never
    fails the run."""
    global ORIG_AFFINITY
    note = []
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        node = -1
        try:
            bdf = pynvml.nvmlDeviceGetPciInfo(h).busId
            bdf = (bdf.decode() if isinstance(bdf, bytes) else bdf).lower()
            if len(bdf.split(":")[0]) == 8:          # nvml pads the domain to 8 hex digits, sysfs uses 4
                bdf = bdf[4:]
            with open("/sys/bus/pci/devices/%s/numa_node" % bdf) as fh:
                node = int(fh.read().strip())
        except Exception:  # noqa: BLE001
            node = -1
        if node < 0:
            try:                                      # NVML: bit mask of the NUMA nodes closest to the device
                mask = pynvml.nvmlDeviceGetMemoryAffinity(h, 4, 0)
                bits = [64 * w + b for w, word in enumerate(mask) for b in range(64) if (int(word) >> b) & 1]
                if bits:
                    node = bits[0]
                    note.append("node from NVML")
            except Exception:  # noqa: BLE001
                pass
        cpus = set()
        if node >= 0:
            try:
                with open("/sys/devices/system/node/node%d/cpulist" % node) as fh:
                    for part in fh.read().strip().split(","):
                        lo, _, hi = part.partition("-")
                        cpus.update(range(int(lo), int(hi or lo) + 1))
            except Exception:  # noqa: BLE001
                pass
        if not cpus:
            try:                                      # NVML: the device's ideal CPU set
                words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
                cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
                if cpus:
                    note.append("cpus from NVML")
            except Exception:  # noqa: BLE001
                pass
        ORIG_AFFINITY = set(os.sched_getaffinity(0))
        allowed = cpus & ORIG_AFFINITY
        if allowed and allowed != ORIG_AFFINITY:
            os.sched_setaffinity(0, allowed)
            note.append("%d cpus" % len(allowed))
        elif cpus and not allowed:
            note.append("the node's cpus are outside this container's cpuset")
        if node >= 0:
            try:                                      # set_mempolicy(MPOL_PREFERRED, {node}) -- x86-64 syscall 238
                import ctypes
                libc = ctypes.CDLL(None, use_errno=True)
                nodemask = ctypes.c_ulong(1 << node)
                rc = libc.syscall(238, 1, ctypes.byref(nodemask), ctypes.c_ulong(65))
                note.append("mempolicy preferred" if rc == 0 else "mempolicy refused (errno %d)" % ctypes.get_errno())
            except Exception:  # noqa: BLE001
                pass
            return "NUMA node %d (%s)" % (node, ", ".join(note) or "no binding possible")
        return "numa node unknown" + (" (%s)" % ", ".join(note) if note else "")
    except Exception as e:  # noqa: BLE001
        return "not bound (%s)" % type(e).__name__


# ----------------------------------------------------------- CPU baselines ---
def host_threads():
    return os.cpu_count() or 1


def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1 to its workers: the CPU arm must not inherit that
    (nor the NUMA binding the GPU arm gave itself)."""
    if ORIG_AFFINITY:
        try:
            os.sched_setaffinity(0, ORIG_AFFINITY)
        except Exception:  # noqa: BLE001
            pass
    n = host_threads()
    os.environ["OMP_NUM_THREADS"] = str(n)
    os.environ.pop("OMP_THREAD_LIMIT", None)
    try:
        import ctypes
        ctypes.CDLL("libgomp.so.1").omp_set_num_threads(n)
    except Exception:  # noqa: BLE001
        pass
    return n


class CpuPort:
    """The oracle port (C + OpenMP) of the reference path on the host cores: per user
    decompress(compress(g)) over every tensor, then apply() (ps_quantizer.py:27-65 /
    ring_quantizer.py:25-49).  Inputs are generated once; step() is what gets timed."""

    def __init__(self, a, n_users):
        import numpy as np
        from oracle import gq_oracle as O
        self.O, self.a, self.n_users = O, a, n_users
        self.threads = use_all_host_threads()
        O.lib()
        use_all_host_threads()
        shapes = workload_shapes(a.workload)
        sizes = [int(np.prod(s)) for s in shapes]
        rs = np.random.RandomState(1)
        base = [(rs.standard_normal(n) * 0.01).astype(np.float32).reshape(s) for s, n in zip(shapes, sizes)]
        # users share the tensor values up to a cheap, user-specific perturbation (generating
        # 8 x 23.5M normals costs more than the timed work); the codec cost does not depend on it
        self.grads = [base] + [[g * np.float32(1.0 + 0.01 * u) for g in base] for u in range(1, n_users)]
        cbdir = os.path.join(ROOT, "gradient-quantization_b200", "codebooks", "learned_codebook")
        self.codecs = []
        n_draws = 0
        for s, n in zip(shapes, sizes):
            if n <= 1000:
                self.codecs.append(O.Identity())
            elif a.codec == "hsq":
                d = O.chunk_dim(n, a.c_dim)
                cb = O.normalize(O.fvecs_read(os.path.join(cbdir, "angular_dim_%d_Ks_%d.fvecs" % (d, 2 ** a.k_bit))))[1]
                self.codecs.append(O.HSQ(n, s, cb, a.n_bit, True))
                n_draws += n // d
            elif a.codec in ("qsgd", "terngrad"):
                self.codecs.append(O.QSGD(n, s, a.c_dim, a.n_bit, True))
                n_draws += n
            elif a.codec == "sign":
                self.codecs.append(O.Sign(n, s))
            else:
                self.codecs.append(O.TopK(n, s, a.cr))
        self.draws = rs.random_sample(n_draws * n_users).astype(np.float32)
        self.elems = sum(sizes) * n_users
        self.out = None

    def step(self):
        O = self.O
        t0 = time.perf_counter()
        if self.a.mode == "ps":
            self.out = O.ps_step(self.codecs, self.grads, O.UniformStream(self.draws))
        else:
            self.out = O.ring_step(self.codecs, self.grads, O.UniformStream(self.draws))
        return time.perf_counter() - t0


def reference_python(a, n_users, steps=2, warmup=1, timeout=900):
    """The UNMODIFIED reference (baseline/_ref) in a subprocess, all host threads; dict or None."""
    runner = os.path.join(ROOT, "baseline", "ref_runner.py")
    if not os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "compressors")):
        return None
    env = dict(os.environ)
    env["OMP_NUM_THREADS"] = str(host_threads())
    env["MKL_NUM_THREADS"] = str(host_threads())
    cmd = [sys.executable, runner, "--codec", a.codec, "--mode", a.mode, "--users", str(n_users), "--steps", str(steps),
           "--warmup", str(warmup), "--workload", a.workload, "--c-dim", str(a.c_dim), "--k-bit", str(a.k_bit),
           "--n-bit", str(a.n_bit), "--cr", str(a.cr)]
    if a.codec == "hsq" and a.k_bit > 8:
        cmd += ["--max-elems", "3000000"]     # the reference materialises [N/d, K] fp32 scores: bounded sample
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)
        for line in reversed(out.stdout.strip().splitlines()):
            if line.startswith("{"):
                r = json.loads(line)
                return None if "unavailable" in r else r
    except Exception:  # noqa: BLE001
        return None
    return None


def run_reference_arm(a):
    """--impl reference: rank 0 runs the CPU path with every host thread on the FULL workload
    (all `gpus` users) for exactly `steps` timed steps; the other ranks exit."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import numpy as np
    n_users = a.gpus
    port = CpuPort(a, n_users)
    W, K = max(a.warmup, 1), max(a.steps, 1)
    budget = 240.0                       # the whole arm must end within a few minutes
    t_first = port.step()
    done_w = 1
    while done_w < W and t_first * (done_w + 1 + K) < budget:
        port.step()
        done_w += 1
    k_eff = K if t_first * K < budget else max(int(budget / max(t_first, 1e-6)), 1)
    times = [port.step() for _ in range(k_eff)]
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, np.concatenate([o.reshape(-1) for o in port.out]))
    t = float(np.mean(times))
    value = port.elems / t
    ref_py = reference_python(a, n_users, steps=1 if n_users > 2 else 2, warmup=1)
    cpu = {"value": value, "unit": UNIT, "cores": port.threads, "kind": "port",
           "sample": "%d users x %d elements per step, %d timed steps, C/OpenMP oracle port of the reference path, %d threads"
                     % (n_users, port.elems // n_users, len(times), port.threads)}
    if ref_py is not None:
        cpu["reference_py_value"] = ref_py["value"]
        cpu["reference_py"] = {k: ref_py[k] for k in ("seconds_per_step", "steps", "elements_per_user", "users", "cores",
                                                      "torch_threads", "torch", "kind")}
    line = {
        "impl": "reference", "metric": metric_name(a), "value": value, "unit": UNIT, "n_gpus": a.gpus,
        "steps": len(times), "warmup": done_w, "ms_per_step": t * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_label(a, n_users), "elements_per_user": port.elems // n_users,
                   "users": n_users, "codec": a.codec, "mode": a.mode},
        "cpu_baseline": cpu,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# -------------------------------------------------------------- GPU arm ---
def main():
    a = parse_args()
    if a.impl == "reference":
        return run_reference_arm(a)

    import numpy as np
    import torch
    import torch.distributed as dist

    import gq_b200
    from gq_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a.gpus and a.gpus > 1:
        raise SystemExit("bench.py --gpus %d needs WORLD_SIZE == %d (launch with torch.distributed.run)"
                         % (a.gpus, a.gpus))
    numa = bind_to_gpu_numa(local_rank)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # torch seeds its default generators at random in every process; the stochastic-rounding draws
    # (Philox keyed by the CUDA generator's seed, mixed with the user) must be the same in every run
    torch.manual_seed(1)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W, K = max(a.warmup, 3), a.steps

    shapes = workload_shapes(a.workload)
    args = make_args(a, world)
    args.hsq_algo = {"auto": _lib.ALGO_AUTO, "exact": _lib.ALGO_EXACT, "tc": _lib.ALGO_TC}[a.algo]
    Comp = {"hsq": gq_b200.NearestNeighborCompressor, "qsgd": gq_b200.QSGDCompressor,
            "terngrad": gq_b200.QSGDCompressor, "sign": gq_b200.SignSGDCompressor,
            "topk": gq_b200.TopKSparsificationCompressor}[a.codec]
    params = [torch.nn.Parameter(torch.empty(0, device=dev)) for _ in shapes]
    for p, s in zip(params, shapes):
        p.data = torch.zeros(s, device=dev)
    q = gq_b200.Quantizer(Comp, params, args)
    plan = q.plan
    n_total = plan.total_elems()
    n_comp = plan.compressed_elems()
    grp = plan.groups[0]

    # synthetic gradients, resident in HBM, rotating so that the inputs exceed L2 (126 MB)
    ROT = 4
    gen = torch.Generator(device=dev)
    gen.manual_seed(1 + rank)
    inputs = [torch.randn(plan.arena_elems, device=dev, generator=gen) * 0.01 for _ in range(ROT)]
    outputs = [torch.empty(plan.arena_elems, device=dev) for _ in range(ROT)]

    if a.mode == "ps":
        def step(i):
            q.encode_local(rank, src=inputs[i % ROT])          # fused encode into the local packed record
            q.exchange_and_decode(out=outputs[i % ROT])        # exchange of the records + fused decode-and-average
    else:
        def step(i):
            q.step_buffers(src=inputs[i % ROT], out=outputs[i % ROT])   # chained decode-add-encode + final decode

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def all_max(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return t.item()
        return ms

    sampler = ClockSampler(local_rank)
    for i in range(W):
        step(i)
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        step(i)
    e1.record()
    barrier()
    ms_per_step = all_max(e0.elapsed_time(e1)) / K
    value = world * n_total / (ms_per_step * 1e-3)
    if a.dump_outputs and rank == 0:
        # the buffer of the last timed step, before the per-kernel and end-to-end loops below reuse it
        last = plan.views(outputs[(K - 1) % ROT])
        dump_outputs(a.dump_outputs, torch.cat([v.reshape(-1) for v in last]).cpu().numpy())

    # ---- per-kernel timing (same rotation; every rank runs them, rank 0 reports) ----
    def time_loop(fn, iters):
        for i in range(3):
            fn(i)
        torch.cuda.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for i in range(iters):
            fn(i)
        a1.record()
        torch.cuda.synchronize()
        return a0.elapsed_time(a1) / iters

    slot = q.p2p.row() if getattr(q, "p2p", None) is not None else rank
    encode_ms = time_loop(lambda i: plan.encode(slot, src=inputs[i % ROT]), K)
    if a.mode == "ps":
        decode_ms = time_loop(lambda i: q.decode_exchanged(outputs[i % ROT]), K)
    else:
        decode_ms = time_loop(lambda i: plan.decode(first_user=0, n_users=1, mean=False, out=outputs[i % ROT]), K)
    search_ms = None
    if a.codec == "hsq":
        st = _lib.stream()
        ws = plan.workspace
        codes_ptr = plan.records[slot].data_ptr() + grp.codes_off
        keys_ptr = ws.data_ptr()          # the real per-tensor min/max keys ride along (reset every call by a tiny fill)

        def search_only(i):
            _lib.call("gq_hsq_search", inputs[i % ROT].data_ptr() + grp.arena_off * 4, grp.n_chunks, grp.dim,
                      grp.codebook.data_ptr(), grp.K, codes_ptr, grp.code_bytes, plan.u_scratch.data_ptr(),
                      grp.seg_start.data_ptr(), grp.n_seg, keys_ptr, ws.data_ptr() + 8192, ws.numel() - 8192,
                      args.hsq_algo, st)
        if ws.numel() > 16384:
            search_ms = time_loop(search_only, K)

    # ---- end to end through the public quantizer API with HOST buffers ----
    # Every step copies its gradient from pinned host memory (H2D), hands it to the quantizer as ordinary
    # per-parameter .grad tensors (views of a staging buffer in MODEL order -- not the codec arena's
    # order, so record() runs its multi-tensor gather kernel like it would after a real backward()),
    # and reads the averaged gradient back to pinned host memory (D2H).  Software-pipelined over two
    # device buffers: H2D of step i+1 and D2H of step i-1 overlap the codec work of step i.
    sizes = [int(np.prod(s)) for s in shapes]
    flat_elems = sum(sizes)

    def model_views(buf):
        out, o = [], 0
        for s, n in zip(shapes, sizes):
            out.append(buf[o:o + n].view(s))
            o += n
        return out

    host_in = [torch.empty(flat_elems, dtype=torch.float32).pin_memory() for _ in range(2)]
    for h in host_in:
        h.normal_(0.0, 0.01)
    host_out = [torch.empty(plan.arena_elems, dtype=torch.float32).pin_memory() for _ in range(2)]
    dev_in = [torch.empty(flat_elems, device=dev) for _ in range(2)]
    dev_in_views = [model_views(b) for b in dev_in]
    dev_out = [torch.empty(plan.arena_elems, device=dev) for _ in range(2)]
    s_h2d, s_d2h = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    main_s = torch.cuda.current_stream()
    ev_in = [torch.cuda.Event() for _ in range(2)]
    ev_in_free = [torch.cuda.Event() for _ in range(2)]
    ev_out = [torch.cuda.Event() for _ in range(2)]
    ev_out_free = [torch.cuda.Event() for _ in range(2)]

    def issue_h2d(i):
        b = i % 2
        with torch.cuda.stream(s_h2d):
            s_h2d.wait_event(ev_in_free[b])
            dev_in[b].copy_(host_in[b], non_blocking=True)
            ev_in[b].record(s_h2d)

    def e2e_step(i):
        b = i % 2
        main_s.wait_event(ev_in[b])
        for p, v in zip(params, dev_in_views[b]):
            p.grad = v                                            # this step's gradient, per parameter
        q.record(rank, epoch=1)                                   # public API: gather + fused encode (+ ring hop)
        ev_in_free[b].record(main_s)
        q.apply()                                                 # exchange + decode-and-average
        main_s.wait_event(ev_out_free[b])
        dev_out[b].copy_(plan.arena, non_blocking=True)
        ev_out[b].record(main_s)
        with torch.cuda.stream(s_d2h):
            s_d2h.wait_event(ev_out[b])
            host_out[b].copy_(dev_out[b], non_blocking=True)      # D2H of the averaged gradient
            ev_out_free[b].record(s_d2h)

    for b in range(2):
        ev_in_free[b].record(main_s)
        ev_out_free[b].record(main_s)
    KE = max(min(K, 20), 4)

    def e2e_loop(n):
        issue_h2d(0)
        for i in range(n):
            if i + 1 < n:
                issue_h2d(i + 1)
            e2e_step(i)
        main_s.wait_stream(s_d2h)

    e2e_loop(3)
    barrier()
    b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    b0.record()
    e2e_loop(KE)
    b1.record()
    barrier()
    e2e_ms = all_max(b0.elapsed_time(b1)) / KE
    e2e_value = world * n_total / (e2e_ms * 1e-3)
    for p, v in zip(params, plan.views()):
        p.grad = v

    # keep the same loop running (~0.6 s) so that the sampler sees the clocks under load; the number
    # of extra steps is derived from the all-reduced step time, hence identical on every rank
    n_extra = int(min(max(0.6 / (ms_per_step * 1e-3), 50), 20000))
    for i in range(n_extra):
        step(i)
        if i % 200 == 199:
            torch.cuda.synchronize()
    barrier()
    clocks = sampler.finish()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks, peak_kind = measured_peaks()
    traffic = ncu_traffic_bytes(a.codec)
    hbm_peak = float(peaks["hbm_gbs"])
    enc_b, dec_b, step_b = algorithmic_bytes(a, n_comp, world)
    ident_b = (n_total - n_comp) * 4
    dom_ms = search_ms if search_ms is not None else encode_ms
    if a.codec == "hsq":
        # dominant kernel = the tcgen05 search + fused tail launch; SURVEY 8(d): read 4 B/elem, write
        # code + norm code per chunk.  (The fp32 u intermediate it also writes/reads is not algorithmic.)
        dom_name = "hsq_encode (%s)" % a.algo
        dom_ms = encode_ms
    else:
        dom_name = "%s encode" % a.codec
    achieved = enc_b / (dom_ms * 1e-3) / 1e9
    roofline = {
        "bound": "hbm", "kernel": dom_name, "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
        "frac": achieved / hbm_peak, "traffic": traffic[0] if traffic else None,
        "traffic_source": traffic[1] if traffic else None, "peak_source": peak_kind,
        "kernel_ms": dom_ms, "algorithmic_bytes_per_launch": enc_b,
        "step_hbm_frac": (step_b + 2 * ident_b) / (ms_per_step * 1e-3) / 1e9 / hbm_peak,
        "encode_ms": encode_ms, "decode_ms": decode_ms,
        "decode_achieved": dec_b / (decode_ms * 1e-3) / 1e9, "decode_frac": dec_b / (decode_ms * 1e-3) / 1e9 / hbm_peak,
    }
    if a.codec == "hsq":
        roofline["search_ms"] = search_ms
        roofline["tensor_flops_per_launch"] = 2.0 * grp.K * grp.n
        roofline["tensor_tflops_achieved"] = 2.0 * grp.K * grp.n / (dom_ms * 1e-3) / 1e12
    if getattr(q, "p2p", None) is not None:
        exch = "peer-to-peer (%s): packed records cross NVLink through peer-mapped memory" % q.exchange_name()
    elif world > 1:
        exch = "NCCL (%s)" % ("all-gather of packed records" if a.mode == "ps" else q.exchange_name() + ", packed records")
    else:
        exch = "none (1 user)"
    line = {
        "metric": metric_name(a), "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_label(a, world), "elements_per_user": n_total,
                   "compressed_elements": n_comp, "users": world, "codec": a.codec, "mode": a.mode,
                   "wire_bytes_per_user": plan.wire_bytes(), "algo": a.algo, "exchange": exch,
                   "l2": "inputs/outputs rotate over %d buffers of %.0f MB each (> 126 MB L2)"
                         % (ROT, plan.arena_elems * 4 / 1e6)},
        "roofline": roofline,
        "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": flat_elems * 4, "d2h_bytes_per_step": plan.arena_elems * 4,
                "api": "Quantizer.record(rank)/apply() on ordinary per-parameter .grad tensors (model order, copied "
                       "from pinned host memory each step; record() gathers them into the codec arena with one "
                       "multi-tensor kernel), averaged gradient copied back to pinned host memory each step",
                "pipelining": "double-buffered: H2D of step i+1 and D2H of step i-1 overlap step i",
                "host": numa},
        "gpu_launches": K * q.launches_per_step(),
        "clocks": clocks,
    }
    if not a.no_cpu_baseline and world == 1:
        port = CpuPort(a, 1)
        port.step()
        dt = min(port.step() for _ in range(3))
        cpu = {"value": port.elems / dt, "unit": UNIT, "cores": port.threads, "kind": "port",
               "sample": "1 user-pass (encode+decode) of the full %d-element gradient, best of 3, "
                         "C/OpenMP oracle port, %d threads (%.3f s)" % (port.elems, port.threads, dt)}
        ref_py = reference_python(a, 1, steps=2, warmup=1)
        if ref_py is not None:
            cpu["reference_py_value"] = ref_py["value"]
            cpu["reference_py"] = {k: ref_py[k] for k in ("seconds_per_step", "steps", "elements_per_user", "users",
                                                          "cores", "torch_threads", "torch", "kind")}
        line["cpu_baseline"] = cpu
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
