#!/usr/bin/env python
# -*- coding: utf-8 -*-
"""bench.py -- lasso sweeps/s on B200 (BASELINE.json metric) with roofline and CPU baseline.

    python bench.py --gpus 1 --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path
    python bench.py --steps K --warmup W --dump-outputs DIR  # also writes x and r of the last timed sweep

A "step" is one sweep: BLOCK block steps, each reading the column block A_m for the block
gradient A_m^T r and again for A_m D (prox, line search, error and updates fused).  The
workload is BASELINE.json configs[1]: dense fp32 lasso 10,000 x 100,000, 100 column
blocks, synthetic Gaussian A with unit-l2 rows (reference recipe parameters.py:20-33),
generated on the device.  A (4 GB) is far larger than L2 (126 MB), so nothing is flushed
between timed steps.

`value`  : sweeps/s with everything resident in HBM (K fused launches, CUDA events).
`e2e`    : sweeps/s through the reference-facing API, ClassLasso.run(): host b -> device,
           the solve, x -> host, all inside the timed region (A is uploaded once by
           GPU_Calculation(A, BLOCK), exactly as in the reference driver cpu_vs_gpu.py:131);
           10 sweeps per call by default -- a solve of C2 to eps = 1e-4 takes 9.
`roofline`: algorithmic bytes of a sweep (SURVEY.md section 8(d)) / kernel time vs the
           measured HBM copy peak of MEASURED_PEAKS.json.
`cpu_baseline`: the reference's own ClassLassoCPU.run (oracle/_ref, an unmodified copy made by
           oracle/make_ref.py) on a bounded sample; the NumPy port of the same loop beside it.
N > 1 (torchrun): one C2-sized column shard per GPU (weak scaling); the line also carries an
oracle-checked parity record of a small sharded solve and a C4-shard leg (50,000 x 125,000 fp32
per GPU: 8 GPUs = BASELINE.json configs[3]).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# The CPU arm uses every host core it can: torchrun exports OMP_NUM_THREADS=1 to its workers, which
# would pin NumPy's BLAS to one thread before it is even imported (round 1: the N>=2 reference
# arm ran 7x slower than the N=1 one for this reason).
if "reference" in sys.argv[1:]:
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_v] = str(os.cpu_count() or 1)

import numpy as np  # noqa: E402

METRIC = "lasso_sweeps_per_s"
UNIT = "sweeps/s"
# BASELINE.json configs[1]
C2 = dict(N=10000, K=100000, BLOCK=100, den=0.01, seed=2, dtype="float")
FALLBACK_HBM_GBS = 6650.0     # /opt/skills/guides/B200_PROFILING.md fallback


def sweep_bytes(N, K, BLOCK, s):
    return 2 * N * K * s + 5 * BLOCK * N * s + 4 * K * s


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def ncu_traffic(config, layout):
    """dram bytes per sweep from the committed ncu --set full capture of this workload, if any"""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    key = layout if config == "c2" else "%s_%s" % (config, layout)
    try:
        with open(path) as f:
            return json.load(f).get(key)
    except Exception:
        return None


# ------------------------------------------------------------------------------ clocks
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML polled from a thread
    every ~4 ms (nvidia_ml_py), nvidia-smi -lms as a fallback."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []          # (time, sm_mhz, max_mhz, [reasons])
        self.proc = None
        self.nvml = None
        self.stop_flag = False

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll(self):
        nv = self.nvml
        bits = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        while not self.stop_flag:
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM))
                mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                self.rows.append((time.time(), sm, self.max_mhz, [n for n, b in bits.items() if mask & b]))
            except Exception:
                pass
            time.sleep(0.004)

    def _pump(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.proc.stdout:
            f = [x.strip() for x in line.strip().split(",")]
            try:
                self.rows.append((time.time(), float(f[0]), float(f[1]),
                                  [n for n, v in zip(names, f[2:6]) if v.lower().startswith("active")]))
            except Exception:
                continue

    def stop(self, t0, t1):
        if self.nvml is None and self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml / nvidia-smi unavailable"], "samples": 0}
        if self.nvml is not None:
            self.stop_flag = True
            self.thread.join(timeout=1.0)
        else:
            time.sleep(0.05)
            self.proc.terminate()
        # NVML queries can stall while the process sits in a stream synchronisation, so samples
        # up to 10 ms before / after the region count as "during" (clocks do not move that fast)
        inside = [r for r in self.rows if t0 - 0.010 <= r[0] <= t1 + 0.010]
        rows = inside or self.rows          # (a region shorter than the sampling period: nearest samples)
        reasons = sorted({n for r in rows for n in r[3]})
        return {"sm_mhz": float(np.median([r[1] for r in rows])) if rows else None,
                "sm_max_mhz": float(max(r[2] for r in rows)) if rows else None,
                "reasons": reasons, "samples": len(inside),
                "source": "nvml, 4 ms period" if self.nvml is not None else "nvidia-smi -lms 20"}


# ------------------------------------------------------------------------------ data
def make_device_instance(torch, device, N, K, BLOCK, den, seed, torch_dtype, ld, layout="row",
                         dist=None, rank=0):
    """reference recipe (parameters.py:20-33) on the device: Gaussian A, unit-l2 rows,
    sparse x_true, b = A x_true + e, mu = 0.1 |A^T b|_inf.  Returns (store, b, mu).
    With ``dist`` (multi-GPU) every rank generates its own column shard (K local columns,
    seed + rank); row norms, b and mu are combined over the ranks, the noise e is the same
    on every rank."""
    w = K // BLOCK
    gen = torch.Generator(device=device)
    gen.manual_seed(seed + 1000 * rank)
    gen_common = torch.Generator(device=device)
    gen_common.manual_seed(seed + 77)
    rows = N if layout == "row" else w
    store = torch.zeros((BLOCK, rows, ld), dtype=torch_dtype, device=device)
    sq = torch.zeros(N, dtype=torch.float64, device=device)
    for m in range(BLOCK):
        blk = torch.randn((N, w), generator=gen, dtype=torch_dtype, device=device)
        sq += (blk.double() ** 2).sum(dim=1)
        if layout == "row":
            store[m, :, :w] = blk
        else:
            store[m, :, :N] = blk.t()
    if dist is not None:
        dist.all_reduce(sq)
    inv = (1.0 / sq.sqrt()).to(torch_dtype)
    x_true = torch.randn(K, generator=gen, dtype=torch.float64, device=device)
    x_true *= (torch.rand(K, generator=gen, dtype=torch.float64, device=device) < den)
    b = torch.zeros(N, dtype=torch.float64, device=device)
    for m in range(BLOCK):
        if layout == "row":
            store[m, :, :w] *= inv[:, None]
            b += store[m, :, :w].double() @ x_true[m * w:(m + 1) * w]
        else:
            store[m, :, :N] *= inv[None, :]
            b += store[m, :, :N].double().t() @ x_true[m * w:(m + 1) * w]
    if dist is not None:
        dist.all_reduce(b)
    b += 1e-2 * torch.randn(N, generator=gen_common, dtype=torch.float64, device=device)
    gmax = 0.0
    for m in range(BLOCK):
        if layout == "row":
            g = store[m, :, :w].double().t() @ b
        else:
            g = store[m, :, :N].double() @ b
        gmax = max(gmax, float(g.abs().max()))
    if dist is not None:
        t = torch.tensor([gmax], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        gmax = float(t.item())
    return store, b.cpu().numpy().reshape(-1, 1), 0.1 * gmax


# ------------------------------------------------------------------------------ CPU arm
C2_SAMPLE = dict(N=10000, K=3000, BLOCK=3)       # same block shape as C2 (10000 x 1000), 3 of its 100 blocks


def blas_threads(n=None):
    """set (when n is given) and return the BLAS thread count actually in use"""
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        if n:
            threadpool_limits(limits=int(n))
        info = [p.get("num_threads") for p in threadpool_info() if p.get("user_api") == "blas"]
        return int(max(info)) if info else None
    except Exception:
        return None


def cpu_sample(N, K, BLOCK, seed=2):
    """C2-shaped sample on the host (reference recipe parameters.py:20-33, pinned seed)"""
    rng = np.random.RandomState(seed)
    A = rng.standard_normal((N, K))
    A /= np.linalg.norm(A, axis=1, keepdims=True)
    xt = rng.standard_normal((K, 1)) * (rng.rand(K, 1) < 0.01)
    b = A @ xt + 1e-2 * rng.standard_normal((N, 1))
    mu = 0.1 * np.max(np.abs(A.T @ b))
    return A, b, float(mu)


def largest_divisor(n, limit):
    return max(d for d in range(1, max(1, limit) + 1) if n % d == 0)


class RefCPU:
    """the UNMODIFIED reference ClassLassoCPU (oracle/_ref/lasso.py:25-169; Pool(P) forked per
    run(), lasso.py:101) on the C2-shaped sample.  One step = run() for BLOCK iterations = one
    sweep of the sample; the time is what run() itself returns (lasso.py:98,164)."""

    def __init__(self, P):
        from oracle import make_ref
        self.ref_lasso, _, self.ref_cpu = make_ref.import_reference()
        N, K, BLOCK = C2_SAMPLE["N"], C2_SAMPLE["K"], C2_SAMPLE["BLOCK"]
        self.A, self.b, self.mu = cpu_sample(N, K, BLOCK)
        self.P, self.BLOCK, self.K = P, BLOCK, K
        self.A_block_p = self.ref_cpu.A_bp_get(self.A, BLOCK, P)
        self.d_ATA = self.ref_cpu.fun_diag_ATA(self.A_block_p)

    def sweep_seconds(self):
        solver = self.ref_lasso.ClassLassoCPU(self.A_block_p, self.d_ATA, self.A, self.b, self.mu,
                                              self.BLOCK, self.P, self.BLOCK)
        return float(solver.run(SILENCE=True))


def port_sweeps_per_s(seconds):
    """the NumPy port of the same loop (oracle/lasso_oracle.py), BLAS on all host threads, without
    the reference's per-call Pool pickling: sample sweeps/s"""
    from oracle import lasso_oracle as orc
    N, K, BLOCK = C2_SAMPLE["N"], C2_SAMPLE["K"], C2_SAMPLE["BLOCK"]
    A, b, mu = cpu_sample(N, K, BLOCK)
    orc.lasso_oracle(A, b, mu, BLOCK, BLOCK, None, faithful=False)
    o = orc.lasso_oracle(A, b, mu, BLOCK, BLOCK * 100000, None, faithful=False, time_limit=seconds)
    return o["iters"] / float(BLOCK) / o["elapsed"]


def ref_available():
    try:
        from oracle import make_ref
        return make_ref.available()
    except Exception:
        return False


def cpu_baseline_block(seconds=10.0):
    """~20 s of CPU work on rank 0: the reference's own class on the sample (3 sweeps) and the port"""
    cores = os.cpu_count() or 1
    frac = C2_SAMPLE["K"] / float(C2["K"])
    blas_threads(cores)
    port = port_sweeps_per_s(min(seconds, 6.0)) * frac
    shape = "%dx%d, %d blocks of w=%d (%d/100 of the C2 columns, same block shape)" % (
        C2_SAMPLE["N"], C2_SAMPLE["K"], C2_SAMPLE["BLOCK"], C2_SAMPLE["K"] // C2_SAMPLE["BLOCK"], C2_SAMPLE["BLOCK"])
    if not ref_available():
        return {"value": port, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": "oracle port (NumPy fp64, BLAS on %d threads) on %s; scaled by bytes (x%.3f) to C2; "
                          "oracle/_ref is not populated on this box, so the reference class itself was not timed"
                          % (cores, shape, frac)}
    P = largest_divisor(C2_SAMPLE["K"] // C2_SAMPLE["BLOCK"], cores)
    blas_threads(1)                                  # one BLAS thread per Pool worker
    ref = RefCPU(P)
    ref.sweep_seconds()
    ts = [ref.sweep_seconds() for _ in range(2)]
    value = frac / float(np.mean(ts))
    return {"value": value, "unit": UNIT, "cores": P, "kind": "reference",
            "sample": "unmodified ClassLassoCPU.run (oracle/_ref/lasso.py:70-169, Pool(P=%d), 1 BLAS thread per "
                      "worker) on %s: %.2f s per sample sweep; scaled by bytes (x%.3f) to the C2 sweep"
                      % (P, shape, float(np.mean(ts)), frac),
            "port": {"value": port, "unit": UNIT, "cores": cores,
                     "what": "the NumPy port of the same loop (oracle/lasso_oracle.py), BLAS on all host threads, "
                             "no Pool pickling; same sample and scaling"}}


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    frac = C2_SAMPLE["K"] / float(C2["K"])
    shape = "%dx%d / %d-block sample of C2 (block shape 10000x1000 as in C2)" % (
        C2_SAMPLE["N"], C2_SAMPLE["K"], C2_SAMPLE["BLOCK"])
    extra = {}
    if ref_available():
        P = largest_divisor(C2_SAMPLE["K"] // C2_SAMPLE["BLOCK"], cores)
        nblas = blas_threads(1)
        ref = RefCPU(P)
        for _ in range(max(args.warmup, 1)):
            ref.sweep_seconds()
        dt = sum(ref.sweep_seconds() for _ in range(args.steps))
        kind, used = "reference", P
        how = ("unmodified ClassLassoCPU.run (oracle/_ref/lasso.py:70-169) with Pool(P=%d) on %d host cores, %s BLAS "
               "thread(s) per worker; each step = one sweep of a %s, scaled by bytes (x%.3f)" % (P, cores, nblas, shape, frac))
        if args.gpus == 1 and not args.small:
            # the driver's default worker count (cpu_vs_gpu.py:74) as a second point
            P4 = largest_divisor(C2_SAMPLE["K"] // C2_SAMPLE["BLOCK"], min(4, cores))
            r4 = RefCPU(P4)
            r4.sweep_seconds()
            extra["reference_P%d" % P4] = {"value": frac / r4.sweep_seconds(), "unit": UNIT, "cores": P4}
            nb = blas_threads(cores)
            extra["port"] = {"value": port_sweeps_per_s(6.0) * frac, "unit": UNIT, "cores": cores, "blas_threads": nb,
                             "what": "NumPy port of the same loop, no Pool pickling"}
            extra["c1_time_to_eps"] = c1_reference_time_to_eps(min(4, cores))
    else:
        from oracle import lasso_oracle as orc
        nblas = blas_threads(cores)
        A, b, mu = cpu_sample(C2_SAMPLE["N"], C2_SAMPLE["K"], C2_SAMPLE["BLOCK"])
        BLOCK = C2_SAMPLE["BLOCK"]

        def one():
            return orc.lasso_oracle(A, b, mu, BLOCK, BLOCK, None, faithful=False)["elapsed"]
        for _ in range(max(args.warmup, 1)):
            one()
        dt = sum(one() for _ in range(args.steps))
        kind, used = "port", cores
        how = ("oracle port (NumPy fp64, %s BLAS threads; oracle/_ref is not populated on this box); each step = one "
               "sweep of a %s, scaled by bytes (x%.3f)" % (nblas, shape, frac))
    value = args.steps / dt * frac
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps / frac * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": "dense lasso 10000x100000, 100 column blocks (C2); " + how},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": used, "kind": kind, "sample": how},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    line.update(extra)
    print(json.dumps(line))
    return 0


def c1_reference_time_to_eps(P):
    """BASELINE.json configs[0] on the reference itself: the default instance (cpu_vs_gpu.py:57-74) solved by
    the unmodified ClassLassoCPU to ERR_BOUND = 1e-4"""
    try:
        from oracle import make_ref
        ref_lasso, ref_par, ref_cpu = make_ref.import_reference()
        ref_par.time = lambda: 1234
        A, _, b, mu = ref_par.parameters(1024, 4096, 0.4, False, False, SILENCE=True)
        Abp = ref_cpu.A_bp_get(A, 2, P)
        solver = ref_lasso.ClassLassoCPU(Abp, ref_cpu.fun_diag_ATA(Abp), A, b, mu, 2, P, 1000)
        err = np.zeros(1000)
        secs = float(solver.run(1e-4, err_iter=err, SILENCE=True))
        return {"workload": "default instance 1024x4096, BLOCK=2, P=%d, fp64, ERR_BOUND=1e-4" % P, "seconds": secs,
                "iterations": int(np.count_nonzero(err))}
    except Exception as e:                                  # pragma: no cover
        return {"skipped": repr(e)}


def c1_time_to_eps(device_index):
    """BASELINE.json configs[0]: the reference's default instance (cpu_vs_gpu.py:57-74: N=1024, K=4096,
    BLOCK=2, den=0.4, fp64, ERR_BOUND=1e-4, seed 1234) solved through ClassLasso.run() from host
    arrays; the reference arm times the unmodified ClassLassoCPU on the same instance.  Never fatal."""
    try:
        from convex_optimization_b200 import lasso, parameters
        from convex_optimization_b200.gpu_calculation import GPU_Calculation

        class Cal(GPU_Calculation):
            TYPE = "double"
            LAYOUT = "row"
            DEVICE = device_index
        A, _, b, mu = parameters.parameters(1024, 4096, 0.4, False, False, SILENCE=True, seed=1234)
        t0 = time.time()
        cal = Cal(A, 2)
        d = cal.diag_ATA
        solver = lasso.ClassLasso(cal, d, A, b, mu, 2, 1000)
        solver.run(1e-4, SILENCE=True)                      # includes module load / first launch
        first = time.time() - t0
        t0 = time.time()
        solver.run(1e-4, SILENCE=True)
        dt = time.time() - t0
        return {"workload": "default instance 1024x4096, BLOCK=2, fp64, ERR_BOUND=1e-4 (cpu_vs_gpu.py:57-74)",
                "seconds": dt, "seconds_first_call_incl_upload": first, "iterations": int(solver.iters),
                "nnz_x": int(np.count_nonzero(solver.x)), "api": "ClassLasso.run() (host b in, x out)",
                "reference_cpu_seconds_survey": 52.45, "reference_iterations_survey": 128}
    except Exception as e:                                  # pragma: no cover
        sys.stderr.write("c1_time_to_eps skipped: %r\n" % (e,))
        return None


# ------------------------------------------------------------------------------ GPU arm
CONFIGS = {
    "c2": dict(N=10000, K=100000, BLOCK=100, den=0.01, seed=2, dtype="float"),
    # BASELINE.json configs[2]: fp64 20,000 x 200,000 (32 GB)
    "c3": dict(N=20000, K=200000, BLOCK=100, den=0.01, seed=3, dtype="double"),
    # one GPU's share of configs[3] on 8 GPUs: 50,000 x 125,000 fp32 (25 GB)
    "c4shard": dict(N=50000, K=125000, BLOCK=100, den=0.01, seed=4, dtype="float"),
}


class Ctx:
    """what every leg needs: torch, ranks, device, barrier, timing helpers"""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
        torch.cuda.set_device(self.local_rank)
        self.device = torch.device("cuda", self.local_rank)
        self.peak, self.peak_src = measured_peak()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.device)

    def max_over_ranks(self, v):
        if self.world == 1:
            return float(v)
        t = self.torch.tensor([v], device=self.device, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())


def cal_class(cfg, layout, local_rank):
    from convex_optimization_b200.gpu_calculation import GPU_Calculation

    class Cal(GPU_Calculation):
        TYPE = cfg["dtype"]
        LAYOUT = layout
        DEVICE = local_rank
    return Cal


def build_instance(cx, cfg, layout, instance, connect=True):
    """(cal, b, mu): the local column shard of the instance on this rank's GPU"""
    import ctypes
    from convex_optimization_b200 import _lib
    torch = cx.torch
    Cal = cal_class(cfg, layout, cx.local_rank)
    N, K, BLOCK = cfg["N"], cfg["K"], cfg["BLOCK"]
    if instance == "philox":
        # the library's generator: the same global matrix for every world size (DESIGN.md 5c)
        from convex_optimization_b200 import parameters as pm
        cal, _, b, mu = pm.parameters_device(N, K * cx.world, BLOCK, cfg["den"], cfg["seed"], gpu_cal_cls=Cal)
    else:
        tdt = torch.float32 if cfg["dtype"] == "float" else torch.float64
        ld = Cal.padded_ld(N, K, BLOCK)
        store, b, mu = make_device_instance(torch, cx.device, N, K, BLOCK, cfg["den"], cfg["seed"], tdt, ld, layout,
                                            cx.dist if cx.world > 1 else None, cx.rank)
        cal = Cal.from_device_blocks(store, N, K, BLOCK)
    stream = torch.cuda.current_stream(cx.device)
    _lib.check(cal._lib.b200l_ctx_set_stream(cal.ctx, ctypes.c_void_p(stream.cuda_stream)))
    transport = "single"
    if cx.world > 1 and connect:
        from convex_optimization_b200 import distributed as dd
        transport = dd.connect(cal)
    return cal, b, float(mu), transport


def time_sweeps(cx, cal, b, mu, BLOCK, steps, warmup, single_launch=False, sampler=None):
    """device-timed sweeps of the fused kernel with everything resident: (ms per sweep, max over ranks)"""
    import ctypes
    from convex_optimization_b200 import _lib
    torch = cx.torch
    lib, ctx = cal._lib, cal.ctx
    bb = np.ascontiguousarray(b.reshape(-1))
    _lib.check(lib.b200l_set_problem(ctx, _lib.dptr(bb)))

    def sweeps(n):
        if not single_launch:
            for _ in range(n):
                _lib.check(lib.b200l_run(ctx, None, BLOCK, float(mu), -1.0, None, None, None, None, None))
        elif n > 0:
            _lib.check(lib.b200l_run(ctx, None, BLOCK * n, float(mu), -1.0, None, None, None, None, None))
    sweeps(warmup)
    cx.barrier()
    ev0 = torch.cuda.Event(enable_timing=True)
    ev1 = torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    ev0.record()
    sweeps(steps)
    ev1.record()
    cx.barrier()
    t1 = time.time()
    ms = cx.max_over_ranks(ev0.elapsed_time(ev1))
    clocks = sampler.stop(t0, t1) if sampler is not None else None
    return ms / steps, clocks


DUMP_BYTES = 64 << 20


def dump_outputs(cx, cal, BLOCK, directory):
    """write the solution x and the residual r = Ax - b, as the last timed sweep left them on the device,
    to directory/x.npy and directory/r.npy (float64).  Several GPUs: x is gathered into global column
    order and rank 0 writes.  An array larger than its share of DUMP_BYTES is replaced by a fixed sample
    of its entries (sorted indices drawn by np.random.RandomState(0)), the same for every run of a shape."""
    from convex_optimization_b200 import _lib
    x = np.empty(cal.MAT_WIDTH_ALL)
    r = np.empty(cal.MAT_HEIGHT)
    _lib.check(cal._lib.b200l_get_x(cal.ctx, _lib.dptr(x)))
    _lib.check(cal._lib.b200l_get_r(cal.ctx, _lib.dptr(r)))
    if cx.world > 1:
        from convex_optimization_b200 import distributed as dd
        x = dd.gather_x(x, BLOCK).reshape(-1)
    if cx.rank != 0:
        return
    os.makedirs(directory, exist_ok=True)
    outputs = {"x": x, "r": r}
    for name, a in outputs.items():
        limit = DUMP_BYTES // len(outputs) // a.itemsize
        if a.size > limit:
            a = a[np.sort(np.random.RandomState(0).choice(a.size, limit, replace=False))]
        np.save(os.path.join(directory, name + ".npy"), a)


def roofline_record(cx, cfg, layout, ms_per_sweep, sweeps_per_launch, traffic_key, l2_bytes):
    N, K, BLOCK = cfg["N"], cfg["K"], cfg["BLOCK"]
    s = 4 if cfg["dtype"] == "float" else 8
    W = sweep_bytes(N, K, BLOCK, s)
    achieved = W / (ms_per_sweep * 1e-3) / 1e9
    traffic_sweep = ncu_traffic(*traffic_key) if traffic_key else None
    block_mb = N * (K // BLOCK) * s / 1e6
    resident = 2 * N * (K // BLOCK) * s <= l2_bytes * 3 // 4
    rec = {"bound": "hbm", "achieved": achieved, "peak": cx.peak, "unit": "GB/s", "frac": achieved / cx.peak,
           "traffic": None if traffic_sweep is None else traffic_sweep * sweeps_per_launch,
           "kernel": "lasso_fused<%s,%s>" % ("float" if s == 4 else "double", "TRANS" if layout == "transposed" else "ROWMAJOR"),
           "kernel_ms_per_launch": ms_per_sweep * sweeps_per_launch, "sweeps_per_launch": sweeps_per_launch,
           "algorithmic_bytes_per_launch": W * sweeps_per_launch, "algorithmic_bytes_per_sweep": W,
           "traffic_per_sweep": traffic_sweep, "peak_source": cx.peak_src,
           "frac_of_nominal_8TBs": achieved / 8000.0,
           "frac_dram": None if traffic_sweep is None else traffic_sweep / (ms_per_sweep * 1e-3) / 1e9 / cx.peak,
           "note": ("algorithmic bytes count A twice per sweep (SURVEY 8d); a %.0f MB block and its successor fit in L2, so "
                    "the second pass is served by L2 and DRAM moves about half of the algorithmic bytes: frac_dram is "
                    "the DRAM bytes of the committed ncu capture / time / peak" % block_mb) if resident else
                   ("algorithmic bytes count A twice per sweep (SURVEY 8d); a %.0f MB block does not stay in L2, both "
                    "passes stream from HBM: DRAM traffic = algorithmic bytes" % block_mb)}
    return rec


def parity_record(cx):
    """a small column-sharded solve on this world size against the oracle with P = world (the reference's
    own P-way split, lasso.py:107-126): iterations, support, x; rc != 0 on mismatch"""
    from oracle import lasso_oracle as orc
    from convex_optimization_b200 import distributed as dd
    from convex_optimization_b200 import lasso
    world, rank = cx.world, cx.rank
    out = []
    for (N, K, BLOCK, den, TYPE, seed) in [(600, 512 * world, 4, 0.05, "double", 7), (1000, 1000 * world, 2, 0.02, "float", 5)]:
        A, _, b, mu = orc.make_problem(N, K, den, seed=seed)
        if TYPE == "float":
            A = A.astype(np.float32).astype(np.float64)
        ITER_MAX = 100 * BLOCK if TYPE == "double" else 12 * BLOCK
        bound = 1e-4 if TYPE == "double" else None
        o = orc.lasso_oracle(A, b, mu, BLOCK, ITER_MAX, bound, P=world, faithful=False)
        Cal = cal_class(dict(dtype=TYPE), "row", cx.local_rank)
        A_loc = dd.shard_columns(A, BLOCK, rank, world) if world > 1 else A
        cal = Cal(A_loc, BLOCK)
        if world > 1:
            dd.connect(cal)
        solver = lasso.ClassLasso(cal, cal.diag_ATA, A_loc, b, mu, BLOCK, ITER_MAX)
        solver.run(bound, SILENCE=True)
        x = dd.gather_x(solver.x, BLOCK) if world > 1 else solver.x
        obj = dd.objective(cal, mu)
        xo = o["x"]
        rel = float(np.abs(x - xo).max() / np.abs(xo).max())
        small = np.abs(xo) < 1e-5 * np.abs(xo).max()
        mism = (x != 0) != (xo != 0)
        obj_o = 0.5 * float(np.sum((A @ xo - b) ** 2)) + mu * float(np.abs(xo).sum())
        tol = 1e-10 if TYPE == "double" else 1e-5
        ok = (rel < tol and solver.iters == o["iters"] and abs(obj - obj_o) <= tol * abs(obj_o)
              and (not mism.any() if TYPE == "double" else bool(np.all(small[mism]))))
        out.append({"shape": "%dx%d b%d %s" % (N, K, BLOCK, TYPE), "world": world, "rel_x": rel, "rel_obj": abs(obj - obj_o) / abs(obj_o),
                    "support_equal": bool(not mism.any()), "support_mismatches_all_below_1e-5_of_max": bool(np.all(small[mism])),
                    "iters": int(solver.iters), "iters_oracle": int(o["iters"]), "ok": bool(ok)})
        if world > 1:
            dd.disconnect(cal)
        del solver, cal
    return out


def leg(cx, name, cfg, layout, instance, steps, warmup, traffic_key, l2_bytes, standalone_first=False):
    """one timed configuration as a sub-record"""
    torch = cx.torch
    cal, b, mu, transport = build_instance(cx, cfg, layout, instance, connect=False)
    rec = {"workload": "dense %s lasso %dx%d, %d column blocks, %s layout%s" % (
        "fp32" if cfg["dtype"] == "float" else "fp64", cfg["N"], cfg["K"] * cx.world, cfg["BLOCK"], layout,
        (", column-sharded over %d GPUs (%dx%d per GPU)" % (cx.world, cfg["N"], cfg["K"])) if cx.world > 1 else ""),
        "instance": instance}
    ms1 = None
    if cx.world > 1 and standalone_first:
        # this rank's shard as a 1-GPU problem (the same matrix), then the sharded solve: efficiency
        ms1, _ = time_sweeps(Ctx1(cx), cal, b, mu, cfg["BLOCK"], steps, warmup)
        rec["ms_per_sweep_1gpu_shard"] = cx.max_over_ranks(ms1)
    if cx.world > 1:
        from convex_optimization_b200 import distributed as dd
        rec["transport"] = dd.connect(cal)
    ms, _ = time_sweeps(cx, cal, b, mu, cfg["BLOCK"], steps, warmup)
    rec.update({"ms_per_sweep": ms, "value": cx.world * 1e3 / ms, "unit": UNIT, "instance_sweeps_per_s": 1e3 / ms,
                "launch": cal.run_config()})
    roof = roofline_record(cx, cfg, layout, ms, 1, traffic_key, l2_bytes)
    rec["roofline"] = {k: roof[k] for k in ("achieved", "peak", "frac", "frac_dram", "traffic_per_sweep", "algorithmic_bytes_per_sweep", "note")}
    if ms1 is not None:
        rec["efficiency_vs_1gpu_shard"] = rec["ms_per_sweep_1gpu_shard"] / ms
        rec["frac_of_aggregate_roofline"] = roof["frac"]
    if cx.world > 1:
        from convex_optimization_b200 import distributed as dd
        dd.disconnect(cal)
    del cal
    torch.cuda.empty_cache()
    return rec


class Ctx1:
    """a view of Ctx that behaves like a single-GPU run (no cross-rank barrier inside the timing)"""

    def __init__(self, cx):
        self.torch, self.device, self.world = cx.torch, cx.device, 1

    def barrier(self):
        self.torch.cuda.synchronize(self.device)

    def max_over_ranks(self, v):
        return float(v)


def main_gpu(args):
    import ctypes
    from convex_optimization_b200 import _lib, lasso
    cx = Ctx()
    torch, world, rank, local_rank, device = cx.torch, cx.world, cx.rank, cx.local_rank, cx.device
    l2_bytes = torch.cuda.get_device_properties(device).L2_cache_size

    cfg = dict(CONFIGS[args.config])
    if args.small:
        cfg.update(N=2000, K=20000, BLOCK=20)
    if args.shape:              # diagnostics only: N,K,BLOCK[,dtype]
        f = args.shape.split(",")
        cfg.update(N=int(f[0]), K=int(f[1]), BLOCK=int(f[2]))
        if len(f) > 3:
            cfg["dtype"] = f[3]
    N, K, BLOCK = cfg["N"], cfg["K"], cfg["BLOCK"]
    s = 4 if cfg["dtype"] == "float" else 8
    layout = args.layout
    quick = args.small or bool(args.shape) or args.quick

    # ---- parity first: a wrong kernel must not print a number -------------------------------
    parity = None
    if not args.no_parity:
        parity = parity_record(cx)
        if not all(p["ok"] for p in parity):
            if rank == 0:
                print(json.dumps({"metric": METRIC, "error": "parity check against the oracle failed", "parity": parity}))
            return 3

    # ---- headline: C2 (one C2-sized shard per GPU), resident, device-timed --------------------
    cal, b, mu, transport = build_instance(cx, cfg, layout, args.instance)
    if args.slot_bytes or args.inflight:
        cal.set_tuning(args.slot_bytes, args.inflight)
    lib, ctx = cal._lib, cal.ctx
    if args.dbg:
        _lib.check(lib.b200l_debug_flags(ctx, args.dbg))
    t0 = time.time()
    d_ATA = cal.diag_ATA
    torch.cuda.synchronize(device)
    setup_ms = (time.time() - t0) * 1e3
    geo = cal.run_config()
    # (the sampler starts before the warm-up: its start-up must not delay rank 0 behind the others)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # several GPUs: the K timed sweeps run in ONE launch per rank, the way a solve runs (every launch
    # boundary makes the ranks meet again after the host-side launch skew of 8 processes); one GPU:
    # one launch per sweep, the unit the roofline record and the committed ncu launch list refer to
    single_launch = args.single_launch or world > 1
    ms_per_step, clocks = time_sweeps(cx, cal, b, mu, BLOCK, args.steps, args.warmup, single_launch,
                                      sampler if rank == 0 else None)
    if args.dump_outputs:
        dump_outputs(cx, cal, BLOCK, args.dump_outputs)
    value = world * 1e3 / ms_per_step
    sweeps_per_launch = args.steps if single_launch else 1
    n_launches = args.steps // sweeps_per_launch
    kms = ctypes.c_double()
    ktimes = []
    for _ in range(min(args.steps, 10)):
        _lib.check(lib.b200l_run(ctx, None, BLOCK, float(mu), -1.0, None, None, None, None, ctypes.byref(kms)))
        ktimes.append(kms.value)
    from convex_optimization_b200 import distributed as dd
    obj_bench = dd.objective(cal, mu)

    # ---- e2e: through ClassLasso.run(), host b in, host x out -------------------------------
    e2e_sweeps = args.e2e_sweeps

    class HostShape:            # the solver only needs A.shape on the fused path (lasso.py:32)
        shape = (N, K)
    solver = lasso.ClassLasso(cal, d_ATA, HostShape, b, mu, BLOCK, BLOCK * e2e_sweeps)
    for _ in range(2):
        solver.run(SILENCE=True)
    cx.barrier()
    t0 = time.time()
    e2e_steps = max(3, min(args.steps, 10))
    e2e_kernel_ms = 0.0
    for _ in range(e2e_steps):
        solver.run(SILENCE=True)
        e2e_kernel_ms += solver.kernel_ms
    cx.barrier()
    e2e_dt = cx.max_over_ranks(time.time() - t0)
    e2e_value = world * e2e_steps * e2e_sweeps / e2e_dt
    nnz = int(np.count_nonzero(solver.x))

    # ---- time-to-eps: cold start (x = 0) to the reference's stop rule (lasso.py:141-150) ----
    tte = None
    if args.eps > 0:
        bb = np.ascontiguousarray(b.reshape(-1))
        x_host = np.empty((K, 1))
        cx.barrier()
        t0 = time.time()
        _lib.check(lib.b200l_set_problem(ctx, _lib.dptr(bb)))
        steps_done, stopped = ctypes.c_int64(), ctypes.c_int32()
        _lib.check(lib.b200l_run(ctx, None, BLOCK * args.eps_max_sweeps, float(mu), float(args.eps), None, None,
                                 ctypes.byref(steps_done), ctypes.byref(stopped), ctypes.byref(kms)))
        _lib.check(lib.b200l_get_x(ctx, _lib.dptr(x_host)))
        wall_ms = (time.time() - t0) * 1e3
        tte = {"eps": args.eps, "ms": kms.value, "sweeps": steps_done.value / BLOCK,
               "reached": bool(stopped.value), "objective": dd.objective(cal, mu),
               "e2e_ms": wall_ms + setup_ms, "setup_ms": setup_ms,
               "note": "ms: device time of the one launch from x = 0 until every block of a sweep has error_crit < eps; "
                       "e2e_ms: diag(A^T A) (one pass over A, setup_ms) + b to the device + that launch + x to the host"}

    line = None
    if rank == 0:
        roof = roofline_record(cx, cfg, layout, ms_per_step, sweeps_per_launch,
                               None if quick else (args.config, layout), l2_bytes)
        roof["ms_per_single_sweep_launch_alone"] = float(np.mean(ktimes))
        roof["dram_single_pass_GBs"] = (roof["algorithmic_bytes_per_sweep"] - N * K * s) / (ms_per_step * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32" if s == 4 else "f64",
            "data": "synthetic",
            "config": {"workload": "dense %s lasso %dx%d, %d column blocks, %s A layout; 1 step = 1 sweep, the timed "
                                   "sweeps run in %d launch(es) of the persistent kernel; "
                                   "A=%.1f GB per GPU >> L2 so no flush between steps%s"
                                   % ("fp32" if s == 4 else "fp64", N, K * world, BLOCK, layout, n_launches,
                                      N * K * s / 1e9,
                                      ("; column-sharded over %d GPUs (slice g of every block on GPU g, partial "
                                       "A_m D summed in-kernel over NVLink peer memory, transport %s); value counts "
                                       "C2-sized shard sweeps: %d per sweep of the %dx%d instance"
                                       % (world, transport, world, N, K * world)) if world > 1 else ""),
                       "launch": geo, "objective_after_bench": obj_bench},
            "roofline": roof,
            "e2e": {"value": e2e_value, "unit": UNIT,
                    "h2d_bytes_per_step": int(N * 8),
                    "d2h_bytes_per_step": int(K * 8 + 24),
                    "sweeps_per_call": e2e_sweeps, "calls": e2e_steps, "nnz_x": nnz,
                    "wall_ms_per_call": e2e_dt * 1e3 / e2e_steps, "kernel_ms_per_call": e2e_kernel_ms / e2e_steps,
                    "api": "ClassLasso.run() (host b -> device, fused solve, x -> host)"},
            "gpu_launches": n_launches,
            "clocks": clocks,
        }
        if world > 1:
            line["value_counts"] = "C2-sized shard sweeps summed over the GPUs (weak scaling)"
            line["instance_sweeps_per_s"] = 1e3 / ms_per_step
        if parity is not None:
            line["parity"] = parity
        if tte:
            line["time_to_eps"] = tte
    if world > 1:
        dd.disconnect(cal)
    del solver, cal
    torch.cuda.empty_cache()

    # ---- the other configurations of BASELINE.json as sub-records ---------------------------------
    others = {}
    if not quick and args.config == "c2":
        nsw = max(3, min(args.steps, 5))
        if world == 1:
            others["c2_transposed"] = leg(cx, "c2_transposed", CONFIGS["c2"], "transposed", "torch", args.steps, 3,
                                          ("c2", "transposed"), l2_bytes)
            others["c3_fp64"] = leg(cx, "c3", CONFIGS["c3"], "row", "torch", nsw, 2, ("c3", "row"), l2_bytes)
        # C4: one 50,000 x 125,000 shard per GPU (8 GPUs = the 50k x 1M instance), Philox instance: the same
        # global matrix for every world size
        others["c4_shard_per_gpu"] = leg(cx, "c4shard", CONFIGS["c4shard"], "row", "philox", nsw, 2,
                                         ("c4shard", "row"), l2_bytes, standalone_first=True)
        if world == 1:
            # the same shard pre-transposed: N / #SM = 338 entries per CTA, i.e. two TMA boxes per tile and four
            # threads per column in pass 1 (the general tile shape of the pre-transposed layout)
            others["c4_shard_transposed"] = leg(cx, "c4shard", CONFIGS["c4shard"], "transposed", "philox", nsw, 2,
                                                ("c4shard", "transposed"), l2_bytes)
    if rank == 0:
        if others:
            line["configs"] = others
        if world == 1 and not quick and args.eps > 0:
            c1 = c1_time_to_eps(local_rank)
            if c1:
                line["c1_time_to_eps"] = c1
        if not args.no_cpu and world == 1:
            line["cpu_baseline"] = cpu_baseline_block()
        print(json.dumps(line))
    if world > 1:
        cx.dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--layout", default="row", choices=["row", "transposed"])
    ap.add_argument("--small", action="store_true", help="2000x20000 debug size (not a bench value)")
    ap.add_argument("--quick", action="store_true", help="headline leg only (no sub-records of the other configurations)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle-checked solve in front of the timing")
    ap.add_argument("--e2e-sweeps", type=int, default=10,
                    help="sweeps per ClassLasso.run() call of the e2e leg (a C2 solve to eps = 1e-4 takes 9)")
    ap.add_argument("--instance", default="torch", choices=["torch", "philox"],
                    help="how the synthetic instance is generated on the device: torch RNG per rank (default) or "
                         "b200l_gen_gaussian (Philox keyed by seed/row/global column)")
    ap.add_argument("--single-launch", action="store_true",
                    help="run the K timed sweeps in one kernel launch instead of one launch per sweep")
    ap.add_argument("--eps", type=float, default=1e-4, help="ERR_BOUND of the time-to-eps leg (0 = skip)")
    ap.add_argument("--eps-max-sweeps", type=int, default=2000)
    ap.add_argument("--slot-bytes", type=int, default=0)
    ap.add_argument("--inflight", type=int, default=0)
    ap.add_argument("--dbg", type=int, default=0, help="diagnostic flags of b200l_debug_flags (not for bench values)")
    ap.add_argument("--shape", default="", help="diagnostics: N,K,BLOCK[,float|double] instead of a named config")
    ap.add_argument("--config", default="c2", choices=["c2", "c3", "c4shard"],
                    help="c2 is the bench workload; the others appear as sub-records of the default run")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed sweeps, write x and r = Ax - b of the last one as DIR/x.npy and DIR/r.npy "
                         "(float64, at most 64 MB in all); the instance depends only on the arguments, so two builds "
                         "can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the CUDA path (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return main_reference(args)
    return main_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
