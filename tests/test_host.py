"""Host logic that must work without a GPU: the NumPy helper mirrors, the problem
recipe, ClassLassoCPU, and that the C-ABI library loads and exports every declared
symbol (no compute calls: those need a device and must fail loudly without one)."""
import ctypes
import os
import re

import numpy as np
import pytest

from conftest import ROOT, golden_names, load_golden
from oracle import lasso_oracle as orc
from convex_optimization_b200 import _lib, cpu_calculation as cc
from convex_optimization_b200.parameters import parameters


def test_helper_parity_random_and_edges():
    rng = np.random.RandomState(0)
    for _ in range(20):
        u = rng.randn(37, 1)
        mu = abs(rng.randn()) * 0.3
        u[3, 0] = mu
        u[4, 0] = -mu
        u[5, 0] = 0.0
        u[6, 0] = -0.0
        assert np.array_equal(cc.soft_thresholding(u, mu), orc.soft_thresholding(u, mu))
        x = rng.randn(37, 1) * (rng.rand(37, 1) < 0.5)
        assert cc.error_crit(u, x, mu) == orc.error_crit(u, x, mu)
        assert np.array_equal(cc.element_proj(u, -mu, mu), orc.element_proj(u, -mu, mu))


def test_layout_helpers_match_reference_semantics():
    rng = np.random.RandomState(1)
    N, K, BLOCK, P = 6, 24, 3, 2
    A = rng.randn(N, K)
    Abp = cc.A_bp_get(A, BLOCK, P)
    assert Abp.shape == (BLOCK, P, N, K // (BLOCK * P))
    w, wp = K // BLOCK, K // (BLOCK * P)
    for m in range(BLOCK):
        for p in range(P):
            assert np.array_equal(Abp[m, p], A[:, m * w + p * wp: m * w + (p + 1) * wp])
    d = cc.fun_diag_ATA(Abp)
    assert d.shape == (BLOCK, w, 1)
    assert np.allclose(d.reshape(-1), (A * A).sum(axis=0), rtol=1e-14)
    s11 = rng.randn(N, 1)
    assert np.allclose(cc.fun_s12(Abp[1, 0], s11), A[:, w:w + wp].T @ s11)
    dd = rng.randn(w, 1)
    parts = cc.fun_dd_p(P, dd)
    assert parts.shape == (P, wp, 1)
    q = sum(cc.fun_s22(Abp[2, p], parts[p]) for p in range(P))
    assert np.allclose(q, A[:, 2 * w:3 * w] @ dd)
    with pytest.raises(ValueError):
        cc.A_bp_get(A, 5, 1)


@pytest.mark.parametrize("name", golden_names(small_only=True))
def test_parameters_reproduces_reference_instance(name):
    g, A, b, mu = load_golden(name)
    A2, x_true, b2, mu2 = parameters(int(g["N"]), int(g["K"]), float(g["den"]), False, False,
                                     SILENCE=True, seed=int(g["seed"]))
    assert np.array_equal(A2, A) and np.array_equal(np.asarray(b2), b) and mu2 == mu


@pytest.mark.parametrize("name", golden_names(small_only=True))
def test_classlassocpu_matches_reference(name):
    from convex_optimization_b200.lasso import ClassLassoCPU
    g, A, b, mu = load_golden(name)
    BLOCK, P = int(g["BLOCK"]), int(g["P"])
    Abp = cc.A_bp_get(A, BLOCK, P)
    d = cc.fun_diag_ATA(Abp)
    solver = ClassLassoCPU(Abp, d, A, b, mu, BLOCK, P, int(g["ITER_MAX"]))
    err_iter = np.zeros(int(g["ITER_MAX"]))
    time_iter = np.zeros(int(g["ITER_MAX"]) + 1)
    elapsed = solver.run(float(g["ERR_BOUND"]), err_iter=err_iter, time_iter=time_iter, SILENCE=True)
    assert solver.iters == int(g["iters"]) and solver.stopped
    assert np.array_equal(solver.x != 0, g["x"] != 0)
    assert np.abs(solver.x - g["x"]).max() / np.abs(g["x"]).max() < 1e-12
    assert np.abs(err_iter[:solver.iters] - g["err"]).max() < 1e-12
    assert elapsed == time_iter[solver.iters - 1]          # ref lasso.py:161-162


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "b200lasso.h")).read()
    declared = set(re.findall(r"\b(b200l_[A-Za-z_0-9]+)\s*\(", header))
    assert declared, "no declarations found"
    assert declared == set(_lib.PROTOTYPES), declared ^ set(_lib.PROTOTYPES)
    lib = _lib.load()
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.b200l_abi_version() == 1


def test_compute_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    lib = _lib.load()
    n = ctypes.c_int(0)
    assert lib.b200l_device_count(ctypes.byref(n)) != 0
    assert lib.b200l_last_error()
    ctx = ctypes.c_void_p()
    assert lib.b200l_ctx_create(ctypes.byref(ctx), _lib.F64, _lib.ROWMAJOR, 8, 8, 1, 0) != 0
    with pytest.raises(Exception):
        from convex_optimization_b200.gpu_calculation import GPU_Calculation
        GPU_Calculation(np.zeros((8, 8)), 1)


def test_bench_reference_arm_prints_the_contract_line(monkeypatch, capsys):
    """bench.py --impl reference: one JSON line with the keys of the bench contract (small sample here),
    timed on the unmodified reference class when oracle/_ref is populated, else on the port"""
    import argparse
    import json
    import bench

    monkeypatch.setattr(bench, "C2_SAMPLE", dict(N=200, K=400, BLOCK=4))
    monkeypatch.setattr(bench, "c1_reference_time_to_eps", lambda P: {"skipped": "test"})
    monkeypatch.setattr(bench, "port_sweeps_per_s", lambda seconds: 1.0)
    monkeypatch.delenv("RANK", raising=False)
    args = argparse.Namespace(gpus=1, steps=2, warmup=1, small=False)
    assert bench.main_reference(args) == 0
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line
    assert line["impl"] == "reference" and line["metric"] == bench.METRIC and line["value"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] == 0
    assert line["cpu_baseline"]["kind"] == ("reference" if bench.ref_available() else "port")
    assert line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["value"] == line["value"]
    # other ranks of a torchrun launch exit without work
    monkeypatch.setenv("RANK", "1")
    assert bench.main_reference(args) == 0
    assert capsys.readouterr().out == ""


def test_bench_dump_outputs_writes_x_and_r_within_the_budget(monkeypatch, tmp_path):
    """bench.py --dump-outputs: x and r as float64 .npy; past the byte budget a fixed sample of the entries"""
    import types
    import bench
    N, K = 300, 4000
    x_dev, r_dev = np.arange(K) * 0.5, -np.arange(N) - 1.0

    def copy_out(src):
        def get(ctx, ptr):
            np.ctypeslib.as_array(ptr, shape=(src.size,))[:] = src
            return 0
        return get
    lib = types.SimpleNamespace(b200l_get_x=copy_out(x_dev), b200l_get_r=copy_out(r_dev))
    cal = types.SimpleNamespace(_lib=lib, ctx=None, MAT_WIDTH_ALL=K, MAT_HEIGHT=N)
    cx = types.SimpleNamespace(world=1, rank=0)
    bench.dump_outputs(cx, cal, 4, str(tmp_path / "full"))
    x, r = np.load(tmp_path / "full" / "x.npy"), np.load(tmp_path / "full" / "r.npy")
    assert x.dtype == r.dtype == np.float64
    assert np.array_equal(x, x_dev) and np.array_equal(r, r_dev)
    # several GPUs: x is gathered over the ranks and only rank 0 writes
    from convex_optimization_b200 import distributed as dd
    monkeypatch.setattr(dd, "gather_x", lambda x_local, BLOCK: np.concatenate([x_local, x_local + K]).reshape(-1, 1))
    for rank in (1, 0):
        bench.dump_outputs(types.SimpleNamespace(world=2, rank=rank), cal, 4, str(tmp_path / ("rank%d" % rank)))
    assert not (tmp_path / "rank1").exists()
    assert np.array_equal(np.load(tmp_path / "rank0" / "x.npy"), np.concatenate([x_dev, x_dev + K]))
    monkeypatch.setattr(bench, "DUMP_BYTES", 2 * 8 * 1000)            # x over its share, r within it
    for run in ("a", "b"):
        bench.dump_outputs(cx, cal, 4, str(tmp_path / run))
    xa, xb = np.load(tmp_path / "a" / "x.npy"), np.load(tmp_path / "b" / "x.npy")
    assert xa.size == 1000 and np.array_equal(xa, xb)                 # the same sample every run
    assert np.all(np.diff(xa) > 0) and np.all(np.isin(xa, x_dev))     # entries of x, in index order
    assert np.array_equal(np.load(tmp_path / "a" / "r.npy"), r_dev)


@pytest.mark.gpu
def test_bench_dump_outputs_repeat_from_run_to_run(tmp_path):
    """bench.py --dump-outputs on the CUDA path: two runs with the same arguments write the same x and r
    (the fused kernel is bitwise deterministic), and one more timed sweep changes them"""
    import json
    import subprocess
    import sys

    def run(tag, steps):
        out = tmp_path / tag
        cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--small", "--quick", "--no-cpu", "--no-parity",
               "--eps", "0", "--steps", str(steps), "--warmup", "3", "--dump-outputs", str(out)]
        proc = subprocess.run(cmd, cwd=str(tmp_path), capture_output=True, text=True, timeout=600)
        assert proc.returncode == 0, proc.stdout[-2000:] + proc.stderr[-2000:]
        assert json.loads(proc.stdout.strip().splitlines()[-1])["steps"] == steps
        return np.load(out / "x.npy"), np.load(out / "r.npy")
    xa, ra = run("a", 2)
    xb, rb = run("b", 2)
    xc, _ = run("c", 3)
    assert xa.shape == (20000,) and ra.shape == (2000,) and xa.dtype == ra.dtype == np.float64
    assert np.count_nonzero(xa) > 0 and np.all(np.isfinite(ra))
    assert np.array_equal(xa, xb) and np.array_equal(ra, rb)
    assert not np.array_equal(xc, xa)
