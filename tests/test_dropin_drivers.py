"""The reference's own drivers, UNMODIFIED, against this package (SURVEY.md section 8b / VERDICT round 1
"missing" 1): ``cpu_vs_gpu.py`` and ``compare.py`` run through the drop-in directory
(convex_optimization_b200/dropin: flat module names + pycuda / skcuda shims + a headless matplotlib
fallback).  The scripts come from oracle/_ref, an unmodified copy of the reference's files that
oracle/make_ref.py makes from a checkout of the reference; the reference's sources are not part of
this repository, so without that copy the tests skip."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, load_golden

REF_DIR = os.path.join(ROOT, "oracle", "_ref")


def ref_script(name):
    p = os.path.join(REF_DIR, name)
    if not os.path.exists(p):
        pytest.skip("oracle/_ref does not hold %s (run oracle/make_ref.py with B200L_REFERENCE set to a "
                    "checkout of the reference)" % name)
    return p


def run_dropin(script, env_extra, timeout=600):
    env = dict(os.environ)
    env.update(env_extra)
    env["PYTHONPATH"] = ROOT + os.pathsep + env.get("PYTHONPATH", "")
    return subprocess.run([sys.executable, "-m", "convex_optimization_b200.dropin", script], cwd=ROOT, env=env,
                          capture_output=True, text=True, timeout=timeout)


def test_oracle_ref_copies_are_unmodified():
    from oracle import make_ref
    if not make_ref.available():
        pytest.skip("oracle/_ref is not populated")
    assert make_ref.check()
    with open(os.path.join(make_ref.DEST, make_ref.MANIFEST)) as f:
        source = json.load(f)["source"]             # the checkout the copies were made from
    if os.path.isdir(source):
        for name in make_ref.FILES:
            with open(os.path.join(source, name), "rb") as f1, \
                    open(os.path.join(make_ref.DEST, name), "rb") as f2:
                assert f1.read() == f2.read(), name


def test_shim_namespaces_import_without_a_gpu():
    """everything the drivers import resolves to the drop-in modules; no CUDA needed to import them"""
    code = ("import convex_optimization_b200.dropin as d, os; d.install();"
            "import pycuda, pycuda.autoinit, pycuda.driver as cuda, pycuda.gpuarray, pycuda.elementwise;"
            "from skcuda import cublas; import matplotlib.pyplot as plt;"
            "import lasso, gpu_calculation, cpu_calculation, parameters, settings, average;"
            "h = cublas.cublasCreate(); cublas.cublasDestroy(h);"
            "assert cublas._CUBLAS_OP['N'] == 0 and cublas._CUBLAS_OP['T'] == 1;"
            "assert all(os.path.abspath(m.__file__).startswith(d.DIR) for m in (lasso, gpu_calculation, pycuda, cublas));"
            "from average import list_aver; assert list_aver([[1, 2], [3]]) == [2.0, 2.0];"
            "settings.init(); assert settings.Dir_PERFORMANCE.endswith('Performance');"
            "print('matplotlib from', os.path.dirname(plt.__file__)); print('SHIMS OK')")
    proc = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=300,
                          env=dict(os.environ, PYTHONPATH=ROOT))
    assert proc.returncode == 0 and "SHIMS OK" in proc.stdout, proc.stdout + proc.stderr


def test_compare_py_runs_unmodified_on_saved_traces(tmp_path):
    """compare.py:7-10 loads GPU_/CPU_ time and error traces from settings.Dir_PERFORMANCE; the traces
    come from path.save_traces (here: the host solver twice), the plot goes to the headless fallback
    when matplotlib is not installed"""
    from convex_optimization_b200 import cpu_calculation as cc
    from convex_optimization_b200 import lasso, path, settings
    script = ref_script("compare.py")
    g, A, b, mu = load_golden("g_128x512_b2_p4")
    BLOCK, P, ITER_MAX = int(g["BLOCK"]), int(g["P"]), int(g["ITER_MAX"])
    Abp = cc.A_bp_get(A, BLOCK, P)
    os.environ["B200L_HOME"] = str(tmp_path)
    try:
        settings.init()
        for prefix in ("CPU", "GPU"):
            solver = lasso.ClassLassoCPU(Abp, cc.fun_diag_ATA(Abp), A, b, mu, BLOCK, P, ITER_MAX)
            err, tim = np.zeros(ITER_MAX), np.zeros(ITER_MAX + 1)
            solver.run(float(g["ERR_BOUND"]), err_iter=err, time_iter=tim, SILENCE=True)
            path.save_traces(prefix, tim, err, solver.iters)
    finally:
        del os.environ["B200L_HOME"]
    proc = run_dropin(script, {"B200L_HOME": str(tmp_path), "B200L_PLOT_DIR": str(tmp_path / "plots"), "MPLBACKEND": "Agg"})
    assert proc.returncode == 0, proc.stdout + proc.stderr
    try:
        import matplotlib  # noqa: F401
    except ImportError:
        assert "[headless plot]" in proc.stdout and "CPU" in proc.stdout and "GPU" in proc.stdout
        assert (tmp_path / "plots" / "figure_0.txt").exists()


@pytest.mark.gpu
def test_cpu_vs_gpu_py_runs_unmodified(tmp_path):
    """the reference's benchmark driver (cpu_vs_gpu.py: 1024 x 4096, BLOCK = 2, ClassLassoCB_v1 and
    ClassLassoCB_v2, 4 warm-up runs + 1 timed run of 1000 iterations each) exits 0 against the package"""
    script = ref_script("cpu_vs_gpu.py")
    proc = run_dropin(script, {"B200L_HOME": str(tmp_path)}, timeout=900)
    assert proc.returncode == 0, proc.stdout[-3000:] + proc.stderr[-3000:]
    out = proc.stdout
    assert "Parameters @@created with N: 1024" in out
    assert "Cublas CPU combined" in out and "Pure Cublas" in out
    assert out.count("time used") >= 4                      # two rlt_display lines per class (run + summary)


@pytest.mark.gpu
def test_reference_solver_class_on_the_shims(tmp_path):
    """the drop-in boundary itself (SURVEY.md 8b): the REFERENCE's own ClassLassoCB_v1 (oracle/_ref/lasso.py:
    310-353, cublasDgemv on gpu_cal.A_b_gpu[m].gpudata with gpuarray vectors) runs on this package's
    GPU_Calculation + the pycuda / skcuda shims and reproduces the golden iterates of the reference's CPU path"""
    ref_lasso_py = ref_script("lasso.py")
    only = tmp_path / "ref_only"
    only.mkdir()
    (only / "lasso.py").write_bytes(open(ref_lasso_py, "rb").read())
    code = r'''
import sys, os, numpy as np
root, only, name = sys.argv[1:4]
sys.path.insert(0, root)
import convex_optimization_b200.dropin as d
d.install()
sys.path.insert(0, only)                      # the reference's lasso.py wins over the drop-in one
sys.path.insert(0, os.path.join(root, "tests"))
import lasso
assert os.path.dirname(os.path.abspath(lasso.__file__)) == only
from gpu_calculation import GPU_Calculation
from skcuda import cublas
from conftest import load_golden
g, A, b, mu = load_golden(name)
BLOCK, ITER_MAX = int(g["BLOCK"]), int(g["ITER_MAX"])
cal = GPU_Calculation(A, BLOCK)
h = cublas.cublasCreate()
xs = {}
class Hooked(lasso.ClassLassoCB_v1):
    def err_record(self, err_iter, s13, x_block_m, t):
        xs["x"] = x_block_m.base
        lasso.ClassLassoCB_v1.err_record(self, err_iter, s13, x_block_m, t)
solver = Hooked(h, cal, cal.diag_ATA, A, b, mu, BLOCK, ITER_MAX)
err = np.zeros(ITER_MAX)
solver.run(float(g["ERR_BOUND"]), err_iter=err, SILENCE=True)
x = np.array(xs["x"]).reshape(-1, 1)
n = int(g["iters"])
assert np.count_nonzero(err) == n, (np.count_nonzero(err), n)
assert np.array_equal(x != 0, g["x"] != 0)
assert np.abs(x - g["x"]).max() / np.abs(g["x"]).max() < 1e-10
assert np.abs(err[:n] - g["err"]).max() < 1e-10
cublas.cublasDestroy(h)
print("REFERENCE CLASS ON SHIMS OK", n)
'''
    proc = subprocess.run([sys.executable, "-c", code, ROOT, str(only), "g_128x512_b2_p4"], cwd=ROOT,
                          capture_output=True, text=True, timeout=600, env=dict(os.environ, B200L_HOME=str(tmp_path)))
    assert proc.returncode == 0 and "REFERENCE CLASS ON SHIMS OK" in proc.stdout, proc.stdout[-3000:] + proc.stderr[-3000:]
