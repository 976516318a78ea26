"""Parity of the CUDA path (through the C ABI / the reference-facing classes) against the
oracle and the golden vectors minted from the unmodified reference.

Bars (BASELINE.json north_star): support set exactly; x and objective within 1e-10
relative in fp64 and 1e-5 in fp32."""
import ctypes

import numpy as np
import pytest

from conftest import assert_support, golden_names, load_golden
from oracle import lasso_oracle as orc

pytestmark = pytest.mark.gpu

TOL = {"double": 1e-10, "float": 1e-5}


def make_gpu_cal(A, BLOCK, TYPE="double", LAYOUT="row"):
    from convex_optimization_b200.gpu_calculation import GPU_Calculation

    class Cal(GPU_Calculation):
        pass
    Cal.TYPE = TYPE
    Cal.LAYOUT = LAYOUT
    return Cal(A, BLOCK)


def rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


# ---------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("TYPE", ["double", "float"])
@pytest.mark.parametrize("LAYOUT", ["row", "transposed"])
# (the two large shapes: several column slabs x many row chunks in the single-launch column sums, rows
# shared by 2 and 8 warps in the row dots, vector kept in registers or not)
@pytest.mark.parametrize("shape", [(64, 256, 1), (257, 1002, 3), (1000, 4096, 2), (33, 35, 5), (5, 7, 7),
                                   (5000, 3000, 2), (300, 40000, 2), (2000, 12000, 2)])
def test_matvec_kernels_vs_numpy(TYPE, LAYOUT, shape):
    check_matvec_kernels(TYPE, LAYOUT, shape, 0)


# the load-batch kernels (the fallback of the TMA-streamed mat-vec for small or very wide matrices) at shapes that
# the streamed kernel would otherwise take
@pytest.mark.parametrize("TYPE", ["double", "float"])
@pytest.mark.parametrize("LAYOUT", ["row", "transposed"])
@pytest.mark.parametrize("shape", [(1000, 4096, 2), (5000, 3000, 2), (300, 40000, 2)])
def test_matvec_load_batch_kernels_vs_numpy(TYPE, LAYOUT, shape):
    check_matvec_kernels(TYPE, LAYOUT, shape, 262144)


def check_matvec_kernels(TYPE, LAYOUT, shape, dbg):
    N, K, BLOCK = shape
    rng = np.random.RandomState(N + K)
    A = rng.randn(N, K)
    if TYPE == "float":
        A = A.astype(np.float32).astype(np.float64)      # same matrix on both sides
    cal = make_gpu_cal(A, BLOCK, TYPE, LAYOUT)
    if dbg:
        from convex_optimization_b200 import _lib
        _lib.check(cal._lib.b200l_debug_flags(cal.ctx, dbg))
    w = K // BLOCK
    assert cal.MAT_HEIGHT == N and cal.MAT_WIDTH == w and cal.MAT_WIDTH_ALL == K
    assert tuple(cal.A_b_gpu[0].shape) == (N, w)
    assert np.array_equal(cal.A_b_gpu[BLOCK - 1].get().astype(np.float64), A[:, (BLOCK - 1) * w:])
    assert int(cal.A_b_gpu[0].gpudata) == cal._A_store.data_ptr() and len(cal.A_b_gpu) == BLOCK
    d = cal.diag_ATA
    assert d.shape == (BLOCK, w, 1) and d.dtype == np.float64
    assert rel(d.reshape(-1), (A * A).sum(axis=0)) < 1e-13
    for m in {0, BLOCK - 1}:
        Am = A[:, m * w:(m + 1) * w]
        s11 = rng.randn(N, 1)
        s13 = np.zeros((w, 1))
        cal.mat_tMulVec_DiffSize(s13, m, s11)
        assert rel(s13, Am.T @ s11) < 1e-13
        dd = rng.randn(w, 1)
        s23 = np.zeros((N, 1))
        cal.matMulVec_DiffSize(s23, m, dd)
        assert rel(s23, Am @ dd) < 1e-13


# ---------------------------------------------------------------------------- iterates
def run_fused(cls_name, A, b, mu, BLOCK, ITER_MAX, ERR_BOUND, TYPE="double", LAYOUT="row", **kw):
    from convex_optimization_b200 import lasso
    cal = make_gpu_cal(A, BLOCK, TYPE, LAYOUT)
    d = cal.diag_ATA
    cls = getattr(lasso, cls_name)
    if cls_name.startswith("ClassLassoCB"):
        solver = cls(None, cal, d, A, b, mu, BLOCK, ITER_MAX)
    else:
        solver = cls(cal, d, A, b, mu, BLOCK, ITER_MAX)
    err_iter = np.zeros(ITER_MAX)
    time_iter = np.zeros(ITER_MAX + 1)
    elapsed = solver.run(ERR_BOUND, err_iter=err_iter, time_iter=time_iter, SILENCE=True, **kw)
    return solver, err_iter, time_iter, elapsed


@pytest.mark.parametrize("name", golden_names())
@pytest.mark.parametrize("cls_name", ["ClassLasso", "ClassLassoCB_v2"])
def test_fused_fp64_matches_reference_golden(name, cls_name):
    g, A, b, mu = load_golden(name)
    solver, err_iter, time_iter, elapsed = run_fused(
        cls_name, A, b, mu, int(g["BLOCK"]), int(g["ITER_MAX"]), float(g["ERR_BOUND"]))
    n = int(g["iters"])
    assert solver.iters == n and solver.stopped
    assert np.array_equal(solver.x != 0, g["x"] != 0)                 # support exactly
    assert rel(solver.x, g["x"]) < TOL["double"]
    obj = orc.objective(A, b, solver.x, mu)
    assert abs(obj - float(g["objective"])) / float(g["objective"]) < TOL["double"]
    assert np.abs(err_iter[:n] - g["err"]).max() < 1e-10
    assert np.all(err_iter[n:] == 0)
    assert np.all(np.diff(time_iter[:n]) >= 0) and elapsed == time_iter[n - 1]


@pytest.mark.parametrize("name", golden_names())
def test_fused_fp32_matches_reference_golden(name):
    g, A, b, mu = load_golden(name)
    solver, err_iter, _, _ = run_fused("ClassLasso", A, b, mu, int(g["BLOCK"]), int(g["ITER_MAX"]),
                                       float(g["ERR_BOUND"]), TYPE="float")
    n = int(g["iters"])
    x = g["x"]
    assert_support(solver.x, x, "float")           # the fp32 support rule (conftest.assert_support)
    assert rel(solver.x, x) < TOL["float"]
    obj = orc.objective(A, b, solver.x, mu)
    assert abs(obj - float(g["objective"])) / float(g["objective"]) < TOL["float"]
    assert abs(solver.iters - n) <= int(g["BLOCK"])
    m = min(n, solver.iters)
    assert np.abs(err_iter[:m] - g["err"][:m]).max() < 1e-5


@pytest.mark.parametrize("name", golden_names(small_only=True))
def test_stepwise_cb_v1_matches_reference_golden(name):
    g, A, b, mu = load_golden(name)
    solver, err_iter, _, _ = run_fused("ClassLassoCB_v1", A, b, mu, int(g["BLOCK"]),
                                       int(g["ITER_MAX"]), float(g["ERR_BOUND"]))
    n = int(g["iters"])
    assert solver.iters == n and solver.stopped
    assert np.array_equal(solver.x != 0, g["x"] != 0)
    assert rel(solver.x, g["x"]) < TOL["double"]
    assert np.abs(err_iter[:n] - g["err"]).max() < 1e-10


def test_hooks_force_stepwise_and_are_called():
    from convex_optimization_b200 import lasso
    g, A, b, mu = load_golden("g_128x512_b2_p4")
    cal = make_gpu_cal(A, 2)
    calls = []

    class Hooked(lasso.ClassLasso):
        def err_record(self, err_iter, s13, x_block, t):
            calls.append(t)
            lasso.ClassLasso.err_record(self, err_iter, s13, x_block, t)
    solver = Hooked(cal, cal.diag_ATA, A, b, mu, 2, int(g["ITER_MAX"]))
    solver.run(float(g["ERR_BOUND"]), SILENCE=True)
    assert calls == list(range(int(g["iters"])))
    assert rel(solver.x, g["x"]) < TOL["double"]


def test_unbounded_run_and_no_records():
    g, A, b, mu = load_golden("g_64x256_b1_p1")
    o = orc.lasso_oracle(A, b, mu, 1, 25, None, faithful=False)
    from convex_optimization_b200 import lasso
    cal = make_gpu_cal(A, 1)
    solver = lasso.ClassLasso(cal, cal.diag_ATA, A, b, mu, 1, 25)
    solver.run(SILENCE=True)
    assert solver.iters == 25 and not solver.stopped
    assert rel(solver.x, o["x"]) < TOL["double"]
    assert np.array_equal(solver.x != 0, o["x"] != 0)


def test_random_order_matches_oracle_with_same_order():
    import random
    from convex_optimization_b200 import lasso
    g, A, b, mu = load_golden("g_256x1024_b8_p4")
    BLOCK, ITER_MAX = 8, 400
    cal = make_gpu_cal(A, BLOCK)
    solver = lasso.ClassLassoR(cal, cal.diag_ATA, A, b, mu, BLOCK, ITER_MAX)
    random.seed(5)
    err_iter = np.zeros(ITER_MAX)
    solver.run(1e-4, err_iter=err_iter, SILENCE=True)
    # replay the same shuffles for the oracle
    random.seed(5)
    idx = np.arange(BLOCK)
    order = []
    for t in range(ITER_MAX):
        if t % BLOCK == 0:
            random.shuffle(idx)
        order.append(int(idx[t % BLOCK]))
    o = orc.lasso_oracle(A, b, mu, BLOCK, ITER_MAX, 1e-4, order=order, faithful=False)
    assert solver.iters == o["iters"] and solver.stopped == o["stopped"]
    assert np.array_equal(solver.x != 0, o["x"] != 0)
    assert rel(solver.x, o["x"]) < TOL["double"]
    assert np.abs(err_iter[:o["iters"]] - o["err"]).max() < 1e-10


@pytest.mark.parametrize("shape", [(257, 1002, 3, 0.05), (33, 70, 5, 0.2), (100, 2048, 1, 0.05),
                                   (1500, 3000, 2, 0.02), (300, 8000, 2, 0.01)])
@pytest.mark.parametrize("TYPE", ["double", "float"])
def test_ragged_shapes_vs_oracle(shape, TYPE):
    """N not a multiple of the SM count or the tile, N < SM count, odd w (padded ld),
    w beyond one column-group per thread."""
    from convex_optimization_b200 import lasso
    N, K, BLOCK, den = shape
    A, _, b, mu = orc.make_problem(N, K, den, seed=N + K)
    if TYPE == "float":
        A = A.astype(np.float32).astype(np.float64)
    ITER_MAX = 60 * BLOCK
    o = orc.lasso_oracle(A, b, mu, BLOCK, ITER_MAX, 1e-4, faithful=False)
    cal = make_gpu_cal(A, BLOCK, TYPE)
    solver = lasso.ClassLasso(cal, cal.diag_ATA, A, b, mu, BLOCK, ITER_MAX)
    err_iter = np.zeros(ITER_MAX)
    solver.run(1e-4, err_iter=err_iter, SILENCE=True)
    tol = TOL[TYPE]
    if TYPE == "double":
        assert solver.iters == o["iters"] and solver.stopped == o["stopped"]
    else:
        assert abs(solver.iters - o["iters"]) <= BLOCK
    assert_support(solver.x, o["x"], TYPE)
    assert rel(solver.x, o["x"]) < tol
    assert abs(orc.objective(A, b, solver.x, mu) - o["objective"]) / o["objective"] < tol


def test_run_to_run_bitwise_determinism_and_step_by_step_equivalence():
    from convex_optimization_b200 import _lib, lasso
    g, A, b, mu = load_golden("g_200x1200_b4_p2")
    BLOCK, ITER_MAX = 4, int(g["ITER_MAX"])
    cal = make_gpu_cal(A, BLOCK)
    xs = []
    for _ in range(3):
        solver = lasso.ClassLasso(cal, cal.diag_ATA, A, b, mu, BLOCK, ITER_MAX)
        solver.run(1e-4, SILENCE=True)
        xs.append(solver.x.copy())
    assert np.array_equal(xs[0], xs[1]) and np.array_equal(xs[0], xs[2])
    # the same solve as ITER_MAX launches of one block step each (state carried on the device)
    lib = cal._lib
    bb = np.ascontiguousarray(b, dtype=np.float64).reshape(-1)
    _lib.check(lib.b200l_set_problem(cal.ctx, _lib.dptr(bb)))
    steps = ctypes.c_int64()
    stopped = ctypes.c_int32()
    n = 0
    for t in range(ITER_MAX):
        _lib.check(lib.b200l_run(cal.ctx, None, 1, float(mu), 1e-4, None, None,
                                 ctypes.byref(steps), ctypes.byref(stopped), None))
        n += 1
        if stopped.value:
            break
    x = np.empty((A.shape[1], 1))
    _lib.check(lib.b200l_get_x(cal.ctx, _lib.dptr(x)))
    assert n == int(g["iters"])
    assert rel(x, xs[0]) < 1e-13 and np.array_equal(x != 0, xs[0] != 0)


def test_warm_start_and_objective():
    from convex_optimization_b200 import _lib
    g, A, b, mu = load_golden("g_128x512_b2_p4")
    cal = make_gpu_cal(A, 2)
    lib = cal._lib
    bb = np.ascontiguousarray(b, dtype=np.float64).reshape(-1)
    _lib.check(lib.b200l_set_problem(cal.ctx, _lib.dptr(bb)))
    x0 = np.ascontiguousarray(g["x"], dtype=np.float64).reshape(-1)
    _lib.check(lib.b200l_set_x(cal.ctx, _lib.dptr(x0)))
    r = np.empty(A.shape[0])
    _lib.check(lib.b200l_get_r(cal.ctx, _lib.dptr(r)))
    assert rel(r, (A @ g["x"] - b).reshape(-1)) < 1e-12
    val = ctypes.c_double()
    _lib.check(lib.b200l_objective(cal.ctx, float(mu), ctypes.byref(val)))
    assert abs(val.value - float(g["objective"])) / float(g["objective"]) < 1e-12
    # from the converged point one more sweep stops immediately (idempotence)
    steps = ctypes.c_int64()
    stopped = ctypes.c_int32()
    _lib.check(lib.b200l_run(cal.ctx, None, 2, float(mu), 1e-4, None, None,
                             ctypes.byref(steps), ctypes.byref(stopped), None))
    assert stopped.value == 1 and steps.value == 2


def test_error_paths():
    from convex_optimization_b200 import _lib
    from convex_optimization_b200.gpu_calculation import GPU_Calculation
    with pytest.raises(ValueError):
        GPU_Calculation(np.zeros((8, 10)), 3)
    cal = make_gpu_cal(np.eye(8), 2)
    with pytest.raises(_lib.B200LassoError):
        _lib.check(cal._lib.b200l_run(cal.ctx, None, 4, 0.1, -1.0, None, None, None, None, None))
    with pytest.raises(_lib.B200LassoError):
        cal.mat_tMulVec_DiffSize(np.zeros((4, 1)), 7, np.zeros((8, 1)))
    # debug flags: the knock-outs (bits 0-2) and the load-batch mat-vecs (bit 18) only; the tuning
    # call takes a slot size but no cap on the bulk copies in flight
    for flags in (1, 2, 4, 7, 262144, 262144 | 7, 0):
        _lib.check(cal._lib.b200l_debug_flags(cal.ctx, flags))
    for flags in (8, 32, 64, 128, 256, 512, 4096, 1 << 20, 7 << 20, 262144 | 4096, -1):
        with pytest.raises(_lib.B200LassoError, match="bits 0-2"):
            _lib.check(cal._lib.b200l_debug_flags(cal.ctx, flags))
    cal.set_tuning(49152, 0)
    with pytest.raises(_lib.B200LassoError, match="max_inflight_tiles"):
        cal.set_tuning(0, 2)
    cal.set_tuning(0, 0)
    # a block row beyond 32 KiB: the C entry point of the fused kernel refuses it loudly; the solver
    # classes (which accept any block width in the reference) warn and run the step-wise DEVICE path
    # (two library mat-vecs per iteration) -- never a CPU fallback
    from convex_optimization_b200 import lasso
    A, _, b, mu = orc.make_problem(16, 6000, 0.01, seed=1)
    wide = make_gpu_cal(A, 1)
    bb = np.ascontiguousarray(b.reshape(-1))
    _lib.check(wide._lib.b200l_set_problem(wide.ctx, _lib.dptr(bb)))
    with pytest.raises(_lib.B200LassoError, match="32 KiB"):
        _lib.check(wide._lib.b200l_run(wide.ctx, None, 4, mu, -1.0, None, None, None, None, None))
    solver = lasso.ClassLasso(wide, wide.diag_ATA, A, b, mu, 1, 6)
    with pytest.warns(UserWarning, match="32 KiB"):
        solver.run(SILENCE=True)
    o = orc.lasso_oracle(A, b, mu, 1, 6, None, faithful=False)
    assert solver.iters == 6 and rel(solver.x, o["x"]) < 1e-10


def test_lambda_path_warm_starts_match_oracle(tmp_path):
    """20 decreasing lambdas, each warm-started from the previous solution (BASELINE config 5
    at oracle size): every point of the path must match the oracle run with the same x0."""
    from convex_optimization_b200 import path as bpath
    N, K, BLOCK = 200, 1600, 4
    A, _, b, mu = orc.make_problem(N, K, 0.05, seed=33)
    mus = bpath.lambda_grid(mu / 0.1, n=20)
    assert mus[0] > mus[-1] and abs(mus[0] - 0.9 * mu / 0.1) < 1e-12
    cal = make_gpu_cal(A, BLOCK)
    ITER_MAX = 400 * BLOCK
    res = bpath.lasso_path(cal, b, mus, BLOCK, ITER_MAX, 1e-5)
    x0 = None
    cold_iters = warm_iters = 0
    for r, m in zip(res, mus):
        o = orc.lasso_oracle(A, b, m, BLOCK, ITER_MAX, 1e-5, faithful=False, x0=x0)
        assert r["iters"] == o["iters"] and r["stopped"] == o["stopped"]
        assert np.array_equal(r["x"] != 0, o["x"] != 0)
        assert rel(r["x"], o["x"]) < TOL["double"] or np.abs(o["x"]).max() == 0
        assert abs(r["objective"] - o["objective"]) <= 1e-10 * max(1.0, abs(o["objective"]))
        x0 = o["x"]
        warm_iters += o["iters"]
        cold_iters += orc.lasso_oracle(A, b, m, BLOCK, ITER_MAX, 1e-5, faithful=False)["iters"]
    assert warm_iters < cold_iters                    # warm starts pay
    nnz = [int(np.count_nonzero(r["x"])) for r in res]
    assert nnz[0] <= nnz[-1]                          # the support grows along the path


def test_traces_written_for_compare_py(tmp_path):
    from convex_optimization_b200 import path as bpath
    g, A, b, mu = load_golden("g_128x512_b2_p4")
    solver, err_iter, time_iter, _ = run_fused("ClassLasso", A, b, mu, 2, int(g["ITER_MAX"]), float(g["ERR_BOUND"]))
    pt, pe = bpath.save_traces("GPU", time_iter, err_iter, solver.iters, directory=str(tmp_path))
    t, e = np.loadtxt(pt), np.loadtxt(pe)
    assert t.shape == e.shape and len(t) == solver.iters
    assert np.all(np.diff(t) >= 0) and np.all(e > 0)
    assert np.all(np.isfinite(np.log10(e)))           # what compare.py:12-13 computes


@pytest.mark.parametrize("TYPE", ["double", "float"])
@pytest.mark.parametrize("shape", [(300, 2400, 4, 0.05), (257, 1002, 3, 0.05), (1000, 4000, 2, 0.02),
                                   (33, 70, 5, 0.2), (2000, 3000, 1, 0.02),
                                   (20000, 600, 2, 0.02), (40000, 768, 2, 0.02)])
def test_fused_transposed_layout_vs_oracle(shape, TYPE):
    """the pre-transposed (BLOCK, w, N) layout through the fused kernel (2-D TMA boxes); the two tall shapes:
    2, 4 or 8 threads per column in pass 1, and a CTA's share of a column fetched as two boxes"""
    from convex_optimization_b200 import lasso
    N, K, BLOCK, den = shape
    A, _, b, mu = orc.make_problem(N, K, den, seed=N + K + 1)
    if TYPE == "float":
        A = A.astype(np.float32).astype(np.float64)
    ITER_MAX = 60 * BLOCK if TYPE == "double" else 10 * BLOCK
    bound = 1e-4 if TYPE == "double" else None          # fp32: fixed iteration count
    o = orc.lasso_oracle(A, b, mu, BLOCK, ITER_MAX, bound, faithful=False)
    cal = make_gpu_cal(A, BLOCK, TYPE, LAYOUT="transposed")
    solver = lasso.ClassLasso(cal, cal.diag_ATA, A, b, mu, BLOCK, ITER_MAX)
    err_iter = np.zeros(ITER_MAX)
    solver.run(bound, err_iter=err_iter, SILENCE=True)
    assert solver.iters == o["iters"] and solver.stopped == o["stopped"]
    assert_support(solver.x, o["x"], TYPE)
    assert rel(solver.x, o["x"]) < TOL[TYPE]
    assert abs(orc.objective(A, b, solver.x, mu) - o["objective"]) / o["objective"] < TOL[TYPE]
    assert np.abs(err_iter[:o["iters"]] - o["err"]).max() < max(TOL[TYPE], 1e-10)
    # and the row-major run of the same instance gives the same iterates
    cal2 = make_gpu_cal(A, BLOCK, TYPE, LAYOUT="row")
    s2 = lasso.ClassLasso(cal2, cal2.diag_ATA, A, b, mu, BLOCK, ITER_MAX)
    s2.run(bound, SILENCE=True)
    assert s2.iters == solver.iters and rel(s2.x, solver.x) < TOL[TYPE]


def test_full_size_c2_properties_fp32_vs_fp64():
    """BASELINE.json configs[1] at full size (10,000 x 100,000, 100 blocks) where no CPU oracle can
    follow: the fp32 and the fp64 device solves of the same fp32-representable matrix must agree
    (x to 1e-5, same support above the fp32 resolution), the objective must decrease from sweep to
    sweep (exact line search), and a warm restart from the fp64 solution must not move."""
    import torch
    from bench import make_device_instance
    from convex_optimization_b200 import _lib
    from convex_optimization_b200.gpu_calculation import GPU_Calculation
    N, K, BLOCK, sweeps = 10000, 100000, 100, 3
    dev = torch.device("cuda", 0)
    store32, b, mu = make_device_instance(torch, dev, N, K, BLOCK, 0.01, 2, torch.float32, K // BLOCK)
    res = {}
    for TYPE in ("float", "double"):
        class Cal(GPU_Calculation):
            pass
        Cal.TYPE = TYPE
        store = store32 if TYPE == "float" else store32.double()
        cal = Cal.from_device_blocks(store, N, K, BLOCK)
        lib, ctx = cal._lib, cal.ctx
        bb = np.ascontiguousarray(b.reshape(-1))
        _lib.check(lib.b200l_set_problem(ctx, _lib.dptr(bb)))
        objs = []
        val = ctypes.c_double()
        for _ in range(sweeps):
            _lib.check(lib.b200l_run(ctx, None, BLOCK, float(mu), -1.0, None, None, None, None, None))
            _lib.check(lib.b200l_objective(ctx, float(mu), ctypes.byref(val)))
            objs.append(val.value)
        x = np.empty((K, 1))
        _lib.check(lib.b200l_get_x(ctx, _lib.dptr(x)))
        r = np.empty(N)
        _lib.check(lib.b200l_get_r(ctx, _lib.dptr(r)))
        res[TYPE] = (x, objs, r)
        assert all(objs[i + 1] <= objs[i] * (1 + 1e-12) for i in range(sweeps - 1)), objs
        del cal, store
    x32, o32, r32 = res["float"]
    x64, o64, r64 = res["double"]
    assert rel(x32, x64) < TOL["float"]
    big = np.abs(x64) > 1e-4 * np.abs(x64).max()
    assert np.array_equal((x32 != 0)[big], (x64 != 0)[big])
    assert abs(o32[-1] - o64[-1]) / o64[-1] < TOL["float"]
    assert rel(r32, r64) < 1e-4
    assert 0 < np.count_nonzero(x64) < K // 10            # a sparse solution


def _device_blocks(cal):
    """(BLOCK, N, w) float64 copy of the device matrix, whatever the layout"""
    t = cal._A_store.cpu().numpy().astype(np.float64)
    if cal.LAYOUT == "row":
        return t[:, :, :cal.MAT_WIDTH]
    return np.transpose(t[:, :, :cal.MAT_HEIGHT], (0, 2, 1))


@pytest.mark.gpu
@pytest.mark.parametrize("TYPE", ["float", "double"])
@pytest.mark.parametrize("LAYOUT", ["row", "transposed"])
def test_device_generator_matches_restatement_and_any_sharding(TYPE, LAYOUT):
    """b200l_gen_gaussian: entries = f(seed, row, global column); checked against the NumPy
    restatement (published Philox KATs in test_oracle) and across column shardings"""
    import torch
    from oracle import philox
    from convex_optimization_b200 import _lib
    from convex_optimization_b200.gpu_calculation import GPU_Calculation
    N, K, BLOCK, seed = 203, 1200, 3, 0x1234567890ABCDEF
    w = K // BLOCK

    def fill(rank, world):
        class Cal(GPU_Calculation):
            pass
        Cal.TYPE, Cal.LAYOUT = TYPE, LAYOUT
        Kl = K // world
        ld = Cal.padded_ld(N, Kl, BLOCK)
        rows = N if LAYOUT == "row" else Kl // BLOCK
        store = torch.zeros((BLOCK, rows, ld), dtype=torch.float32 if TYPE == "float" else torch.float64, device="cuda")
        cal = Cal.from_device_blocks(store, N, Kl, BLOCK)
        _lib.check(cal._lib.b200l_gen_gaussian(cal.ctx, seed, rank, world))
        return cal, _device_blocks(cal)

    cal, full = fill(0, 1)
    want = philox.gauss_matrix(seed, N, np.arange(K)).astype(np.float64).reshape(N, BLOCK, w).transpose(1, 0, 2)
    assert np.abs(full - want).max() < 2e-5          # logf / sincospif on the device vs NumPy
    for world in (2, 4):
        wl = w // world
        for rank in range(world):
            _, part = fill(rank, world)
            assert np.array_equal(part, full[:, :, rank * wl:(rank + 1) * wl])
    # row norms and scaling (parameters.py:22-23)
    ss = np.empty(N)
    _lib.check(cal._lib.b200l_row_sumsq(cal.ctx, _lib.dptr(ss)))
    assert np.allclose(ss, (full ** 2).sum(axis=(0, 2)), rtol=1e-12)
    scale = np.ascontiguousarray(1.0 / np.sqrt(ss))
    _lib.check(cal._lib.b200l_scale_rows(cal.ctx, _lib.dptr(scale)))
    scaled = _device_blocks(cal)
    tol = 1e-6 if TYPE == "float" else 1e-14
    assert np.allclose((scaled ** 2).sum(axis=(0, 2)), 1.0, atol=10 * tol)
    # padding stays zero
    assert float(cal._A_store.cpu().numpy().astype(np.float64).__abs__().sum()) == pytest.approx(np.abs(scaled).sum(), rel=1e-12)


@pytest.mark.gpu
def test_parameters_device_instance_solves_like_the_oracle():
    """parameters_device(): unit rows, b, mu as in parameters.py:20-33, and the instance solved by the
    fused kernel matches the oracle run on the downloaded matrix"""
    from convex_optimization_b200 import lasso, parameters
    from convex_optimization_b200.gpu_calculation import GPU_Calculation

    class Cal(GPU_Calculation):
        pass
    Cal.TYPE, Cal.LAYOUT = "double", "row"
    N, K, BLOCK = 300, 1800, 3
    cal, x_true, b, mu = parameters.parameters_device(N, K, BLOCK, 0.05, 11, gpu_cal_cls=Cal)
    blocks = _device_blocks(cal)
    A = np.concatenate([blocks[m] for m in range(BLOCK)], axis=1)
    assert np.allclose(np.linalg.norm(A, axis=1), 1.0, atol=1e-12)
    assert mu == pytest.approx(0.1 * np.max(np.abs(A.T @ b)), rel=1e-12)
    assert np.linalg.norm(b[:, 0] - (A @ x_true)[:, 0]) < 0.05 * np.sqrt(N)      # noise sd 1e-2
    ITER_MAX = 300 * BLOCK
    o = orc.lasso_oracle(A, b, mu, BLOCK, ITER_MAX, 1e-4, faithful=False)
    s = lasso.ClassLasso(cal, cal.diag_ATA, A, b, mu, BLOCK, ITER_MAX)
    s.run(1e-4, SILENCE=True)
    assert s.iters == o["iters"]
    assert np.array_equal(s.x != 0, o["x"] != 0)
    assert rel(s.x, o["x"]) < 1e-10
