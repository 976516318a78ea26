"""Every shipping instantiation and geometry regime of the fused kernel against the fp64 oracle.

plan_geometry (csrc/b200lasso.cu) picks, from the shape alone, among numerically distinct code paths: the
column groups per thread (CPT), row groups combined through shared memory or a direct publish from registers,
the slice width cs (1..64; cs > 32 publishes D from two warps and sums two l1/err partials), the packing of
the step D (dpw, dsec), the tile rows TR, the ring slots S, the L2 gates, and for the pre-transposed layout
the threads per column P1 and the boxes per tile NBX.  REGIMES lists one row per regime with what the planner
chooses for it.  test_regime_table_matches_the_planner_and_reaches_every_regime checks the table against a
restatement of the planner (_plan) and that it reaches every value of every choice;
test_regime_table_matches_run_config_on_the_b200 checks it against b200l_run_config.  If the planner changes,
these two tests name the rows to move."""
import ctypes

import numpy as np
import pytest

from conftest import assert_support
from oracle import lasso_oracle as orc
from test_gpu_geometry import _instance
from test_gpu_parity import TOL, make_gpu_cal, rel

pytestmark = pytest.mark.gpu

# B200: 148 SMs, 227 KiB of opt-in shared memory per block, 126.5 MiB of L2 (cudaDeviceProp)
B200 = dict(sm=148, optin=232448, l2=132644864)


# ----------------------------------------------------------------------------- restated planner
def _ru(x, m):
    return (x + m - 1) // m * m


def _plan(N, K, BLOCK, TYPE, LAYOUT, sm, optin, l2):
    """plan_geometry (csrc/b200lasso.cu) for world = 1 and the default tuning, restated: the launch values
    b200l_run_config reports (TR, S, tiles, smem) and the choices it does not (cpt, nrg, cs, mw, direct,
    dpw, dsec, gate2, l2_ahead, P1, NBX), plus NK, the pass-2 load batch of CPT = 1 (the kernel's row_pair:
    8 / 4 / 2 loads per row from dk_n = ceil(ncg / 32)).  None when the planner refuses the shape."""
    NTC, GMAX, MAX_CS, NW = 256, 160, 64, 8
    trans = LAYOUT == "transposed"
    es = 8 if TYPE == "double" else 4
    V = 16 // es
    w = K // BLOCK
    c_ld = _ru(N if trans else w, V)                     # ctx ld: the stored row of a block
    ld = _ru(w, V) if trans else c_ld                    # columns of a block incl. padding (xld)
    rowbytes = ld * es
    if not trans and rowbytes > 32768:                   # the 32 KiB row limit
        return None
    G = min(sm, GMAX)
    rows_max = V * ((-(-N // V) + G - 1) // G) if trans else -(-N // G)
    ncg = ld // V
    cpt = 1
    while not trans and cpt * NTC < ncg:
        cpt *= 2
    nrg = max(1, NTC // ncg) if (not trans and cpt == 1) else 1
    brows = w if trans else N
    l2_resident = 2 * brows * c_ld * es <= l2 * 3 // 4
    slot_target = 49152 if (l2_resident and not trans) else 65536
    TR = min(64, max(1, slot_target // rowbytes))
    TR = min(TR, _ru(max(rows_max, 1), 4))
    if TR >= 4:
        TR &= ~3
    cs = 1
    while cs * G < ld:
        cs *= 2
    if cs > MAX_CS:                                      # the slice width limit: G * 64 columns
        return None
    direct = 1 if (trans or (nrg == 1 and cs * (es // 4) >= 4)) else 0

    def fixed(rows_pad, redT, red2):
        parts = [2 * 64 * 8, 184, rows_pad * 8, rows_pad * 8, rows_pad * es, rows_pad * es, redT, red2,
                 NTC * 16, (2 * MAX_CS + 2 * NW) * 8, rows_pad * 8, 128 * 4]   # (184 = sizeof(Ctl))
        return sum(_ru(p, 128) for p in parts)

    P1 = NBX = 1
    if trans:
        need = -(-rows_max // V)
        maxb = 256 // V
        best, pick = 1e30, None
        for p1 in (1, 2, 4, 8):
            nb0 = -(-need // maxb)
            for nb in range(nb0, nb0 + 3):
                k = -(-(-(-need // nb)) // p1)
                if not k & 1:
                    k += 1
                bxvb = p1 * k
                if bxvb > maxb or nb * bxvb > NTC:
                    continue
                BXV = nb * bxvb
                TJ = NTC // p1
                nt_t = -(-w // TJ)
                nparts = max(1, min(NTC // BXV, 32))
                slot = _ru(TJ * BXV * V * es, 128)
                slots = (optin - fixed(_ru(BXV * V, 8), nt_t * TJ * es, nparts * BXV * V * es)) // slot
                if slots < 2:
                    continue
                cost = BXV / need * (1.0 if slots >= 3 else 1.03) * (1.0 + 1e-3 * (nb - nb0)) * (1.0 + 1e-4 * p1)
                if cost < best:
                    best, pick = cost, (p1, nb, BXV, TJ, nt_t, nparts, slot)
        if pick is None:                                 # the N / #SM limit of the transposed layout
            return None
        P1, NBX, BXV, TJ, nt_max, nparts, slot = pick
        cpt = 1 if (P1 == 1 and NBX == 1) else 2
        fx = fixed(_ru(BXV * V, 8), nt_max * TJ * es, nparts * BXV * V * es)
    else:
        slot = _ru(TR * rowbytes, 128)
        fx = fixed(_ru(max(rows_max, 1), max(TR, 8)), ld * es if direct else nrg * 2 * ld * es, 16)
        nt_max = -(-rows_max // TR)
    S = min((optin - fx) // slot, 60)
    if S < 2:                                            # the ring: the row-major slab height limit
        return None
    S = min(S, 2 * nt_max + 2)
    dpw = 2 if (es == 4 and cs >= 4) else 1
    dk_n = (ncg + 31) >> 5
    return dict(TR=TR, S=S, tiles=nt_max, smem=S * slot + fx, grid=G, cpt=cpt, nrg=nrg, cs=cs,
                mw=cs * es // 4, direct=direct, dpw=dpw, dsec=1 if cs >= 2 * dpw else 0,
                gate2=1 if (l2_resident and not trans and S >= 4) else 0, l2_ahead=1 if l2_resident else 0,
                P1=P1, NBX=NBX,
                NK=(8 if dk_n > 4 else 4 if dk_n > 2 else 2) if (cpt == 1 and not trans) else None)


# ----------------------------------------------------------------------------- the regime table
# (N, K, BLOCK, TYPE, LAYOUT, kind, (TR, S, tiles per slab) on the B200, what the row is for).
# kind "plan": a fused shape another test solves, only planned here; "solve": solved here against the oracle
# (test_solve_row_vs_oracle); "prop": the shape of one kernel instantiation in the property tests below.
REGIMES = [
    (64, 256, 1, "double", "row", "plan", (4, 4, 1), "golden vectors (test_gpu_parity)"),
    (64, 256, 1, "float", "row", "plan", (4, 4, 1), "golden vectors (test_gpu_parity)"),
    (128, 512, 2, "double", "row", "plan", (4, 4, 1), "golden vectors (test_gpu_parity)"),
    (128, 512, 2, "float", "row", "plan", (4, 4, 1), "golden vectors (test_gpu_parity)"),
    (200, 1200, 4, "double", "row", "plan", (4, 4, 1), "golden vectors (test_gpu_parity)"),
    (200, 1200, 4, "float", "row", "plan", (4, 4, 1), "golden vectors (test_gpu_parity)"),
    (256, 1024, 8, "double", "row", "plan", (4, 4, 1), "golden vectors (test_gpu_parity)"),
    (256, 1024, 8, "float", "row", "plan", (4, 4, 1), "golden vectors (test_gpu_parity)"),
    (1024, 4096, 2, "double", "row", "plan", (3, 4, 3), "golden vectors (test_gpu_parity)"),
    (1024, 4096, 2, "float", "row", "plan", (4, 6, 2), "golden vectors (test_gpu_parity)"),
    (257, 1002, 3, "double", "row", "plan", (4, 4, 1), "ragged and transposed-layout tests"),
    (257, 1002, 3, "float", "row", "plan", (4, 4, 1), "ragged and transposed-layout tests"),
    (33, 70, 5, "double", "row", "plan", (4, 4, 1), "ragged and transposed-layout tests"),
    (33, 70, 5, "float", "row", "plan", (4, 4, 1), "ragged and transposed-layout tests"),
    (100, 2048, 1, "double", "row", "plan", (3, 4, 1), "test_ragged_shapes_vs_oracle"),
    (100, 2048, 1, "float", "row", "plan", (4, 4, 1), "test_ragged_shapes_vs_oracle"),
    (1500, 3000, 2, "double", "row", "plan", (4, 4, 3), "test_ragged_shapes_vs_oracle"),
    (1500, 3000, 2, "float", "row", "plan", (8, 4, 2), "test_ragged_shapes_vs_oracle"),
    (300, 8000, 2, "double", "row", "plan", (1, 6, 3), "test_ragged_shapes_vs_oracle"),
    (300, 8000, 2, "float", "row", "plan", (3, 4, 1), "test_ragged_shapes_vs_oracle"),
    (300, 2400, 4, "double", "row", "plan", (4, 4, 1), "test_fused_transposed_layout_vs_oracle"),
    (300, 2400, 4, "double", "transposed", "plan", (4, 12, 5), "test_fused_transposed_layout_vs_oracle"),
    (300, 2400, 4, "float", "row", "plan", (4, 4, 1), "test_fused_transposed_layout_vs_oracle"),
    (300, 2400, 4, "float", "transposed", "plan", (4, 8, 3), "test_fused_transposed_layout_vs_oracle"),
    (1000, 4000, 2, "double", "row", "plan", (3, 4, 3), "test_fused_transposed_layout_vs_oracle"),
    (1000, 4000, 2, "double", "transposed", "plan", (4, 50, 32), "test_fused_transposed_layout_vs_oracle"),
    (1000, 4000, 2, "float", "row", "plan", (4, 6, 2), "test_fused_transposed_layout_vs_oracle"),
    (1000, 4000, 2, "float", "transposed", "plan", (8, 34, 16), "test_fused_transposed_layout_vs_oracle"),
    (2000, 3000, 1, "double", "row", "plan", (2, 4, 7), "test_fused_transposed_layout_vs_oracle"),
    (2000, 3000, 1, "double", "transposed", "plan", (2, 6, 12), "test_fused_transposed_layout_vs_oracle"),
    (2000, 3000, 1, "float", "row", "plan", (4, 4, 4), "test_fused_transposed_layout_vs_oracle"),
    (2000, 3000, 1, "float", "transposed", "plan", (4, 51, 47), "test_fused_transposed_layout_vs_oracle"),
    (20000, 600, 2, "double", "row", "plan", (20, 4, 7), "test_fused_transposed_layout_vs_oracle"),
    (20000, 600, 2, "double", "transposed", "plan", (24, 3, 5), "test_fused_transposed_layout_vs_oracle"),
    (20000, 600, 2, "float", "row", "plan", (40, 4, 4), "test_fused_transposed_layout_vs_oracle"),
    (20000, 600, 2, "float", "transposed", "plan", (52, 3, 3), "test_fused_transposed_layout_vs_oracle"),
    (40000, 768, 2, "double", "row", "plan", (20, 3, 14), "test_fused_transposed_layout_vs_oracle"),
    (40000, 768, 2, "double", "transposed", "plan", (20, 2, 12), "test_fused_transposed_layout_vs_oracle"),
    (40000, 768, 2, "float", "row", "plan", (40, 3, 7), "test_fused_transposed_layout_vs_oracle"),
    (40000, 768, 2, "float", "transposed", "plan", (40, 5, 12), "test_fused_transposed_layout_vs_oracle"),
    (257, 1002, 3, "double", "transposed", "plan", (4, 6, 2), "test_fused_transposed_layout_vs_oracle"),
    (257, 1002, 3, "float", "transposed", "plan", (4, 6, 2), "test_fused_transposed_layout_vs_oracle"),
    (33, 70, 5, "double", "transposed", "plan", (4, 4, 1), "test_fused_transposed_layout_vs_oracle"),
    (33, 70, 5, "float", "transposed", "plan", (4, 4, 1), "test_fused_transposed_layout_vs_oracle"),
    (10000, 10000, 10, "double", "row", "plan", (8, 3, 9), "C2 block shape (test_gpu_geometry)"),
    (10000, 10000, 10, "double", "transposed", "plan", (8, 3, 8), "C2 block shape (test_gpu_geometry)"),
    (10000, 10000, 10, "float", "row", "plan", (12, 4, 6), "C2 block shape (test_gpu_geometry)"),
    (10000, 10000, 10, "float", "transposed", "plan", (16, 3, 4), "C2 block shape (test_gpu_geometry)"),
    (20000, 4000, 2, "double", "row", "plan", (4, 3, 34), "C3 block shape (test_gpu_geometry)"),
    (10000, 100000, 100, "double", "row", "plan", (8, 3, 9), "C2 at full size (test_gpu_parity)"),
    (10000, 100000, 100, "float", "row", "plan", (12, 4, 6), "C2 at full size (test_gpu_parity)"),
    (2000, 12000, 2, "float", "row", "solve", (2, 4, 7), "CPT 8, cs 64, dpw 2, TR 2, in L2: 48 KiB slots, gate2"),
    (12000, 12000, 2, "float", "row", "solve", (2, 4, 41), "CPT 8, cs 64, not in L2: no gate2 / l2_ahead"),
    (300, 8192, 1, "float", "row", "solve", (1, 5, 3), "widest fp32 row: 32,768-byte rows, TR 1"),
    (300, 4096, 1, "double", "row", "solve", (1, 5, 3), "widest fp64 row: CPT 8, cs 32, mw 64"),
    (1000, 8000, 2, "float", "row", "solve", (3, 4, 3), "CPT 4, TR 3 with three tiles per slab"),
    (600, 9472, 1, "float", "transposed", "solve", (1, 45, 74), "widest transposed block: cs 64, P1 2"),
    (600, 9472, 1, "double", "transposed", "solve", (1, 12, 37), "widest transposed block: cs 64, mw 128"),
    (3000, 12000, 2, "double", "transposed", "solve", (1, 3, 24), "cs 64, mw 128, not L2-resident"),
    (384800, 128, 2, "double", "row", "solve", (64, 3, 41), "tall slab: nrg 8, three ring slots for 41 tiles"),
    (740000, 128, 2, "float", "row", "solve", (64, 3, 79), "tall slab: nrg 16, three ring slots for 79 tiles"),
    (1000, 600, 2, "float", "row", "solve", (8, 4, 1), "nrg 3, cs 4: smem publish + packed D, NK 4"),
    (3000, 300, 3, "double", "row", "solve", (24, 4, 1), "nrg 5, NK 2, cs 1: D one column per sector (dsec 0)"),
    (200, 900, 3, "double", "row", "prop", (4, 4, 1), "fp64 row-major CPT 1 (nrg 1, NK 8)"),
    (200, 2400, 3, "double", "row", "prop", (4, 4, 1), "fp64 row-major CPT 2"),
    (200, 4500, 3, "double", "row", "prop", (4, 4, 1), "fp64 row-major CPT 4"),
    (200, 9000, 3, "double", "row", "prop", (2, 4, 1), "fp64 row-major CPT 8"),
    (200, 1800, 3, "float", "row", "prop", (4, 4, 1), "fp32 row-major CPT 1 (nrg 1, NK 8)"),
    (200, 4500, 3, "float", "row", "prop", (4, 4, 1), "fp32 row-major CPT 2"),
    (200, 9000, 3, "float", "row", "prop", (4, 4, 1), "fp32 row-major CPT 4"),
    (200, 18000, 3, "float", "row", "prop", (2, 4, 1), "fp32 row-major CPT 8, cs 64"),
    (3000, 600, 3, "double", "transposed", "prop", (24, 4, 1), "fp64 transposed CPT 1 (P1 1, one box), cs 2"),
    (8000, 768, 3, "double", "transposed", "prop", (32, 7, 4), "fp64 transposed CPT 2 (P1 4)"),
    (300, 600, 3, "float", "transposed", "prop", (4, 4, 1), "fp32 transposed CPT 1 (P1 1, one box), cs 2"),
    (8000, 768, 3, "float", "transposed", "prop", (56, 6, 2), "fp32 transposed CPT 2 (P1 2)"),
]

_SOLVE = [r for r in REGIMES if r[5] == "solve"]
# one shape per MODE-0 instantiation: T in {float, double} x CPT in {1, 2, 4, 8} row-major, CPT in {1, 2} transposed
_PROPS = [r for r in REGIMES if r[5] == "prop"]


def _rid(r):
    return "%dx%d_b%d_%s_%s" % (r[0], r[1], r[2], "f32" if r[3] == "float" else "f64", r[4])


def _device():
    from convex_optimization_b200 import _lib
    lib = _lib.load()
    name = ctypes.create_string_buffer(256)
    sm, optin, l2 = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    _lib.check(lib.b200l_device_info(0, name, 256, ctypes.byref(sm), ctypes.byref(optin), ctypes.byref(l2)))
    return dict(name=name.value.decode(), sm=sm.value, optin=optin.value, l2=l2.value)


def _cal_cls(TYPE, LAYOUT):
    from convex_optimization_b200.gpu_calculation import GPU_Calculation

    class Cal(GPU_Calculation):
        pass
    Cal.TYPE, Cal.LAYOUT = TYPE, LAYOUT
    return Cal


def _bind_zeros(N, K, BLOCK, TYPE, LAYOUT):
    """a context with an all-zero A bound: enough for b200l_run_config"""
    import torch
    Cal = _cal_cls(TYPE, LAYOUT)
    rows = N if LAYOUT == "row" else K // BLOCK
    store = torch.zeros((BLOCK, rows, Cal.padded_ld(N, K, BLOCK)),
                        dtype=torch.float64 if TYPE == "double" else torch.float32, device="cuda")
    return Cal.from_device_blocks(store, N, K, BLOCK)


def test_regime_table_matches_the_planner_and_reaches_every_regime():
    """every row plans as the table states, and the table reaches every value of every choice"""
    bad = []
    seen = {}
    for r in REGIMES:
        p = _plan(*r[:5], **B200)
        if p is None or (p["TR"], p["S"], p["tiles"]) != r[6]:
            bad.append("%s: table says (TR, S, tiles) = %s, the planner %s" % (
                _rid(r), r[6], None if p is None else (p["TR"], p["S"], p["tiles"])))
            continue
        TYPE, LAYOUT = r[3], r[4]
        for key in ("cpt", "cs", "nrg", "direct", "gate2", "l2_ahead", "P1", "NBX", "NK", "mw"):
            seen.setdefault((key, LAYOUT, TYPE), set()).add(p[key])
        seen.setdefault(("dpw/dsec", LAYOUT, TYPE), set()).add((p["dpw"], p["dsec"]))
        seen.setdefault(("TR", LAYOUT, TYPE), set()).add(min(p["TR"], 4))
    assert not bad, "\n".join(bad)

    def union(key, layouts=("row", "transposed"), types=("float", "double")):
        return set().union(*(seen.get((key, lay, t), set()) for lay in layouts for t in types))
    missing = []
    for TYPE in ("float", "double"):
        if union("cpt", ["row"], [TYPE]) != {1, 2, 4, 8}:
            missing.append("row-major %s CPT: %s" % (TYPE, sorted(union("cpt", ["row"], [TYPE]))))
    for LAYOUT in ("row", "transposed"):
        if union("cs", [LAYOUT]) != {1, 2, 4, 8, 16, 32, 64}:
            missing.append("%s cs: %s" % (LAYOUT, sorted(union("cs", [LAYOUT]))))
    want = {"direct": {0, 1}, "dpw/dsec": {(1, 0), (1, 1), (2, 1)}, "gate2": {0, 1}, "l2_ahead": {0, 1},
            "TR": {1, 2, 3, 4}, "NK": {None, 2, 4, 8}}
    for key, vals in want.items():
        if union(key) != vals:
            missing.append("%s: %s of %s" % (key, sorted(union(key), key=str), sorted(vals, key=str)))
    if union("P1", ["transposed"]) != {1, 2, 4, 8} or max(union("NBX", ["transposed"])) < 2:
        missing.append("transposed P1 %s NBX %s" % (sorted(union("P1", ["transposed"])),
                                                    sorted(union("NBX", ["transposed"]))))
    if 128 not in union("mw", ["transposed"], ["double"]):
        missing.append("fp64 transposed mw = 128")
    assert not missing, "regimes no row reaches:\n" + "\n".join(missing)


def test_regime_table_matches_run_config_on_the_b200():
    """b200l_run_config gives the (TR, S, tiles per slab) of the table, and the shared memory the restated
    planner computes, for every row"""
    dev = _device()
    if (dev["sm"], dev["optin"]) != (B200["sm"], B200["optin"]):
        pytest.skip("the table is for the B200 (148 SMs, 232,448 B of opt-in shared memory); this device "
                    "has %d SMs and %d B" % (dev["sm"], dev["optin"]))
    assert dev["l2"] == B200["l2"], dev
    bad = []
    for r in REGIMES:
        cal = _bind_zeros(*r[:5])
        geo = cal.run_config()
        p = _plan(*r[:5], **B200)
        got = (geo["tile_rows"], geo["ring_slots"], geo["tiles_per_slab"])
        if got != r[6] or geo["smem_bytes"] != p["smem"] or geo["grid"] != p["grid"]:
            bad.append("%s: run_config %s, table %s / smem %d" % (_rid(r), geo, r[6], p["smem"]))
        del cal
    assert not bad, "\n".join(bad)


# ----------------------------------------------------------------------------- oracle parity of the solve rows
_cache = {}


def _oracle(N, K, BLOCK, TYPE, iters, order=None, bound=None):
    """the instance of test_gpu_geometry and the oracle's solve of it; one instance at a time (the tall
    and the wide rows hold up to 1.2 GB on the host)"""
    den = 0.05 if K <= 1024 else 0.01
    key = (N, K, BLOCK, TYPE)
    if key not in _cache:
        _cache.clear()
        _cache[key] = (_instance(N, K, den, N + K, TYPE), {})
    (A, b, mu), solves = _cache[key]
    skey = (iters, None if order is None else tuple(order), bound)
    if skey not in solves:
        solves[skey] = orc.lasso_oracle(A, b, mu, BLOCK, iters, bound, order=order, faithful=False)
    return A, b, mu, solves[skey]


def _sweeps(N):
    return 2 if N > 100000 else 4


def _assert_matches_oracle(x, err, iters, o, A, b, mu, TYPE):
    assert iters == o["iters"]
    assert_support(x, o["x"], TYPE)
    assert rel(x, o["x"]) < TOL[TYPE]
    assert abs(orc.objective(A, b, x, mu) - o["objective"]) / o["objective"] < TOL[TYPE]
    if err is not None:
        assert np.abs(err[:iters] - o["err"]).max() / np.abs(o["err"]).max() < max(TOL[TYPE], 1e-10)


def _fused_solve(A, b, mu, BLOCK, iters, TYPE, LAYOUT, bound=None):
    """ClassLasso on the fused kernel; fails if the shape would take the step-wise path"""
    import warnings
    from convex_optimization_b200 import lasso
    cal = make_gpu_cal(A, BLOCK, TYPE, LAYOUT)
    cal.run_config()
    solver = lasso.ClassLasso(cal, cal.diag_ATA, A, b, mu, BLOCK, iters)
    err = np.zeros(iters)
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        solver.run(bound, err_iter=err, SILENCE=True)
    return solver, err


@pytest.mark.parametrize("row", _SOLVE, ids=_rid)
def test_solve_row_vs_oracle(row):
    """a fixed number of sweeps against the oracle; where the other layout takes the shape too, both
    layouts give the same iterates"""
    from convex_optimization_b200 import _lib
    N, K, BLOCK, TYPE, LAYOUT = row[:5]
    iters = BLOCK * _sweeps(N)
    A, b, mu, o = _oracle(N, K, BLOCK, TYPE, iters)
    solver, err = _fused_solve(A, b, mu, BLOCK, iters, TYPE, LAYOUT)
    _assert_matches_oracle(solver.x, err, solver.iters, o, A, b, mu, TYPE)
    assert solver.iters == iters and not solver.stopped
    other = "transposed" if LAYOUT == "row" else "row"
    try:
        s2, _ = _fused_solve(A, b, mu, BLOCK, iters, TYPE, other)
    except _lib.B200LassoError:
        assert _plan(N, K, BLOCK, TYPE, other, **B200) is None
        return
    assert s2.iters == solver.iters and rel(s2.x, solver.x) < TOL[TYPE]


# ----------------------------------------------------------------------------- properties per instantiation
def _prop_cal(row):
    N, K, BLOCK, TYPE, LAYOUT = row[:5]
    A, b, mu = _oracle(N, K, BLOCK, TYPE, 1)[:3]
    cal = make_gpu_cal(A, BLOCK, TYPE, LAYOUT)
    p = _plan(N, K, BLOCK, TYPE, LAYOUT, **B200)
    assert p is not None
    return cal, A, b, mu, p


class _Ctx:
    """b200l_* calls on one context: launches of the fused kernel and the state they leave"""

    def __init__(self, cal, b, mu):
        from convex_optimization_b200 import _lib
        self.cal, self.lib, self.ctx, self.mu, self._lib = cal, cal._lib, cal.ctx, float(mu), _lib
        self.b = np.ascontiguousarray(b, dtype=np.float64).reshape(-1)
        _lib.check(self.lib.b200l_set_problem(self.ctx, _lib.dptr(self.b)))

    def reset(self):
        self._lib.check(self.lib.b200l_reset(self.ctx))

    def run(self, n, bound=-1.0, order=None, err=None):
        """one launch of n steps: (steps_done, stopped)"""
        steps, stopped = ctypes.c_int64(), ctypes.c_int32()
        o = None
        if order is not None:
            order = np.ascontiguousarray(order, dtype=np.int32)
            o = order.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))
        self._lib.check(self.lib.b200l_run(self.ctx, o, n, self.mu, bound,
                                           None if err is None else self._lib.dptr(err), None,
                                           ctypes.byref(steps), ctypes.byref(stopped), None))
        return int(steps.value), int(stopped.value)

    def chunks(self, sizes, bound=-1.0, order=None):
        """the same solve as consecutive launches of the given sizes, from x = 0; stops where a launch
        reports the stop rule: (steps_done, stopped, x, r)"""
        self.reset()
        done, stopped, at = 0, 0, 0
        for n in sizes:
            s, stopped = self.run(n, bound, None if order is None else order[at:at + n])
            done += s
            at += n
            if stopped:
                break
            assert s == n
        return done, stopped, self.x(), self.r()

    def x(self):
        x = np.empty(self.cal.MAT_WIDTH_ALL)
        self._lib.check(self.lib.b200l_get_x(self.ctx, self._lib.dptr(x)))
        return x

    def r(self):
        r = np.empty(self.cal.MAT_HEIGHT)
        self._lib.check(self.lib.b200l_get_r(self.ctx, self._lib.dptr(r)))
        return r


def _close(a, b, TYPE):
    """same steps and stop, x and r equal up to rounding: inside a launch the next block gradient is formed as
    A_m^T r + gamma A_m^T q while gamma is being resolved, a launch boundary applies r += gamma q first (r is
    rounded to T for pass 1), so a split launch is not bit for bit the single one -- about 1e-15 relative in fp64
    and 1e-7 in fp32 (measured on a B200)"""
    tol = 1e-13 if TYPE == "double" else 2e-6
    return a[:2] == b[:2] and rel(a[2], b[2]) < tol and rel(a[3], b[3]) < tol


@pytest.mark.parametrize("row", _PROPS, ids=_rid)
def test_launch_granularity_changes_nothing_but_rounding(row):
    """INTEGRATION.md section 3: a solve split into launches of 1, 2, 7 and the remaining steps continues the
    single launch -- unbounded, and bounded with the stop firing inside the launch of 7 steps (at step 6 or 9
    of the 3-block sweeps) or alone in a launch of one step"""
    cal, A, b, mu, p = _prop_cal(row)
    TYPE, BLOCK = row[3], row[2]
    assert BLOCK == 3
    c = _Ctx(cal, b, mu)
    T = 8 * BLOCK
    err = np.zeros(T)
    c.reset()
    c.run(T, err=err)
    one = c.chunks([T])
    assert one[:2] == (T, 0)
    assert _close(c.chunks([1, 2, 7, T - 10]), one, TYPE)
    # a bound between the largest error of sweep s (s = 2 or 3) and the smallest of the largest errors of the
    # sweeps before it: the stop rule fires at the end of sweep s
    M = err.reshape(-1, BLOCK).max(axis=1)
    gap, s = max((M[:s - 1].min() / M[s - 1], s) for s in (2, 3))
    assert gap > 1.5, M
    bound = float(np.sqrt(M[s - 1] * M[:s - 1].min()))
    one = c.chunks([T], bound)
    assert one[:2] == (s * BLOCK, 1)
    assert _close(c.chunks([1, 2, 7, T - 10], bound), one, TYPE)
    assert _close(c.chunks([s * BLOCK - 1, 1, T], bound), one, TYPE)      # the stopping step alone


def _order(T):
    """nblocks = 3: block 1 never runs, blocks 0 and 2 repeat back to back (0 0 2 | 2 0 2 | ..)"""
    return np.array([(0, 0, 2, 2, 0, 2)[t % 6] for t in range(T)], np.int32)


def _bound_between_errors(err, order, BLOCK, TYPE):
    """an error bound that stops the run at some sweep, placed in a gap of the error trace at least a
    factor 1.5 wide (so that the fp32 iterates take the same decisions as the fp64 oracle's): the stop
    rule counts the steps below the bound since the last step of block nblocks - 1 and stops there when
    the count is nblocks (lasso.py:141-150)"""
    def stop_at(bound):
        cnt = 0
        for t, m in enumerate(order):
            cnt += err[t] < bound
            if m == BLOCK - 1:
                if cnt == BLOCK:
                    return t + 1
                cnt = 0
        return None
    floor = 1e-3 * err.max() if TYPE == "float" else 0.0
    v = np.unique(err[err > floor])
    best = None
    for lo, hi in zip(v[:-1], v[1:]):
        bound = float(np.sqrt(lo * hi))
        t = stop_at(bound)
        if hi / lo >= 1.5 and t and (best is None or (t, hi / lo) > best[:2]):
            best = (t, hi / lo, bound)                   # the latest stop, then the widest gap
    assert best is not None, "no usable gap in the error trace"
    return best[2]


@pytest.mark.parametrize("row", _PROPS, ids=_rid)
def test_explicit_order_vs_oracle(row):
    """an explicit block order (b200l_run's order_host) with a block repeated back to back and a block
    that never runs, against the oracle with the same order: unbounded, and bounded (the stop rule on
    the steps of block nblocks - 1)"""
    N, K, BLOCK, TYPE, LAYOUT = row[:5]
    cal, A, b, mu, p = _prop_cal(row)
    c = _Ctx(cal, b, mu)
    T = 4 * BLOCK          # (further on, the fp64 transposed instances reach errors of 1e-10 and below, where the
    order = _order(T)      # line search divides rounding noise by |q|^2 ~ 1e-18 and no two summation orders agree)
    A, b, mu, o = _oracle(N, K, BLOCK, TYPE, T, order=order)
    err = np.zeros(T)
    c.reset()
    done, stopped = c.run(T, order=order, err=err)
    assert (done, stopped) == (T, 0)
    _assert_matches_oracle(c.x().reshape(-1, 1), err, done, o, A, b, mu, TYPE)
    bound = _bound_between_errors(o["err"], order, BLOCK, TYPE)
    A, b, mu, o = _oracle(N, K, BLOCK, TYPE, T, order=order, bound=bound)
    assert o["stopped"]
    c.reset()
    err[:] = 0
    done, stopped = c.run(T, bound, order=order, err=err)
    assert stopped == 1
    _assert_matches_oracle(c.x().reshape(-1, 1), err, done, o, A, b, mu, TYPE)


@pytest.mark.parametrize("row", _PROPS, ids=_rid)
def test_traced_instantiation_matches_run(row):
    """b200l_run_traced (the MODE 2 instantiations) computes what b200l_run computes, bit for bit, and
    every CTA's step-start stamps do not decrease"""
    from convex_optimization_b200 import _lib
    cal, A, b, mu, p = _prop_cal(row)
    c = _Ctx(cal, b, mu)
    T = 6 * row[2]
    c.reset()
    c.run(T)
    x1, r1 = c.x(), c.r()
    c.reset()
    G = cal.run_config()["grid"]
    tr = np.zeros((G, T, _lib.NTRACE), np.uint64)
    g_out = ctypes.c_int32()
    _lib.check(c.lib.b200l_run_traced(c.ctx, T, c.mu, tr.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)), None,
                                      ctypes.byref(g_out), None))
    assert g_out.value == G
    assert np.array_equal(c.x(), x1) and np.array_equal(c.r(), r1)
    start = tr[:, :, 0].astype(np.int64)
    assert np.all(np.diff(start, axis=1) >= 0)
    assert np.all(start[:, -1] > 0)


# ----------------------------------------------------------------------------- shape limits and the fallback
def _limit_edge(N, K, BLOCK, TYPE, LAYOUT, accepted, match):
    """accepted: the fused kernel plans and solves the shape like the oracle.  Rejected: b200l_run fails
    with a message naming the limit, ClassLasso warns and runs the step-wise device path, which matches
    the oracle too."""
    from convex_optimization_b200 import _lib, lasso
    iters = 2 * BLOCK
    A, b, mu, o = _oracle(N, K, BLOCK, TYPE, iters)
    if accepted:
        solver, err = _fused_solve(A, b, mu, BLOCK, iters, TYPE, LAYOUT)
        _assert_matches_oracle(solver.x, err, solver.iters, o, A, b, mu, TYPE)
        return
    cal = make_gpu_cal(A, BLOCK, TYPE, LAYOUT)
    with pytest.raises(_lib.B200LassoError, match=match):
        cal.run_config()
    bb = np.ascontiguousarray(b.reshape(-1))
    _lib.check(cal._lib.b200l_set_problem(cal.ctx, _lib.dptr(bb)))
    with pytest.raises(_lib.B200LassoError, match=match):
        _lib.check(cal._lib.b200l_run(cal.ctx, None, iters, float(mu), -1.0, None, None, None, None, None))
    solver = lasso.ClassLasso(cal, cal.diag_ATA, A, b, mu, BLOCK, iters)
    err = np.zeros(iters)
    with pytest.warns(UserWarning, match=match):
        solver.run(err_iter=err, SILENCE=True)
    _assert_matches_oracle(solver.x, err, solver.iters, o, A, b, mu, TYPE)


@pytest.mark.parametrize("accepted", [True, False], ids=["widest", "first_rejected"])
@pytest.mark.parametrize("TYPE,LAYOUT", [("float", "row"), ("double", "row"), ("float", "transposed"),
                                         ("double", "transposed")])
def test_block_width_limit(TYPE, LAYOUT, accepted):
    """row-major: rows of up to 32 KiB (w = 8192 fp32, 4096 fp64); pre-transposed: the #SM CTAs own at most
    64 columns of a block each (w = 148 * 64 = 9472 on the B200)"""
    if LAYOUT == "row":
        w, match = (8192 if TYPE == "float" else 4096), "32 KiB"
    else:
        w, match = min(_device()["sm"], 160) * 64, "too wide for the fused kernel"
    _limit_edge(96, w + (0 if accepted else 1), 1, TYPE, LAYOUT, accepted, match)


def _tallest_row_slab(TYPE, dev):
    """largest N the row-major planner takes for w = 64 (K = 128, two blocks): a CTA's rows (N / #SM) must
    leave room for two ring slots next to the per-row buffers"""
    R = 1
    while _plan(dev["sm"] * 2 * R, 128, 2, TYPE, "row", **dev) is not None:
        R *= 2
    lo, hi = R, 2 * R                                    # accepted at lo rows per CTA, refused at hi
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if _plan(dev["sm"] * mid, 128, 2, TYPE, "row", **dev) is not None else (lo, mid)
    return dev["sm"] * lo


@pytest.mark.parametrize("accepted", [True, False], ids=["tallest", "first_rejected"])
@pytest.mark.parametrize("TYPE", ["double", "float"])
def test_row_slab_height_limit(TYPE, accepted):
    """row-major: the rows of a CTA (N / #SM) need per-row buffers in shared memory next to at least two
    ring slots; about 3,800 rows per CTA in fp64 and 5,700 in fp32 at w = 64 on the B200.  The limit the
    restated planner finds is the one b200l_run_config finds on the device."""
    dev = {k: v for k, v in _device().items() if k != "name"}
    N = _tallest_row_slab(TYPE, dev)
    cal = _bind_zeros(N, 128, 2, TYPE, "row")
    assert cal.run_config()["ring_slots"] == 2
    del cal
    cal = _bind_zeros(N + 1, 128, 2, TYPE, "row")
    from convex_optimization_b200 import _lib
    with pytest.raises(_lib.B200LassoError, match="shared memory too small"):
        cal.run_config()
    del cal
    _limit_edge(N + (0 if accepted else 1), 128, 2, TYPE, "row", accepted, "shared memory too small")
