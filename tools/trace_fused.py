#!/usr/bin/env python
"""Phase breakdown of the fused kernel (b200l_run_traced): per block step, where the time
of the median / slowest CTA goes.  Diagnostic tool, not a bench (GPU only)."""
import argparse
import ctypes
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PHASES = ["pass1 (A^T r)", "publish g", "gather g", "combine", "resolve gamma", "prox+publish D",
          "gather D", "pass2 (A D)", "line-search partials"]


def main():
    import torch
    from bench import C2, make_device_instance
    from convex_optimization_b200 import _lib
    from convex_optimization_b200.gpu_calculation import GPU_Calculation
    ap = argparse.ArgumentParser()
    ap.add_argument("--N", type=int, default=C2["N"])
    ap.add_argument("--K", type=int, default=C2["K"])
    ap.add_argument("--block", type=int, default=C2["BLOCK"])
    ap.add_argument("--dtype", default="float")
    ap.add_argument("--sweeps", type=int, default=3)
    ap.add_argument("--layout", default="row", choices=["row", "transposed"])
    ap.add_argument("--slot-bytes", type=int, default=0)
    ap.add_argument("--sweep", default="", help="semicolon list of slot[,dbg] tuples (dbg: b200l_debug_flags bits 0-2)")
    ap.add_argument("--out", default="")
    ap.add_argument("--raw", default="", help="prefix for raw trace dumps (.npy)")
    ap.add_argument("--tiles", action="store_true", help="per-tile durations of the two passes")
    ap.add_argument("--all-ranks", action="store_true", help="under torchrun: every rank prints its line")
    args = ap.parse_args()
    N, K, BLOCK = args.N, args.K, args.block
    # under torchrun: one C2-sized column shard per rank (the instance grows with the world size)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)

    class Cal(GPU_Calculation):
        TYPE = args.dtype
        LAYOUT = args.layout
        DEVICE = local_rank
    dev = torch.device("cuda", local_rank)
    tdt = torch.float32 if args.dtype == "float" else torch.float64
    ld = Cal.padded_ld(N, K, BLOCK)
    store, b, mu = make_device_instance(torch, dev, N, K, BLOCK, 0.01, 2, tdt, ld, args.layout, dist, rank)
    cal = Cal.from_device_blocks(store, N, K, BLOCK)
    if world > 1:
        from convex_optimization_b200 import distributed as dd
        dd.connect(cal)
    lib, ctx = cal._lib, cal.ctx
    bb = np.ascontiguousarray(b.reshape(-1))
    NT = _lib.NTRACE
    combos = [(args.slot_bytes, 0)]
    if args.sweep:
        combos = [tuple(int(v) for v in c.split(",")) for c in args.sweep.split(";") if c]
    results = []
    for combo in combos:
        slot = combo[0]
        dbg = combo[1] if len(combo) > 1 else 0
        cal.set_tuning(slot)
        _lib.check(lib.b200l_debug_flags(ctx, dbg))
        _lib.check(lib.b200l_set_problem(ctx, _lib.dptr(bb)))
        geo = cal.run_config()
        G = geo["grid"]
        for _ in range(2):
            _lib.check(lib.b200l_run(ctx, None, BLOCK, float(mu), -1.0, None, None, None, None, None))
        nsteps = BLOCK * args.sweeps
        tr = np.zeros((G, nsteps, NT), np.uint64)
        kms = ctypes.c_double()
        g_out = ctypes.c_int32()
        tt = np.zeros((G, nsteps, _lib.NTTRACE), np.uint64) if (args.raw or args.tiles) else None
        _lib.check(lib.b200l_run_traced(ctx, nsteps, float(mu),
                                        tr.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)),
                                        tt.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)) if tt is not None else None,
                                        ctypes.byref(g_out), ctypes.byref(kms)))
        # untraced timing of the same configuration
        k2 = ctypes.c_double()
        ts = []
        for _ in range(5):
            _lib.check(lib.b200l_run(ctx, None, BLOCK, float(mu), -1.0, None, None, None, None,
                                     ctypes.byref(k2)))
            ts.append(k2.value)
        # stamps are SM cycles since the CTA's start; every CTA carries a (globaltimer, cycle) pair
        # at both ends of the launch (slots 13 / 14 of the first and the last step)
        trf = tr.astype(np.float64)
        ns_per_cycle = (trf[:, -1, 13] - trf[:, 0, 13]) / trf[:, -1, 11]
        scale = (ns_per_cycle * 1e-3)[:, None, None]         # us per cycle, per CTA
        g0 = (trf[:, 0, 13] - trf[:, 0, 13].min()) * 1e-3    # start of the CTA on the common clock, us
        t = trf[:, :, :10] * scale
        t_abs = t + g0[:, None, None]
        s = t[:, BLOCK:, :]                        # skip the first sweep of the launch
        s_abs = t_abs[:, BLOCK:, :]
        dur = np.diff(s, axis=2)
        step_len = s[:, 1:, 0] - s[:, :-1, 0]
        out = {"tuning": {"slot_bytes": slot, "dbg": dbg}, "geo": geo,
               "ms_per_sweep_traced": kms.value / args.sweeps, "ms_per_sweep": float(np.median(ts)),
               "sweeps_per_s": 1e3 / float(np.median(ts)),
               "us_per_block_step": float(step_len.mean()),
               "us_per_block_step_by_sweep": [round(float(step_len[:, i * BLOCK:(i + 1) * BLOCK].mean()), 2)
                                              for i in range(max(1, step_len.shape[1] // BLOCK))],
               "phases_us_mean_over_ctas": {n: round(float(dur[:, :, i].mean()), 3) for i, n in enumerate(PHASES)},
               "phases_us_max_cta": {n: round(float(dur[:, :, i].mean(axis=1).max()), 3) for i, n in enumerate(PHASES)},
               "phases_us_min_cta": {n: round(float(dur[:, :, i].mean(axis=1).min()), 3) for i, n in enumerate(PHASES)},
               "sm_mhz_from_trace": float(1e3 / np.median(ns_per_cycle)),
               "skew_us_pass1_end": float((s_abs[:, :, 1].max(axis=0) - s_abs[:, :, 1].min(axis=0)).mean()),
               "skew_us_step_start": float((s_abs[:, :, 0].max(axis=0) - s_abs[:, :, 0].min(axis=0)).mean())}
        if NT >= 15:        # inside "gather g": every word valid, combined over the threads, final sums
            f = trf[:, BLOCK:, :] * scale
            out["gather_g_detail_us"] = {
                "publish end -> every word of this thread valid (L2 loads + polls)": round(float((f[:, :, 10] - f[:, :, 2]).mean()), 3),
                "shuffle tree + barrier": round(float((f[:, :, 12] - f[:, :, 10]).mean()), 3),
                "sums over the warps": round(float((f[:, :, 3] - f[:, :, 12]).mean()), 3),
                "words polled again per thread and step (thread 0)": round(float(tr[:, BLOCK:-1, 11].mean()), 3)}
            out["gather D end -> pass-2 loop entered (r update, l1/err terms, D to registers)"] = \
                round(float((f[:, :, 14] - f[:, :, 7]).mean()), 3)
        if world > 1 and NT >= 16:
            f = trf[:, BLOCK:, :] * scale
            out["peer_rows_us"] = {
                "pass 2 end -> all peer rows summed (collector warp)": round(float((f[:, :, 15] - f[:, :, 8]).mean()), 3),
                "max over CTAs": round(float((f[:, :, 15] - f[:, :, 8]).max(axis=0).mean()), 3)}
        if args.tiles:
            ft = tt.astype(np.float64)[:, BLOCK:, :] * scale
            ntile = min(16, geo["tiles_per_slab"])
            out["tiles_us"] = {
                "pass1 tile (data landed -> done, incl. wait for peer rows)":
                    [round(float((ft[:, :, 16 + t] - ft[:, :, t]).mean()), 3) for t in range(ntile)],
                "pass1 tile end -> next tile landed":
                    [round(float((ft[:, :, t + 1] - ft[:, :, 16 + t]).mean()), 3) for t in range(ntile - 1)],
                "pass2 tile": [round(float((ft[:, :, 48 + t] - ft[:, :, 32 + t]).mean()), 3) for t in range(ntile)]}
            # the tile stamps are absolute, the phase stamps relative to the kernel start of the CTA
            fp = trf[:, BLOCK:, :] * scale
            off = ft[:, :, 16 + ntile - 1] - fp[:, :, 1]
            if world > 1:
                # my send of tile t -> my release of the peers' tile t; summed over two ranks it is the sum of
                # the two one-way latencies "tile finished there -> row usable here" (the clocks cancel)
                out["tiles_us"]["my rows of tile t sent -> all ranks' rows of tile t released here"] = \
                    [round(float((ft[:, :, 80 + t] - ft[:, :, 64 + t]).mean()), 3) for t in range(ntile)]
                out["tiles_us"]["pass2 tile t done -> my rows of tile t sent (sender warp)"] = \
                    [round(float((ft[:, :, 64 + t] - ft[:, :, 48 + t]).mean()), 3) for t in range(ntile)]
                out["tiles_us"]["all ranks' rows of tile t released -> next pass 1 reaches tile t"] = \
                    [round(float((ft[:, 1:, t] - ft[:, :-1, 80 + t]).mean()), 3) for t in range(ntile)]
            out["tiles_us"]["pass2 tile 0 issued by the producer, after the end of gather g"] = \
                round(float((ft[:, :, 80] - off - fp[:, :, 3]).mean()), 3)
            out["tiles_us"]["pass2 tile 0 landed, after the end of gather D"] = \
                round(float((ft[:, :, 32] - off - fp[:, :, 7]).mean()), 3)
            out["tiles_us"]["pass2 tile 0 landed, after its issue"] = round(float((ft[:, :, 32] - ft[:, :, 80]).mean()), 3)
            out["tiles_us"]["pass2 tile end -> next tile start"] = \
                [round(float((ft[:, :, 32 + t + 1] - ft[:, :, 48 + t]).mean()), 3) for t in range(ntile - 1)]
        results.append(out)
        if args.raw:
            np.save("%s_%d_%d.npy" % (args.raw, slot, dbg), tr)
            np.save("%s_tiles_%d_%d.npy" % (args.raw, slot, dbg), tt[::16])
        if world > 1:
            out["rank"] = rank
        if rank == 0 or args.all_ranks:
            print(json.dumps({k: out[k] for k in ("tuning", "ms_per_sweep", "ms_per_sweep_traced", "sweeps_per_s", "us_per_block_step", "us_per_block_step_by_sweep", "sm_mhz_from_trace",
                                                   "phases_us_mean_over_ctas", "skew_us_pass1_end",
                                                   "gather_g_detail_us", "gather D end -> pass-2 loop entered (r update, l1/err terms, D to registers)", "peer_rows_us", "tiles_us", "rank") if k in out}))
        sys.stdout.flush()
    out = results if len(results) > 1 else results[0]
    if world > 1:
        dd.disconnect(cal)
        dist.destroy_process_group()
    if args.out and rank == 0:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
