"""Algorithmic bytes, CUDA-event time and rate of every operator of the bench hierarchy (256^3 Poisson by default, one
GPU), the transfer operators P and R included: bench.py prints GB/s for A only.

The hierarchy is built, uploaded and mapping-autotuned as bench.py does it.  Every operator is then timed as one
application with a plain epilogue (`saena_b200_time_matvec`), every A also as one fused Chebyshev sweep
(`saena_b200_time_smooth_sweep`); 20 launches each, median, L2 flushed between launches where the operator's bytes fit
in L2.  On a level that runs on the route (level 1 of the bench hierarchy) "A" is R A P of the level above, as in the
solve.  Bytes are SURVEY 8d's formulas on the uploaded sizes (`saena_b200_operator_bytes`), the sweep's as in bench.py
(+ 24 bytes a row).  "stored/nnz" is the entries the sliced layout streams, padding included, over the non-zeros (from
the row lengths, for the operators on a sliced mapping).  With --sorted, every operator on the sliced layout is also
timed on the sorted sliced layout (mapping 101) and put back.

    python tools/transfer_rates.py [--n 256] [--sorted] > profiles/<name>.md
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from saena_b200 import native  # noqa: E402
from saena_b200.hierarchy import KIND_A, KIND_P, KIND_R  # noqa: E402
from saena_b200.sa_setup import build_device_hierarchy, poisson3d_coo  # noqa: E402

SELL, SELLP, SYMDIAG = 100, 101, 103
REPS = 20
L2_BYTES = 300e6   # below this an operator's stream could stay in the 126 MB L2 between launches: flush


def mapping_name(m: int) -> str:
    if m == SELL:
        return "sliced"
    if m == SELLP:
        return "sorted sliced"
    if m == SYMDIAG:
        return "symmetric diagonals"
    if m < 0:
        return f"stream/{-m}"
    return f"{m} lanes/row" if m < 32 else f"{m} thr/row"


def stored_over_nnz(lengths: np.ndarray, sorted_windows: bool) -> float:
    """entries of the sliced layout (every 32-row slice padded to its longest row) over the non-zeros; sorted: rows
    sorted by length inside windows of 256 rows first"""
    n = len(lengths)
    if n == 0 or lengths.sum() == 0:
        return float("nan")
    w = 256 if sorted_windows else 32
    pad = (-n) % w
    x = np.concatenate([lengths.astype(np.int64), np.zeros(pad, np.int64)]).reshape(-1, w)
    if sorted_windows:
        x = -np.sort(-x, axis=1)
    return float(x.reshape(-1, 32).max(axis=1).sum() * 32) / float(lengths.sum())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=256)
    ap.add_argument("--sorted", action="store_true", help="also time the sorted sliced layout of every sliced operator")
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    dh = build_device_hierarchy(*poisson3d_coo(args.n))
    hier = dh.to_rank(0, 1)
    del dh
    torch.cuda.empty_cache()
    ctx = native.Context()
    ctx.upload_hierarchy(hier)
    ctx.autotune_mapping_native(10, 0.03)
    route = [l for l in range(len(hier.levels)) if ctx.get_level_route(l)]

    rows = []
    for l, lv in enumerate(hier.levels):
        for kind, op in ((KIND_A, lv.A), (KIND_P, lv.P), (KIND_R, lv.R)):
            if op is None or op.M == 0:
                continue
            b = ctx.operator_bytes(l, kind)
            flush = b < L2_BYTES
            ctx.time_matvec(l, kind, 3)   # warm-up
            ms = ctx.time_matvec(l, kind, REPS, flush_l2=flush)
            m = ctx.get_mapping(l, kind)
            on_route = kind == KIND_A and l in route
            r = {"level": l, "op": "APR"[kind], "rows": op.M, "nnz": op.nnz_local,
                 "mapping": "R A P of the level above" if on_route else mapping_name(m),
                 "bytes": b, "ms": ms, "GBs": b / ms / 1e6}
            if m in (SELL, SELLP) and not on_route:
                r["stored_over_nnz"] = stored_over_nnz(np.asarray(op.nnzPerRow_local), m == SELLP)
            if kind == KIND_A:
                sb = b + 24 * op.M
                ctx.time_smooth_sweep(l, "chebyshev", 3)
                sw = ctx.time_smooth_sweep(l, "chebyshev", REPS, flush_l2=flush)
                r.update(sweep_bytes=sb, sweep_ms=sw, sweep_GBs=sb / sw / 1e6)
            if args.sorted and m == SELL and not on_route:
                r["sorted_stored_over_nnz"] = stored_over_nnz(np.asarray(op.nnzPerRow_local), True)
                ctx.set_mapping(l, kind, SELLP)
                if ctx.get_mapping(l, kind) == SELLP:
                    ctx.time_matvec(l, kind, 3)
                    r["sorted_ms"] = ctx.time_matvec(l, kind, REPS, flush_l2=flush)
                    if kind == KIND_A:
                        ctx.time_smooth_sweep(l, "chebyshev", 3)
                        r["sorted_sweep_ms"] = ctx.time_smooth_sweep(l, "chebyshev", REPS, flush_l2=flush)
                ctx.set_mapping(l, kind, SELL)
            rows.append(r)
            print(json.dumps(r), file=sys.stderr, flush=True)
    ctx.close()

    print(f"# Operator rates of the {args.n}^3 Poisson bench hierarchy, one GPU\n")
    print(f"GPU (name, power limit, max SM clock): {gpu}. CUDA events around single launches, {REPS} launches each "
          f"(median), L2 flushed between launches below {L2_BYTES / 1e6:.0f} MB. Plain application (w = Op x) and, for A, "
          f"one fused Chebyshev sweep. Level(s) on the route: {route}.\n")
    sorted_cols = args.sorted
    head = "| level | op | rows | nnz | mapping | stored/nnz | MB | SpMV ms | SpMV GB/s | sweep ms | sweep GB/s |"
    sep = "|---:|---|---:|---:|---|---:|---:|---:|---:|---:|---:|"
    if sorted_cols:
        head += " sorted stored/nnz | sorted ms | sorted sweep ms |"
        sep += "---:|---:|---:|"
    print(head)
    print(sep)
    f = lambda v, p: "" if v is None else f"{v:.{p}f}"   # noqa: E731
    for r in rows:
        line = (f"| {r['level']} | {r['op']} | {r['rows']} | {r['nnz']} | {r['mapping']} | {f(r.get('stored_over_nnz'), 3)} "
                f"| {r['bytes'] / 1e6:.1f} | {r['ms']:.4f} | {r['GBs']:.0f} | {f(r.get('sweep_ms'), 4)} "
                f"| {f(r.get('sweep_GBs'), 0)} |")
        if sorted_cols:
            line += (f" {f(r.get('sorted_stored_over_nnz'), 3)} | {f(r.get('sorted_ms'), 4)} "
                     f"| {f(r.get('sorted_sweep_ms'), 4)} |")
        print(line)
    print("\n" + json.dumps({"gpu": gpu, "n": args.n, "route_levels": route, "operators": rows}))


if __name__ == "__main__":
    main()
