"""Cost of a value update (saena_b200_update_values) against a full re-setup at 256^3 Poisson (one GPU): the bench's
hierarchy is built, uploaded, finalized and mapping-autotuned, then for two new value sets on the same pattern -- a shift
A0 + sigma I (the mass term of an implicit time step, sigma = a fifth of the diagonal) and a symmetric rescaling D A0 D,
D = 1 + 0.5 sin(2 pi x) sin(2 pi y) sin(2 pi z) on the grid (changes every off-diagonal) -- it reports the update's
host-clock time ending in a synchronise and its phases, the peak device memory in use during the update (cudaMemGetInfo
polled every ms, above what was in use before), the lumped fractions per level, the PCG iterations and ms per solve
after the update; and the same for a full re-setup on the same values (setup + upload + finalize + autotune).

    python tools/update_time.py [n] > profiles/r03_update_time.json
"""
import json
import math
import subprocess
import sys
import threading
import time

sys.path.insert(0, ".")
import numpy as np  # noqa: E402
import torch  # noqa: E402

from saena_b200 import sa_setup  # noqa: E402
from saena_b200.native import Context  # noqa: E402

OPTS = dict(max_iter=50, tol=1e-8, smoother="chebyshev", pre=3, post=3)   # bench.py's
n = int(sys.argv[1]) if len(sys.argv) > 1 else 256
out = {"n": n, "gpu": subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                     capture_output=True, text=True).stdout.strip()}
sync = torch.cuda.synchronize


def build(N, row, col, val):
    t = time.perf_counter()
    dh = sa_setup.build_device_hierarchy(N, row, col, val, device="cuda")
    hier = dh.to_rank(0, 1)
    del dh
    torch.cuda.empty_cache()
    t_setup = time.perf_counter() - t
    ctx = Context()
    ctx.upload_hierarchy(hier)
    t_upload = time.perf_counter() - t - t_setup
    ctx.autotune_mapping_native(10, 0.03)
    sync()
    return ctx, hier, {"setup_s": round(t_setup, 2), "upload_finalize_s": round(t_upload, 2),
                       "autotune_s": round(time.perf_counter() - t - t_setup - t_upload, 2),
                       "total_s": round(time.perf_counter() - t, 2)}


def solve_cost(ctx, rhs_dev, reps=5):
    u_dev = torch.zeros_like(rhs_dev)
    it, hist = ctx.solve_pcg_dev(rhs_dev.data_ptr(), u_dev.data_ptr(), **OPTS)   # warm-up (graph capture)
    sync()
    t = time.perf_counter()
    for _ in range(reps):
        ctx.solve_pcg_dev(rhs_dev.data_ptr(), u_dev.data_ptr(), **OPTS)
    sync()
    return {"iters": it, "rel_res": float(hist[-1] / hist[0]), "ms_per_solve": round((time.perf_counter() - t) / reps * 1e3, 2)}


def peak_during(fn):
    free0, total = torch.cuda.mem_get_info()
    peak, stop = [total - free0], threading.Event()

    def poll():
        while not stop.is_set():
            f, _ = torch.cuda.mem_get_info()
            peak[0] = max(peak[0], total - f)
            time.sleep(0.001)

    th = threading.Thread(target=poll)
    th.start()
    try:
        r = fn()
    finally:
        stop.set()
        th.join()
    return r, (peak[0] - (total - free0)) / 1e9


N, row, col, val = sa_setup.poisson3d_coo(n)
rhs_dev = torch.as_tensor(sa_setup.poisson3d_rhs(n), device="cuda")
ctx, hier, cost0 = build(N, row, col, val)
out["initial_setup"] = cost0
out["levels"] = [(lv.A.M, int(lv.A.nnz_local)) for lv in hier.levels]
out["solve_before"] = solve_cost(ctx, rhs_dev)

A0 = hier.levels[0].A
urow = np.repeat(np.arange(A0.M), A0.nnzPerRow_local)
ucol = np.asarray(A0.col_local, np.int64)
sigma = 0.2 * float(np.mean(val[row == col]))
t = np.arange(1, n + 1, dtype=np.float64) / (n + 1)
s = np.sin(2 * math.pi * t)
idx = np.arange(N)
D = 1.0 + 0.5 * s[idx % n] * s[(idx // n) % n] * s[idx // (n * n)]
value_sets = {
    "shift": ((row, col, val, idx, idx, np.full(N, sigma)), A0.val_local + sigma * (urow == ucol)),
    "dad": ((row, col, val * D[row] * D[col]), A0.val_local * D[urow] * D[ucol]),
}
for name, (coo, uploaded_order) in value_sets.items():
    res = {}
    v_dev = torch.as_tensor(uploaded_order, device="cuda")
    sync()

    def update():
        t0 = time.perf_counter()
        fr = ctx.update_values(v_dev, 20, 0)
        sync()
        return fr, time.perf_counter() - t0

    (fracs, sec), peak_gb = peak_during(update)
    res["update"] = {"wall_ms": round(sec * 1e3, 1), "phases_ms": {k: round(v, 1) for k, v in ctx.update_values_times().items()},
                     "peak_device_GB_above_before": round(peak_gb, 2), "lumped_fraction_per_level": [float(f) for f in fracs]}
    res["solve_after_update"] = solve_cost(ctx, rhs_dev)
    del v_dev
    if len(coo) == 6:   # shift: the diagonal entries are added to the COO (duplicates are summed by the setup)
        r2, c2, v2 = np.concatenate([coo[0], coo[3]]), np.concatenate([coo[1], coo[4]]), np.concatenate([coo[2], coo[5]])
    else:
        r2, c2, v2 = coo
    ctx2, _, cost = build(N, r2, c2, v2)
    res["full_resetup"] = cost
    res["solve_after_resetup"] = solve_cost(ctx2, rhs_dev)
    ctx2.close()
    del ctx2
    torch.cuda.empty_cache()
    out[name] = res
    print(json.dumps({name: res}), file=sys.stderr, flush=True)
ctx.close()
print(json.dumps(out))
