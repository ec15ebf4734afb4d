"""Flexible GMRES (saena_b200_solve_gmres) on one GPU: what it costs against PCG on an SPD problem, what it buys on a
nonsymmetric one, and what its orthogonalisation kernels reach against their byte model.

1. 256^3 Poisson with bench.py's hierarchy, options and mapping autotune: PCG and GMRES(30) at preconditioner precision
   64 and 32 (one context each), alternated `reps` times after a warm-up, host clock around work that ends in a device
   synchronise; iterations and ||b - A u|| / ||b|| recomputed with the FP64 operator.
2. The nonsymmetric convection-diffusion operator (sa_setup.convdiff3d_coo) at nc^3, Jacobi smoother (2 + 2 sweeps):
   GMRES(10), GMRES(30), and the plain V-cycle iteration (solve_vcycle) for contrast, same timing.
3. One orthogonalisation step at 256^3 for nv = j + 1 basis vectors, j = 0 .. 29 (saena_b200_time_gmres_step: the three
   CGS2 passes and the normalisation, median of `kreps` CUDA-event-timed steps, no L2 flush -- the working set is
   (j + 2) x 134 MB, above the 126 MB L2 from j = 0), against the byte model (3 j + 11) x 8 n: the multi-dot reads
   j + 2 vectors, the fused update j + 2 and writes 1, the correction the same, the normalisation reads 1 and writes 2.
   Next to it: one level-0 SpMV and one V-cycle of the same hierarchy, the rest of an iteration.
The card's name, power limit and clocks are read in the same process.

    python tools/gmres_time.py [n] [nc] [reps] > profiles/r08_gmres.json
"""
import json
import subprocess
import sys
import time

sys.path.insert(0, ".")
import numpy as np  # noqa: E402
import torch  # noqa: E402

from saena_b200 import sa_setup  # noqa: E402
from saena_b200.native import Context  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 256
nc = int(sys.argv[2]) if len(sys.argv) > 2 else 128
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 3
sync = torch.cuda.synchronize
POISSON = dict(max_iter=50, tol=1e-8, smoother="chebyshev", pre=3, post=3)   # bench.py's
CONVDIFF = dict(max_iter=300, tol=1e-8, smoother="jacobi", pre=2, post=2)


def gpu_info():
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm,clocks.mem",
                           "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()


def hierarchy(coo):
    dh = sa_setup.build_device_hierarchy(*coo, device="cuda")
    h = dh.to_rank(0, 1)
    del dh
    torch.cuda.empty_cache()
    return h


def timed(solvers, reps):
    """solvers: name -> f() returning (iters, hist, u as numpy); one warm-up each, then `reps` alternated rounds"""
    out = {k: {"ms_all": []} for k in solvers}
    for k, f in solvers.items():
        it, hist, _ = f()
        out[k].update(iters=int(it), history=[float(x) for x in hist])
    for _ in range(reps):
        for k, f in solvers.items():
            sync()
            t = time.perf_counter()
            f()
            sync()
            out[k]["ms_all"].append(round(1e3 * (time.perf_counter() - t), 2))
    for k in solvers:
        out[k]["ms"] = float(np.median(out[k]["ms_all"]))
    return out


def dev_solver(ctx, method, bd, **kw):
    u = torch.zeros_like(bd)

    def f():
        if method == "pcg":
            it, hist = ctx.solve_pcg_dev(bd.data_ptr(), u.data_ptr(), **kw)
        else:
            it, hist = ctx.solve_gmres_dev(bd.data_ptr(), u.data_ptr(), **kw)
        return it, hist, u
    return f


def true_residual(ctx, res, solvers, b):
    nb = np.linalg.norm(b)
    for k, f in solvers.items():
        u = f()[2]
        u = u.cpu().numpy() if hasattr(u, "cpu") else u
        res[k]["true_rel_residual"] = float(np.linalg.norm(ctx.residual(0, u, b)) / nb)


out = {"n": n, "nc": nc, "reps": reps, "gpu": gpu_info()}

# ---- 1. Poisson: GMRES(30) against PCG at both preconditioner precisions
hier = hierarchy(sa_setup.poisson3d_coo(n))
b = sa_setup.poisson3d_rhs(n)
bd = torch.from_numpy(b).cuda()
c64 = Context()
c64.upload_hierarchy(hier)
c64.autotune_mapping_native(10, 0.03)
c32 = Context()
c32.upload_hierarchy(hier)
for l, lv in enumerate(hier.levels):
    for kind, op in ((0, lv.A), (1, lv.P), (2, lv.R)):
        if op is not None and c32.get_mapping(l, kind) != c64.get_mapping(l, kind):
            c32.set_mapping(l, kind, c64.get_mapping(l, kind))
for l in range(1, len(hier.levels)):
    if c64.get_level_route(l) != c32.get_level_route(l):
        c32.set_level_route(l, c64.get_level_route(l))
c32.set_precond_precision(32)
solvers = {"pcg_fp64": dev_solver(c64, "pcg", bd, **POISSON),
           "gmres30_fp64": dev_solver(c64, "gmres", bd, restart=30, **POISSON),
           "pcg_fp32": dev_solver(c32, "pcg", bd, **POISSON),
           "gmres30_fp32": dev_solver(c32, "gmres", bd, restart=30, **POISSON)}
res = timed(solvers, reps)
true_residual(c64, res, solvers, b)
out["poisson"] = {"problem": f"poisson3d_{n}", "rows": [lv.A.M for lv in hier.levels], "opts": POISSON, "solves": res}
print(json.dumps({k: (v["iters"], v["ms"], v["true_rel_residual"]) for k, v in res.items()}), file=sys.stderr, flush=True)

# ---- 3. the orthogonalisation step against its byte model, with the rest of an iteration next to it
N = hier.levels[0].A.M
steps = []
for j in range(30):
    ms = c64.time_gmres_step(j + 1, reps=20)
    model = (3 * j + 11) * 8 * N
    steps.append({"j": j, "ms": round(ms, 4), "model_bytes": model, "gbps": round(model / ms / 1e6, 1)})
out["orth_step"] = steps
out["spmv_l0_ms"] = round(c64.time_matvec(0, 0, reps=20, flush_l2=True), 4)
out["vcycle_ms"] = round(c64.time_vcycle(0, "chebyshev", 3, 3, reps=10), 4)
print(json.dumps(steps[::5]), file=sys.stderr, flush=True)
c64.close()
c32.close()
del hier, bd
torch.cuda.empty_cache()

# ---- 2. the nonsymmetric problem
hier = hierarchy(sa_setup.convdiff3d_coo(nc))
b = np.random.default_rng(nc).uniform(-1, 1, nc ** 3)
bd = torch.from_numpy(b).cuda()
ctx = Context()
ctx.upload_hierarchy(hier)
ctx.autotune_mapping_native(10, 0.03)


def vcycle_solver():
    u, it, hist = ctx.solve_vcycle(b, **CONVDIFF)
    return it, hist, u


solvers = {"gmres10": dev_solver(ctx, "gmres", bd, restart=10, **CONVDIFF),
           "gmres30": dev_solver(ctx, "gmres", bd, restart=30, **CONVDIFF),
           "vcycle": vcycle_solver}
res = timed(solvers, reps)
true_residual(ctx, res, solvers, b)
out["convdiff"] = {"problem": f"convdiff3d_{nc}", "rows": [lv.A.M for lv in hier.levels], "opts": CONVDIFF,
                   "solves": res}
print(json.dumps({k: (v["iters"], v["ms"], v["true_rel_residual"]) for k, v in res.items()}), file=sys.stderr, flush=True)
ctx.close()
out["gpu_after"] = gpu_info()
print(json.dumps(out, indent=1))
