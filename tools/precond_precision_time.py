"""AMG-PCG with the FP32 preconditioner (saena_b200_set_precond_precision 32) against the FP64 one on one GPU.

Two problems: 256^3 Poisson with bench.py's hierarchy, options and mapping autotune, and bench.py's one-GPU
unstructured2d hierarchy (g = 2828, 8.0 M rows).  Two contexts hold the same hierarchy with the same mappings and
routes (the FP64 one is autotuned, the FP32 one takes its choices); FP64 and FP32 solves are alternated `reps` times
after a warm-up of each, timed with the host clock around work that ends in a device synchronise.  Reported per
problem: iterations, residual histories and ms per solve of each precision; ||b - A u|| / ||b|| of each returned u,
recomputed with the FP64 operator; max|u32 - u64| / max|u64|; the device memory the FP32 state adds (cudaMemGetInfo
around the switch and the first FP32 solve); per level the FP64 and FP32 V-cycle cost from time_vcycle differences and
the byte model of one V-cycle at both precisions (SURVEY.md 8d per operator application: 6 applications of A -- 3 pre
sweeps, the first from zero needs none, the residual, 3 post sweeps -- plus R and P).  The card's name, power limit and
clocks are read in the same process.

    python tools/precond_precision_time.py [n] [reps] [g] > profiles/r07_f32_precond.json
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

OPTS = dict(max_iter=50, tol=1e-8, smoother="chebyshev", pre=3, post=3)   # bench.py's
n = int(sys.argv[1]) if len(sys.argv) > 1 else 256
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
g = int(sys.argv[3]) if len(sys.argv) > 3 else 2828
sync = torch.cuda.synchronize


def gpu_info():
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm,clocks.mem",
                           "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()


def copy_configuration(src, dst, hier):
    for l, lv in enumerate(hier.levels):
        for kind, op in ((0, lv.A), (1, lv.P), (2, lv.R)):
            if op is not None and dst.get_mapping(l, kind) != src.get_mapping(l, kind):
                dst.set_mapping(l, kind, src.get_mapping(l, kind))
    for l in range(1, len(hier.levels)):
        if src.get_level_route(l) != dst.get_level_route(l):
            dst.set_level_route(l, src.get_level_route(l))


def vcycle_bytes(ctx, hier, vb):
    """per level l < coarsest: 6 x A_l + P_l + R_l, operator_bytes at the context's precision"""
    out = []
    for l, lv in enumerate(hier.levels[:-1]):
        out.append(6 * ctx.operator_bytes(l, 0) + ctx.operator_bytes(l, 1) + ctx.operator_bytes(l, 2))
    return out


def per_level_ms(ctx, L):
    t = [ctx.time_vcycle(l, "chebyshev", 3, 3, reps=10) for l in range(L)]
    return [round(t[l] - (t[l + 1] if l + 1 < L else 0.0), 4) for l in range(L)], [round(x, 4) for x in t]


def run(name, hier, b):
    L = len(hier.levels)
    c64 = Context()
    c64.upload_hierarchy(hier)
    c64.autotune_mapping_native(10, 0.03)
    c32 = Context()
    c32.upload_hierarchy(hier)
    copy_configuration(c64, c32, hier)
    res = {"problem": name, "rows": [lv.A.M for lv in hier.levels],
           "mapping": [[c64.get_mapping(l, k) for k in range(3)] for l in range(L)],
           "route": [c64.get_level_route(l) for l in range(L)]}
    bd = torch.from_numpy(b).cuda()
    u64d, u32d = torch.zeros_like(bd), torch.zeros_like(bd)
    sync()
    free0 = torch.cuda.mem_get_info()[0]
    c32.set_precond_precision(32)
    it32, h32 = c32.solve_pcg_dev(bd.data_ptr(), u32d.data_ptr(), **OPTS)   # warm-up: copies, graph capture
    sync()
    res["fp32_state_gb"] = round((free0 - torch.cuda.mem_get_info()[0]) / 1e9, 3)
    it64, h64 = c64.solve_pcg_dev(bd.data_ptr(), u64d.data_ptr(), **OPTS)
    t64, t32 = [], []
    for _ in range(reps):
        for ctx, u, ts in ((c64, u64d, t64), (c32, u32d, t32)):
            sync()
            t = time.perf_counter()
            ctx.solve_pcg_dev(bd.data_ptr(), u.data_ptr(), **OPTS)
            sync()
            ts.append(1e3 * (time.perf_counter() - t))
    u64, u32 = u64d.cpu().numpy(), u32d.cpu().numpy()
    nb = np.linalg.norm(b)
    res.update({
        "iters": {"fp64": it64, "fp32": it32},
        "history": {"fp64": h64.tolist(), "fp32": h32.tolist()},
        "ms": {"fp64": round(float(np.median(t64)), 2), "fp32": round(float(np.median(t32)), 2),
               "fp64_all": [round(x, 2) for x in t64], "fp32_all": [round(x, 2) for x in t32]},
        "true_rel_residual": {"fp64": float(np.linalg.norm(c64.residual(0, u64, b)) / nb),
                              "fp32": float(np.linalg.norm(c64.residual(0, u32, b)) / nb)},
        "u_rel_diff": float(np.abs(u32 - u64).max() / np.abs(u64).max()),
    })
    lv64, cum64 = per_level_ms(c64, L)
    lv32, cum32 = per_level_ms(c32, L)
    res["vcycle_ms_by_level"] = {"fp64": lv64, "fp32": lv32, "fp64_from_level": cum64, "fp32_from_level": cum32}
    res["vcycle_bytes_by_level"] = {"fp64": vcycle_bytes(c64, hier, 8), "fp32": vcycle_bytes(c32, hier, 4)}
    c64.close()
    c32.close()
    print(json.dumps({k: v for k, v in res.items() if k != "history"}), file=sys.stderr, flush=True)
    return res


out = {"n": n, "g": g, "reps": reps, "opts": OPTS, "gpu": gpu_info(), "runs": []}
dh = sa_setup.build_device_hierarchy(*sa_setup.poisson3d_coo(n), device="cuda")
hier = dh.to_rank(0, 1)
del dh
torch.cuda.empty_cache()
out["runs"].append(run(f"poisson3d_{n}", hier, sa_setup.poisson3d_rhs(n)))
del hier
torch.cuda.empty_cache()
N, row, col, val = sa_setup.unstructured2d_coo(g, row_lengths=(6, 8, 10), weights=(16, 48, 20))   # bench.py's
dh = sa_setup.build_device_hierarchy(N, row, col, val, device="cuda")
del row, col, val
hier = dh.to_rank(0, 1)
del dh
torch.cuda.empty_cache()
out["runs"].append(run(f"unstructured2d_{g}", hier, sa_setup.unstructured2d_rhs(N)))
out["gpu_after"] = gpu_info()
print(json.dumps(out, indent=1))
