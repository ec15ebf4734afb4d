"""Block AMG-PCG (saena_b200_solve_pcg_block) against k single solves at 256^3 Poisson on one GPU.

The bench's hierarchy is built, uploaded and mapping-autotuned as bench.py does; the right-hand sides are the Poisson
rhs and seeded random columns.  For each k in (1, 2, 4, 8): one block solve of k columns and k single solves, alternated
`reps` times after a warm-up of each, timed with the host clock around work that ends in a device synchronise.  Reported:
ms per solve and per right-hand side, the speed-up, per-column bitwise agreement (iterations, history, u), device memory
in use after the block buffers for k exist (cudaMemGetInfo, above what was in use before the first block call), and the
algorithmic bytes of one V-cycle of each path (SURVEY.md 8d: per operator application the stored matrix once plus x and
w per column; vector-only kernels not counted).  The card's name, power limit and clocks are read in the same process.

    python tools/block_solve_time.py [n] [reps] > profiles/r06_block_pcg.json
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
out = {"n": n, "reps": reps, "gpu": subprocess.run(
    ["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm,clocks.mem", "--format=csv,noheader"],
    capture_output=True, text=True).stdout.strip()}
sync = torch.cuda.synchronize

dh = sa_setup.build_device_hierarchy(*sa_setup.poisson3d_coo(n), device="cuda")
hier = dh.to_rank(0, 1)
del dh
torch.cuda.empty_cache()
ctx = Context()
ctx.upload_hierarchy(hier)
ctx.autotune_mapping_native(10, 0.03)
L = len(hier.levels)
M0 = hier.levels[0].A.M
out["levels"] = [{"rows": lv.A.M, "route": ctx.get_level_route(l),
                  "mapping": [ctx.get_mapping(l, kind) for kind in range(3) if (lv.A, lv.P, lv.R)[kind] is not None]}
                 for l, lv in enumerate(hier.levels)]


def vcycle_bytes(k):
    """per level: 6 applications of A (3 pre sweeps, the first from zero needs none; residual; 3 post), R and P"""
    per_level = []
    for l, lv in enumerate(hier.levels[:-1]):
        tot = 0
        for kind, op, times in ((0, lv.A, 6), (1, lv.P, 1), (2, lv.R, 1)):
            b = ctx.operator_bytes(l, kind)
            vec = 8 * (op.n_local_cols + op.M)   # on a route level the intermediates' traffic stays in b - vec
            tot += times * ((b - vec) + k * vec)
        per_level.append(tot)
    return per_level


rng = np.random.default_rng(2024)
cols = np.stack([sa_setup.poisson3d_rhs(n)] + [rng.standard_normal(M0) for _ in range(7)])
rhs_dev = torch.from_numpy(cols).cuda()
free0, total = torch.cuda.mem_get_info()
u1 = torch.zeros(M0, dtype=torch.float64, device="cuda")


def singles(k):
    res = []
    for j in range(k):
        it, hist = ctx.solve_pcg_dev(rhs_dev[j].data_ptr(), u1.data_ptr(), **OPTS)
        res.append((it, hist, u1.cpu().numpy()))
    return res


out["runs"] = []
for k in (1, 2, 4, 8):
    rhs_k = rhs_dev[:k].contiguous()
    ub, itb, hb = ctx.solve_pcg_block(rhs_k, **OPTS)          # warm-up: buffers, graph capture
    ref = singles(k)
    sync()
    mem_gb = (total - torch.cuda.mem_get_info()[0] - (total - free0)) / 1e9
    agree = [bool(itb[j] == ref[j][0] and np.array_equal(hb[j], ref[j][1]) and
                  np.array_equal(ub[j].cpu().numpy(), ref[j][2])) for j in range(k)]
    t_block, t_single = [], []
    for _ in range(reps):
        sync()
        t = time.perf_counter()
        ctx.solve_pcg_block(rhs_k, **OPTS)
        sync()
        t_block.append(time.perf_counter() - t)
        t = time.perf_counter()
        for j in range(k):
            ctx.solve_pcg_dev(rhs_dev[j].data_ptr(), u1.data_ptr(), **OPTS)
        sync()
        t_single.append(time.perf_counter() - t)
    mb, ms = 1e3 * float(np.median(t_block)), 1e3 * float(np.median(t_single))
    vb1, vbk = vcycle_bytes(1), vcycle_bytes(k)
    out["runs"].append({
        "k": k, "iters": [int(i) for i in itb], "bitwise_equal_to_single": agree,
        "ms_block": round(mb, 2), "ms_k_singles": round(ms, 2), "ms_per_rhs_block": round(mb / k, 2),
        "ms_per_rhs_single": round(ms / k, 2), "speedup": round(ms / mb, 3),
        "ms_block_all": [round(1e3 * t, 2) for t in t_block], "ms_singles_all": [round(1e3 * t, 2) for t in t_single],
        "device_mem_gb_above_start": round(mem_gb, 2),
        "vcycle_bytes_block_by_level": vbk, "vcycle_bytes_k_singles": k * sum(vb1), "vcycle_bytes_block": sum(vbk),
        "byte_model_speedup": round(k * sum(vb1) / sum(vbk), 3)})
    print(json.dumps(out["runs"][-1]), file=sys.stderr, flush=True)
ctx.close()
print(json.dumps(out, indent=1))
