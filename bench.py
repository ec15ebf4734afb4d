#!/usr/bin/env python
"""bench.py -- AMG-PCG solve of the 3D 7-point Poisson problem on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--n 256] [--dump-outputs DIR]

A "step" is one complete `solve_pCG` (zero initial guess, AMG V-cycle preconditioner with 3+3
Chebyshev sweeps, stop at ||r||/||r0|| < 1e-8: the reference's experiments/Poisson.cpp loop with
data/options006_poisson.xml) on synthetic data: the 256^3-unknown Poisson operator and the
sin*sin*sin right-hand side of laplacian3D_set_rhs.  The hierarchy is built once, untimed (setup is
outside the hot path; saena_b200/sa_setup.py restates the reference's setup so the hierarchy has
the reference's shape), uploaded once, and stays resident in HBM.

Printed JSON line (rank 0): `value` = unknowns solved per second, whole job, inputs resident in
HBM, CUDA events on the library's compute stream, max over ranks; `e2e` = the same through the
host-buffer entry point (pinned host rhs -> H2D -> solve -> D2H u inside the timed region);
`roofline` = the dominant kernel's algorithmic bytes / its CUDA-event duration against the
measured HBM peak; `cpu_baseline` = the reference's own CPU solve (oracle/_ref, the compiled
reference) on a bounded sample.  `--impl reference` times only that CPU arm.

`--dump-outputs DIR` writes what the last timed solve returned, as float64 .npy files: `u` (the
solution, or a fixed seeded sample of at most DUMP_SAMPLE of its entries), `u_index` (their global
row indices), `residual_history` and `iterations`.  The inputs depend only on the arguments, so two
builds run with the same arguments can be compared output for output (to rounding: the setup picks
each operator's kernel mapping by timing it).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "AMG-PCG solve throughput, 3D 7-pt Poisson, rel. residual 1e-8 (unknowns solved per second)"
UNIT = "Munknowns/s"
OPTS = dict(max_iter=50, tol=1e-8, smoother="chebyshev", pre=3, post=3)   # data/options006_poisson.xml
# reference arm: laplacian3D(mx) -> (mx-2)^3 = 48^3 unknowns (env override only for the contract test)
CPU_SAMPLE_MX = int(os.environ.get("SAENA_BENCH_CPU_MX", 50))
# --dump-outputs: entries of u written at most (16 MB of values + 16 MB of indices, whatever the problem size)
DUMP_SAMPLE = 1 << 21


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json, copy bandwidth)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# clocks during the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device, self.proc, self.path = device, None, f"/tmp/saena_bench_clocks_{os.getpid()}.csv"

    def __enter__(self):
        try:
            self.out = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.out,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *exc):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
            self.out.close()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 6:
                    continue
                sm.append(float(f[0])); mx.append(float(f[1]))
                for n, v in zip(names, f[2:6]):
                    if v == "Active":
                        reasons.add(n)
            os.remove(self.path)
        except Exception:
            pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# the reference arm: the reference's own CPU implementation (compiled from /root/reference into
# oracle/_ref by oracle/Makefile), one MPI rank = one core (no MPI in this image; the reference's
# OpenMP is off by default, CMakeLists.txt:27).  Falls back to the C oracle port.
# ------------------------------------------------------------------------------------------------
def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_reference_solve_multirank(reps: int, warmup: int, ranks: int, mx: int):
    """The reference's own MPI solve on `ranks` host cores: the UNMODIFIED sources built against the
    multi-process MPI stand-in (oracle/ref_shim_mp, make -C oracle ref_mp), one process per rank started
    by oracle/mprun.py -- row partitioning, float halo, repartition / shrink, distributed setup and all."""
    import shutil
    import tempfile
    from oracle import mprun
    out = tempfile.mkdtemp(prefix="saena_ref_mp_")
    try:
        t = time.perf_counter()
        rc = mprun.run(ranks, [sys.executable, "-m", "oracle.mp_worker", "poisson", str(mx), out, str(max(reps, 1)),
                               str(warmup)], timeout=600, env=dict(os.environ, PYTHONPATH=ROOT))
        wall = time.perf_counter() - t
        if rc:
            raise RuntimeError(f"multi-rank reference run exited with {rc}")
        parts = [np.load(os.path.join(out, f"rank{r}.npz")) for r in range(ranks)]
    finally:
        shutil.rmtree(out, ignore_errors=True)
    sec = max(float(p["sec_per_solve"][0]) for p in parts)   # max over ranks, as Poisson.cpp:216-246 reports
    iters = int(parts[0]["iters"][0])
    setup_s = max(float(p["setup_s"][0]) for p in parts) if all("setup_s" in p.files for p in parts) else None
    n = (mx - 2) ** 3
    # the other half of BASELINE.json's metric on the CPU: level-0 SpMV as saena_object::profile_matvecs times it
    # (20 applications after a warm-up, max over ranks), in the algorithmic bytes of SURVEY 8d: 12 nnz + 20 M,
    # nnz = 7 n - 6 (mx-2)^2; at 96^3 / 128^3 the operator (130 / 310 MB with its vectors) is beyond the host's caches
    spmv_gbs = None
    if all("sec_per_matvec0" in p.files for p in parts):
        mv = max(float(p["sec_per_matvec0"][0]) for p in parts)
        if mv > 0:
            spmv_gbs = (12.0 * (7 * n - 6 * (mx - 2) ** 2) + 20.0 * n) / mv / 1e9
    what = (f"the reference's own solve_pCG (oracle/_ref/libsaena_ref_mp.so = unmodified paralab/Saena sources, -Ofast) "
            f"on {ranks} MPI ranks = {ranks} host cores (multi-process MPI stand-in over Unix sockets, oracle/ref_shim_mp), "
            f"3D Poisson {mx - 2}^3 = {n} unknowns (laplacian3D mx={mx}), same options; {reps} solves, {iters} "
            f"iterations each, max over ranks; the reference's own setup ({setup_s if setup_s is None else round(setup_s, 1)} s) "
            f"and the warm-up are not timed (whole run {wall:.0f} s)")
    return dict(value=n / sec / 1e6, unit=UNIT, cores=ranks, kind="reference", sample=what,
                spmv_level0_GBs=spmv_gbs, unknowns=n, setup_s=setup_s, ms_per_solve=sec * 1e3), sec, iters, n


def cpu_sample_mx(ranks: int, arm: bool) -> int:
    """laplacian3D(mx) size of the CPU sample: what the reference's own HOST SETUP lets a bounded run afford (the setup
    is what costs: 40 s for 96^3 on 8 ranks in this image, the solves are 0.9 s each).  The reference arm
    (--impl reference) takes the larger sample; the in-run cpu_baseline of the default bench run the smaller one."""
    if os.environ.get("SAENA_BENCH_CPU_MX_MP"):
        return int(os.environ["SAENA_BENCH_CPU_MX_MP"])
    if ranks >= 16:
        return 130 if arm else 98     # 128^3 = 2.1 M unknowns / 96^3 = 0.88 M
    if ranks >= 8:
        return 98 if arm else 66
    return 66


def cpu_reference_solve(reps: int, warmup: int = 0, mx: int = CPU_SAMPLE_MX, arm: bool = False):
    from oracle import ref
    n = (mx - 2) ** 3
    ranks = min(host_cores(), int(os.environ.get("SAENA_BENCH_CPU_RANKS", 32)))
    if ref.mp_available() and ranks > 1:
        try:
            # far larger samples than the one-rank arm can set up: 96^3 / 128^3 unknowns -- every rank's share of every
            # fine level is beyond its core's caches, as at the bench's own 256^3
            return cpu_reference_solve_multirank(reps, warmup, ranks, cpu_sample_mx(ranks, arm))
        except Exception as e:   # fall back to the one-rank build below
            log(f"[reference arm] multi-rank run failed ({e!r}); falling back to one rank")
    if ref.available():
        t = time.perf_counter()
        s = ref.RefSolver.poisson(mx)
        setup_s = time.perf_counter() - t
        u, iters, hist = s.solve_pcg()
        for _ in range(warmup):
            s.time_solve_pcg(1)
        sec = s.time_solve_pcg(reps) / reps
        s.close()
        kind = "reference"
        what = (f"the reference's own solve_pCG (oracle/_ref = unmodified paralab/Saena sources, -Ofast, 1 MPI rank) "
                f"on 3D Poisson {mx - 2}^3 = {n} unknowns (laplacian3D mx={mx}), same options; {reps} solves, "
                f"{iters} iterations each; host setup {setup_s:.1f} s not timed")
    else:
        from oracle.oracle import Oracle
        from saena_b200.sa_setup import build_hierarchy, poisson3d_coo, poisson3d_rhs
        h = build_hierarchy(*poisson3d_coo(mx - 2), device="cpu")
        o, rhs = Oracle(h), poisson3d_rhs(mx - 2)
        u, iters, hist = o.solve_pcg(rhs, **OPTS)
        t = time.perf_counter()
        for _ in range(reps):
            o.solve_pcg(rhs, **OPTS)
        sec = (time.perf_counter() - t) / reps
        kind = "port"
        what = (f"C restatement of the reference solve (oracle/saena_oracle.c) on 3D Poisson {mx - 2}^3 = {n} unknowns, "
                f"same options; {reps} solves, {iters} iterations each")
    return dict(value=n / sec / 1e6, unit=UNIT, cores=1, kind=kind, sample=what), sec, iters, n


def run_reference_arm(args, rank):
    if rank != 0:
        return
    base, sec, iters, n = cpu_reference_solve(max(args.steps, 1), args.warmup, arm=True)
    # the trend with the problem size (one more, smaller sample; SAENA_BENCH_CPU_SWEEP=0 skips it): the CPU's
    # unknowns/s is nearly flat in n, so the sample stands for the 256^3 workload it cannot set up in a bounded run
    sweep = [{"unknowns": n, "value": base["value"], "ms_per_solve": sec * 1e3, "iterations": iters}]
    if base.get("cores", 1) > 1 and os.environ.get("SAENA_BENCH_CPU_SWEEP", "1") != "0" and n > 64 ** 3:
        try:
            b2, s2, i2, n2 = cpu_reference_solve_multirank(3, 1, base["cores"], 66)
            sweep.insert(0, {"unknowns": n2, "value": b2["value"], "ms_per_solve": s2 * 1e3, "iterations": i2})
        except Exception as e:
            log(f"[reference arm] size sweep point failed: {e!r}")
    base["size_sweep"] = sweep
    line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"3D 7-point Poisson AMG-PCG, bounded sample {round(n ** (1 / 3))}^3 unknowns of the "
                                   f"256^3 workload, {base['cores']} host core(s)",
                       "same_config_as_gpu_arm": False,
                       "why_a_sample": "the reference's own host setup for 256^3 takes the better part of an hour; "
                                       "throughput in unknowns/s is compared, see cpu_baseline.size_sweep for its trend in n",
                       "options": "data/options006_poisson.xml values"},
            "iterations": iters, "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def autotune_mapping_collective(ctx, hier, world, reps=10, min_gain=0.03):
    """The setup-time row-mapping autotuner on several ranks (opt-in A/B, SAENA_BENCH_AUTOTUNE_MAP): every timed
    application is an exchange, so all ranks walk the same candidates -- rank 0's current mapping of the operator
    and its neighbours -- and decide on the slowest rank's time (all-reduce MAX): one mapping per operator, the same
    on every rank.  Returns [(level, kind, before on this rank, after, ms_before, ms_after)]."""
    import torch
    import torch.distributed as dist

    def agree(vals, op):
        t = torch.tensor(vals, dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=op)
        return t.tolist()

    out = []
    for l, lv in enumerate(hier.levels):
        for kind, op in ((0, lv.A), (1, lv.P), (2, lv.R)):
            if op is None:
                continue
            mine = ctx.get_mapping(l, kind) if op.M else 0
            lead = torch.tensor([mine], dtype=torch.int64, device="cuda")
            dist.broadcast(lead, 0)
            cur = int(lead.item())
            rows = int(agree([float(op.M)], dist.ReduceOp.MIN)[0])
            if cur <= 0 or cur >= 100 or rows == 0:
                continue            # sliced / streaming choices and levels some rank holds nothing of: left alone
            cands = [cur] + sorted({c for c in (cur // 4, cur // 2, cur * 2, cur * 4) if 1 <= c <= 256 and c != cur})
            times = []
            for c in cands:
                ctx.set_mapping(l, kind, c)
                times.append(ctx.time_matvec(l, kind, reps, flush_l2=ctx.operator_bytes(l, kind) < 300e6))
            times = agree(times, dist.ReduceOp.MAX)
            k = int(np.argmin(times))
            if times[k] > (1.0 - min_gain) * times[0]:
                k = 0
            ctx.set_mapping(l, kind, cands[k])
            out.append((l, kind, mine, cands[k], times[0], times[k]))
    return out


def verify_properties(ctx, hier, rank, world):
    """SAENA_BENCH_VERIFY=1 (untimed, collective): size-independent properties of the uploaded, row-partitioned
    hierarchy -- what stands in for the oracle at sizes it cannot run (tests/full_size_properties.py is the one-rank
    version): <A x, y> = <x, A y> and <R x, e> = <x, P e> on every level, dots summed over the ranks."""
    import torch
    import torch.distributed as dist
    from saena_b200.hierarchy import KIND_A, KIND_P, KIND_R

    def gsum(*vals):
        t = torch.tensor(list(vals), dtype=torch.float64, device="cuda" if torch.cuda.is_available() else "cpu")
        if world > 1:
            dist.all_reduce(t)
        return t.tolist()

    out = {}
    for l, lv in enumerate(hier.levels):
        rng = np.random.default_rng(1000 * l + rank)
        x, y = rng.uniform(-1, 1, lv.A.M), rng.uniform(-1, 1, lv.A.M)
        ax, ay = ctx.matvec(l, KIND_A, x), ctx.matvec(l, KIND_A, y)
        axy, xay, nax, ny = gsum(float(ax @ y), float(x @ ay), float(ax @ ax), float(y @ y))
        out[f"L{l}.symmetry"] = abs(axy - xay) / max(np.sqrt(nax * ny), 1e-300)
        if lv.P is not None:
            e = rng.uniform(-1, 1, lv.P.n_local_cols)
            rx, pe = ctx.matvec(l, KIND_R, x), ctx.matvec(l, KIND_P, e)
            rxe, xpe, nrx, ne = gsum(float(rx @ e), float(x @ pe), float(rx @ rx), float(e @ e))
            out[f"L{l}.adjoint"] = abs(rxe - xpe) / max(np.sqrt(nrx * ne), 1e-300)
    out["worst"] = max(out.values())
    out["ok"] = bool(out["worst"] <= 1e-6 if any(not lv.A.use_double for lv in hier.levels) and world > 1 else out["worst"] <= 1e-12)
    return out


def nvlink_counters(device: int):
    """cumulative NVLink data counters of one GPU, summed over its links, in KiB: (tx, rx); None if unavailable"""
    import re
    try:
        out = subprocess.run(["nvidia-smi", "nvlink", "-gt", "d", "-i", str(device)], capture_output=True, text=True,
                             timeout=20).stdout
        tx = sum(int(x) for x in re.findall(r"Data Tx:\s*(\d+)\s*KiB", out))
        rx = sum(int(x) for x in re.findall(r"Data Rx:\s*(\d+)\s*KiB", out))
        return (tx, rx) if ("Data Tx" in out) else None
    except Exception:
        return None


def dump_outputs(out_dir: str, u_dev, iters: int, hist, row_offset: int, n_global: int, rank: int, world: int):
    """--dump-outputs: u of the last solve at a fixed seeded sample of global rows (all rows when there are at most
    DUMP_SAMPLE), gathered from the ranks' row blocks; rank 0 writes the files."""
    import torch
    if n_global > DUMP_SAMPLE:
        idx = np.sort(np.random.default_rng(0).choice(n_global, DUMP_SAMPLE, replace=False))
    else:
        idx = np.arange(n_global)
    lo, hi = (int(x) for x in np.searchsorted(idx, [row_offset, row_offset + u_dev.numel()]))
    mine = u_dev[torch.from_numpy(idx[lo:hi] - row_offset).to(u_dev.device)].cpu().numpy()
    parts = [(lo, mine)]
    if world > 1:
        import torch.distributed as dist
        parts = [None] * world
        dist.all_gather_object(parts, (lo, mine))
    if rank != 0:
        return
    u = np.full(len(idx), np.nan)
    for start, vals in parts:
        u[start:start + len(vals)] = vals
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("u", u), ("u_index", idx), ("residual_history", hist), ("iterations", [iters])):
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


# ------------------------------------------------------------------------------------------------
def main():
    def at_least_one(s):
        if int(s) < 1:
            raise argparse.ArgumentTypeError(f"must be at least 1, got {s}")
        return int(s)

    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=at_least_one, default=10, help="timed solves")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", "--size", dest="n", type=int, default=int(os.environ.get("SAENA_BENCH_N", 256)),
                    help="unknowns per dimension (256 = BASELINE.json configs[1]); under torchrun write --size (its own "
                         "parser reads a bare --n as an abbreviation of --nnodes / --nproc-per-node)")
    ap.add_argument("--workload", default="poisson3d", choices=["poisson3d", "unstructured2d"],
                    help="poisson3d = BASELINE.json configs[1] (the bench line); unstructured2d = configs[4]'s synthetic "
                         "2-D Helmholtz-like matrix with irregular rows (same solve, same JSON keys, its own metric name)")
    ap.add_argument("--g", type=int, default=2828, help="unstructured2d: g*g nodes (2828^2 = 8.0 M rows)")
    ap.add_argument("--row-lengths", default="6,8,10", help="unstructured2d: entries per row drawn from these "
                                                            "(donor P2: 6,8,10; P8: 24,32,40)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dist-setup", default="auto", choices=["auto", "on", "off"],
                    help="N>1: build the hierarchy row-partitioned over the ranks (saena_b200/sa_setup_dist.py) instead of "
                         "redundantly on every GPU; auto = on when the problem is beyond one GPU's setup (n > 320: "
                         "BASELINE.json configs[2], 512^3 on 8 GPUs)")
    ap.add_argument("--agglomerate-below", type=int, default=10_000,
                    help="N>1: levels with fewer global rows live on rank 0 (the reference's shrink-to-one-rank)")
    ap.add_argument("--rebalance-above", type=float, default=float(os.environ.get("SAENA_BENCH_REBALANCE", 1.10)),
                    help="N>1: a coarse level whose aligned row blocks leave one rank above this multiple of the mean "
                         "nnz is split by its own nnz balance (0: never)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed solves, write what the last one returned to DIR/<name>.npy (see the top of "
                         "this file)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU solve (--impl b200)")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    if args.warmup < 3:
        log("warm-up raised to 3 (timing rules)")
        args.warmup = 3

    import torch
    import torch.distributed as dist
    from saena_b200 import native
    from saena_b200.distributed import all_ranks_ok, exchange_nccl_id, setup_p2p_halo
    from saena_b200.hierarchy import KIND_A, KIND_P, KIND_R
    from saena_b200.sa_setup import (build_device_hierarchy, poisson3d_coo, poisson3d_rhs, unstructured2d_coo,
                                     unstructured2d_rhs)

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the solve path has no CPU fallback")
    torch.cuda.set_device(local)
    nccl_id = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        nccl_id = exchange_nccl_id(native.nccl_unique_id)

    # ---- setup (untimed): hierarchy of the reference's shape, built on this rank's GPU
    n = args.n
    t0 = time.perf_counter()
    dist_setup = world > 1 and (args.dist_setup == "on" or
                                (args.dist_setup == "auto" and args.workload == "poisson3d" and n > 320))
    verbose = rank == 0 and bool(os.environ.get("SAENA_BENCH_VERBOSE"))
    agg_sweep = []
    if args.workload == "poisson3d" and n > 320 and not dist_setup:
        # 256^3 already takes 17 GB of operators and ~100 GB of setup buffers on one device (DESIGN.md section 6)
        raise SystemExit(f"bench.py: a {n}^3 hierarchy cannot be built on one device; run on 8 GPUs (torchrun, "
                         f"--gpus 8) where the setup is row-partitioned (--dist-setup)")
    if dist_setup:
        # every rank generates and coarsens only its own rows; what comes out is already this rank's share
        from saena_b200 import sa_setup_dist as sd
        comm = sd.Comm(torch.device("cuda", local))
        if args.workload == "poisson3d":
            N = n ** 3
            A0 = sd.poisson3d_dcsr(n, comm)
        else:
            # every rank generates the whole synthetic matrix on the host (numpy, seeded) and keeps its rows
            lengths = tuple(int(x) for x in args.row_lengths.split(","))
            weights = (16, 48, 20) if len(lengths) == 3 else (1,) * len(lengths)
            N, row, col, val = unstructured2d_coo(args.g, row_lengths=lengths, weights=weights)
            A0 = sd.coo_dcsr(N, row, col, val, comm)
            del row, col, val
        hier, summary = sd.build_distributed_hierarchy(A0, agglomerate_below=args.agglomerate_below,
                                                       rebalance_above=args.rebalance_above, verbose=verbose, comm=comm)
        del A0
        if rank == 0:
            log(f"[setup] hierarchy built on {world} ranks in {time.perf_counter() - t0:.1f}s\n" + "\n".join(summary))
    else:
        if args.workload == "poisson3d":
            N, row, col, val = poisson3d_coo(n)
        else:
            lengths = tuple(int(x) for x in args.row_lengths.split(","))
            weights = (16, 48, 20) if len(lengths) == 3 else (1,) * len(lengths)   # the donors' 16:48:20 proportions
            N, row, col, val = unstructured2d_coo(args.g, row_lengths=lengths, weights=weights)
        dh = build_device_hierarchy(N, row, col, val, verbose=verbose)
        del row, col, val
        if rank == 0:
            log(f"[setup] hierarchy built in {time.perf_counter() - t0:.1f}s\n{dh.summary()}")
        hier = dh.to_rank(rank, world, agglomerate_below=args.agglomerate_below if world > 1 else 0,
                          rebalance_above=args.rebalance_above if world > 1 else 0.0)
        agg_sweep = [int(x) for x in filter(None, os.environ.get("SAENA_BENCH_AGG_SWEEP", "").split(","))] if world > 1 else []
        if not agg_sweep:
            del dh
    import gc
    gc.collect()                 # the setup's tensors go back to the driver before the library allocates
    torch.cuda.empty_cache()
    ctx = native.Context(device=local, rank=rank, nranks=world, nccl_id=nccl_id)
    ctx.upload_hierarchy(hier)
    # Halo transport (N > 1).  Default: NVLink peer memory, fused kernel, per-operator choice fused / separate launches
    # measured at setup.  Every step below is agreed across the ranks: if the peer-memory exchange cannot be set up, or
    # its autotune / trial solve fails or times out on ANY rank (csrc/halo_sync.cuh bounds every wait), ALL ranks switch
    # to the NCCL transport together and the line says so ("halo_fallback").
    halo_transport, halo_fallback = "none", None

    def fall_back_to_nccl(why: str):
        nonlocal halo_transport, halo_fallback
        log(f"[rank {rank}] peer-memory halo -> NCCL: {why}")
        try:
            ctx.clear_fault()
            ctx.p2p_enable(0)
        except native.NativeError as e:
            log(f"[rank {rank}] could not switch the transport: {e}")
        halo_transport = "nccl"
        halo_fallback = why

    p2p_up = world > 1 and os.environ.get("SAENA_B200_HALO", "p2p") == "p2p" and setup_p2p_halo(ctx, log)
    # every operator's row mapping chosen by measurement at setup (saena_b200_autotune_mapping, collective; untimed like
    # the rest of the setup -- the adaptor does the same after its upload); SAENA_BENCH_MAPPING_AUTOTUNE=0: nnz/row rule only
    mapping_tuned = None
    if os.environ.get("SAENA_BENCH_MAPPING_AUTOTUNE", "1") != "0":
        before = {(l, k): ctx.get_mapping(l, k) for l in range(len(hier.levels)) for k in (KIND_A, KIND_P, KIND_R)}
        for attempt in (0, 1):
            ok, why = True, "on another rank"
            try:
                ctx.autotune_mapping_native(10, 0.03)
            except native.NativeError as e:
                ok, why = False, f"mapping autotune: {e}"
            if world == 1 and not ok:
                raise SystemExit(f"bench.py: {why}")
            if world == 1 or all_ranks_ok(ok):
                break
            if attempt == 1 or not p2p_up:
                raise SystemExit(f"bench.py: mapping autotune failed over NCCL too ({why})")
            fall_back_to_nccl(why)   # its timed applications are the first exchanges over peer memory
            p2p_up = False
        mapping_tuned = [{"level": l, "kind": "APR"[k], "rule": b, "measured": ctx.get_mapping(l, k)}
                         for (l, k), b in before.items() if b != 0 and ctx.get_mapping(l, k) != b]
    if world > 1:
        if halo_fallback is None:
            halo_transport = "nccl"
        if p2p_up:
            if os.environ.get("SAENA_B200_HALO_FUSED", "1") != "0":
                halo_transport = ("nvlink peer memory, fused: pack + peer stores + interior rows + ghost rows "
                                  "in one kernel per operator application")
                if os.environ.get("SAENA_B200_HALO_AUTOTUNE", "1") != "0":
                    ok, why = True, "on another rank"
                    try:
                        ctx.autotune_halo(10)   # per operator: fused kernel or separate launches, whichever measured faster
                    except native.NativeError as e:
                        ok, why = False, f"autotune: {e}"
                    if all_ranks_ok(ok):
                        halo_transport += "; per-operator choice fused / separate launches measured at setup"
                    else:
                        fall_back_to_nccl(why)
            else:
                ctx.p2p_enable(1)
                halo_transport = "nvlink peer memory, separate launches (pack kernel stores into the neighbour's landing area)"
    for spec in filter(None, os.environ.get("SAENA_BENCH_MAP", "").split(",")):   # tuning: "level:kind:mapping"
        lvl, kind, mp = (int(x) for x in spec.split(":"))
        ctx.set_mapping(lvl, kind, mp)
    if rank == 0:
        log(f"[setup] uploaded in {time.perf_counter() - t0:.1f}s total")
    l0 = hier.levels[0].A
    if dist_setup and args.workload == "poisson3d":
        rhs_host = torch.from_numpy(sd.poisson3d_rhs_rows(n, l0.row_offset, l0.row_offset + l0.M)).pin_memory()
    else:
        rhs_full = poisson3d_rhs(n) if args.workload == "poisson3d" else unstructured2d_rhs(N)
        rhs_host = torch.from_numpy(rhs_full[l0.row_offset:l0.row_offset + l0.M].copy()).pin_memory()
        del rhs_full
    u_host = torch.empty(l0.M, dtype=torch.float64).pin_memory()
    rhs_dev = rhs_host.cuda()
    u_dev = torch.zeros(l0.M, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    if world > 1 and halo_transport != "nccl":
        # trial solve over the chosen transport before anything is timed
        ok, why = True, "on another rank"
        try:
            ctx.solve_pcg_dev(rhs_dev.data_ptr(), u_dev.data_ptr(), **OPTS)
        except native.NativeError as e:
            ok, why = False, f"trial solve: {e}"
        if not all_ranks_ok(ok):
            fall_back_to_nccl(why)

    # ---- warm-up (the clock sampler starts here: nvidia-smi needs ~0.2 s before its first sample,
    #      longer than a multi-GPU timed region; every sample is taken under the same solve load)
    def timed_region():
        it_ = hist_ = None
        with ClockSampler(local) as clocks_:
            for _ in range(args.warmup):
                it_, hist_ = ctx.solve_pcg_dev(rhs_dev.data_ptr(), u_dev.data_ptr(), **OPTS)
            # ---- timed: K solves, inputs resident in HBM, CUDA events on the library's compute stream
            l0_ = ctx.launch_count()
            barrier()
            ctx.timer_start()
            for _ in range(args.steps):
                it_, hist_ = ctx.solve_pcg_dev(rhs_dev.data_ptr(), u_dev.data_ptr(), **OPTS)
            ms_ = ctx.timer_stop()
            barrier()
        return it_, hist_, ms_, l0_, clocks_

    ok, why = True, "on another rank"
    try:
        iters, hist, ms_total, launches0, clocks = timed_region()
    except native.NativeError as e:
        if world == 1:
            raise
        ok, why = False, f"timed region: {e}"
    if world > 1 and not all_ranks_ok(ok):
        if halo_transport == "nccl":
            raise SystemExit(f"bench.py: the solve failed over the NCCL transport too ({why})")
        fall_back_to_nccl(why)
        iters, hist, ms_total, launches0, clocks = timed_region()
    launches = ctx.launch_count() - launches0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, u_dev, iters, hist, l0.row_offset, N, rank, world)
    ms_step = max_over_ranks(ms_total / args.steps)
    clk = clocks.summary()
    graph_info = {"vcycles_replayed_from_graph": ctx.graph_replays()}
    map_tune = None
    if os.environ.get("SAENA_BENCH_AUTOTUNE_MAP"):
        # in-run A/B (not the bench value, off by default until measured): per-operator row mapping picked by timing the
        # neighbours of the heuristic's choice, then the same solves again.  SAENA_BENCH_AUTOTUNE_MAP=keep leaves the tuned
        # mappings in place for the per-level tables below; anything else restores the heuristic's.
        table = ctx.autotune_mapping(10) if world == 1 else autotune_mapping_collective(ctx, hier, world)
        for _ in range(2):
            ctx.solve_pcg_dev(rhs_dev.data_ptr(), u_dev.data_ptr(), **OPTS)
        barrier()
        ctx.timer_start()
        for _ in range(args.steps):
            ctx.solve_pcg_dev(rhs_dev.data_ptr(), u_dev.data_ptr(), **OPTS)
        tuned_ms = max_over_ranks(ctx.timer_stop() / args.steps)
        barrier()
        map_tune = {"ms_per_step_heuristic": ms_step, "ms_per_step_autotuned": tuned_ms,
                    "changed": [dict(zip(("level", "kind", "before", "after", "ms_before", "ms_after"), (l, "APR"[k], a, b, t0, t1)))
                                for l, k, a, b, t0, t1 in table if a != b]}
        if os.environ["SAENA_BENCH_AUTOTUNE_MAP"] != "keep":
            for l, k, a, b, _, _ in table:
                ctx.set_mapping(l, k, a)
    # (opt-in since round 2, SAENA_BENCH_AB=1: the default run carries the bench value and the per-level tables only)
    if world > 1 and ctx.graph_replays() > 0 and os.environ.get("SAENA_BENCH_AB") and not os.environ.get("SAENA_BENCH_NO_AB"):
        # A/B on the same uploaded hierarchy: the same solves with eager launches (not the bench value)
        ctx.set_graphs(False)
        ctx.solve_pcg_dev(rhs_dev.data_ptr(), u_dev.data_ptr(), **OPTS)
        barrier()
        ctx.timer_start()
        for _ in range(args.steps):
            ctx.solve_pcg_dev(rhs_dev.data_ptr(), u_dev.data_ptr(), **OPTS)
        eager_ms = ctx.timer_stop()
        barrier()
        graph_info["eager_ms_per_step"] = max_over_ranks(eager_ms / args.steps)
        ctx.set_graphs(True)
        if halo_transport.startswith("nvlink peer memory, fused"):
            # the autotuner's per-operator choices (rank 0's timings), then the same solves with every
            # operator on the fused kernel / on the separate launches (pack kernel, memory-op flags, boundary kernel)
            graph_info["halo_autotune"] = [
                dict(zip(("level", "kind", "fused", "ms_fused", "ms_separate"), (l, "APR"[k], *ctx.halo_choice(l, k))))
                for l in range(len(hier.levels)) for k in (KIND_A, KIND_P, KIND_R) if ctx.halo_choice(l, k)[1] > 0]
            for label, mode in (("all_fused_ms_per_step", 2), ("all_separate_ms_per_step", 1)):
                ctx.p2p_enable(mode)
                for _ in range(2):
                    ctx.solve_pcg_dev(rhs_dev.data_ptr(), u_dev.data_ptr(), **OPTS)
                barrier()
                ctx.timer_start()
                for _ in range(args.steps):
                    ctx.solve_pcg_dev(rhs_dev.data_ptr(), u_dev.data_ptr(), **OPTS)
                ab_ms = ctx.timer_stop()
                barrier()
                graph_info[label] = max_over_ranks(ab_ms / args.steps)
            ctx.p2p_enable(2)
            if "per-operator" in halo_transport:
                ctx.autotune_halo(10)

    # ---- e2e: host buffers through the reference-facing entry point, copies inside the timed region
    diag_error = None
    e2e_ms = e2e_pageable_ms = None
    try:
        ctx._ck(ctx._L.saena_b200_solve_pcg(ctx._h, rhs_host.data_ptr(), u_host.data_ptr(), OPTS["max_iter"], OPTS["tol"],
                                            1, OPTS["pre"], OPTS["post"], *_iters_hist_args()))
        barrier()
        t = time.perf_counter()
        for _ in range(args.steps):
            ctx._ck(ctx._L.saena_b200_solve_pcg(ctx._h, rhs_host.data_ptr(), u_host.data_ptr(), OPTS["max_iter"],
                                                OPTS["tol"], 1, OPTS["pre"], OPTS["post"], *_iters_hist_args()))
        barrier()
        e2e_ms = max_over_ranks((time.perf_counter() - t) * 1e3 / args.steps)
        # the same with the caller's PAGEABLE buffers: what the drop-in receives from saena_aligned_alloc'ed vectors
        # (adaptor/saena_b200_adaptor.cpp:run_solver); not the e2e value, reported beside it
        rhs_pg, u_pg = np.array(rhs_host.numpy(), copy=True), np.empty(l0.M)
        barrier()
        t = time.perf_counter()
        for _ in range(args.steps):
            ctx._ck(ctx._L.saena_b200_solve_pcg(ctx._h, rhs_pg.ctypes.data, u_pg.ctypes.data, OPTS["max_iter"],
                                                OPTS["tol"], 1, OPTS["pre"], OPTS["post"], *_iters_hist_args()))
        barrier()
        e2e_pageable_ms = max_over_ranks((time.perf_counter() - t) * 1e3 / args.steps)
        del rhs_pg, u_pg
    except native.NativeError as e:
        diag_error = f"e2e: {e}"
        log(f"[rank {rank}] {diag_error}")

    # ---- check the answer we timed: the recurrence's last <r,r>, and ||rhs - A u|| / ||rhs|| recomputed from the u the
    #      host-buffer solve returned (one more operator application, untimed; collective on several ranks)
    rel_res = float(hist[-1] / hist[0])
    true_rel_res = None
    try:
        au = ctx.matvec(0, KIND_A, u_host.numpy())
        sums = torch.tensor([float(np.sum((rhs_host.numpy() - au) ** 2)), float(np.sum(rhs_host.numpy() ** 2))],
                            dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(sums)
        true_rel_res = float(torch.sqrt(sums[0] / sums[1]).item())
        del au
    except Exception as e:   # the bench line must still come out
        log(f"[verify] recomputing the residual failed: {e!r}")

    # ---- per-level kernel table + roofline of the dominant kernel (CUDA events per launch)
    peak, peak_src = measured_peaks()
    levels_tbl, dominant = [], None
    try:
        for l, lv in enumerate(hier.levels):
            if lv.A.M == 0:
                continue
            a_bytes = ctx.operator_bytes(l, KIND_A)
            # first Chebyshev sweep (SURVEY 8d): 12 nnz + M*(4 + 8*[u gathered, rhs, inv_diag, d out, u out]) = SpMV + 24 M
            sweep_bytes = a_bytes + 24 * lv.A.M
            big = a_bytes > 300e6   # larger than L2: no flush needed; smaller levels are flushed between launches
            ms_mv = ctx.time_matvec(l, KIND_A, 20, flush_l2=not big)
            ms_sw = ctx.time_smooth_sweep(l, "chebyshev", 20, flush_l2=not big)
            ent = {"level": l, "rows": lv.A.M, "nnz": lv.A.nnz, "mapping": ctx.get_mapping(l, KIND_A), "spmv_ms": ms_mv, "spmv_GBs": a_bytes / ms_mv / 1e6,
                   "cheb_sweep_ms": ms_sw, "cheb_sweep_GBs": sweep_bytes / ms_sw / 1e6,
                   "frac_of_peak": sweep_bytes / ms_sw / 1e6 / peak}
            if lv.P is not None and lv.P.M:
                ent["P_ms"] = ctx.time_matvec(l, KIND_P, 20, flush_l2=not big)
                ent["R_ms"] = ctx.time_matvec(l, KIND_R, 20, flush_l2=not big)
                ent["P_mapping"], ent["R_mapping"] = ctx.get_mapping(l, KIND_P), ctx.get_mapping(l, KIND_R)
            levels_tbl.append(ent)
            # share of a V-cycle: 5 fused sweeps + residual ~ 6 passes
            if dominant is None or ms_sw * 5 > dominant[0]:
                dominant = (ms_sw * 5, l, sweep_bytes, ms_sw)
    except native.NativeError as e:
        diag_error = diag_error or f"per-level table: {e}"
        log(f"[rank {rank}] per-level table: {e}")
    have_dominant = dominant is not None
    if not have_dominant:   # nothing could be timed: the roofline object says so
        dominant = (0.0, 0, 0, 1.0)
    _, dl, dbytes, dms = dominant
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")   # dram bytes per launch from the committed ncu capture
    if os.path.exists(tp) and world == 1:
        traffic = json.load(open(tp)).get(f"n{n}_level{dl}_cheb_sweep") if args.workload == "poisson3d" else None
    roofline = {"bound": "hbm", "achieved": dbytes / dms / 1e6, "peak": peak, "unit": "GB/s",
                "frac": dbytes / dms / 1e6 / peak, "traffic": traffic,
                "kernel": f"fused Chebyshev sweep (SpMV + update epilogue) on level {dl}", "peak_source": peak_src,
                "algorithmic_bytes_per_launch": dbytes, "launch_ms": dms}
    if not have_dominant:
        roofline.update(achieved=None, frac=None, launch_ms=None, kernel="not measured: " + str(diag_error))

    # whole-solve algorithmic bytes (SURVEY 8d formulas on the uploaded sizes) -> effective bandwidth
    pre, post = OPTS["pre"], OPTS["post"]
    vcycle_bytes = 0
    for l, lv in enumerate(hier.levels[:-1]):
        M = lv.A.M
        a = ctx.operator_bytes(l, KIND_A)
        vcycle_bytes += 32 * M                              # first pre-sweep from a zero iterate: rhs, inv_diag in; d, u out
        vcycle_bytes += (pre - 1 + post) * (a + 32 * M)      # fused sweeps: SpMV + rhs, inv_diag, d in; d, u out
        vcycle_bytes += a + 8 * M                            # residual
        vcycle_bytes += ctx.operator_bytes(l, KIND_R)        # restriction
        vcycle_bytes += ctx.operator_bytes(l, KIND_P) + 8 * M  # prolongation + correction (u read)
    M0, a0 = hier.levels[0].A.M, ctx.operator_bytes(0, KIND_A)
    krylov_bytes = a0 + 16 * M0 + 48 * M0 + 16 * M0 + 24 * M0  # h = A p, <p,h>, update + <r,r>, <r,rho>, p update
    solve_bytes = (iters + 1) * vcycle_bytes + iters * krylov_bytes
    solve_gbs = solve_bytes / ms_step / 1e6

    # ---- what each level costs inside a solve: V-cycles entered at level l, consecutive differences
    vcycle_levels, halo = None, None
    try:
        if diag_error is None:
            vc = [max_over_ranks(ctx.time_vcycle(l, OPTS["smoother"], OPTS["pre"], OPTS["post"], 10))
                  for l in range(len(hier.levels))]
            vcycle_levels = {"unit": "ms per V-cycle, eager launches, max over ranks",
                             "entered_at_level": vc,
                             "level_share": [vc[l] - (vc[l + 1] if l + 1 < len(vc) else 0.0) for l in range(len(vc))]}
        if world > 1 and diag_error is None:
            full_ms, local_ms, halo_ms = ctx.time_matvec_parts(0, KIND_A, 20)
            full_ms, local_ms, halo_ms = max_over_ranks(full_ms), max_over_ranks(local_ms), max_over_ranks(halo_ms)
            halo = {"level": 0, "spmv_full_ms": full_ms, "spmv_local_only_ms": local_ms, "pack_exchange_only_ms": halo_ms,
                    "hidden_frac": max(0.0, min(1.0, 1.0 - (full_ms - local_ms) / halo_ms)) if halo_ms > 0 else None,
                    "transport": halo_transport,
                    "ghost_values_per_rank": int(hier.levels[0].A.col_remote_size),
                    "ghost_dtype": "f64" if hier.levels[0].A.use_double else "f32 (float_level 0)"}
        if world > 1 and diag_error is None and os.environ.get("SAENA_BENCH_NVLINK"):
            # NVLink evidence for the fused compute + exchange kernel: the GPU's own link counters around 500
            # applications of the level-0 operator (every application is one exchange); expected = what the plan sends
            apps = 500
            barrier()
            c0 = nvlink_counters(local)
            ctx.time_matvec(0, KIND_A, apps)
            barrier()
            c1 = nvlink_counters(local)
            sent = int(hier.levels[0].A.vIndexSize) * 8   # doubles on the wire (rounded through float by the sender)
            if c0 and c1:
                halo["nvlink_rank0"] = {"applications": apps, "tx_KiB": c1[0] - c0[0], "rx_KiB": c1[1] - c0[1],
                                        "tx_bytes_per_application": (c1[0] - c0[0]) * 1024 / apps,
                                        "rx_bytes_per_application": (c1[1] - c0[1]) * 1024 / apps,
                                        "payload_bytes_sent_per_application_by_plan": sent,
                                        "source": "nvidia-smi nvlink -gt d, summed over the links of this rank's GPU"}
    except native.NativeError as e:
        diag_error = diag_error or f"per-level V-cycle / halo timing: {e}"
        log(f"[rank {rank}] per-level V-cycle / halo timing: {e}")

    total_unknowns = int(N)
    if args.workload == "poisson3d":
        metric = METRIC
        workload = (f"3D 7-point Poisson {n}^3 = {total_unknowns} unknowns, AMG-PCG to 1e-8 "
                    + ("(BASELINE.json configs[2])" if n == 512 else "(BASELINE.json configs[1] at n=256)"))
    else:
        metric = "AMG-PCG solve throughput, synthetic 2D Helmholtz-like unstructured matrix, rel. residual 1e-8 (unknowns solved per second)"
        workload = (f"synthetic 2D Helmholtz-like matrix, unstructured-mesh pattern, {args.g}^2 = {total_unknowns} rows, "
                    f"row lengths drawn from {args.row_lengths} (BASELINE.json configs[4] shape, seed 2024), AMG-PCG to 1e-8")
    line = {"metric": metric, "value": total_unknowns / (ms_step / 1e3) / 1e6, "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload,
                       "options": "options006_poisson.xml: chebyshev 3+3, conn_str 0.2, float_level 0, max_iter 50",
                       "levels": len(hier.levels),
                       "setup": ("row-partitioned over the ranks (saena_b200/sa_setup_dist.py), untimed" if dist_setup else
                                 "on one device (saena_b200/sa_setup.py), every rank keeps its share, untimed"),
                       "partition": f"{world} row block(s), nnz-balanced" + (
                           f"; coarse levels follow the level above, re-split when a rank exceeds "
                           f"{args.rebalance_above:g}x the mean nnz; levels under {args.agglomerate_below} rows on rank 0"
                           if world > 1 else ""),
                       "l2": "inputs larger than L2 (level-0/1 operators are GBs); per-kernel timings of "
                             "L2-sized levels flush L2 between launches"},
            "solve_s": ms_step / 1e3, "iterations": iters, "rel_residual": rel_res, "true_rel_residual": true_rel_res,
            "solve_algorithmic_GB": solve_bytes / 1e9, "solve_effective_GBs": solve_gbs,
            "solve_frac_of_hbm_peak": solve_gbs / peak,
            "e2e": {"value": total_unknowns / (e2e_ms / 1e3) / 1e6 if e2e_ms else None, "unit": UNIT, "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": 8 * total_unknowns, "d2h_bytes_per_step": 8 * total_unknowns,
                    "timer": "wall clock between device synchronisations (host copies included)",
                    "buffers": "pinned host memory",
                    "pageable_ms_per_step": e2e_pageable_ms,
                    "pageable_value": total_unknowns / (e2e_pageable_ms / 1e3) / 1e6 if e2e_pageable_ms else None},
            "gpu_launches": int(launches), "vcycle_graph": graph_info, "vcycle_levels": vcycle_levels, "clocks": clk, "roofline": roofline,
            "levels": levels_tbl}
    if halo is not None:
        line["halo_overlap"] = halo
    line["row_mappings_changed_by_setup_autotune"] = mapping_tuned
    if world > 1:
        line["halo_transport"] = halo_transport
        line["halo_fallback"] = halo_fallback
    if map_tune is not None:
        line["mapping_autotune"] = map_tune
    if os.environ.get("SAENA_BENCH_VERIFY"):
        try:
            line["verify"] = verify_properties(ctx, hier, rank, world)
        except Exception as e:
            line["verify"] = {"ok": False, "error": repr(e)}
    if rank == 0 and world == 1 and not args.no_cpu_baseline and args.workload == "poisson3d":
        try:
            line["cpu_baseline"], _, cpu_iters, _ = cpu_reference_solve(5)
            line["cpu_baseline"]["iterations"] = cpu_iters
        except Exception as e:  # the bench line must still come out
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 1, "kind": "unavailable", "sample": repr(e)}
    # tuning only (SAENA_BENCH_AGG_SWEEP="2000,50000"): the same solves with other agglomeration thresholds
    for thr in agg_sweep:
        hier2 = dh.to_rank(rank, world, agglomerate_below=thr, rebalance_above=args.rebalance_above)
        barrier()
        ctx.upload_hierarchy(hier2)
        if halo_transport != "nccl":
            if not setup_p2p_halo(ctx, log):
                raise SystemExit("bench.py: agglomeration sweep: the peer-memory halo could not be set up again")
            if "per-operator" in halo_transport:
                ctx.autotune_halo(10)
        for _ in range(3):
            ctx.solve_pcg_dev(rhs_dev.data_ptr(), u_dev.data_ptr(), **OPTS)
        barrier()
        ctx.timer_start()
        for _ in range(args.steps):
            it2, _ = ctx.solve_pcg_dev(rhs_dev.data_ptr(), u_dev.data_ptr(), **OPTS)
        ms2 = max_over_ranks(ctx.timer_stop() / args.steps)
        barrier()
        line.setdefault("agglomerate_sweep", []).append({"agglomerate_below": thr, "ms_per_step": ms2, "iterations": it2})
    if diag_error is not None:
        # a diagnostic after the timed region failed on this rank: the ranks may no longer be in step, so the line goes
        # out first and nobody waits for anybody (a clean shutdown would synchronise with a stream that may never drain)
        line["diagnostics_error"] = diag_error
        if rank == 0:
            print(json.dumps(line), flush=True)
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()   # nobody unmaps a peer's arena while that peer may still write into it
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def _iters_hist_args():
    import ctypes
    it, n = ctypes.c_int(0), ctypes.c_int(0)
    hist = (ctypes.c_double * 64)()
    _iters_hist_args.keep = (it, n, hist)
    return ctypes.byref(it), hist, 64, ctypes.byref(n)


if __name__ == "__main__":
    main()
