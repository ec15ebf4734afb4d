"""bench.py's reference arm (CPU only) prints one JSON line with the contract's keys."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


import pytest


@pytest.mark.parametrize("ranks", [1, 3])
def test_reference_arm_prints_one_contract_line(ranks):
    # 10^3 / 16^3 unknowns: seconds instead of half a minute; ranks > 1 = the reference on several MPI ranks
    # (multi-process MPI stand-in), what the arm uses on a multi-core host
    env = dict(os.environ, SAENA_BENCH_CPU_MX="12", SAENA_BENCH_CPU_MX_MP="18", SAENA_BENCH_CPU_RANKS=str(ranks))
    if ranks > 1:
        from oracle import ref
        if not ref.mp_available():
            pytest.skip("oracle/_ref/libsaena_ref_mp.so not built (make -C oracle ref_mp)")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                          "--warmup", "1"], capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "Munknowns/s"
    for k in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "dtype", "data", "config",
              "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["cpu_baseline"]["kind"] in ("reference", "port")
    assert d["cpu_baseline"]["cores"] == (ranks if d["cpu_baseline"]["kind"] == "reference" else 1)
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"] > 0
    assert "workload" in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, SAENA_BENCH_CPU_MX="12", RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_bench_rejects_zero_steps_and_a_dump_of_the_reference_arm():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True,
                             timeout=120)
        assert out.returncode == 2 and out.stdout == "", (extra, out.stderr[-2000:])


@pytest.mark.parametrize("n", [1000, 3_000_000])
def test_dump_outputs_writes_a_fixed_sample_of_u(n, tmp_path):
    """--dump-outputs without a GPU: the whole u up to bench.DUMP_SAMPLE entries, else the same seeded sample every run,
    every file float64, at most 64 MB in all"""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    u = torch.from_numpy(np.random.default_rng(n).standard_normal(n))
    hist = np.array([1.0, 0.1, 1e-9])
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), u, 2, hist, 0, n, 0, 1)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["iterations.npy", "residual_history.npy", "u.npy", "u_index.npy"]
    got = {f: np.load(tmp_path / "a" / f) for f in files}
    assert all(a.dtype == np.float64 for a in got.values())
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 << 20
    idx = got["u_index.npy"].astype(np.int64)
    assert len(idx) == min(n, bench.DUMP_SAMPLE) and np.all(np.diff(idx) > 0) and idx[-1] < n
    assert np.array_equal(got["u.npy"], u.numpy()[idx])
    assert np.array_equal(got["residual_history.npy"], hist) and got["iterations.npy"].tolist() == [2.0]
    for f in files:
        assert np.array_equal(np.load(tmp_path / "b" / f), got[f])


def test_dump_outputs_assembles_the_sample_from_every_ranks_row_block(tmp_path, monkeypatch):
    """--dump-outputs on three ranks (all_gather_object stood in for): rank 0 writes the same files as one rank would"""
    import numpy as np
    import torch
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    import bench
    n, cuts = 3_000_000, [0, 1_000_003, 2_400_000, 3_000_000]
    full = np.random.default_rng(7).standard_normal(n)
    hist = np.array([1.0, 1e-9])
    sent = {}

    def all_gather_object(parts, obj):   # ranks 2 and 1 call first, so rank 0 receives every block
        sent[rank] = obj
        parts[:] = [sent.get(r) for r in range(3)]

    monkeypatch.setattr(dist, "all_gather_object", all_gather_object)
    for rank in (2, 1, 0):
        u = torch.from_numpy(full[cuts[rank]:cuts[rank + 1]].copy())
        bench.dump_outputs(str(tmp_path / "three"), u, 5, hist, cuts[rank], n, rank, 3)
    bench.dump_outputs(str(tmp_path / "one"), torch.from_numpy(full), 5, hist, 0, n, 0, 1)
    for f in ("u", "u_index", "residual_history", "iterations"):
        assert np.array_equal(np.load(tmp_path / "three" / f"{f}.npy"), np.load(tmp_path / "one" / f"{f}.npy")), f
    assert not np.isnan(np.load(tmp_path / "three" / "u.npy")).any()


def _bench_line(*args, env=None):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                         timeout=600, env=env)
    assert out.returncode == 0, out.stderr[-3000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


@pytest.mark.gpu
def test_bench_times_the_requested_solves_and_dumps_the_last_ones_solution(tmp_path):
    """two small bench runs: the kernel launches of the timed region grow with --steps (one solve's worth per step),
    and the dumped u solves the system"""
    import numpy as np
    import scipy.sparse as sp
    from saena_b200.sa_setup import poisson3d_coo, poisson3d_rhs
    n = 24
    # the row mappings by the nnz/row rule, not by timing: both runs then launch the same kernels per solve
    env = dict(os.environ, SAENA_BENCH_MAPPING_AUTOTUNE="0")
    common = ["--n", str(n), "--warmup", "3", "--no-cpu-baseline"]
    one = _bench_line(*common, "--steps", "1", env=env)
    three = _bench_line(*common, "--steps", "3", "--dump-outputs", str(tmp_path), env=env)
    assert one["iterations"] == three["iterations"]
    assert one["gpu_launches"] > 0 and three["gpu_launches"] == 3 * one["gpu_launches"], (one["gpu_launches"],
                                                                                             three["gpu_launches"])
    u, idx = np.load(tmp_path / "u.npy"), np.load(tmp_path / "u_index.npy")
    hist, iters = np.load(tmp_path / "residual_history.npy"), np.load(tmp_path / "iterations.npy")
    assert np.array_equal(idx, np.arange(n ** 3)) and int(iters[0]) == three["iterations"]
    assert hist[-1] < 1e-8 * hist[0]
    N, row, col, val = poisson3d_coo(n)
    A = sp.csr_matrix((val, (row, col)), shape=(N, N))
    rhs = poisson3d_rhs(n)
    assert np.linalg.norm(A @ u - rhs) / np.linalg.norm(rhs) < 1e-7


def test_bench_verify_properties_through_the_oracle():
    """bench.py's SAENA_BENCH_VERIFY check (symmetry / R = P^T adjointness on every level) is implementation-agnostic:
    here through the C oracle on one rank"""
    sys.path.insert(0, ROOT)
    import bench
    from oracle.oracle import Oracle
    from tests.util import GOLDEN, Golden
    g = Golden(GOLDEN[1])
    out = bench.verify_properties(Oracle(g.hier), g.hier, 0, 1)
    assert out["ok"] and out["worst"] <= 1e-14, out
