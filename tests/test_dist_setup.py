"""The row-partitioned setup (saena_b200/sa_setup_dist.py) on N CPU processes over gloo, against the same setup on
one rank (sa_setup.build_device_hierarchy) -- tests/dist_setup_check.py does the comparing."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("world,args,env", [
    (2, ["poisson", "12", "esc", "double"], {}),
    (2, ["poisson", "16", "dense", "double"], {}),          # sparse x dense column blocks on every level
    # many narrow column blocks (the width is agreed between the ranks) / many small product chunks
    (3, ["poisson", "12", "dense", "double"], {"SAENA_SETUP_DENSE_BUDGET": "400000"}),
    (3, ["poisson", "12", "esc", "double"], {"SAENA_SETUP_CHUNK_PRODUCTS": "5000"}),
    (3, ["poisson", "20"], {}),                             # float halo (float_level 0, the drivers' value)
    (3, ["unstructured", "60", "double"], {"DSC_AGG_BELOW": "50"}),
    (4, ["poisson", "14", "double"], {"DSC_AGG_BELOW": "20"}),   # nothing agglomerated but the coarsest level
    (3, ["poisson", "10", "double", "skew"], {}),                # lopsided input partition, one rank starts empty
], ids=["np2-poisson12-esc", "np2-poisson16-dense", "np3-narrow-dense-blocks", "np3-small-esc-chunks", "np3-poisson20-floathalo", "np3-unstructured60", "np4-poisson14", "np3-skewed-input"])
def test_distributed_setup_equals_the_one_process_setup(world, args, env):
    port = 29720 + world + 7 * len(args) + len(env) * 13 + len(args[1])
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                          "--master-addr", "127.0.0.1", "--master-port", str(port),
                          os.path.join(ROOT, "tests", "dist_setup_check.py"), *args],
                         capture_output=True, text=True, timeout=900,
                         env=dict(os.environ, MASTER_ADDR="127.0.0.1", OMP_NUM_THREADS="1", **env))
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-6000:]
    assert "DIST_SETUP_OK" in out.stdout


def test_one_rank_distributed_setup_is_the_one_process_setup():
    """no process group: on a single rank the two layout paths -- each rank's operators from its own rows
    (build_distributed_hierarchy, rank_operator) and from the global matrices (build_hierarchy, to_rank) -- give the
    same hierarchy, array by array and bit for bit"""
    import numpy as np
    from saena_b200 import sa_setup, sa_setup_dist as sd
    from saena_b200.hierarchy import hierarchy_to_arrays
    n, row, col, val = sa_setup.poisson3d_coo(14)
    comm = sd.Comm()
    assert comm.world == 1
    h, summary = sd.build_distributed_hierarchy(sd.poisson3d_dcsr(14, comm), comm=comm)
    ref = sa_setup.build_hierarchy(n, row, col, val, device="cpu")
    a, b = hierarchy_to_arrays(h), hierarchy_to_arrays(ref)
    assert a.keys() == b.keys() and len(summary) == len(ref.levels)
    for k in a:
        assert a[k].dtype == b[k].dtype and a[k].shape == b[k].shape and np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("world", [2, 4])
def test_distributed_operator_builder_equals_split_operator(world):
    """sa_setup_dist.rank_operator (each rank from its own rows) = hierarchy.split_operator (from the global matrix),
    array by array, on random rectangular operators and partitions with empty blocks (tests/dist_rank_operator_check.py)"""
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                          "--master-addr", "127.0.0.1", "--master-port", str(29790 + world),
                          os.path.join(ROOT, "tests", "dist_rank_operator_check.py")],
                         capture_output=True, text=True, timeout=300,
                         env=dict(os.environ, MASTER_ADDR="127.0.0.1", OMP_NUM_THREADS="1"))
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-4000:]
    assert "RANK_OPERATOR_OK" in out.stdout
