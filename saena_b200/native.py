"""ctypes binding of libsaena_b200.so -- exactly the C ABI of include/saena_b200.h.

There is no fallback: if the library is missing it is built with nvcc (saena_b200/build.py);
if no CUDA device is usable `saena_b200_init` fails and `Context()` raises.
"""
from __future__ import annotations

import ctypes
import os
from typing import List, Optional, Sequence

import numpy as np

from .hierarchy import F64, I32, Hierarchy, Level, Operator

c_i32_p = ctypes.POINTER(ctypes.c_int32)
c_f64_p = ctypes.POINTER(ctypes.c_double)

JACOBI, CHEBYSHEV = 0, 1
NCCL_ID_BYTES = 128


class OperatorDesc(ctypes.Structure):
    _fields_ = [("kind", ctypes.c_int32), ("level", ctypes.c_int32), ("M", ctypes.c_int32),
                ("n_local_cols", ctypes.c_int32), ("col_offset", ctypes.c_int32), ("use_double", ctypes.c_int32),
                ("nnz_local", ctypes.c_int64), ("nnzPerRow_local", c_i32_p), ("col_local", c_i32_p),
                ("val_local", c_f64_p), ("nnz_remote", ctypes.c_int64), ("col_remote_size", ctypes.c_int32),
                ("row_remote", c_i32_p), ("val_remote", c_f64_p), ("nnzPerCol_remote", c_i32_p),
                ("vIndexSize", ctypes.c_int32), ("vIndex", c_i32_p), ("numSendProc", ctypes.c_int32),
                ("sendProcRank", c_i32_p), ("sendProcCount", c_i32_p), ("vdispls", c_i32_p),
                ("numRecvProc", ctypes.c_int32), ("recvProcRank", c_i32_p), ("recvProcCount", c_i32_p),
                ("rdispls", c_i32_p)]


class Block(ctypes.Structure):
    _fields_ = [("peer", ctypes.c_int32), ("offset", ctypes.c_int32), ("count", ctypes.c_int32)]


class NativeError(RuntimeError):
    pass


_lib = None


def load_library(path: Optional[str] = None):
    """Loads (building first if needed) libsaena_b200.so and declares the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if path is None:
        from . import build
        path = build.LIB if os.path.exists(build.LIB) and not build._stale() else build.build_library()
    L = ctypes.CDLL(path)
    vp, i, d = ctypes.c_void_p, ctypes.c_int, ctypes.c_double
    ip, dp = ctypes.POINTER(ctypes.c_int), c_f64_p
    L.saena_b200_last_error.restype = ctypes.c_char_p
    L.saena_b200_last_error.argtypes = [vp]
    L.saena_b200_nccl_unique_id.argtypes = [vp]
    L.saena_b200_init.argtypes = [ctypes.POINTER(vp), i, i, i, vp]
    L.saena_b200_init_detached.argtypes = [ctypes.POINTER(vp), i, i, i]
    L.saena_b200_destroy.argtypes = [vp]
    L.saena_b200_upload_operator.argtypes = [vp, ctypes.POINTER(OperatorDesc)]
    L.saena_b200_upload_band_operator.argtypes = [vp, i, i, i, i]
    L.saena_b200_upload_level_aux.argtypes = [vp, i, dp, d, i, i, i, ctypes.POINTER(Block), i, ctypes.POINTER(Block)]
    L.saena_b200_upload_level_scale.argtypes = [vp, i, dp]
    L.saena_b200_upload_coarsest.argtypes = [vp, i, ctypes.c_int64, c_i32_p, c_i32_p, dp]
    L.saena_b200_set_coarsest_solver.argtypes = [vp, i]
    L.saena_b200_set_operator_dense.argtypes = [vp, i, i, i]
    L.saena_b200_sellp_layout.argtypes = [i, vp, vp, vp]
    L.saena_b200_symdiag_plan.argtypes = [i, i, vp, ctypes.c_int64, ctypes.c_int64, vp]
    L.saena_b200_set_graphs.argtypes = [vp, i]
    L.saena_b200_finalize.argtypes = [vp]
    L.saena_b200_p2p_export.argtypes = [vp, vp, ctypes.c_int64, ctypes.POINTER(ctypes.c_int64)]
    L.saena_b200_p2p_import.argtypes = [vp, vp, ctypes.c_int64]
    L.saena_b200_find_eig.argtypes = [vp, i, i, vp, ctypes.c_uint64, i, ctypes.POINTER(ctypes.c_double),
                                      ctypes.POINTER(ctypes.c_int)]
    L.saena_b200_update_values.argtypes = [vp, vp, ctypes.c_int64, i, ctypes.c_uint64, dp, i]
    L.saena_b200_update_values_dev.argtypes = [vp, vp, ctypes.c_int64, i, ctypes.c_uint64, dp, i]
    L.saena_b200_update_values_times.argtypes = [vp, dp, i]
    L.saena_b200_p2p_enable.argtypes = [vp, i]
    L.saena_b200_fault_status.argtypes = [vp]
    L.saena_b200_clear_fault.argtypes = [vp]
    L.saena_b200_set_timeouts.argtypes = [vp, ctypes.c_double, ctypes.c_double]
    L.saena_b200_autotune_halo.argtypes = [vp, i]
    L.saena_b200_halo_choice.argtypes = [vp, i, i, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float)]
    solve_args = [vp, vp, vp, i, d, i, i, i, ip, dp, i, ip]
    L.saena_b200_solve_pcg.argtypes = solve_args
    L.saena_b200_solve_pcg_dev.argtypes = solve_args
    L.saena_b200_solve_vcycle.argtypes = solve_args
    L.saena_b200_solve_smoother.argtypes = solve_args
    L.saena_b200_solve_cg.argtypes = [vp, vp, vp, i, d, ip, dp, i, ip]
    L.saena_b200_matvec.argtypes = [vp, i, i, vp, vp]
    L.saena_b200_residual.argtypes = [vp, i, vp, vp, vp]
    L.saena_b200_smooth.argtypes = [vp, i, i, i, vp, vp]
    L.saena_b200_vcycle.argtypes = [vp, i, i, i, i, vp, vp]
    L.saena_b200_coarsest_solve.argtypes = [vp, vp, vp]
    L.saena_b200_dot.argtypes = [vp, vp, vp, i, dp]
    block_solve_args = [vp, i, vp, vp, i, d, i, i, i, ip, dp, i, ip]
    L.saena_b200_solve_pcg_block.argtypes = block_solve_args
    L.saena_b200_solve_pcg_block_dev.argtypes = block_solve_args
    L.saena_b200_matvec_block.argtypes = [vp, i, i, i, vp, vp]
    L.saena_b200_residual_block.argtypes = [vp, i, i, vp, vp, vp]
    L.saena_b200_smooth_block.argtypes = [vp, i, i, i, i, vp, vp]
    L.saena_b200_vcycle_block.argtypes = [vp, i, i, i, i, i, vp, vp]
    L.saena_b200_time_matvec.argtypes = [vp, i, i, i, i, ctypes.POINTER(ctypes.c_float)]
    L.saena_b200_time_smooth_sweep.argtypes = [vp, i, i, i, i, ctypes.POINTER(ctypes.c_float)]
    L.saena_b200_time_matvec_parts.argtypes = [vp, i, i, i] + [ctypes.POINTER(ctypes.c_float)] * 3
    L.saena_b200_time_vcycle.argtypes = [vp, i, i, i, i, i, ctypes.POINTER(ctypes.c_float)]
    L.saena_b200_time_matvec_compute_only.argtypes = [vp, i, i, i, i, i, ctypes.POINTER(ctypes.c_float)]
    L.saena_b200_timer_start.argtypes = [vp]
    L.saena_b200_timer_stop.argtypes = [vp, ctypes.POINTER(ctypes.c_float)]
    L.saena_b200_launch_count.restype = ctypes.c_int64
    L.saena_b200_launch_count.argtypes = [vp]
    L.saena_b200_graph_replays.restype = ctypes.c_int64
    L.saena_b200_graph_replays.argtypes = [vp]
    L.saena_b200_set_mapping.argtypes = [vp, i, i, i]
    L.saena_b200_set_fused_restrict.argtypes = [vp, i]
    L.saena_b200_spgemm_symbolic.argtypes = [i, i, i, vp, vp, vp, vp, vp, ctypes.POINTER(ctypes.c_int64)]
    L.saena_b200_spgemm_numeric.argtypes = [i, i, i, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.saena_b200_time_residual_restrict.argtypes = [vp, i, vp, vp, i, ctypes.POINTER(ctypes.c_float),
                                                    ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_double)]
    L.saena_b200_autotune_mapping.argtypes = [vp, i, ctypes.c_double, ip]
    L.saena_b200_set_mapping_deferred.argtypes = [vp, i, i, i]
    L.saena_b200_get_mapping.argtypes = [vp, i, i]
    L.saena_b200_set_level_route.argtypes = [vp, i, i]
    L.saena_b200_get_level_route.argtypes = [vp, i, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float)]
    L.saena_b200_operator_bytes.restype = ctypes.c_int64
    L.saena_b200_operator_bytes.argtypes = [vp, i, i]
    L.saena_b200_set_precond_precision.argtypes = [vp, i]
    L.saena_b200_get_precond_precision.argtypes = [vp]
    L.saena_b200_matvec_f32.argtypes = [vp, i, i, vp, vp]
    L.saena_b200_residual_f32.argtypes = [vp, i, vp, vp, vp]
    L.saena_b200_smooth_f32.argtypes = [vp, i, i, i, vp, vp]
    L.saena_b200_vcycle_f32.argtypes = [vp, i, i, i, i, vp, vp]
    _lib = L
    return L


EXPORTED_SYMBOLS = [
    "saena_b200_nccl_unique_id", "saena_b200_init", "saena_b200_init_detached", "saena_b200_time_matvec_compute_only", "saena_b200_destroy", "saena_b200_last_error",
    "saena_b200_upload_operator", "saena_b200_upload_band_operator", "saena_b200_upload_level_aux", "saena_b200_upload_level_scale",
    "saena_b200_upload_coarsest",
    "saena_b200_set_coarsest_solver", "saena_b200_set_operator_dense", "saena_b200_sellp_layout", "saena_b200_symdiag_plan", "saena_b200_set_graphs", "saena_b200_finalize",
    "saena_b200_p2p_export", "saena_b200_p2p_import", "saena_b200_find_eig", "saena_b200_update_values", "saena_b200_update_values_dev", "saena_b200_update_values_times", "saena_b200_p2p_enable", "saena_b200_fault_status", "saena_b200_clear_fault", "saena_b200_set_timeouts", "saena_b200_autotune_halo", "saena_b200_halo_choice", "saena_b200_solve_pcg", "saena_b200_solve_vcycle", "saena_b200_solve_smoother", "saena_b200_solve_cg",
    "saena_b200_solve_pcg_dev", "saena_b200_matvec", "saena_b200_residual", "saena_b200_smooth",
    "saena_b200_vcycle", "saena_b200_coarsest_solve", "saena_b200_dot", "saena_b200_time_matvec",
    "saena_b200_time_smooth_sweep", "saena_b200_time_matvec_parts", "saena_b200_time_vcycle", "saena_b200_timer_start", "saena_b200_timer_stop", "saena_b200_launch_count", "saena_b200_graph_replays", "saena_b200_set_mapping", "saena_b200_set_fused_restrict", "saena_b200_spgemm_symbolic", "saena_b200_spgemm_numeric", "saena_b200_time_residual_restrict", "saena_b200_autotune_mapping", "saena_b200_set_mapping_deferred", "saena_b200_get_mapping",
    "saena_b200_set_level_route", "saena_b200_get_level_route", "saena_b200_operator_bytes",
    "saena_b200_solve_pcg_block", "saena_b200_solve_pcg_block_dev", "saena_b200_matvec_block",
    "saena_b200_residual_block", "saena_b200_smooth_block", "saena_b200_vcycle_block",
    "saena_b200_set_precond_precision", "saena_b200_get_precond_precision", "saena_b200_matvec_f32",
    "saena_b200_residual_f32", "saena_b200_smooth_f32", "saena_b200_vcycle_f32",
]


def nccl_unique_id() -> bytes:
    L = load_library()
    buf = ctypes.create_string_buffer(NCCL_ID_BYTES)
    if L.saena_b200_nccl_unique_id(buf):
        raise NativeError(L.saena_b200_last_error(None).decode())
    return buf.raw


def _i32p(a: np.ndarray):
    return a.ctypes.data_as(c_i32_p)


def _f64p(a: np.ndarray):
    return a.ctypes.data_as(c_f64_p)


def _vp(a):
    if a is None:
        return None
    if isinstance(a, int):
        return ctypes.c_void_p(a)
    return a.ctypes.data_as(ctypes.c_void_p)


def smoother_id(name) -> int:
    if isinstance(name, int):
        return name
    if name == "chebyshev":
        return CHEBYSHEV
    if name == "jacobi":
        return JACOBI
    raise ValueError(f"unknown smoother {name!r}")  # the reference: "Error: Unknown smoother" then exit


def sellp_layout(rowptr: np.ndarray):
    """host-only half of mapping 101 (saena_b200_sellp_layout): (perm, slice_ptr) for CSR row offsets"""
    rp = np.ascontiguousarray(rowptr, np.int64)
    M = len(rp) - 1
    n_slots = (M + 255) // 256 * 256
    perm = np.full(max(n_slots, 1), -1, I32)
    sp = np.zeros(n_slots // 32 + 1, np.int64)
    L = load_library()
    if L.saena_b200_sellp_layout(M, _vp(rp), _vp(perm), _vp(sp)):
        raise RuntimeError("saena_b200_sellp_layout failed")
    return perm[:n_slots], sp


def symdiag_plan(M: int, offsets, nnz: int, padded_est: int):
    """host-only rule of mapping 103 (saena_b200_symdiag_plan): the stored diagonals (0, then the positive offsets
    ascending) for an operator with these distinct offsets col - row, or None where the layout does not apply"""
    off = np.ascontiguousarray(offsets, I32)
    stored = np.zeros(16, I32)
    L = load_library()
    nd = L.saena_b200_symdiag_plan(int(M), len(off), _vp(off), int(nnz), int(padded_est), _vp(stored))
    if nd < 0:
        raise RuntimeError("saena_b200_symdiag_plan: bad arguments")
    return stored[:nd].tolist() if nd else None


def spgemm_csr(M: int, K: int, N: int, a_rowptr, a_col, a_val, b_rowptr, b_col, b_val):
    """C = A B on the device (saena_b200_spgemm_symbolic / _numeric, csrc/spgemm.cu).  Operands: torch CUDA tensors --
    int64 row offsets, int32 columns, float64 values, contiguous.  Returns (c_rowptr int64[M + 1], c_col int32, c_val
    float64), every row with ascending columns.  torch is only the owner of the buffers here: the products are the
    library's kernels on raw device pointers."""
    import torch
    L = load_library()
    for t, dt in ((a_rowptr, torch.int64), (a_col, torch.int32), (a_val, torch.float64), (b_rowptr, torch.int64),
                  (b_col, torch.int32), (b_val, torch.float64)):
        if not (t.is_cuda and t.dtype == dt and t.is_contiguous()):
            raise ValueError("spgemm_csr: operands must be contiguous CUDA tensors (int64 offsets, int32 columns, float64 values)")
    dev = a_val.device
    with torch.cuda.device(dev):
        torch.cuda.current_stream().synchronize()   # the kernels run on the default stream
        c_rowptr = torch.empty(M + 1, dtype=torch.int64, device=dev)
        nnz = ctypes.c_int64(0)
        if L.saena_b200_spgemm_symbolic(M, K, N, a_rowptr.data_ptr(), a_col.data_ptr(), b_rowptr.data_ptr(), b_col.data_ptr(),
                                        c_rowptr.data_ptr(), ctypes.byref(nnz)):
            raise NativeError(L.saena_b200_last_error(None).decode())
        c_col = torch.empty(nnz.value, dtype=torch.int32, device=dev)
        c_val = torch.empty(nnz.value, dtype=torch.float64, device=dev)
        if L.saena_b200_spgemm_numeric(M, K, N, a_rowptr.data_ptr(), a_col.data_ptr(), a_val.data_ptr(), b_rowptr.data_ptr(),
                                       b_col.data_ptr(), b_val.data_ptr(), c_rowptr.data_ptr(), c_col.data_ptr(), c_val.data_ptr()):
            raise NativeError(L.saena_b200_last_error(None).decode())
    return c_rowptr, c_col, c_val


class Context:
    """One rank's device context: an uploaded hierarchy and the solve entry points."""

    def __init__(self, device: int = 0, rank: int = 0, nranks: int = 1, nccl_id: Optional[bytes] = None,
                 detached: bool = False):
        """detached=True: this rank's share of an nranks-way partition with no peer behind it (profiling of the
        compute side of the distributed kernels on one GPU; anything that needs a peer fails)"""
        self._L = load_library()
        self._h = ctypes.c_void_p()
        idbuf = ctypes.create_string_buffer(nccl_id, NCCL_ID_BYTES) if nccl_id else None
        if detached:
            rc = self._L.saena_b200_init_detached(ctypes.byref(self._h), device, rank, nranks)
        else:
            rc = self._L.saena_b200_init(ctypes.byref(self._h), device, rank, nranks, idbuf)
        if rc:
            raise NativeError(self._L.saena_b200_last_error(None).decode())
        self.rank, self.nranks, self.device = rank, nranks, device
        self.level_rows: List[int] = []
        self.hier: Optional[Hierarchy] = None

    def _ck(self, rc: int):
        if rc:
            raise NativeError(self._L.saena_b200_last_error(self._h).decode())

    def close(self):
        if self._h:
            self._L.saena_b200_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- upload ----
    def upload_operator(self, op: Operator):
        a = [np.ascontiguousarray(x, I32) for x in
             (op.nnzPerRow_local, op.col_local, op.row_remote, op.nnzPerCol_remote, op.vIndex, op.sendProcRank,
              op.sendProcCount, op.vdispls, op.recvProcRank, op.recvProcCount, op.rdispls)]
        vl, vr = np.ascontiguousarray(op.val_local, F64), np.ascontiguousarray(op.val_remote, F64)
        d = OperatorDesc(kind=op.kind, level=op.level, M=op.M, n_local_cols=op.n_local_cols,
                         col_offset=op.col_offset, use_double=int(op.use_double), nnz_local=op.nnz_local,
                         nnzPerRow_local=_i32p(a[0]), col_local=_i32p(a[1]), val_local=_f64p(vl),
                         nnz_remote=op.nnz_remote, col_remote_size=op.col_remote_size, row_remote=_i32p(a[2]),
                         val_remote=_f64p(vr), nnzPerCol_remote=_i32p(a[3]), vIndexSize=op.vIndexSize,
                         vIndex=_i32p(a[4]), numSendProc=len(a[5]), sendProcRank=_i32p(a[5]),
                         sendProcCount=_i32p(a[6]), vdispls=_i32p(a[7]), numRecvProc=len(a[8]),
                         recvProcRank=_i32p(a[8]), recvProcCount=_i32p(a[9]), rdispls=_i32p(a[10]))
        self._ck(self._L.saena_b200_upload_operator(self._h, ctypes.byref(d)))

    def upload_hierarchy(self, h: Hierarchy):
        """Upload once: what the adaptor does at the end of amg::set_matrix (INTEGRATION.md)."""
        for lv in h.levels:
            self.upload_operator(lv.A)
            if lv.A.use_dense:   # saena_matrix::use_dense: the reference's dense product (float input when !use_double)
                self._ck(self._L.saena_b200_set_operator_dense(self._h, lv.level, lv.A.kind, 1))
            if lv.P is not None:
                self.upload_operator(lv.P)
                self.upload_operator(lv.R)
            inv = np.ascontiguousarray(lv.inv_diag, F64)
            send = (Block * max(len(lv.repart_send), 1))(*[Block(*b) for b in lv.repart_send])
            recv = (Block * max(len(lv.repart_recv), 1))(*[Block(*b) for b in lv.repart_recv])
            self._ck(self._L.saena_b200_upload_level_aux(self._h, lv.level, _f64p(inv), float(lv.eig_max),
                                                        lv.M_coarse_old, lv.M_coarse, len(lv.repart_send), send,
                                                        len(lv.repart_recv), recv))
        if h.scale:
            for lv in h.levels:
                if lv.inv_sq_diag is None:
                    raise ValueError("scale=true hierarchy without inv_sq_diag on a level")
                isq = np.ascontiguousarray(lv.inv_sq_diag, F64)
                self._ck(self._L.saena_b200_upload_level_scale(self._h, lv.level, _f64p(isq)))
        owns_coarsest = h.levels[-1].A.M > 0
        if owns_coarsest:
            r, c = np.ascontiguousarray(h.coarse_row, I32), np.ascontiguousarray(h.coarse_col, I32)
            v = np.ascontiguousarray(h.coarse_val, F64)
            self._ck(self._L.saena_b200_upload_coarsest(self._h, h.coarse_n, len(v), _i32p(r), _i32p(c), _f64p(v)))
        else:
            self._ck(self._L.saena_b200_upload_coarsest(self._h, 0, 0, None, None, None))
        self._ck(self._L.saena_b200_finalize(self._h))
        self.hier = h
        self.level_rows = [lv.A.M for lv in h.levels]

    def upload_band(self, n: int, half_bandwidth: int, eig_max: float = 2.0, mapping: int = 0, sliced_only: bool = False):
        """A lone level-0 operator generated on the device with saena::band_matrix's pattern and values
        (BASELINE.json configs[3]); matvec / residual / smooth hooks only.  inv_diag = 1/diag = 2i+1."""
        from .hierarchy import KIND_A, Level
        self._ck(self._L.saena_b200_upload_band_operator(self._h, 0, int(n), int(half_bandwidth), int(sliced_only)))
        inv = 2.0 * np.arange(n, dtype=F64) + 1.0
        none = (Block * 1)()
        self._ck(self._L.saena_b200_upload_level_aux(self._h, 0, _f64p(inv), float(eig_max), 0, 0, 0, none, 0, none))
        if mapping:
            # forced before finalize so that no sliced copy is built first (77 GB at the full size)
            self._ck(self._L.saena_b200_set_mapping_deferred(self._h, 0, KIND_A, int(mapping)))
        self._ck(self._L.saena_b200_upload_coarsest(self._h, 0, 0, None, None, None))
        self._ck(self._L.saena_b200_finalize(self._h))
        b = int(half_bandwidth)
        i = np.arange(n, dtype=np.int64)
        counts = (np.minimum(i + b, n - 1) - np.maximum(i - b, 0) + 1)
        op = Operator(kind=KIND_A, level=0, M=n, Mbig=n, Nbig=n, row_offset=0, col_offset=0, n_local_cols=n,
                      nnzPerRow_local=np.zeros(0, I32), col_local=np.zeros(0, I32), val_local=np.zeros(0, F64))
        self.hier = Hierarchy([Level(0, op, inv_diag=inv, eig_max=eig_max)], coarse_n=0, coarse_row=np.zeros(0, I32),
                              coarse_col=np.zeros(0, I32), coarse_val=np.zeros(0, F64))
        self.level_rows = [n]
        return int(counts.sum())

    def set_coarsest_solver(self, name: str):
        """'SuperLU' (default: direct solve) or 'CG' -- saena_object::direct_solver"""
        if name not in ("SuperLU", "CG"):
            raise ValueError("Error: Unknown direct solver!")   # saena_object_solve.cpp:1011-1013
        self._ck(self._L.saena_b200_set_coarsest_solver(self._h, int(name == "CG")))

    # ---- peer-memory halo ----
    def p2p_export(self) -> bytes:
        n = ctypes.c_int64(0)
        self._ck(self._L.saena_b200_p2p_export(self._h, None, 0, ctypes.byref(n)))
        buf = ctypes.create_string_buffer(n.value)
        self._ck(self._L.saena_b200_p2p_export(self._h, buf, n.value, ctypes.byref(n)))
        return buf.raw

    def p2p_import(self, blobs):
        """blobs: every rank's p2p_export(), in rank order"""
        assert len(blobs) == self.nranks and len({len(b) for b in blobs}) == 1
        joined = b"".join(blobs)
        self._ck(self._L.saena_b200_p2p_import(self._h, ctypes.create_string_buffer(joined, len(joined)), len(blobs[0])))

    def p2p_enable(self, on: int):
        """2: fused halo kernel (default after p2p_import), 1: peer stores with separate launches, 0: NCCL"""
        self._ck(self._L.saena_b200_p2p_enable(self._h, int(on)))

    def fault_status(self) -> bool:
        """True once a device-side wait of the halo exchange (or a host wait) of this context has timed out"""
        return bool(self._L.saena_b200_fault_status(self._h))

    def set_timeouts(self, halo_timeout_ms: float = -1.0, sync_timeout_s: float = 180.0):
        self._ck(self._L.saena_b200_set_timeouts(self._h, float(halo_timeout_ms), float(sync_timeout_s)))

    def clear_fault(self):
        """after a timed-out exchange: every rank calls this, then p2p_enable(0) (NCCL) or a new p2p export/import"""
        self._ck(self._L.saena_b200_clear_fault(self._h))

    def autotune_halo(self, reps: int = 10):
        """collective: keep, per operator, the faster of the fused kernel and the separate launches"""
        self._ck(self._L.saena_b200_autotune_halo(self._h, reps))

    def halo_choice(self, level: int, kind: int):
        """-> (choice, ms_fused, ms_unfused); choice 1 fused kernel, 0 separate launches / NCCL, -1 absent"""
        a, b = ctypes.c_float(0), ctypes.c_float(0)
        c = int(self._L.saena_b200_halo_choice(self._h, level, kind, ctypes.byref(a), ctypes.byref(b)))
        return c, a.value, b.value

    def find_eig(self, level: int, max_iter: int = 20, start=None, seed: int = 0, store: bool = False):
        """saena_object::find_eig on the device -> (1.0001 * lambda_max(D^-1/2 A D^-1/2), Lanczos steps)"""
        eig, it = ctypes.c_double(0), ctypes.c_int(0)
        arr = None if start is None else np.ascontiguousarray(start, F64)   # kept alive across the call
        self._ck(self._L.saena_b200_find_eig(self._h, level, int(max_iter), _vp(arr), int(seed), int(store),
                                             ctypes.byref(eig), ctypes.byref(it)))
        return eig.value, it.value

    def update_values(self, val_local, max_eig_iter: int = 20, seed: int = 0) -> np.ndarray:
        """New values for level 0's A on its uploaded pattern (saena_b200_update_values): val_local in the uploaded
        order (row-major, the nnzPerRow_local / col_local given at upload), a numpy array or a CUDA torch tensor (float64,
        contiguous; it goes to the device-pointer entry).  Every coarse level is recomputed as R A P on its stored
        pattern, with inv_diag, the Chebyshev bounds (find_eig with max_eig_iter and seed), the sliced layouts and the
        coarsest factor.  Returns, per level, the share ||C - C|pattern||_F / ||C||_F of R A P lumped into the
        diagonal (entry 0 is 0).  `self.hier` keeps the uploaded host arrays: it does not follow the update."""
        out = np.zeros(len(self.level_rows), F64)
        if hasattr(val_local, "is_cuda") and val_local.is_cuda:
            import torch
            if val_local.dtype != torch.float64 or not val_local.is_contiguous():
                raise ValueError("update_values: a device tensor must be contiguous float64")
            with torch.cuda.device(val_local.device):
                torch.cuda.current_stream().synchronize()   # the values are complete before the library reads them
            self._ck(self._L.saena_b200_update_values_dev(self._h, ctypes.c_void_p(val_local.data_ptr()),
                                                          int(val_local.numel()), int(max_eig_iter), int(seed),
                                                          _f64p(out), len(out)))
        else:
            v = np.ascontiguousarray(val_local, F64)
            self._ck(self._L.saena_b200_update_values(self._h, _vp(v), len(v), int(max_eig_iter), int(seed), _f64p(out),
                                                      len(out)))
        return out

    def update_values_times(self) -> dict:
        """host-clock ms of the last update_values, by phase"""
        ms = np.zeros(5, F64)
        self._ck(self._L.saena_b200_update_values_times(self._h, _f64p(ms), 5))
        return dict(zip(("products", "pattern_map", "layouts", "eig", "coarsest"), ms.tolist()))

    def set_graphs(self, on: bool):
        self._ck(self._L.saena_b200_set_graphs(self._h, int(on)))

    # ---- solvers ----
    def _solve(self, fn, rhs, u, max_iter, tol, smoother, pre, post):
        iters, n = ctypes.c_int(0), ctypes.c_int(0)
        hist = np.zeros(max_iter + 2, F64)
        self._ck(fn(self._h, _vp(rhs), _vp(u), int(max_iter), float(tol), smoother_id(smoother), int(pre), int(post),
                    ctypes.byref(iters), _f64p(hist), len(hist), ctypes.byref(n)))
        return iters.value, hist[:n.value]

    def solve_pcg(self, rhs: np.ndarray, max_iter=50, tol=1e-8, smoother="chebyshev", pre=3, post=3):
        rhs = np.ascontiguousarray(rhs, F64)
        u = np.zeros(self.level_rows[0], F64)
        it, hist = self._solve(self._L.saena_b200_solve_pcg, rhs, u, max_iter, tol, smoother, pre, post)
        return u, it, hist

    def solve_pcg_dev(self, rhs_ptr: int, u_ptr: int, max_iter=50, tol=1e-8, smoother="chebyshev", pre=3, post=3):
        """rhs / u are raw device pointers (e.g. torch.Tensor.data_ptr())."""
        return self._solve(self._L.saena_b200_solve_pcg_dev, rhs_ptr, u_ptr, max_iter, tol, smoother, pre, post)

    def solve_vcycle(self, rhs, max_iter=50, tol=1e-8, smoother="chebyshev", pre=3, post=3):
        rhs = np.ascontiguousarray(rhs, F64)
        u = np.zeros(self.level_rows[0], F64)
        it, hist = self._solve(self._L.saena_b200_solve_vcycle, rhs, u, max_iter, tol, smoother, pre, post)
        return u, it, hist

    def solve_smoother(self, rhs, max_iter=50, tol=1e-8, smoother="chebyshev", pre=3, post=3):
        """saena_object::solve_smoother: the smoother alone as a stationary iteration on level 0"""
        rhs = np.ascontiguousarray(rhs, F64)
        u = np.zeros(self.level_rows[0], F64)
        it, hist = self._solve(self._L.saena_b200_solve_smoother, rhs, u, max_iter, tol, smoother, pre, post)
        return u, it, hist

    def solve_cg(self, rhs, max_iter=500, tol=1e-8):
        rhs = np.ascontiguousarray(rhs, F64)
        u = np.zeros(self.level_rows[0], F64)
        iters, n = ctypes.c_int(0), ctypes.c_int(0)
        hist = np.zeros(max_iter + 2, F64)
        self._ck(self._L.saena_b200_solve_cg(self._h, _vp(rhs), _vp(u), int(max_iter), float(tol),
                                             ctypes.byref(iters), _f64p(hist), len(hist), ctypes.byref(n)))
        return u, iters.value, hist[:n.value]

    # ---- block solve: k = 1..8 right-hand sides as (k, n) arrays (row j = column j of the C ABI's block) ----
    @staticmethod
    def _block(a, n: int) -> np.ndarray:
        a = np.ascontiguousarray(a, F64)
        if a.ndim != 2 or a.shape[1] != n:
            raise ValueError(f"expected a (k, {n}) array, got shape {a.shape}")
        return a

    def solve_pcg_block(self, rhs, max_iter=50, tol=1e-8, smoother="chebyshev", pre=3, post=3):
        """saena_b200_solve_pcg_block: rhs (k, n) -> (u (k, n), iters [k], [history of each column]); column j is
        bit for bit what solve_pcg(rhs[j]) gives.  rhs may be a CUDA torch tensor (float64, contiguous): it then goes
        to the device-pointer entry and u comes back as a torch tensor on the same device."""
        n = self.level_rows[0]
        dev = hasattr(rhs, "is_cuda") and rhs.is_cuda
        if dev:
            import torch
            if rhs.dtype != torch.float64 or not rhs.is_contiguous() or rhs.dim() != 2 or rhs.shape[1] != n:
                raise ValueError(f"solve_pcg_block: a device tensor must be contiguous float64 of shape (k, {n})")
            u = torch.zeros_like(rhs)
            with torch.cuda.device(rhs.device):
                torch.cuda.current_stream().synchronize()   # rhs and u are complete before the library reads them
            fn, a, b = self._L.saena_b200_solve_pcg_block_dev, ctypes.c_void_p(rhs.data_ptr()), ctypes.c_void_p(u.data_ptr())
        else:
            rhs = self._block(rhs, n)
            u = np.zeros_like(rhs)
            fn, a, b = self._L.saena_b200_solve_pcg_block, _vp(rhs), _vp(u)
        k = int(rhs.shape[0])
        iters, lens = np.zeros(max(k, 1), np.int32), np.zeros(max(k, 1), np.int32)
        cap = max_iter + 2
        hist = np.zeros((max(k, 1), cap), F64)
        self._ck(fn(self._h, k, a, b, int(max_iter), float(tol), smoother_id(smoother), int(pre), int(post),
                    _i32p(iters), _f64p(hist), cap, _i32p(lens)))
        return u, iters[:k].tolist(), [hist[j, :lens[j]] for j in range(k)]

    def matvec_block(self, level: int, kind: int, v) -> np.ndarray:
        op = self._op(level, kind)
        v = self._block(v, op.n_local_cols)
        w = np.zeros((v.shape[0], op.M), F64)
        self._ck(self._L.saena_b200_matvec_block(self._h, level, kind, v.shape[0], _vp(v), _vp(w)))
        return w

    def residual_block(self, level, u, rhs) -> np.ndarray:
        n = self.level_rows[level]
        u, rhs = self._block(u, n), self._block(rhs, n)
        res = np.zeros_like(u)
        self._ck(self._L.saena_b200_residual_block(self._h, level, u.shape[0], _vp(u), _vp(rhs), _vp(res)))
        return res

    def smooth_block(self, level, smoother, iters, u, rhs) -> np.ndarray:
        n = self.level_rows[level]
        u, rhs = self._block(u, n).copy(), self._block(rhs, n)
        self._ck(self._L.saena_b200_smooth_block(self._h, level, smoother_id(smoother), int(iters), u.shape[0], _vp(u),
                                                 _vp(rhs)))
        return u

    def vcycle_block(self, level, u, rhs, pre=3, post=3, smoother="chebyshev") -> np.ndarray:
        n = self.level_rows[level]
        u, rhs = self._block(u, n).copy(), self._block(rhs, n)
        self._ck(self._L.saena_b200_vcycle_block(self._h, level, smoother_id(smoother), int(pre), int(post),
                                                 u.shape[0], _vp(u), _vp(rhs)))
        return u

    # ---- FP32 preconditioner ----
    def set_precond_precision(self, bits: int):
        """64 (default) or 32: solve_pcg / solve_pcg_dev apply the preconditioner as an FP32 V-cycle (the Krylov loop
        stays FP64).  Raises, leaving 64, where the hierarchy cannot run it (see saena_b200_set_precond_precision)."""
        self._ck(self._L.saena_b200_set_precond_precision(self._h, int(bits)))

    def get_precond_precision(self) -> int:
        return int(self._L.saena_b200_get_precond_precision(self._h))

    def matvec_f32(self, level: int, kind: int, v) -> np.ndarray:
        """the hooks below on the FP32 path (precision 32 only): float32 arrays in and out"""
        op = self._op(level, kind)
        v = np.ascontiguousarray(v, np.float32)
        assert len(v) == op.n_local_cols
        w = np.zeros(op.M, np.float32)
        self._ck(self._L.saena_b200_matvec_f32(self._h, level, kind, _vp(v), _vp(w)))
        return w

    def residual_f32(self, level, u, rhs) -> np.ndarray:
        u, rhs = np.ascontiguousarray(u, np.float32), np.ascontiguousarray(rhs, np.float32)
        res = np.zeros_like(u)
        self._ck(self._L.saena_b200_residual_f32(self._h, level, _vp(u), _vp(rhs), _vp(res)))
        return res

    def smooth_f32(self, level, smoother, iters, u, rhs) -> np.ndarray:
        u = np.array(u, np.float32, copy=True)
        rhs = np.ascontiguousarray(rhs, np.float32)
        self._ck(self._L.saena_b200_smooth_f32(self._h, level, smoother_id(smoother), int(iters), _vp(u), _vp(rhs)))
        return u

    def vcycle_f32(self, level, u, rhs, pre=3, post=3, smoother="chebyshev") -> np.ndarray:
        u = np.array(u, np.float32, copy=True)
        rhs = np.ascontiguousarray(rhs, np.float32)
        self._ck(self._L.saena_b200_vcycle_f32(self._h, level, smoother_id(smoother), int(pre), int(post), _vp(u),
                                               _vp(rhs)))
        return u

    # ---- hooks ----
    def _op(self, level, kind) -> Operator:
        lv = self.hier.levels[level]
        return (lv.A, lv.P, lv.R)[kind]

    def matvec(self, level: int, kind: int, v: np.ndarray) -> np.ndarray:
        v = np.ascontiguousarray(v, F64)
        op = self._op(level, kind)
        assert len(v) == op.n_local_cols
        w = np.zeros(op.M, F64)
        self._ck(self._L.saena_b200_matvec(self._h, level, kind, _vp(v), _vp(w)))
        return w

    def residual(self, level, u, rhs):
        u, rhs = np.ascontiguousarray(u, F64), np.ascontiguousarray(rhs, F64)
        res = np.zeros_like(u)
        self._ck(self._L.saena_b200_residual(self._h, level, _vp(u), _vp(rhs), _vp(res)))
        return res

    def smooth(self, level, smoother, iters, u, rhs):
        u = np.array(u, F64, copy=True)
        rhs = np.ascontiguousarray(rhs, F64)
        self._ck(self._L.saena_b200_smooth(self._h, level, smoother_id(smoother), int(iters), _vp(u), _vp(rhs)))
        return u

    def vcycle(self, level, u, rhs, pre=3, post=3, smoother="chebyshev"):
        u = np.array(u, F64, copy=True)
        rhs = np.ascontiguousarray(rhs, F64)
        self._ck(self._L.saena_b200_vcycle(self._h, level, smoother_id(smoother), int(pre), int(post), _vp(u),
                                           _vp(rhs)))
        return u

    def coarsest_solve(self, rhs):
        rhs = np.ascontiguousarray(rhs, F64)
        u = np.zeros_like(rhs)
        self._ck(self._L.saena_b200_coarsest_solve(self._h, _vp(rhs), _vp(u)))
        return u

    def dot(self, a, b) -> float:
        a, b = np.ascontiguousarray(a, F64), np.ascontiguousarray(b, F64)
        out = ctypes.c_double(0)
        self._ck(self._L.saena_b200_dot(self._h, _vp(a), _vp(b), len(a), ctypes.byref(out)))
        return out.value

    # ---- measurement ----
    def time_matvec(self, level, kind, reps=20, flush_l2=False) -> float:
        ms = ctypes.c_float(0)
        self._ck(self._L.saena_b200_time_matvec(self._h, level, kind, reps, int(flush_l2), ctypes.byref(ms)))
        return ms.value

    def time_smooth_sweep(self, level, smoother="chebyshev", reps=20, flush_l2=False) -> float:
        ms = ctypes.c_float(0)
        self._ck(self._L.saena_b200_time_smooth_sweep(self._h, level, smoother_id(smoother), reps, int(flush_l2),
                                                      ctypes.byref(ms)))
        return ms.value

    def time_matvec_parts(self, level, kind, reps=20):
        """-> (full_ms, local_only_ms, halo_only_ms); collective when nranks > 1"""
        f, l, h = ctypes.c_float(0), ctypes.c_float(0), ctypes.c_float(0)
        self._ck(self._L.saena_b200_time_matvec_parts(self._h, level, kind, reps, ctypes.byref(f), ctypes.byref(l),
                                                      ctypes.byref(h)))
        return f.value, l.value, h.value

    def time_matvec_compute_only(self, level, kind, fused: bool, reps=20, flush_l2=False) -> float:
        ms = ctypes.c_float(0)
        self._ck(self._L.saena_b200_time_matvec_compute_only(self._h, level, kind, int(fused), reps, int(flush_l2),
                                                             ctypes.byref(ms)))
        return ms.value

    def time_vcycle(self, level: int, smoother="chebyshev", pre=3, post=3, reps=10) -> float:
        ms = ctypes.c_float(0)
        self._ck(self._L.saena_b200_time_vcycle(self._h, level, smoother_id(smoother), pre, post, reps, ctypes.byref(ms)))
        return ms.value

    def timer_start(self):
        self._ck(self._L.saena_b200_timer_start(self._h))

    def timer_stop(self) -> float:
        ms = ctypes.c_float(0)
        self._ck(self._L.saena_b200_timer_stop(self._h, ctypes.byref(ms)))
        return ms.value

    def launch_count(self) -> int:
        return int(self._L.saena_b200_launch_count(self._h))

    def graph_replays(self) -> int:
        return int(self._L.saena_b200_graph_replays(self._h))

    def set_mapping(self, level, kind, mapping: int):
        """mapping > 0: that many lanes per row (sub-warp mapping); < 0: streaming row blocks with
        -mapping lanes per row in the reduce phase; 100 / 101: the sliced layouts; 103: symmetric diagonals (where
        the operator is eligible, else the heuristic's choice); 0: heuristic from nnz/row."""
        self._ck(self._L.saena_b200_set_mapping(self._h, level, kind, int(mapping)))

    def get_mapping(self, level, kind) -> int:
        return int(self._L.saena_b200_get_mapping(self._h, level, kind))

    def set_level_route(self, level: int, on: bool):
        """apply level `level`'s operator as R A P of the level above (True) or stream its stored A (False); raises
        where the route is not allowed or R A P differs from the stored operator by more than 1e-12"""
        self._ck(self._L.saena_b200_set_level_route(self._h, int(level), int(on)))

    def get_level_route(self, level: int) -> bool:
        return self.level_route_choice(level)[0] == 1

    def level_route_choice(self, level: int):
        """-> (choice, ms_stored, ms_route); choice 1 on the route, 0 not, -1 no such level; the two times are the
        autotune's medians of a Chebyshev sweep each way (0: the level was not timed)"""
        a, b = ctypes.c_float(0), ctypes.c_float(0)
        c = int(self._L.saena_b200_get_level_route(self._h, int(level), ctypes.byref(a), ctypes.byref(b)))
        return c, a.value, b.value

    def set_fused_restrict(self, levels: int):
        """levels [0, levels) of the V-cycle: residual + restriction as one scatter kernel where eligible (0: off)"""
        self._ck(self._L.saena_b200_set_fused_restrict(self._h, int(levels)))

    def time_residual_restrict(self, level: int, u: np.ndarray, rhs: np.ndarray, reps: int = 10):
        """-> (ms of residual kernel + R kernel, ms of the fused scatter kernel, relative difference of the results)"""
        u, rhs = np.ascontiguousarray(u, F64), np.ascontiguousarray(rhs, F64)
        a, b, d = ctypes.c_float(0), ctypes.c_float(0), ctypes.c_double(0)
        self._ck(self._L.saena_b200_time_residual_restrict(self._h, int(level), _vp(u), _vp(rhs), int(reps),
                                                           ctypes.byref(a), ctypes.byref(b), ctypes.byref(d)))
        return a.value, b.value, d.value

    def autotune_mapping_native(self, reps: int = 10, min_gain: float = 0.03) -> int:
        """saena_b200_autotune_mapping: the library's own setup-time choice of every operator's row mapping by
        measurement (collective on several ranks); returns how many operators changed on this rank"""
        n = ctypes.c_int(0)
        self._ck(self._L.saena_b200_autotune_mapping(self._h, int(reps), float(min_gain), ctypes.byref(n)))
        return n.value

    def autotune_mapping(self, reps: int = 10, min_gain: float = 0.03):
        """One rank only (setup time, untimed): for every uploaded operator, time the row mappings around the one
        `sb_choose_mapping` picked from nnz/row (half / double / four times the threads per row; the sorted sliced
        layout, mapping 101, where many short irregular rows run on a sub-warp mapping) with the library's own
        per-launch timer and keep the fastest if it wins by more than `min_gain`.  Composes saena_b200_set_mapping and
        saena_b200_time_matvec; returns [(level, kind, before, after, ms_before, ms_after)].
        Not collective-safe: with several ranks every timed application is an exchange and the candidate lists
        would have to agree -- callers gate on nranks == 1."""
        if self.nranks != 1:
            raise RuntimeError("autotune_mapping: one rank only")
        out = []
        for l, lv in enumerate(self.hier.levels):
            for kind, op in ((0, lv.A), (1, lv.P), (2, lv.R)):
                if op is None or op.M == 0:
                    continue
                cur = self.get_mapping(l, kind)
                if cur <= 0 or cur == 101:
                    continue                       # streaming (forced by hand) / already the sorted layout
                flush = self.operator_bytes(l, kind) < 300e6
                if cur == 100:
                    # sliced layout: measured choice; the only candidate is its sorted variant, and only where the
                    # slices are padded (rows of unequal length) and the operator has no halo
                    n = np.asarray(op.nnzPerRow_local, np.int64)
                    pad = np.zeros((len(n) + 31) // 32 * 32, np.int64)
                    pad[:len(n)] = n
                    padded = int(pad.reshape(-1, 32).max(axis=1).sum()) * 32
                    cands = [101] if (op.nnz_remote == 0 and n.sum() > 0 and padded > 1.03 * n.sum()) else []
                    if not cands:
                        continue
                else:
                    cands = sorted({c for c in (cur // 4, cur // 2, cur * 2, cur * 4) if 1 <= c <= 256 and c != cur})
                    if cur < 32 and op.M >= 150_000 and op.nnz_remote == 0:
                        cands.append(101)          # many short irregular rows: the sorted sliced layout
                best, t0 = cur, self.time_matvec(l, kind, reps, flush_l2=flush)
                tb = t0
                for c in cands:
                    self.set_mapping(l, kind, c)
                    t = self.time_matvec(l, kind, reps, flush_l2=flush)
                    if t < tb:
                        best, tb = c, t
                if tb > (1.0 - min_gain) * t0:
                    best, tb = cur, t0
                self.set_mapping(l, kind, best)
                out.append((l, kind, cur, best, t0, tb))
        return out

    def operator_bytes(self, level, kind) -> int:
        return int(self._L.saena_b200_operator_bytes(self._h, level, kind))
