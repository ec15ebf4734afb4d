"""Cases for the device SpGEMM (saena_b200/csrc/spgemm.cu), the dispatch that decides which kernel handles each of
their rows, and an exact reference of C = A B.

Both passes of the SpGEMM send every row to one of seven bins, and three of the bins' kernels loop over rows with a
grid stride, so one CTA clears and reuses its structure for row after row.  Which rows reach which kernel, and
whether a CTA gets a second row, depends on the SM count and the opt-in shared memory of the card.  The dispatch is
restated below in plain Python, line by line from spgemm.cu, so that every case can say what it covers and a test
can check that claim without a GPU (tests/test_spgemm_cases.py, at the B200's constants) and again on the card that
runs the products (tests/test_zzz_spgemm_gpu.py).

The cases use exact values: A's entries are in {±1, ±2, ±3} and B's in {±0.25, ±0.5, ±1}, so every product is a
multiple of 1/16 and every partial sum is a double without rounding, in any summation order (B = I, where each entry
of C is one product, takes any A).  A lost or double-counted product then shows in the value, and C must equal the
reference bit for bit.
"""
import dataclasses
from typing import Optional

import numpy as np
import scipy.sparse as sp

B200_SMS = 148
B200_SMEM_OPTIN = 232_448   # cudaDevAttrMaxSharedMemoryPerBlockOptin of a B200, bytes

SCAN_BLOCK = 1024                # spgemm.cu:214
SLAB_BUDGET_BYTES = 2 << 30      # spgemm.cu:465
A_EXACT = np.array([-3.0, -2.0, -1.0, 1.0, 2.0, 3.0])
B_EXACT = np.array([-1.0, -0.5, -0.25, 0.25, 0.5, 1.0])


# ---------------------------------------------------------------------------------------------------------------------
# the dispatch of spgemm.cu
# ---------------------------------------------------------------------------------------------------------------------
def sg_hash(c, mask):
    """home slot of column c in a hash table of mask + 1 slots (spgemm.cu:51), in uint32 arithmetic"""
    c = np.atleast_1d(np.asarray(c)).astype(np.uint32)
    return ((c * np.uint32(2654435761)) >> np.uint32(7)) & np.uint32(mask)


def _bin_of(size, hi):
    """sg_bin_of (spgemm.cu:77-81): the limits are walked in order and a row stops at the first one its size does
    not exceed; a size above every limit but the last lands in the last bin"""
    size = np.asarray(size, np.int64)
    b = np.zeros(size.shape, np.int64)
    going = np.ones(size.shape, bool)
    for h in hi[:-1]:
        going &= size > h
        b += going
    return b


def symbolic_limits(N, smem):
    """spgemm.cu:485-489: 0 | <= 32 | <= 128 | <= 512 | <= 8192 | bitmask in shared memory | bitmask in global memory;
    without room for a shared bitmask bin 5 takes the limit of bin 4 and stays empty"""
    n_words = (N + 31) // 32
    return (0, 32, 128, 512, 8192, N if n_words * 4 + 64 <= smem else 8192, N)


def symbolic_bin(ub, N, smem):
    """bin of each row in the symbolic pass: by min(ub, N) (spgemm.cu:491 and the cap in sg_bin_count_kernel, :90-91)"""
    return _bin_of(np.minimum(ub, N), symbolic_limits(N, smem))


def numeric_limits(N, smem):
    """spgemm.cu:540-544: 0 | <= 32 | <= 128 | <= 512 | <= 4096 | <= 8192 | dense accumulator"""
    hi4 = 4096 if 8192 * 12 <= smem else 512
    hi5 = 8192 if 16384 * 12 <= smem else hi4
    return (0, 32, 128, 512, hi4, hi5, N)


def numeric_bin(nnz, N, smem):
    """bin of each row in the numeric pass: by the row's exact nnz (spgemm.cu:546)"""
    return _bin_of(np.minimum(nnz, N), numeric_limits(N, smem))


SYMBOLIC_TABLE = {1: 64, 2: 256, 3: 1024, 4: 16384}            # hash-set slots per bin, spgemm.cu:493-499
NUMERIC_TABLE = {1: 64, 2: 256, 3: 1024, 4: 8192, 5: 16384}    # hash-table slots per bin, spgemm.cu:548-565


def numeric_dense_slab(N, smem):
    """spgemm.cu:567-570: the dense accumulator (N doubles and N flag bits) goes to a slab in global memory when it
    does not fit in shared memory with 2 KB to spare"""
    n_words = (N + 31) // 32
    return (N + (n_words + 1) // 2) * 8 + 2048 > smem


def grid(pass_, b, n_rows, N, sms, smem):
    """CTAs of a grid-stride launch: symbolic bins 5 and 6 (spgemm.cu:503, :507) and numeric bin 6 (:572, :576)"""
    n_words = (N + 31) // 32
    if pass_ == "symbolic" and b == 5:
        return min(n_rows, 8 * sms)
    if pass_ == "symbolic" and b == 6:
        return max(1, min(n_rows, 4 * sms, SLAB_BUDGET_BYTES // (n_words * 4)))
    if pass_ == "numeric" and b == 6:
        if not numeric_dense_slab(N, smem):
            return min(n_rows, sms)
        return max(1, min(n_rows, 4 * sms, SLAB_BUDGET_BYTES // ((N + (n_words + 1) // 2) * 8)))
    raise ValueError(f"{pass_} bin {b} launches one CTA or one warp per row")


def scan_blocks(M):
    """CTAs of the row-offset scan (spgemm.cu:515)"""
    return max(1, -(-M // SCAN_BLOCK))


# ---------------------------------------------------------------------------------------------------------------------
# what a case claims to cover
# ---------------------------------------------------------------------------------------------------------------------
@dataclasses.dataclass(frozen=True)
class Rows:
    """At least `at_least` rows in bin `bin` of the pass, counting only rows of exactly this ub or nnz when given.
    `beyond_grid`: the bin has more rows than its grid-stride launch has CTAs, so some CTA handles a second row.
    `slab`: the numeric dense accumulator is in global memory (True) or in shared memory (False)."""
    pass_: str
    bin: int
    at_least: int
    ub: Optional[int] = None
    nnz: Optional[int] = None
    beyond_grid: bool = False
    slab: Optional[bool] = None


@dataclasses.dataclass(frozen=True)
class Wrap:
    """A row of the pass that fills its bin to the bin's limit, whose table has `table` slots, and of whose columns at
    least `at_least` hash to the last slot: linear probing has to wrap around to slot 0."""
    pass_: str
    table: int
    at_least: int


@dataclasses.dataclass(frozen=True)
class Zeros:
    """At least `at_least` entries of C in rows of numeric bin `bin` that are structurally present with value 0."""
    bin: int
    at_least: int


@dataclasses.dataclass(frozen=True)
class Scan:
    """The row-offset scan runs on `blocks` CTAs and the last one holds `tail` rows."""
    blocks: int
    tail: int


@dataclasses.dataclass
class Case:
    name: str
    A: sp.csr_matrix
    B: sp.csr_matrix
    claims: tuple


# ---------------------------------------------------------------------------------------------------------------------
# exact reference
# ---------------------------------------------------------------------------------------------------------------------
def _ones(X, dtype=np.int64):
    return sp.csr_matrix((np.ones(X.nnz, dtype), X.indices, X.indptr), shape=X.shape)


def structure(A, B):
    """spones(A) @ spones(B) in int64: C's pattern, with no cancellation possible, and each entry's product count"""
    S = (_ones(A) @ _ones(B)).tocsr()
    S.sort_indices()
    return S


def upper_bounds(A, B):
    """ub of each row: the products it has, nnz(B_k) summed over its a_ik"""
    return np.asarray(_ones(A) @ np.diff(B.indptr).astype(np.int64)).ravel()


def _on_pattern(S, X):
    """X's values on S's pattern (X's pattern is a subset of S's: scipy drops the entries that sum to 0)"""
    X = X.tocsr()
    X.sort_indices()
    n = S.shape[1]
    key = lambda Y: np.repeat(np.arange(Y.shape[0], dtype=np.int64), np.diff(Y.indptr)) * n + Y.indices
    ks, kx = key(S), key(X)
    pos = np.searchsorted(ks, kx)
    assert len(kx) == 0 or np.array_equal(ks[np.minimum(pos, len(ks) - 1)], kx)
    out = np.zeros(S.nnz, X.dtype)
    out[pos] = X.data
    return out


@dataclasses.dataclass
class Reference:
    indptr: np.ndarray   # int64
    indices: np.ndarray  # int32, ascending in each row
    count: np.ndarray    # k_ij, products per entry
    value: np.ndarray    # long double
    bound: np.ndarray    # long double: (k_ij + 1) 2^-53 (|A| |B|)_ij


def reference(A, B):
    """C = A B exactly in structure and to long-double precision in value.  A double result summed in any order is
    within (k + 1) 2^-53 (|A| |B|)_ij of the exact entry (k products, k - 1 additions); the long-double reference's
    own error, at 2^-64 per operation, stays inside the slack of that bound while k <= 2048."""
    S = structure(A, B)
    Al, Bl = A.astype(np.longdouble), B.astype(np.longdouble)
    value = _on_pattern(S, Al @ Bl)
    mag = _on_pattern(S, abs(Al) @ abs(Bl))
    count = S.data.astype(np.int64)
    bound = (count + 1).astype(np.longdouble) * np.longdouble(2.0) ** -53 * mag
    return Reference(S.indptr.astype(np.int64), S.indices.astype(np.int32), count, value, bound)


def values_are_exact(A, B, count):
    """True when C has no rounding in any summation order: A's and B's values are multiples of 1/4 of magnitude <= 3
    (products are sixteenths of magnitude <= 9, and 9 * 16 * k < 2^53), or every entry of C is one product and B's
    values are +-1"""
    quarters = lambda v: bool(np.all(np.abs(v) <= 3) and np.all(v * 4 == np.round(v * 4)))
    if quarters(A.data) and quarters(B.data) and (len(count) == 0 or 144 * int(count.max()) < 2 ** 53):
        return True
    return bool(np.all(count == 1) and np.all(np.abs(B.data) == 1))


def unmet_claims(case, sms, smem):
    """the claims of `case` that the dispatch of a card with `sms` SMs and `smem` bytes of opt-in shared memory per
    block does not meet (empty when the case covers what it says)"""
    A, B = case.A, case.B
    M, N = A.shape[0], B.shape[1]
    S = structure(A, B)
    ub, nnz = upper_bounds(A, B), np.diff(S.indptr)
    size = {"symbolic": np.minimum(ub, N), "numeric": nnz}
    bins = {"symbolic": symbolic_bin(ub, N, smem), "numeric": numeric_bin(nnz, N, smem)}
    limits = {"symbolic": np.array(symbolic_limits(N, smem)), "numeric": np.array(numeric_limits(N, smem))}
    tables = {"symbolic": SYMBOLIC_TABLE, "numeric": NUMERIC_TABLE}
    entry_row = np.repeat(np.arange(M), nnz)
    zero = None
    out = []
    for c in case.claims:
        if isinstance(c, Rows):
            in_bin = bins[c.pass_] == c.bin
            sel = in_bin.copy()
            if c.ub is not None:
                sel &= ub == c.ub
            if c.nnz is not None:
                sel &= nnz == c.nnz
            if sel.sum() < c.at_least:
                out.append(f"{c}: {int(sel.sum())} rows")
            if c.beyond_grid:
                n_bin = int(in_bin.sum())
                ctas = grid(c.pass_, c.bin, n_bin, N, sms, smem)
                if n_bin <= ctas:
                    out.append(f"{c}: {n_bin} rows in the bin, {ctas} CTAs")
            if c.slab is not None and numeric_dense_slab(N, smem) != c.slab:
                out.append(f"{c}: dense accumulator in {'global' if numeric_dense_slab(N, smem) else 'shared'} memory")
        elif isinstance(c, Wrap):
            with_table = np.isin(bins[c.pass_], [b for b, t in tables[c.pass_].items() if t == c.table])
            full = with_table & (size[c.pass_] == limits[c.pass_][bins[c.pass_]])
            on_last = sg_hash(S.indices, c.table - 1) == c.table - 1
            best = np.bincount(entry_row[on_last & full[entry_row]], minlength=M).max(initial=0)
            if best < c.at_least:
                out.append(f"{c}: at most {int(best)} columns of a full row on the last slot")
        elif isinstance(c, Zeros):
            if zero is None:
                zero = reference(A, B).value == 0
            n = int((zero & (bins["numeric"][entry_row] == c.bin)).sum())
            if n < c.at_least:
                out.append(f"{c}: {n} entries")
        elif isinstance(c, Scan):
            tail = M - (scan_blocks(M) - 1) * SCAN_BLOCK
            if (scan_blocks(M), tail) != (c.blocks, c.tail):
                out.append(f"{c}: {scan_blocks(M)} blocks, {tail} rows in the last")
        else:
            raise TypeError(c)
    return out


# ---------------------------------------------------------------------------------------------------------------------
# generators
# ---------------------------------------------------------------------------------------------------------------------
class _Builder:
    """A's rows as lists of B's rows, B's rows as column sets.  Values not given (NaN) are drawn from A_EXACT and
    B_EXACT when the operands are built."""

    def __init__(self, n_cols):
        self.n_cols = n_cols
        self.b_rows, self.a_rows = [], []

    @staticmethod
    def _entries(idx, vals):
        idx = np.asarray(idx, np.int64)
        vals = np.full(len(idx), np.nan) if vals is None else np.asarray(vals, np.float64)
        o = np.argsort(idx, kind="stable")
        return idx[o], vals[o]

    def b_row(self, cols, vals=None):
        """a new row of B; returns its index (a column of A)"""
        self.b_rows.append(self._entries(cols, vals))
        return len(self.b_rows) - 1

    def a_row(self, b_ids, vals=None):
        assert len(set(np.asarray(b_ids).tolist())) == len(b_ids), "an A row names each B row once"
        self.a_rows.append(self._entries(b_ids, vals))

    def build(self, rng):
        """(A, B) in CSR; A's rows in random order, so the rows of one bin are not contiguous"""
        def csr(rows, shape, choices):
            idx = np.concatenate([r[0] for r in rows] + [np.zeros(0, np.int64)])
            val = np.concatenate([r[1] for r in rows] + [np.zeros(0)])
            draw = np.isnan(val)
            val[draw] = rng.choice(choices, int(draw.sum()))
            ptr = np.concatenate(([0], np.cumsum([len(r[0]) for r in rows], dtype=np.int64)))
            return sp.csr_matrix((val, idx, ptr), shape=shape)
        K = len(self.b_rows)
        rows = [self.a_rows[i] for i in rng.permutation(len(self.a_rows))]
        return csr(rows, (len(rows), K), A_EXACT), csr(self.b_rows, (K, self.n_cols), B_EXACT)


class _Pool:
    """B rows over disjoint column blocks of random sizes 2..96, plus single-column rows: an A row over distinct rows
    of one pool has nnz == ub"""

    def __init__(self, b, rng, cols, n_single):
        self.singles = [b.b_row([c]) for c in cols[:n_single]]
        self.ids, self.sizes, i = [], [], n_single
        while True:
            s = int(rng.integers(2, 97))
            if i + s > len(cols):
                break
            self.ids.append(b.b_row(cols[i:i + s]))
            self.sizes.append(s)
            i += s

    def row(self, rng, n):
        """B-row ids for an A row of exactly n distinct columns: blocks taken in random order while they fit, the
        rest from the single-column rows"""
        ids, left = [], n
        for i in rng.permutation(len(self.ids)):
            if left == 0:
                break
            if self.sizes[i] <= left:
                ids.append(self.ids[i])
                left -= self.sizes[i]
        assert left <= len(self.singles), "pool too small for the row"
        return ids + [self.singles[i] for i in rng.choice(len(self.singles), left, replace=False)]


def _chunked_row(b, rng, cols):
    """an A row of private B rows that split `cols` into chunks of 1..40 columns: nnz == ub == len(cols)"""
    cols = rng.permutation(np.asarray(cols))
    ids, i = [], 0
    while i < len(cols):
        s = int(rng.integers(1, 41))
        ids.append(b.b_row(cols[i:i + s]))
        i += s
    b.a_row(ids)


def _repeated_row(b, cols, ub):
    """an A row of private B rows that repeat `cols`: nnz == len(cols), ub as given"""
    d = len(cols)
    ids = [b.b_row(cols) for _ in range(ub // d)] + ([b.b_row(cols[:ub % d])] if ub % d else [])
    b.a_row(ids)


def _random_csr(rng, n_rows, n_cols, counts):
    """rows with the given entry counts and values from A_EXACT; a row's columns are a random start plus random
    gaps, so they ascend and are distinct without a per-row draw (millions of rows)"""
    counts = np.asarray(counts, np.int64)
    ptr = np.concatenate(([0], np.cumsum(counts)))
    c_max = max(1, int(counts.max(initial=0)))
    step = max(1, n_cols // (c_max + 1))
    gaps = rng.integers(1, step + 1, int(ptr[-1]))
    nz = counts > 0
    starts = ptr[:-1][nz]
    gaps[starts] = rng.integers(0, n_cols - c_max * step, len(starts))
    cs = np.cumsum(gaps)
    cols = cs - np.repeat(cs[starts] - gaps[starts], counts[nz])
    return sp.csr_matrix((rng.choice(A_EXACT, int(ptr[-1])), cols, ptr), shape=(n_rows, n_cols))


CASES = {}


def _case(name, seed):
    def reg(fn):
        def make():
            A, B, claims = fn(np.random.default_rng(seed))
            return Case(name, A, B, tuple(claims))
        CASES[name] = make
        return fn
    return reg


# rows of exactly these nnz (== ub): both sides of every numeric bin limit, and one row well above the last
EDGE_NNZ = (1, 32, 33, 128, 129, 512, 513, 4096, 4097, 8192, 8193, 12000)
EDGE_NUMERIC_BIN = {1: 1, 32: 1, 33: 2, 128: 2, 129: 3, 512: 3, 513: 4, 4096: 4, 4097: 5, 8192: 5, 8193: 6, 12000: 6}


def _numeric_edges(N, big_bin):
    def fn(rng):
        b = _Builder(N)
        pool = _Pool(b, rng, rng.permutation(N)[:16_600], 600)
        for n in EDGE_NNZ:
            for _ in range(3):
                b.a_row(pool.row(rng, n))
        claims = [Rows("numeric", EDGE_NUMERIC_BIN[n], 3, nnz=n) for n in EDGE_NNZ]
        claims += [Rows("symbolic", big_bin, 3, nnz=n) for n in (8193, 12000)]
        claims += [Rows("numeric", 6, 6, slab=big_bin == 6)]
        return (*b.build(rng), claims)
    return fn


# N = 20 000: rows above 8192 take the shared bitmask and the shared dense accumulator; N = 2 000 000: both in global memory
_case("numeric_edges_shared", 11)(_numeric_edges(20_000, 5))
_case("numeric_edges_global", 12)(_numeric_edges(2_000_000, 6))

SYMBOLIC_EDGE_UB = (33, 129, 513, 8193)


def _symbolic_above_numeric(N, big_bin):
    def fn(rng):
        b = _Builder(N)
        for ub in SYMBOLIC_EDGE_UB:
            for d in (1, 7, 32):
                for _ in range(2):
                    _repeated_row(b, rng.choice(N, d, replace=False), ub)
        sym = {33: 2, 129: 3, 513: 4, 8193: big_bin}
        claims = [Rows("symbolic", sym[ub], 6, ub=ub) for ub in SYMBOLIC_EDGE_UB]
        claims += [Rows("numeric", 1, 6, ub=ub) for ub in SYMBOLIC_EDGE_UB]
        return (*b.build(rng), claims)
    return fn


# large ub, 1-32 distinct columns: the symbolic pass takes a bigger structure than the numeric pass
_case("symbolic_above_numeric_shared", 21)(_symbolic_above_numeric(20_000, 5))
_case("symbolic_above_numeric_global", 22)(_symbolic_above_numeric(2_000_000, 6))


@_case("ub_capped_at_n", 23)
def _ub_capped_at_n(rng):
    """N = 40 and ub = 10^4: the symbolic pass bins by min(ub, N) = 40"""
    b = _Builder(40)
    for d in (1, 32, 40):
        for _ in range(3):
            _repeated_row(b, rng.choice(40, d, replace=False), 10_000)
    return (*b.build(rng), [Rows("symbolic", 2, 9, ub=10_000), Rows("numeric", 1, 6, ub=10_000),
                                  Rows("numeric", 2, 3, ub=10_000)])


@_case("probe_wraparound", 31)
def _probe_wraparound(rng):
    """every column of a row on the last slot of its table (warp tables filled to their bin limit), or every such
    column below N in a row padded with others to its bin limit (CTA tables)"""
    N = 2_000_000
    b = _Builder(N)
    every = np.arange(N)
    for table, fill in ((64, 32), (256, 128), (1024, 512), (8192, 4096), (16384, 8192)):
        hot = np.flatnonzero(sg_hash(every, table - 1) == table - 1)
        for _ in range(2):
            if len(hot) >= fill:
                cols = rng.choice(hot, fill, replace=False)
            else:
                other = np.setdiff1d(rng.choice(N, 2 * fill, replace=False), hot)
                cols = np.concatenate((hot, rng.permutation(other)[:fill - len(hot)]))
            _chunked_row(b, rng, cols)
    claims = [Wrap(p, t, n) for t, n in ((64, 32), (256, 128), (1024, 512)) for p in ("symbolic", "numeric")]
    claims += [Wrap("numeric", 8192, 244), Wrap("numeric", 16384, 122), Wrap("symbolic", 16384, 122)]
    return (*b.build(rng), claims)


@_case("bitmask_shared_reused", 41)
def _bitmask_shared_reused(rng):
    """1 600 rows with min(ub, N) > 8192 but 1 280-3 840 distinct columns (8 copies of each block): the shared
    bitmask of the symbolic pass on more rows than its 8 * SMs CTAs"""
    N = 20_000
    b = _Builder(N)
    cols = rng.permutation(N)
    blocks = [[b.b_row(cols[i:i + 64]) for _ in range(8)] for i in range(0, N - 63, 64)]
    for _ in range(1600):
        b.a_row([c for k in rng.choice(len(blocks), int(rng.integers(20, 61)), replace=False) for c in blocks[k]])
    return (*b.build(rng), [Rows("symbolic", 5, 1500, beyond_grid=True), Rows("numeric", 4, 1500)])


def _disjoint_blocks(N, n_blocks, size, n_rows, lo, hi, rng):
    """n_rows rows of lo..hi distinct blocks of `size` columns each, from n_blocks blocks scattered over N columns"""
    b = _Builder(N)
    cols = rng.permutation(N)[:n_blocks * size]
    blocks = [b.b_row(cols[i * size:(i + 1) * size]) for i in range(n_blocks)]
    for _ in range(n_rows):
        b.a_row([blocks[k] for k in rng.choice(n_blocks, int(rng.integers(lo, hi + 1)), replace=False)])
    return b.build(rng)


@_case("dense_shared_reused", 51)
def _dense_shared_reused(rng):
    """450 rows of 8 256-12 800 entries over N = 20 000: the shared dense accumulator on more rows than SMs"""
    A, B = _disjoint_blocks(20_000, 312, 64, 450, 129, 200, rng)
    return A, B, [Rows("numeric", 6, 400, beyond_grid=True, slab=False), Rows("symbolic", 5, 400)]


@_case("global_bitmask_and_slab_reused", 52)
def _global_bitmask_and_slab_reused(rng):
    """720 rows of 8 500-10 000 entries over N = 2 000 000: the global-memory bitmask (4 * SMs CTAs) and the global
    dense slab (2 GiB / 16 MB CTAs), each on more rows than CTAs"""
    A, B = _disjoint_blocks(2_000_000, 3000, 100, 720, 85, 100, rng)
    return A, B, [Rows("symbolic", 6, 700, beyond_grid=True), Rows("numeric", 6, 700, beyond_grid=True, slab=True)]


@_case("scan_many_blocks", 61)
def _scan_many_blocks(rng):
    """M = 3 000 017 rows of 0-6 products (mostly 0-3): 2 930 scan blocks, the last one partial"""
    M, K, N = 3_000_017, 40_000, 50_000
    A = _random_csr(rng, M, K, rng.choice(4, M, p=[0.25, 0.35, 0.25, 0.15]))
    B = _random_csr(rng, K, N, rng.choice(3, K, p=[0.2, 0.6, 0.2]))
    B.data = rng.choice(B_EXACT, B.nnz)
    return A, B, [Scan(2930, 721), Rows("numeric", 1, 2_000_000)]


def _scan_small(M, claim):
    def fn(rng):
        A = _random_csr(rng, M, 500, rng.integers(0, 7, M))
        B = _random_csr(rng, 500, 700, rng.integers(0, 9, 500))
        B.data = rng.choice(B_EXACT, B.nnz)
        return A, B, [claim]
    return fn


for _seed, (_m, _blocks, _tail) in enumerate(((1, 1, 1), (1023, 1, 1023), (1024, 1, 1024), (1025, 2, 1)), 62):
    _case(f"scan_m{_m}", _seed)(_scan_small(_m, Scan(_blocks, _tail)))


@_case("m_zero", 71)
def _m_zero(rng):
    B = _random_csr(rng, 10, 12, rng.integers(0, 4, 10))
    B.data = rng.choice(B_EXACT, B.nnz)
    return sp.csr_matrix((0, 10)), B, [Scan(1, 0)]


@_case("n_one", 72)
def _n_one(rng):
    """B has one column; rows with ub up to 10^4 all land on it"""
    b = _Builder(1)
    full = [b.b_row([0]) for _ in range(12_000)]
    empty = [b.b_row([]) for _ in range(50)]
    for n in (0, 1, 2, 33, 600, 10_000):
        for _ in range(2):
            b.a_row(list(rng.choice(full, n, replace=False)) + list(rng.choice(empty, 3, replace=False)))
    return (*b.build(rng), [Rows("symbolic", 1, 2, ub=10_000), Rows("numeric", 1, 10), Rows("numeric", 0, 2)])


@_case("b_empty", 73)
def _b_empty(rng):
    A = _random_csr(rng, 200, 300, rng.integers(0, 20, 200))
    B = sp.csr_matrix((300, 500))
    return A, B, [Rows("symbolic", 0, 200), Rows("numeric", 0, 200)]


@_case("ub_zero_rows", 74)
def _ub_zero_rows(rng):
    """rows whose every entry names an empty row of B, shuffled among rows with products"""
    b = _Builder(3000)
    empty = [b.b_row([]) for _ in range(400)]
    pool = _Pool(b, rng, rng.permutation(3000), 200)
    for i in range(300):
        if i % 2:
            b.a_row(list(rng.choice(empty, int(rng.integers(1, 40)), replace=False)))
        else:
            b.a_row(pool.row(rng, int(rng.integers(1, 700))) + list(rng.choice(empty, 5, replace=False)))
    return (*b.build(rng), [Rows("symbolic", 0, 150, ub=0), Rows("numeric", 0, 150)])


@_case("b_identity", 75)
def _b_identity(rng):
    """B = I and A with values uniform in [-1, 1]: C == A bit for bit, in every numeric bin"""
    N = 20_000
    row = lambda n: sp.csr_matrix((rng.uniform(-1, 1, n), np.sort(rng.choice(N, n, replace=False)), [0, n]), shape=(1, N))
    A = sp.vstack([row(n) for n in (0, 5, 40, 300, 3000, 6000, 9000) for _ in range(3)]).tocsr()
    A = A[rng.permutation(A.shape[0])]
    return A, sp.identity(N, format="csr"), [Rows("numeric", b, 3) for b in range(7)]


@_case("structural_zeros", 81)
def _structural_zeros(rng):
    """three entries per row that are present in C with value 0: 1 * 0.5 + 1 * (-0.5), a * 0.0 and 0.0 * b"""
    N = 20_000
    b = _Builder(N)
    cols = rng.permutation(N)
    pool = _Pool(b, rng, cols[:18_000], 600)
    spare = iter(cols[18_000:])
    for n in (10, 100, 400, 2000, 6000, 9000):
        for _ in range(2):
            j1, j2, j3 = next(spare), next(spare), next(spare)
            ids = pool.row(rng, n - 3)
            zero = [b.b_row([j1], [0.5]), b.b_row([j1], [-0.5]), b.b_row([j2], [0.0]), b.b_row([j3])]
            b.a_row(ids + zero, [np.nan] * len(ids) + [1.0, 1.0, np.nan, 0.0])
    return (*b.build(rng), [Zeros(k, 6) for k in range(1, 7)])


NAMES = tuple(CASES)


def build(name):
    return CASES[name]()
