"""CPU restatement of the reference's CholInv / CholeskyQR2 hot path.  TEST INFRASTRUCTURE ONLY.

Nothing in the product path (capital_b200/, the C-ABI library, bench.py's GPU arm) may import this
module; it is the checker used by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg.

Each function cites the reference file:line it restates (paths relative to /root/reference).  The
restatement is pinned two ways (tests/test_oracle.py): against the golden dumps produced by the
reference itself, compiled here by oracle/build_ref.sh (tests/golden/*.npz, made by
tests/golden/make_golden.py), and against scipy's LAPACK on the same closed-form inputs.
All arithmetic is FP64; leaves are numpy/scipy BLAS/LAPACK exactly as the reference's leaves are
MKL's (blas/interface.hpp:43-97, lapack/interface.hpp:30-58).
"""
from __future__ import annotations

import json
import math
import numpy as np
import scipy.linalg as sla

_A = 0x5DEECE66D
_C = 0xB
_M48 = (1 << 48) - 1


# --------------------------------------------------------------------------------------------------
# generators  (src/matrix/structure.hpp:69-129)
# --------------------------------------------------------------------------------------------------
def drand48_first(seed: np.ndarray) -> np.ndarray:
    """First drand48() after srand48(seed), vectorised.  glibc: X0 = (seed & 0xFFFFFFFF) << 16 | 0x330E,
    X1 = (a*X0 + c) mod 2^48, value = X1 / 2^48.  Used by _distribute_symmetric (structure.hpp:80-85),
    which re-seeds per element."""
    seed = np.asarray(seed, dtype=np.uint64)
    x0 = ((seed & np.uint64(0xFFFFFFFF)) << np.uint64(16)) | np.uint64(0x330E)
    # 48-bit modular multiply without overflow: split a into 24-bit halves
    a_lo = np.uint64(_A & 0xFFFFFF)
    a_hi = np.uint64(_A >> 24)
    m48 = np.uint64(_M48)
    lo = (x0 * a_lo) & m48
    hi = ((x0 * a_hi) & np.uint64(0xFFFFFF)) << np.uint64(24)
    x1 = (lo + hi + np.uint64(_C)) & m48
    return x1.astype(np.float64) / float(1 << 48)


def spd_global(n: int) -> np.ndarray:
    """Global n x n matrix of A.distribute_symmetric(..., diagonallyDominant=true)
    (structure.hpp:69-103; bench/cholesky/cholinv.cpp:40).  Element (row gy, col gx) is the first
    drand48 after srand48(max(gx,gy) + n*min(gx,gy)); the diagonal gets +n.  Grid-independent."""
    g = np.arange(n, dtype=np.uint64)
    gx, gy = np.meshgrid(g, g, indexing="xy")  # gx = column, gy = row
    hi = np.maximum(gx, gy)
    lo = np.minimum(gx, gy)
    a = drand48_first(hi + np.uint64(n) * lo)
    a[np.arange(n), np.arange(n)] += float(n)
    return a


def local_dim(glob: int, grid: int) -> int:
    """matrix.hpp:8-11: local dimension = ceil(global / grid)."""
    return glob // grid + (1 if glob % grid else 0)


def cyclic_local(a: np.ndarray, d_cols: int, d_rows: int, x: int, y: int) -> np.ndarray:
    """Local block of the element-cyclic distribution (matrix.hpp:6-19): process column x owns global
    columns x, x+d_cols, ...; process row y owns rows y, y+d_rows, ...  Zero padded to ceil dims
    (structure.hpp:92-100).  Returned column-major-in-memory (Fortran order) like the reference."""
    rows, cols = a.shape
    lr, lc = local_dim(rows, d_rows), local_dim(cols, d_cols)
    out = np.zeros((lr, lc), dtype=np.float64, order="F")
    blk = a[y::d_rows, x::d_cols]
    out[: blk.shape[0], : blk.shape[1]] = blk
    return out


def cyclic_assemble(blocks: dict, rows: int, cols: int, d_cols: int, d_rows: int) -> np.ndarray:
    """Inverse of cyclic_local: blocks[(x, y)] -> global matrix."""
    a = np.zeros((rows, cols), dtype=np.float64)
    for (x, y), blk in blocks.items():
        sub = a[y::d_rows, x::d_cols]
        sub[...] = blk[: sub.shape[0], : sub.shape[1]]
    return a


def spd_local(n: int, d: int, x: int, y: int) -> np.ndarray:
    """Local block of distribute_symmetric on process (x, y) of a d x d face."""
    return cyclic_local(spd_global(n), d, d, x, y)


def lcg_stream(key: int, count: int) -> np.ndarray:
    """`count` successive drand48() draws after srand48(key) (structure.hpp:108-117), vectorised by
    jump-ahead: X_k = a^k X_0 + c (a^k - 1)/(a - 1)  (mod 2^48)."""
    x0 = ((key & 0xFFFFFFFF) << 16) | 0x330E
    # sequential in python ints is too slow for 10^7 draws; do block jump-ahead with numpy uint64
    out = np.empty(count, dtype=np.uint64)
    # multipliers a^k, increments c_k for k = 1..B via doubling
    B = 1 << 12
    ak = np.empty(B, dtype=object)
    ck = np.empty(B, dtype=object)
    a, c = 1, 0
    for k in range(B):
        a, c = (a * _A) & _M48, (c * _A + _C) & _M48
        ak[k], ck[k] = a, c
    ak_u = np.array([int(v) for v in ak], dtype=np.uint64)
    ck_u = np.array([int(v) for v in ck], dtype=np.uint64)
    a_lo = ak_u & np.uint64(0xFFFFFF)
    a_hi = ak_u >> np.uint64(24)
    m48 = np.uint64(_M48)
    x = x0
    pos = 0
    while pos < count:
        nb = min(B, count - pos)
        xv = np.uint64(x)
        lo = (xv * a_lo[:nb]) & m48
        hi = ((xv * a_hi[:nb]) & np.uint64(0xFFFFFF)) << np.uint64(24)
        blk = (lo + hi + ck_u[:nb]) & m48
        out[pos : pos + nb] = blk
        x = int(blk[nb - 1])
        pos += nb
    return out.astype(np.float64) / float(1 << 48)


def random_local(m: int, n: int, c: int, d: int, x: int, y: int, key: int) -> np.ndarray:
    """Local block of A.distribute_random(x, y, c, d, key) for an m x n (rows x cols) matrix on a grid of
    c process columns x d process rows (structure.hpp:106-129; bench/qr/cacqr.cpp:33-34, key = rank/c).
    The stream is consumed column by column over the un-padded local extent; pad cells are zero."""
    lr, lc = local_dim(m, d), local_dim(n, c)
    pad_c = lc - 1 if (n % c != 0 and (lc - 1) * c + x >= n) else lc
    pad_r = lr - 1 if (m % d != 0 and (lr - 1) * d + y >= m) else lr
    vals = lcg_stream(key, pad_c * pad_r).reshape(pad_c, pad_r).T  # column-major fill
    out = np.zeros((lr, lc), dtype=np.float64, order="F")
    out[:pad_r, :pad_c] = vals
    return out


# --------------------------------------------------------------------------------------------------
# topology  (src/util/topology.h)
# --------------------------------------------------------------------------------------------------
def topo_square(size: int, rank: int, c: int) -> dict:
    """topo::square, layout 0 (topology.h:76-83): d = ceil(sqrt(size/c)); z = r mod c;
    x = (r mod (c d)) div c; y = r div (c d)."""
    d = int(round(math.ceil(math.sqrt(size // c))))
    return dict(size=size, rank=rank, c=c, d=d, z=rank % c, x=(rank % (c * d)) // c, y=rank // (c * d))


def topo_rect(size: int, rank: int, c: int) -> dict:
    """topo::rect (topology.h:46-50): d = size / c^2; z = r mod c; x = (r mod c^2) div c; y = r div c^2."""
    return dict(size=size, rank=rank, c=c, d=size // (c * c), z=rank % c, x=(rank % (c * c)) // c, y=rank // (c * c))


def transpose_partner(t: dict) -> int:
    """util::transpose partner for layout 0 (util.hpp:237-238): rank of (y, x, z)."""
    return t["x"] * t["c"] * t["d"] + t["y"] * t["c"] + t["z"]


# --------------------------------------------------------------------------------------------------
# packed storage  (src/matrix/structure.h:13,37-39)
# --------------------------------------------------------------------------------------------------
def pack_upper(loc: np.ndarray) -> np.ndarray:
    """rect (col-major) -> uppertri packed: element (col i, row j<=i) at i(i+1)/2 + j."""
    n = loc.shape[0]
    return np.concatenate([loc[: i + 1, i] for i in range(n)]) if n else np.zeros(0)


def unpack_upper(packed: np.ndarray, n: int) -> np.ndarray:
    out = np.zeros((n, n), dtype=np.float64, order="F")
    off = 0
    for i in range(n):
        out[: i + 1, i] = packed[off : off + i + 1]
        off += i + 1
    return out


def load_dump(path: str):
    """(meta, {name: array}) of a reference dump (tests/golden/*.npz).  Blocks that a rank holds identically to a lower rank
    (replicas along z) are stored once; `same_as` names the stored copy of each omitted block."""
    z = np.load(path)
    arrs = {k: z[k] for k in z.files if k not in ("meta", "same_as")}
    if "same_as" in z.files:
        arrs.update({k: arrs[v] for k, v in json.loads(str(z["same_as"])).items()})
    return json.loads(str(z["meta"])), arrs


# --------------------------------------------------------------------------------------------------
# CholInv  (src/alg/cholesky/cholinv/cholinv.hpp)
# --------------------------------------------------------------------------------------------------
def bc_dimension(local_dim_: int, c: int, d: int, bc_mult_dim: int) -> int:
    """Global base-case size, cholinv.hpp:15-18."""
    bc = c * d
    if bc_mult_dim < 0:
        bc <<= -bc_mult_dim
    else:
        bc >>= bc_mult_dim
    bc = max(1, bc)
    bc = min(local_dim_, bc)
    return d * (local_dim_ // bc)


def _base_case(a_blk: np.ndarray):
    """potrf('U') then trtri('U','N') on the gathered dense block (cholinv/policy.h:199-201)."""
    r = sla.cholesky(a_blk, lower=False, check_finite=False)
    rinv, info = sla.lapack.dtrtri(r, lower=0, unitdiag=0)
    assert info == 0
    return np.triu(r), np.triu(rinv)


def cholinv(a: np.ndarray, complete_inv: bool, split: int, bc_dim: int, d: int = 1):
    """Global-view restatement of cholinv::invoke (cholinv.hpp:87-165) on an n x n SPD matrix whose upper
    triangle is read.  Returns (R, Rinv), both upper triangular (A = R^T R).  With complete_inv false the
    top-level block Rinv[0:n1, n1:] stays zero (cholinv.hpp:147).  `d` is the process-face edge: the
    recursion splits the LOCAL dimension (localDim >> split, :92,107) so global split points are d * that."""
    n = a.shape[0]
    w = np.triu(a).copy()
    r = np.zeros_like(w)
    ri = np.zeros_like(w)

    def invoke(lo: int, hi: int, top: bool):
        glob = hi - lo
        loc = glob // d
        s1 = loc >> split
        if glob <= bc_dim or s1 < split:  # cholinv.hpp:93
            blk = w[lo:hi, lo:hi]
            full = blk + np.triu(blk, 1).T
            r[lo:hi, lo:hi], ri[lo:hi, lo:hi] = _base_case(full)
            return
        mid = lo + s1 * d
        invoke(lo, mid, False)  # :107-111
        # "trsm": R12 = Rinv11^T A12 (:116-122)
        r[lo:mid, mid:hi] = ri[lo:mid, lo:mid].T @ w[lo:mid, mid:hi]
        # "tmu": A22 -= R12^T R12 (:131-134)
        w[mid:hi, mid:hi] -= np.triu(r[lo:mid, mid:hi].T @ r[lo:mid, mid:hi])
        invoke(mid, hi, False)  # :139-142
        if not ((not complete_inv) and top):  # :147
            t = ri[lo:mid, lo:mid] @ r[lo:mid, mid:hi]  # :151
            ri[lo:mid, mid:hi] = -(t @ ri[mid:hi, mid:hi])  # :152-155

    invoke(0, n, True)
    return r, ri


def cholesky_residual(a: np.ndarray, r: np.ndarray) -> float:
    """test/cholesky/validate.hpp:7-49 + util::residual_local (util.hpp:25-53):
    sqrt(sum_{upper} (R^T R - A)^2) / sqrt(sum_{upper} A^2)."""
    e = np.triu(r.T @ r - a)
    return float(np.sqrt((e * e).sum()) / np.sqrt((np.triu(a) ** 2).sum()))


# --------------------------------------------------------------------------------------------------
# CholeskyQR2, 1D  (src/alg/qr/cacqr/cacqr.hpp:5-29,172-193; policy.h:78-85)
# --------------------------------------------------------------------------------------------------
def cacqr_1d(blocks: list, num_iter: int = 2):
    """blocks[r] = local rows of rank r (cyclic over d = len(blocks) process rows, c = 1).
    Returns (Q blocks, R) with R the n x n upper factor held by every rank."""
    qs = [np.array(b, dtype=np.float64, order="F") for b in blocks]

    def sweep():
        g = sum(np.triu(q.T @ q) for q in qs)  # dsyrk 'U','T' + Allreduce (cacqr.hpp:15, policy.h:82)
        r = sla.cholesky(g + np.triu(g, 1).T, lower=False, check_finite=False)  # :20
        rinv, info = sla.lapack.dtrtri(r, lower=0, unitdiag=0)  # :22
        assert info == 0
        for i in range(len(qs)):
            qs[i] = qs[i] @ np.triu(rinv)  # dtrmm R/U/N (:25)
        return np.triu(r)

    r1 = sweep()
    if num_iter > 1:
        r2 = sweep()
        return qs, np.triu(r2 @ r1)  # R = R2 R1 (:185-187)
    return qs, r1


# --------------------------------------------------------------------------------------------------
# CA-CholeskyQR2 on the 3D grid, c == d  (src/alg/qr/cacqr/cacqr.hpp:75-120,195-215; solve: :46-71)
# --------------------------------------------------------------------------------------------------
def cacqr_3d(a: np.ndarray, c: int, num_iter: int, complete_inv: bool, split: int, bc_mult_dim: int):
    """Global-view restatement of invoke_3d / sweep_3d for an m x n matrix on a c x c x c grid.  Per sweep: Gram matrix G = Q^T Q
    (row Bcast + gemm + column Reduce + depth Bcast, :92-99), cholinv::factor on G over the same grid (:103), then either
    Q <- Q R^-1 (complete_inv, summa trmm Right/Upper, :106-111) or the block `solve` (:46-71): with n1 = (localN >> split) * c,
    Q1 <- Q1 Rinv11, Q2 <- (Q2 - Q1 R12) Rinv22 -- which needs only the two diagonal blocks of the inverse, the ones
    complete_inv = 0 leaves cholinv to compute.  Two sweeps: R = R2 R1 (:203-209).  Returns (Q, R)."""
    n = a.shape[1]
    q = np.array(a, dtype=np.float64)
    bc = bc_dimension(local_dim(n, c), c, c, bc_mult_dim)

    def sweep():
        g = q.T @ q
        r, ri = cholinv(g, complete_inv, split, bc, c)
        if complete_inv:
            q[...] = q @ ri
        else:
            n1 = (local_dim(n, c) >> split) * c
            q1 = q[:, :n1] @ ri[:n1, :n1]
            q[:, n1:] = (q[:, n1:] - q1 @ r[:n1, n1:]) @ ri[n1:, n1:]
            q[:, :n1] = q1
        return r

    r1 = sweep()
    if num_iter > 1:
        r2 = sweep()
        return q, np.triu(r2 @ r1)
    return q, r1


def qr_residual(a: np.ndarray, q: np.ndarray, r: np.ndarray) -> float:
    """test/qr/validate.hpp:37-52: ||QR - A||_F / ||A||_F."""
    return float(np.linalg.norm(q @ r - a) / np.linalg.norm(a))


def qr_orthogonality(q: np.ndarray) -> float:
    """test/qr/validate.hpp:7-35: ||Q^T Q - I||_F / sqrt(n^2) (control = 1 per entry)."""
    n = q.shape[1]
    return float(np.linalg.norm(q.T @ q - np.eye(n)) / math.sqrt(n * n))
