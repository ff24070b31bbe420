"""Pin the CPU restatement (oracle/capital_oracle.py) against the reference's own outputs
(tests/golden/*.npz, dumped by the reference compiled in oracle/_ref) and against LAPACK."""
import os
import numpy as np
import pytest
import scipy.linalg as sla
from oracle import capital_oracle as co

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def load(name):
    return co.load_dump(os.path.join(GOLD, name + ".npz"))


def test_drand48_known_answers():
    # SURVEY 8d probe values: A[0,0] = n + 0.170828..., A[1,0] = 0.041630... (seed 1 + n*0 = 1)
    assert abs(co.drand48_first(np.array([0]))[0] - 0.17082803610628972) < 1e-15
    assert abs(co.drand48_first(np.array([1]))[0] - 0.0416303447718782) < 1e-15
    a = co.spd_global(8)
    assert np.allclose(a, a.T) and abs(a[0, 0] - 8.170828036106290) < 1e-12


@pytest.mark.parametrize("name", ["cholinv_p1_n96_ci1", "cholinv_p1_n128_ci0", "cholinv_p8_n128_ci0", "cholinv_p8_n192_ci1",
                                  "cholinv_p1_n128_ci0_split2", "cholinv_p8_n256_ci1_split2"])
def test_generator_and_cholinv_match_reference(name):
    meta, z = load(name)
    n, P, c, d = meta["n"], meta["P"], meta["c"], meta["d"]
    a = co.spd_global(n)
    L = co.local_dim(n, d)
    bc = co.bc_dimension(L, c, d, meta["bc_mult_dim"])
    assert bc == meta["bc_dim"]
    r, ri = co.cholinv(a, bool(meta["complete_inv"]), meta["split"], bc, d)
    assert co.cholesky_residual(a, r) < 1e-14
    for rank in range(P):
        t = co.topo_square(P, rank, c)
        # generator: bit-exact
        assert np.array_equal(z[f"A_{rank}"].reshape(L, L, order="F"), co.spd_local(n, d, t["x"], t["y"]))
        # factors: reference packed-upper local blocks vs restatement (unique factors -> elementwise)
        r_ref = co.unpack_upper(z[f"R_{rank}"], L)
        ri_ref = co.unpack_upper(z[f"Rinv_{rank}"], L)
        r_loc = np.triu(co.cyclic_local(r, d, d, t["x"], t["y"]))
        ri_loc = np.triu(co.cyclic_local(ri, d, d, t["x"], t["y"]))
        if t["y"] > t["x"]:  # local diagonal is a global-lower element there: must be zero (SURVEY App. A)
            assert np.all(np.diag(r_ref) == 0) and np.all(np.diag(ri_ref) == 0)
        assert np.abs(r_ref - r_loc).max() <= 1e-13 * np.abs(r).max()
        assert np.abs(ri_ref - ri_loc).max() <= 1e-13 * np.abs(ri).max()


def test_cholinv_vs_lapack_and_incomplete_inverse():
    n = 160
    a = co.spd_global(n)
    r, ri = co.cholinv(a, True, 1, 20)
    assert np.abs(r - sla.cholesky(a)).max() < 1e-13
    assert np.abs(ri @ r - np.eye(n)).max() < 1e-14
    r0, ri0 = co.cholinv(a, False, 1, 20)
    assert np.array_equal(r0, r)
    h = n // 2
    assert np.all(ri0[:h, h:] == 0) and np.array_equal(ri0[:h, :h], ri[:h, :h]) and np.array_equal(ri0[h:, h:], ri[h:, h:])


@pytest.mark.parametrize("name", ["cacqr_p1_m512_n32", "cacqr_p8_1d_m1024_n32", "cacqr_p8_1d_m1024_n32_it1"])
def test_cacqr_1d_matches_reference(name):
    meta, z = load(name)
    m, n, P, c, d = meta["m"], meta["n"], meta["P"], meta["c"], meta["d"]
    lr = co.local_dim(m, d)
    blocks = []
    for rank in range(P):
        t = co.topo_rect(P, rank, c)
        loc = co.random_local(m, n, c, d, t["x"], t["y"], rank // c)
        assert np.array_equal(z[f"A_{rank}"].reshape(lr, n, order="F"), loc)  # generator bit-exact
        blocks.append(loc)
    qs, r = co.cacqr_1d(blocks, meta["variant"])  # the driver's `variant` is num_iter (cacqr.h info::num_iter)
    a = co.cyclic_assemble({(0, y): blocks[y] for y in range(P)}, m, n, 1, d)
    q = co.cyclic_assemble({(0, y): qs[y] for y in range(P)}, m, n, 1, d)
    # one sweep (CholeskyQR) loses orthogonality with cond(A)^2 eps; two sweeps recover it
    assert co.qr_residual(a, q, r) < 1e-14 and co.qr_orthogonality(q) < (1e-15 if meta["variant"] > 1 else 1e-13)
    for rank in range(P):
        if meta["variant"] > 1:
            assert np.abs(co.unpack_upper(z[f"R_{rank}"], n) - r).max() < 1e-12 * np.abs(r).max()
        else:
            # reference quirk: with num_iter = 1 invoke_1d never finalises R (SP::complete_1d sits in the num_iter > 1 branch,
            # cacqr.hpp:180-188) -- args.R comes back holding the Gram matrix (its own validator reads a residual of 65).  Q is right.
            g = np.triu(a.T @ a)
            assert np.abs(co.unpack_upper(z[f"R_{rank}"], n) - g).max() < 1e-12 * np.abs(g).max()
            assert meta["residual"] > 1.0
        assert np.abs(z[f"Q_{rank}"].reshape(lr, n, order="F") - qs[rank]).max() < 1e-12


def test_cacqr_3d_golden_is_consistent():
    """3D (c = d = 2) dump: Q blocks re-assemble to an orthonormal basis with Q R = A."""
    meta, z = load("cacqr_p8_3d_m256_n64")
    m, n, P, c, d = meta["m"], meta["n"], meta["P"], meta["c"], meta["d"]
    lr, lc = co.local_dim(m, d), co.local_dim(n, c)
    ab, qb, rb = {}, {}, {}
    for rank in range(P):
        t = co.topo_rect(P, rank, c)
        loc = co.random_local(m, n, c, d, t["x"], t["y"], rank // c)
        assert np.array_equal(z[f"A_{rank}"].reshape(lr, lc, order="F"), loc)
        if t["z"] == 0:
            ab[(t["x"], t["y"])] = loc
            qb[(t["x"], t["y"])] = z[f"Q_{rank}"].reshape(lr, lc, order="F")
    a = co.cyclic_assemble(ab, m, n, c, d)
    q = co.cyclic_assemble(qb, m, n, c, d)
    assert co.qr_orthogonality(q) < 1e-15
    r = np.triu(q.T @ a)
    assert co.qr_residual(a, q, r) < 1e-14


def test_topology_and_layout_helpers():
    t = co.topo_square(8, 5, 2)
    assert (t["d"], t["x"], t["y"], t["z"]) == (2, 0, 1, 1)
    assert co.transpose_partner(t) == 3  # (x=1,y=0,z=1) -> rank 1*1 + ... = y*cd + x*c + z
    a = np.arange(35.0).reshape(5, 7)
    blocks = {(x, y): co.cyclic_local(a, 3, 2, x, y) for x in range(3) for y in range(2)}
    assert np.array_equal(co.cyclic_assemble(blocks, 5, 7, 3, 2), a)
    u = np.triu(np.arange(16.0).reshape(4, 4))
    assert np.array_equal(co.unpack_upper(co.pack_upper(u), 4), u)


def test_reference_solve_path_yields_the_same_q():
    """cacqr::solve (complete_inv = 0, cacqr.hpp:46-71: block forward substitution with the two diagonal inverse blocks) against the
    reference's own complete_inv = 1 run on the same input: Q agrees to rounding, so applying the complete inverse -- what
    capital_b200's 3D sweep always does (dist.cu) -- is within tolerance of BOTH reference paths.  The multi-GPU tests compare the
    GPU result against each dump."""
    (m0, z0), (_, z1) = load("cacqr_p8_3d_m256_n64_ci0"), load("cacqr_p8_3d_m256_n64")
    assert m0["residual"] < 1e-14 and m0["orthogonality"] < 1e-15
    for r in range(8):
        assert np.array_equal(z0[f"A_{r}"], z1[f"A_{r}"])
        assert np.abs(z0[f"Q_{r}"] - z1[f"Q_{r}"]).max() < 1e-15
        assert np.abs(z0[f"R_{r}"] - z1[f"R_{r}"]).max() <= 1e-13 * np.abs(z1[f"R_{r}"]).max()


@pytest.mark.parametrize("name", ["cacqr_p8_3d_m256_n64", "cacqr_p8_3d_m256_n64_ci0"])
def test_cacqr_3d_restatement_matches_reference(name):
    """the numpy restatement of invoke_3d / sweep_3d / solve against the reference's per-rank dumps, elementwise"""
    meta, z = load(name)
    m, n, P, c, d = meta["m"], meta["n"], meta["P"], meta["c"], meta["d"]
    ci = 0 if name.endswith("ci0") else 1
    lr, lc = co.local_dim(m, d), co.local_dim(n, c)
    ab, qb, rb = {}, {}, {}
    for rank in range(P):
        t = co.topo_rect(P, rank, c)
        if t["z"] == 0:
            ab[(t["x"], t["y"])] = z[f"A_{rank}"].reshape(lr, lc, order="F")
            qb[(t["x"], t["y"])] = z[f"Q_{rank}"].reshape(lr, lc, order="F")
        s = co.topo_square(P, rank, c)
        if s["z"] == 0:
            rb[(s["x"], s["y"])] = co.unpack_upper(z[f"R_{rank}"], lc)
    a = co.cyclic_assemble(ab, m, n, c, d)
    q_ref = co.cyclic_assemble(qb, m, n, c, d)
    r_ref = np.triu(co.cyclic_assemble(rb, n, n, c, c))
    q, r = co.cacqr_3d(a, c, 2, bool(ci), 1, -1)
    assert np.abs(q - q_ref).max() < 1e-13
    assert np.abs(r - r_ref).max() < (1e-13 if ci else 1e-12) * np.abs(r_ref).max()
    assert co.qr_residual(a, q, r) < 1e-14 and co.qr_orthogonality(q) < 1e-15


def test_tf32_gates_have_headroom_over_the_emulated_rounding():
    """tests/test_gpu_zz_late.py gates the experimental TF32 trailing update against the FP64 results; the gates must sit well above what
    a faithful implementation produces.  tools/tf32_emulate.py restates the kernel's arithmetic in numpy (cvt.rna.tf32 on the operands,
    FP32 accumulation, optional hi + lo split)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("tf32_emulate", os.path.join(os.path.dirname(GOLD), "..", "tools", "tf32_emulate.py"))
    em = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(em)
    a = co.spd_global(512)
    res = {p: co.cholesky_residual(a, em.cholesky(a, 64, p, 128)) for p in (0, 1, 3)}
    assert res[0] < 1e-15 and 1e-13 < res[1] < 1e-7 and res[3] < 1e-9
    rng = np.random.default_rng(1)
    A, B = rng.standard_normal((1024, 96)), rng.standard_normal((1024, 160))
    ref, den = A.T @ B, (np.abs(A).T @ np.abs(B)).max()
    assert np.abs(em.product(A, B, 1) - ref).max() / den < 5e-4 / 4
    assert np.abs(em.product(A, B, 3) - ref).max() / den < 2e-6 / 4
