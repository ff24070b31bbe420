"""CholeskyQR2's Gram product at every chunk geometry of the split-K launch, and results that do not depend on earlier calls.

The Gram matrix G = Q^T Q of every 1D sweep, and the Q^T Q - I of the validator, come from gemm_tn_splitk: the k range (the rows
of Q) is cut into `ks` chunks, each chunk stores its partial tile into a grow-only workspace and a second kernel adds the chunks in
order.  The number of chunks depends on the SM count, the tile size, the output's structure flag and k, so the same routine runs
at very different geometries -- one chunk, many full chunks, and chunks that get no k-tile at all (`(ks - 1) * per >= nk`).  The
suite's other QR shapes miss the last kind, where a chunk that skipped its store would let the reduction add a partial sum that an
earlier call left in the workspace.

Here a shape picker aims at each geometry for both tile configurations (128 x 128, 64 x 64) and both structure flags (C_UPPER for
the factor's Gram, none for the validator's), and every result is compared with the numpy restatement
`oracle.capital_oracle.cacqr_1d` (pinned to the reference's dumps) and with numpy norms of the returned factors.  Before a target
with an empty chunk, a *primer* (same n, same number of chunks, none of them empty) runs through factor and validate on the same
context, so that every slice of the workspace holds a real partial sum: a chunk that does not store its slice then corrupts G by a
whole chunk's worth, whatever the allocator returned.

Shapes the picker chose on a B200 (148 SMs), rows m x columns n, primer rows in brackets:
  128 x 128 tiles: 500 x 256 (one chunk), 32768 x 256 (full), 25700 x 256 (factor's Gram has an empty chunk) [131072],
                   19000 x 256 (validator's Gram has an empty chunk) [131072], 25701 x 200 (factor's Gram, odd rows) [131072],
                   8192 x 520 (full; Gram larger than one cluster base case)
  64 x 64 tiles:   500 x 64 (one chunk), 65857 x 100 (full), 51000 x 100 (factor's Gram) [131072],
                   38000 x 100 (validator's Gram) [131072], 152001 x 64 (both Grams) [151041]
"""
import functools
import math

import numpy as np
import pytest
import torch

import capital_b200 as cb
from oracle import capital_oracle as co

gpu = pytest.mark.gpu
KEY = 17  # distribute_random key of every target


# ---- shape picker ------------------------------------------------------------------------------------------------------------
# A copy of the chunk rule of gemm_tn_splitk (capital_b200/csrc/gemm_tn.cu) as it stood when these tests were written.  It only
# CHOOSES shapes; the library may change its rule (for instance never launch an empty chunk) and the tests still hold at these shapes.
def splitk_chunks(n, k, upper, sms):
    """(ks, per, empty) of the n x n Gram product over k rows: number of chunks, k-tiles (16 rows) per chunk, chunks with no k-tile."""
    big = n >= 128
    g = math.ceil(n / (128 if big else 64))
    tiles = g * (g + 1) // 2 if upper else g * g  # with C_UPPER the tiles below the diagonal return at once
    ks = max(1, min(math.ceil(sms * (1 if big else 2) / tiles), math.ceil(k / 512)))  # at least 32 k-tiles per chunk
    nk = math.ceil(k / 16)
    per = math.ceil(nk / ks)
    return ks, per, ks - math.ceil(nk / per)


FLAGS = {"factor": True, "validator": False}  # Gram of the factor's sweeps (C_UPPER) / of the validator (no structure)


def _geometry(n, m, sms):
    return {f: splitk_chunks(n, m, u, sms) for f, u in FLAGS.items()}


KINDS = {
    "ks1": lambda c: all(ks == 1 for ks, _, _ in c.values()),
    "full": lambda c: all(ks > 1 and e == 0 for ks, _, e in c.values()),
    "factor_empty": lambda c: c["factor"][2] > 0,
    "validator_empty": lambda c: c["validator"][2] > 0,
    "both_empty": lambda c: c["factor"][2] > 0 and c["validator"][2] > 0,
}
# name: (n, kind, first m tried, odd rows only)
CASES = {
    "t128-ks1": (256, "ks1", 500, False),
    "t128-full": (256, "full", 32768, False),
    "t128-factor-empty": (256, "factor_empty", 25700, False),
    "t128-validator-empty": (256, "validator_empty", 19000, False),
    "t128-factor-empty-odd": (200, "factor_empty", 25701, True),  # odd rows: the Gram reads an aligned copy of A
    "t128-recursive": (520, "full", 8192, False),  # n > 512: the 1D path factors the Gram matrix by recursion
    "t64-ks1": (64, "ks1", 500, False),
    "t64-full": (100, "full", 65536, False),
    "t64-factor-empty": (100, "factor_empty", 51000, False),
    "t64-validator-empty": (100, "validator_empty", 38000, False),
    "t64-both-empty": (64, "both_empty", 152001, False),
}
EMPTY_CASES = [k for k, v in CASES.items() if v[1].endswith("empty")]
PRIMER_START = 131072


@functools.lru_cache(maxsize=None)
def pick(name, sms):
    """(m, n, primer rows or None) of case `name` on a device with `sms` SMs."""
    n, kind, start, odd = CASES[name]
    m = next((m for m in range(start, 4 * start) if (m % 2 or not odd) and KINDS[kind](_geometry(n, m, sms))), None)
    assert m is not None, f"{name}: no shape of kind {kind} in [{start}, {4 * start}) at {sms} SMs"
    target = _geometry(n, m, sms)
    empty = [f for f, (_, _, e) in target.items() if e]
    if not empty:
        return m, n, None
    for p in range(PRIMER_START, 4 * PRIMER_START):
        c = _geometry(n, p, sms)
        if all(e == 0 for _, _, e in c.values()) and all(c[f][0] == target[f][0] for f in empty):
            return m, n, p
    raise AssertionError(f"{name}: no primer for {m} x {n} at {sms} SMs")


@pytest.fixture(scope="module")
def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---- helpers -----------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=4)
def oracle(m, n, it):
    a = co.random_local(m, n, 1, 1, 0, 0, KEY)
    qs, r = co.cacqr_1d([a], it)
    return a, qs[0], r


def factor(topo, m, n, it=2, host=False, serialize=True, key=KEY):
    A = cb.matrix(n, m, 1, 1).distribute_random(topo, key)
    if host:
        A = cb.matrix(n, m, 1, 1, data=A.data.cpu().pin_memory())
    args = cb.cacqr.info(it, cb.cholinv.info(0, 1, 0, "U"), serialize=serialize)
    cb.cacqr.factor(A, args, topo)
    return A, args


def prime(topo, n, rows):
    """factor + validate at the primer shape: every chunk slice of the split-K workspace then holds a partial sum of this call."""
    A, args = factor(topo, rows, n, key=KEY + 1)
    cb.cacqr.validate(A, args, topo)


def check_against_oracle(m, n, it, Q, R, validated):
    a, q_o, r_o = oracle(m, n, it)
    res, orth = validated
    Q, R = Q.cpu().numpy(), R.cpu().numpy()
    err_r = np.abs(R - r_o).max() / np.abs(r_o).max()
    assert err_r < 1e-11, f"R differs from the oracle by {err_r:.2e} of max|R|"
    err_q = np.abs(Q - q_o).max()
    assert err_q < 1e-11, f"Q differs from the oracle by {err_q:.2e}"
    res_np, orth_np = co.qr_residual(a, Q, R), co.qr_orthogonality(Q)
    assert abs(res - res_np) < 1e-15, f"validate residual {res:.3e}, numpy {res_np:.3e}"
    assert abs(orth - orth_np) < 1e-15, f"validate orthogonality {orth:.3e}, numpy {orth_np:.3e}"


def result(A, args, topo):
    Q, R = cb.cacqr.construct_Q(args).clone(), cb.cacqr.construct_R(args).clone()
    return Q, R, cb.cacqr.validate(A, args, topo)


# ---- CPU: the picker aims at what the GPU cases exist for --------------------------------------------------------------------
def test_shape_picker_aims_at_each_chunk_geometry():
    sms = 148  # B200
    assert splitk_chunks(256, 25700, True, sms) == (50, 33, 1)  # chunk 49 would start at k-tile 1617 of 1607
    covered = set()
    for name, (n, kind, _, odd) in CASES.items():
        m, n, primer = pick(name, sms)
        c = _geometry(n, m, sms)
        assert KINDS[kind](c) and (m % 2 == 1 or not odd), name
        for f, (_, _, e) in c.items():
            if e:
                covered.add((128 if n >= 128 else 64, f))
        assert (primer is not None) == any(e for _, _, e in c.values()), name
        if primer is not None:
            p = _geometry(n, primer, sms)
            assert all(e == 0 for _, _, e in p.values()), name
            assert all(p[f][0] == c[f][0] for f in c if c[f][2]), name
    assert covered == {(t, f) for t in (128, 64) for f in FLAGS}
    # the shapes listed in the module docstring
    assert {k: pick(k, sms) for k in CASES} == {
        "t128-ks1": (500, 256, None), "t128-full": (32768, 256, None), "t128-factor-empty": (25700, 256, 131072),
        "t128-validator-empty": (19000, 256, 131072), "t128-factor-empty-odd": (25701, 200, 131072), "t128-recursive": (8192, 520, None),
        "t64-ks1": (500, 64, None), "t64-full": (65857, 100, None), "t64-factor-empty": (51000, 100, 131072),
        "t64-validator-empty": (38000, 100, 131072), "t64-both-empty": (152001, 64, 151041)}


# ---- GPU -----------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("it", [2, 1])
@pytest.mark.parametrize("case", list(CASES))
def test_cacqr_parity_at_every_splitk_geometry(sms, case, it):
    """Q and R elementwise against the oracle, and validate's residual AND orthogonality against numpy norms of the returned Q, R
    (the orthogonality is the validator's own split-K Gram product).  Empty-chunk targets run after their primer."""
    m, n, primer = pick(case, sms)
    topo = cb.topo.rect(1, 0, 1)
    if primer:
        prime(topo, n, primer)
    A, args = factor(topo, m, n, it)
    check_against_oracle(m, n, it, *result(A, args, topo))


@gpu
@pytest.mark.parametrize("case", EMPTY_CASES)
def test_cacqr_result_does_not_depend_on_earlier_calls(sms, case):
    """The Gram product is deterministic (DESIGN.md section 6): the first call of a new context, a call after the primer and a
    repeated call return the same bits of Q and R, and each of them matches the oracle and the numpy norms.  The validator's sums of
    squares are added across thread blocks with atomics, so its two numbers may differ between calls in the last bits only."""
    m, n, primer = pick(case, sms)
    cb.topo.release_contexts()
    topo = cb.topo.rect(1, 0, 1)
    fresh = result(*factor(topo, m, n), topo)
    prime(topo, n, primer)
    primed = result(*factor(topo, m, n), topo)
    again = result(*factor(topo, m, n), topo)
    for name, other in (("after the primer", primed), ("repeated", again)):
        assert torch.equal(fresh[0], other[0]), f"Q {name} differs from the first call of the context"
        assert torch.equal(fresh[1], other[1]), f"R {name} differs from the first call of the context"
        assert np.allclose(fresh[2], other[2], rtol=1e-12, atol=0), f"validate {name} {other[2]} != first call {fresh[2]}"
    for r in (fresh, primed, again):
        check_against_oracle(m, n, 2, *r)


@gpu
@pytest.mark.parametrize("case", ["t128-factor-empty", "t128-full"])
@pytest.mark.parametrize("path", ["plain-sweep", "host-pointers", "rect-R"])
def test_cacqr_other_paths_into_the_gram_product(sms, case, path, monkeypatch):
    """The same Gram products reached through CAPITAL_QR_TSTORE=0 (the sweep with explicit transposes), pinned host buffers for A, Q
    and R (staged: the last apply does not write the caller's Q in place) and rect R (serialize=False)."""
    if path == "plain-sweep":
        monkeypatch.setenv("CAPITAL_QR_TSTORE", "0")  # read on every call
    m, n, primer = pick(case, sms)
    topo = cb.topo.rect(1, 0, 1)
    if primer:
        prime(topo, n, primer)
    A, args = factor(topo, m, n, host=path == "host-pointers", serialize=path != "rect-R")
    assert args.Q.is_cuda == (path != "host-pointers") and args.R.numel() == (n * n if path == "rect-R" else n * (n + 1) // 2)
    check_against_oracle(m, n, 2, *result(A, args, topo))


@gpu
@pytest.mark.parametrize("n,ci,bcm,serialize", [(1000, 0, -3, False), (777, 1, -2, True), (2048, 0, -2, False)])
def test_cholinv_result_does_not_depend_on_earlier_calls(n, ci, bcm, serialize):
    """cholinv.factor into caller-owned outputs pre-filled with NaN: the first call of a new context and a call after larger
    factorizations with other leading dimensions (which leave their values in every grow-only workspace) return the same bits,
    every output entry is written, and both match the oracle."""
    cb.topo.release_contexts()
    topo = cb.topo.square(1, 0, 1)
    A = cb.matrix(n, n, 1, 1).distribute_symmetric(topo)
    count = n * (n + 1) // 2 if serialize else n * n

    def run():
        args = cb.cholinv.info(ci, 1, bcm, "U", serialize=serialize)
        args.R = torch.full((count,), float("nan"), dtype=torch.float64, device="cuda")
        args.Rinv = torch.full((count,), float("nan"), dtype=torch.float64, device="cuda")
        cb.cholinv.factor(A, args, topo)
        assert not args.R.isnan().any() and not args.Rinv.isnan().any(), "an output entry was not written"
        return args

    fresh = run()
    for pn, pci, pser in ((4096, 1, not serialize), (3000, 0, serialize)):
        P = cb.matrix(pn, pn, 1, 1).distribute_symmetric(topo)
        cb.cholinv.factor(P, cb.cholinv.info(pci, 1, -2, "U", serialize=pser), topo)
    primed = run()
    assert torch.equal(fresh.R, primed.R) and torch.equal(fresh.Rinv, primed.Rinv), "result depends on the earlier factorizations"
    a = co.spd_global(n)
    r_o, ri_o = co.cholinv(a, bool(ci), 1, co.bc_dimension(n, 1, 1, bcm))
    R = cb.cholinv.construct_R(fresh).cpu().numpy()
    Ri = cb.cholinv.construct_Rinv(fresh).cpu().numpy()
    assert np.abs(R - r_o).max() <= 2e-13 * np.abs(r_o).max()
    assert np.abs(Ri - ri_o).max() <= 2e-13 * np.abs(ri_o).max()
    assert np.array_equal(np.tril(R, -1), np.zeros_like(R)) and np.array_equal(np.tril(Ri, -1), np.zeros_like(Ri))
