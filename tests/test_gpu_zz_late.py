"""The newest GPU cases of the suite, in the file that sorts last (a failure here cannot stop the run before the established cases).

1. GATING -- BASELINE-size parity of the default FP64 path: n = 16384 factors elementwise against cuSOLVER potrf + a triangular solve.

2. XPASS/XFAIL -- the EXPERIMENTAL mixed-precision path (BASELINE config 5): trailing updates on the TF32 tensor cores (tcgen05 + TMEM,
   capital_b200/csrc/gemm_tf32.cu), FP64 everywhere else; off by default in the library.  The kernel was written after the round's GPU
   budget was spent: it assembles for sm_100a (UTCHMMA / LDTM / UTMALDG in the SASS) but the run of THIS file is its first execution.
   Hence every case runs in a child process with its own CUDA context and a timeout (the kernel's mbarrier waits are bounded too) and
   is xfail(strict=False): an XPASS in the report means the path computed the right numbers on this device, an XFAIL that it did not;
   neither touches the FP64 product path.  Gates (no reference float path exists, src/blas/interface.hpp:43-97: the FP64 results are
   the yardstick):
     product:       |C - C_fp64| / max(|A|^T |B|) <= 5e-4 (TF32 operands) / 2e-6 (split operands, 3 passes)
     factorization: residual ||A - R^T R||_F / ||A||_F <= 1e-6 (TF32) / 1e-8 (3 x TF32) at n = 4096 (CPU emulation of the rounding,
                    tools/tf32_emulate.py: 5e-9 / 1e-10), and > 1e-13 with the TF32 kernel's launch counter > 0 -- i.e. the
                    tensor-core path really ran.

3. GATING -- split = 2 of the FP64 path against the reference's dump and the oracle."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WHY = "TF32 tcgen05 path: written without GPU access, this run is its first execution (XPASS = it works)"


def worker(*args, timeout=600):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "tf32_worker.py"), *map(str, args)], capture_output=True, text=True,
                       timeout=timeout)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


# ---- gating: BASELINE-size parity of the default FP64 path (placed in the last file: it is the newest test of the suite) ----
@pytest.mark.parametrize("ci", [0, 1])
def test_cholinv_baseline_size_elementwise_against_cusolver(ci):
    """BASELINE config 1 (n = 16384, base case 512): R and R^-1 ELEMENTWISE against an independent FP64 factorization of the same
    matrix on the device (cuSOLVER potrf through torch.linalg.cholesky, then a triangular solve).  The numpy oracle takes minutes at
    this size; at n <= 4096 it agrees with LAPACK to 5e-16 (relative to max |R|), so LAPACK-class results are the same yardstick.
    Tolerance: 1e-12 relative to the largest entry (the matrix is diagonally dominant, cond ~ 2)."""
    import torch
    import capital_b200 as cb
    topo = cb.topo.square(1, 0, 1)
    n, bcm = 16384, -5
    A = cb.matrix(n, n, 1, 1).distribute_symmetric(topo)
    args = cb.cholinv.info(ci, 1, bcm, "U", serialize=False)
    cb.cholinv.factor(A, args, topo)
    R, Ri = cb.cholinv.construct_R(args), cb.cholinv.construct_Rinv(args)
    Rref = torch.linalg.cholesky(A.view2d(), upper=True)
    assert ((R - Rref).abs().max() / Rref.abs().max()).item() < 1e-12
    Riref = torch.linalg.solve_triangular(Rref, torch.eye(n, dtype=torch.float64, device="cuda"), upper=True)
    if not ci:
        Riref[: n // 2, n // 2:] = 0  # the block the reference never forms with complete_inv = 0 (cholinv.hpp:147)
    assert ((Ri - Riref).abs().max() / Riref.abs().max()).item() < 1e-12
    del Rref, Riref, R, Ri
    torch.cuda.empty_cache()


@pytest.mark.xfail(strict=False, reason=WHY)
def test_tf32_product_against_fp64():
    out = worker("gemm")["gemm"]
    for c in out:
        assert c["status"] == 0, c
        assert c["padding_untouched"], c
        assert c["rel_err"] <= (5e-4 if c["passes"] == 1 else 2e-6), c
    # and the tensor cores were really used: TF32 rounding leaves a visible error on a long contraction
    assert any(c["passes"] == 1 and c["rel_err"] > 1e-9 for c in out)


@pytest.mark.xfail(strict=False, reason=WHY)
def test_cholinv_mixed_precision_trailing_update():
    d = worker("cholinv", 4096, -3)
    assert d["tf32_launches"]["f64"] == 0 and d["tf32_launches"]["tf32"] > 0 and d["tf32_launches"]["tf32x3"] > 0
    assert d["residual"]["f64"] <= 1e-14
    assert 1e-13 < d["residual"]["tf32"] <= 1e-6
    assert d["residual"]["tf32x3"] <= 1e-8
    assert d["R_rel_diff"]["tf32"] <= 1e-4 and d["R_rel_diff"]["tf32x3"] <= 1e-6


# ---- not TF32: split = 2 of the FP64 path ----
def test_cholinv_uneven_split_matches_reference_dump_and_oracle():
    """split = 2 (cholinv.hpp:92,107: the left child gets a quarter of the node): the reference's own dump, elementwise, and the numpy
    restatement (pinned to that dump on CPU) at a ragged size."""
    import numpy as np
    import capital_b200 as cb
    from oracle import capital_oracle as co
    topo = cb.topo.square(1, 0, 1)
    z = np.load(os.path.join(ROOT, "tests", "golden", "cholinv_p1_n128_ci0_split2.npz"))
    meta = json.loads(str(z["meta"]))
    n = meta["n"]
    A = cb.matrix(n, n, 1, 1).distribute_symmetric(topo)
    args = cb.cholinv.info(meta["complete_inv"], meta["split"], meta["bc_mult_dim"], "U")
    cb.cholinv.factor(A, args, topo)
    r, ri = args.R.cpu().numpy(), args.Rinv.cpu().numpy()
    assert np.abs(r - z["R_0"]).max() <= 1e-13 * np.abs(z["R_0"]).max()
    assert np.abs(ri - z["Rinv_0"]).max() <= 1e-13 * np.abs(z["Rinv_0"]).max()
    assert np.array_equal(ri == 0, z["Rinv_0"] == 0)  # the skipped block sits at n >> 2 now (cholinv.hpp:147)
    for n, ci, bcm in ((1000, 0, -3), (2048, 1, -3)):
        A = cb.matrix(n, n, 1, 1).distribute_symmetric(topo)
        args = cb.cholinv.info(ci, 2, bcm, "U", serialize=False)
        cb.cholinv.factor(A, args, topo)
        a = co.spd_global(n)
        r_o, ri_o = co.cholinv(a, bool(ci), 2, co.bc_dimension(n, 1, 1, bcm))
        R, Ri = cb.cholinv.construct_R(args).cpu().numpy(), cb.cholinv.construct_Rinv(args).cpu().numpy()
        assert np.abs(R - r_o).max() <= 2e-13 * np.abs(r_o).max()
        assert np.abs(Ri - ri_o).max() <= 2e-13 * np.abs(ri_o).max()
        assert cb.cholinv.residual(A, args, topo) <= 1e-12
