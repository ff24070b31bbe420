"""Generate golden fixtures by running the reference itself (oracle/_ref, built by oracle/build_ref.sh
from /root/reference) and storing its per-rank dumps.  Run in the build container only:

    bash oracle/build_ref.sh && python tests/golden/make_golden.py

Each .npz holds, per rank r: A_r (local rect block of the generator), R_r / Rinv_r (packed upper,
structure.h:37-39) or Q_r / R_r for cacqr, plus the JSON line the driver printed (residuals measured
by the reference's own validators).  Small sizes only -- fixtures are committed.
"""
import json, os, subprocess, sys, tempfile
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.path.join(HERE, "..", "..", "oracle", "_ref")

CHOLINV = [  # name, P, n, complete_inv, split, bc_mult, policy
    ("cholinv_p1_n96_ci1", 1, 96, 1, 1, -2, 0),
    ("cholinv_p1_n128_ci0", 1, 128, 0, 1, -3, 2),
    ("cholinv_p8_n128_ci0", 8, 128, 0, 1, -1, 0),
    ("cholinv_p8_n192_ci1", 8, 192, 1, 1, -2, 0),
    ("cholinv_p1_n128_ci0_split2", 1, 128, 0, 2, -3, 0),  # split = 2: the left child is a quarter (cholinv.hpp:92,107)
    ("cholinv_p8_n256_ci1_split2", 8, 256, 1, 2, -2, 0),
]
CACQR = [  # name, P, variant, m, n, c, complete_inv, split, bc_mult
    ("cacqr_p1_m512_n32", 1, 2, 512, 32, 1, 0, 1, 0),
    ("cacqr_p8_1d_m1024_n32", 8, 2, 1024, 32, 1, 0, 1, 0),
    ("cacqr_p8_3d_m256_n64", 8, 2, 256, 64, 2, 1, 1, -1),
    ("cacqr_p8_3d_m256_n64_ci0", 8, 2, 256, 64, 2, 0, 1, -1),
    ("cacqr_p8_1d_m1024_n32_it1", 8, 1, 1024, 32, 1, 0, 1, 0),  # num_iter = 1: one sweep (CholeskyQR, not QR2)  # complete_inv = 0: the reference's block `solve` (cacqr.hpp:46-71)
]

def run(cmd, np_):
    env = dict(os.environ, MINIMPI_NP=str(np_), OPENBLAS_NUM_THREADS="1")
    out = subprocess.run(cmd, env=env, check=True, capture_output=True, text=True).stdout
    return json.loads(out.strip().splitlines()[-1])

def save(name, meta, arrs):
    """Replicas along z dump identical blocks: each distinct block is stored once and `same_as` maps the others to it (read back by
    oracle.capital_oracle.load_dump), which keeps every fixture under 1 MB."""
    kept, same_as = {}, {}
    for k, a in arrs.items():
        twin = next((j for j, b in kept.items() if np.array_equal(a, b)), None)
        if twin is None:
            kept[k] = a
        else:
            same_as[k] = twin
    np.savez_compressed(os.path.join(HERE, name + ".npz"), meta=json.dumps(meta), same_as=json.dumps(same_as), **kept)

def main():
    only = set(sys.argv[1:])  # optional: regenerate the named fixtures only
    for name, P, n, ci, split, bcm, pol in CHOLINV:
        if only and name not in only:
            continue
        with tempfile.TemporaryDirectory() as td:
            meta = run([os.path.join(REF, "ref_cholinv"), str(n), str(ci), str(split), str(bcm), str(pol), "1", os.path.join(td, "d")], P)
            arrs = {}
            for r in range(P):
                for k in ("A", "R", "Rinv"):
                    arrs[f"{k}_{r}"] = np.fromfile(os.path.join(td, f"d.{k}.{r}.bin"), dtype=np.float64)
            save(name, meta, arrs)
            print(name, meta)
    for name, P, var, m, n, c, ci, split, bcm in CACQR:
        if only and name not in only:
            continue
        with tempfile.TemporaryDirectory() as td:
            meta = run([os.path.join(REF, "ref_cacqr"), str(var), str(m), str(n), str(c), str(ci), str(split), str(bcm), "1", os.path.join(td, "d")], P)
            arrs = {}
            for r in range(P):
                for k in ("A", "Q", "R"):
                    arrs[f"{k}_{r}"] = np.fromfile(os.path.join(td, f"d.{k}.{r}.bin"), dtype=np.float64)
            save(name, meta, arrs)
            print(name, meta)

if __name__ == "__main__":
    main()
