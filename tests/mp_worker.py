"""Multi-GPU parity worker (run under torch.distributed.run, one process per GPU).  Exits non-zero on mismatch.

Checks the distributed CholInv (reference's 2x2x2 grid) and 1D CholeskyQR2 against the reference's own per-rank dumps
(tests/golden/*_p8_*.npz), the oracle restatement, and the validators; rank 0 prints a summary line.
"""
import os, sys
import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import capital_b200 as cb
from oracle import capital_oracle as co

GOLD = os.path.join(ROOT, "tests", "golden")


def load(name):
    return co.load_dump(os.path.join(GOLD, name + ".npz"))


def main():
    rank, world, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    same_dev = bool(os.environ.get("CAPITAL_MP_SAME_DEVICE"))  # all ranks on cuda:0 (1-GPU boxes): same code path, time-sliced
    small = same_dev or bool(os.environ.get("CAPITAL_MP_SMALL"))
    if same_dev:
        torch.cuda.set_device(0)
        dist.init_process_group("gloo")
    else:
        torch.cuda.set_device(lr)
        dist.init_process_group("nccl", device_id=torch.device("cuda", lr))
    ok = True
    msgs = []
    if world == 8:
        topo = cb.topo.square(8, rank, 2)
        # --- reference dumps, elementwise ---
        for name in ("cholinv_p8_n128_ci0", "cholinv_p8_n192_ci1"):
            meta, z = load(name)
            n = meta["n"]
            A = cb.matrix(n, n, 2, 2).distribute_symmetric(topo)
            ok &= np.array_equal(A.data.cpu().numpy(), z[f"A_{rank}"])
            args = cb.cholinv.info(meta["complete_inv"], meta["split"], meta["bc_mult_dim"], "U")
            cb.cholinv.factor(A, args, topo)
            er = np.abs(args.R.cpu().numpy() - z[f"R_{rank}"]).max() / np.abs(z[f"R_{rank}"]).max()
            ei = np.abs(args.Rinv.cpu().numpy() - z[f"Rinv_{rank}"]).max() / np.abs(z[f"Rinv_{rank}"]).max()
            same_zeros = np.array_equal(args.Rinv.cpu().numpy() == 0, z[f"Rinv_{rank}"] == 0)
            res = cb.cholinv.residual(A, args, topo)
            ok &= er < 1e-13 and ei < 1e-13 and same_zeros and res < 1e-14
            msgs.append(f"{name}: dR={er:.1e} dRinv={ei:.1e} zeros={same_zeros} res={res:.1e}")
        # --- split = 2 (left child = a quarter, cholinv.hpp:92,107): reference dump ---
        meta, z = load("cholinv_p8_n256_ci1_split2")
        n = meta["n"]
        A = cb.matrix(n, n, 2, 2).distribute_symmetric(topo)
        args = cb.cholinv.info(meta["complete_inv"], meta["split"], meta["bc_mult_dim"], "U")
        cb.cholinv.factor(A, args, topo)
        er = np.abs(args.R.cpu().numpy() - z[f"R_{rank}"]).max() / np.abs(z[f"R_{rank}"]).max()
        ei = np.abs(args.Rinv.cpu().numpy() - z[f"Rinv_{rank}"]).max() / np.abs(z[f"Rinv_{rank}"]).max()
        same_zeros = np.array_equal(args.Rinv.cpu().numpy() == 0, z[f"Rinv_{rank}"] == 0)
        res = cb.cholinv.residual(A, args, topo)
        ok &= er < 1e-13 and ei < 1e-13 and same_zeros and res < 1e-14
        msgs.append(f"cholinv_p8_n256_ci1_split2: dR={er:.1e} dRinv={ei:.1e} zeros={same_zeros} res={res:.1e}")
        # --- oracle restatement at a size with several distributed levels + ragged local sizes ---
        for n, ci, bcm in (((768, 1, -2), (1536, 0, -3)) if small else ((1024, 1, -2), (1536, 0, -3), (4096, 0, -3))):
            A = cb.matrix(n, n, 2, 2).distribute_symmetric(topo)
            args = cb.cholinv.info(ci, 1, bcm, "U")
            cb.cholinv.factor(A, args, topo)
            L = n // 2
            r_o, ri_o = co.cholinv(co.spd_global(n), bool(ci), 1, co.bc_dimension(L, 2, 2, bcm), d=2)
            R = cb.cholinv.construct_R(args).cpu().numpy()
            Ri = cb.cholinv.construct_Rinv(args).cpu().numpy()
            er = np.abs(R - np.triu(co.cyclic_local(r_o, 2, 2, topo.x, topo.y))).max() / np.abs(r_o).max()
            ei = np.abs(Ri - np.triu(co.cyclic_local(ri_o, 2, 2, topo.x, topo.y))).max() / np.abs(ri_o).max()
            zd = (topo.y <= topo.x) or (np.all(np.diag(R) == 0) and np.all(np.diag(Ri) == 0))
            res = cb.cholinv.residual(A, args, topo)
            ok &= er < 2e-13 and ei < 2e-13 and zd and res < 1e-12
            msgs.append(f"oracle n={n} ci={ci}: dR={er:.1e} dRinv={ei:.1e} zero-diag-slots={zd} res={res:.1e}")
    if world in (2, 4):
        # not reference grids (summa.hpp needs c == d): the library's own 2x1x1 / 1x2x2 schedules, checked against the oracle
        c = 2 if world == 2 else 1
        topo = cb.topo.square(world, rank, c)
        d = topo.d
        sizes = ((512, 1, -2), (1536, 0, -3)) if small else ((512, 1, -2), (2048, 0, -3), (3072, 1, -3), (8192, 1, -4))
        for n, ci, bcm in sizes:
            A = cb.matrix(n, n, d, d).distribute_symmetric(topo)
            args = cb.cholinv.info(ci, 1, bcm, "U")
            cb.cholinv.factor(A, args, topo)
            L = n // d
            r_o, ri_o = co.cholinv(co.spd_global(n), bool(ci), 1, co.bc_dimension(L, c, d, bcm), d=d)
            R = cb.cholinv.construct_R(args).cpu().numpy()
            Ri = cb.cholinv.construct_Rinv(args).cpu().numpy()
            er = np.abs(R - np.triu(co.cyclic_local(r_o, d, d, topo.x, topo.y))).max() / np.abs(r_o).max()
            ei = np.abs(Ri - np.triu(co.cyclic_local(ri_o, d, d, topo.x, topo.y))).max() / np.abs(ri_o).max()
            res = cb.cholinv.residual(A, args, topo)
            ok &= er < 2e-13 and ei < 2e-13 and res < 1e-12
            msgs.append(f"grid {c}x{d}x{d} n={n} ci={ci}: dR={er:.1e} dRinv={ei:.1e} res={res:.1e}")
    if world in (2, 4, 8):
        # --- host-pointer path of the distributed factor (upper-triangle H2D, streamed D2H) == resident path, bit for bit ---
        c = {2: 2, 4: 1, 8: 2}[world]
        topo = cb.topo.square(world, rank, c)
        d = topo.d
        for n, ci in (((2048 * d, 0),) if small else ((4096 * d, 0), (2048 * d, 1))):
            A = cb.matrix(n, n, d, d).distribute_symmetric(topo)
            dev = cb.cholinv.info(ci, 1, -3, "U")
            cb.cholinv.factor(A, dev, topo)
            hostA = cb.matrix(n, n, d, d, data=A.data.cpu().pin_memory())
            hst = cb.cholinv.info(ci, 1, -3, "U")
            cb.cholinv.factor(hostA, hst, topo)
            same = torch.equal(hst.R, dev.R.cpu()) and torch.equal(hst.Rinv, dev.Rinv.cpu())
            ok &= same and not hst.R.is_cuda
            msgs.append(f"host path n={n} ci={ci}: identical={same}")
    if world == 8 and not small:
        # --- the distributed result against the single-GPU one at a size with big products (the generator is grid-independent) ---
        n = 8192
        topo = cb.topo.square(8, rank, 2)
        A = cb.matrix(n, n, 2, 2).distribute_symmetric(topo)
        args = cb.cholinv.info(0, 1, -3, "U")
        cb.cholinv.factor(A, args, topo)
        t1 = cb.topo.square(1, 0, 1)
        A1 = cb.matrix(n, n, 1, 1).distribute_symmetric(t1)
        a1 = cb.cholinv.info(0, 1, -3, "U", serialize=False)
        cb.cholinv.factor(A1, a1, t1)
        R1, Ri1 = cb.cholinv.construct_R(a1), cb.cholinv.construct_Rinv(a1)
        R, Ri = cb.cholinv.construct_R(args), cb.cholinv.construct_Rinv(args)
        sel = (slice(topo.y, None, 2), slice(topo.x, None, 2))
        er = ((R - torch.triu(R1[sel])).abs().max() / R1.abs().max()).item()
        ei = ((Ri - torch.triu(Ri1[sel])).abs().max() / Ri1.abs().max()).item()
        ok &= er < 2e-13 and ei < 2e-13
        msgs.append(f"8 GPUs vs 1 GPU n={n}: dR={er:.1e} dRinv={ei:.1e}")
        del A1, a1, R1, Ri1
    if world in (2, 4, 8):
        # --- SUMMA GEMM entry point (T*N) on the same grid, against the global product ---
        c = {2: 2, 4: 1, 8: 2}[world]
        topo = cb.topo.square(world, rank, c)
        d = topo.d
        m, n, k = 384, 256, 512
        rng = np.random.default_rng(5)
        Ag, Bg, Cg = rng.standard_normal((k, m)), rng.standard_normal((k, n)), rng.standard_normal((m, n))
        mk = lambda G: cb.matrix(G.shape[1], G.shape[0], d, d, data=torch.from_numpy(np.asfortranarray(co.cyclic_local(G, d, d, topo.x, topo.y)).ravel(order="F").copy()).cuda())
        A, B, C = mk(Ag), mk(Bg), mk(Cg)
        cb.summa.invoke(A, B, C, topo, alpha=1.5, beta=-0.5)
        ref = co.cyclic_local(1.5 * Ag.T @ Bg - 0.5 * Cg, d, d, topo.x, topo.y)
        es = np.abs(C.view2d().cpu().numpy() - ref).max()
        ok &= es < 1e-11
        msgs.append(f"summa gemm {c}x{d}x{d}: err={es:.1e}")
    if world == 8:
        # --- 3D CA-CholeskyQR2 (c = d = 2) against the reference's dump ---
        meta, z = load("cacqr_p8_3d_m256_n64")
        m, n = meta["m"], meta["n"]
        t3 = cb.topo.rect(8, rank, 2)
        A = cb.matrix(n, m, 2, 2).distribute_random(t3, rank // 2)
        ok &= np.array_equal(A.data.cpu().numpy(), z[f"A_{rank}"])
        qa = cb.cacqr.info(2, cb.cholinv.info(1, 1, -1, "U"))
        cb.cacqr.factor(A, qa, t3)
        eq = np.abs(qa.Q.cpu().numpy() - z[f"Q_{rank}"]).max()
        res, orth = cb.cacqr.validate(A, qa, t3)
        ok &= eq < 1e-12 and res < 1e-14 and orth < 1e-15
        msgs.append(f"cacqr 3D golden: dQ={eq:.1e} res={res:.1e} orth={orth:.1e}")
        # complete_inv = 0: the reference takes its block `solve` (cacqr.hpp:46-71); here the complete inverse is applied -- same Q
        meta, z = load("cacqr_p8_3d_m256_n64_ci0")
        qa0 = cb.cacqr.info(2, cb.cholinv.info(0, 1, -1, "U"))
        cb.cacqr.factor(A, qa0, t3)
        eq0 = np.abs(qa0.Q.cpu().numpy() - z[f"Q_{rank}"]).max()
        res0, orth0 = cb.cacqr.validate(A, qa0, t3)
        ok &= eq0 < 1e-12 and res0 < 1e-14 and orth0 < 1e-15
        msgs.append(f"cacqr 3D golden (complete_inv=0, reference `solve`): dQ={eq0:.1e} res={res0:.1e}")
    # --- 1D CholeskyQR2 on all ranks ---
    qt = cb.topo.rect(world, rank, 1)
    if world == 8:
        meta, z = load("cacqr_p8_1d_m1024_n32")
        m, n = meta["m"], meta["n"]
        A = cb.matrix(n, m, 1, world).distribute_random(qt, rank)
        ok &= np.array_equal(A.data.cpu().numpy(), z[f"A_{rank}"])
        qa = cb.cacqr.info(2, cb.cholinv.info(0, 1, 0, "U"))
        cb.cacqr.factor(A, qa, qt)
        er = np.abs(qa.R.cpu().numpy() - z[f"R_{rank}"]).max() / np.abs(z[f"R_{rank}"]).max()
        eq = np.abs(qa.Q.cpu().numpy() - z[f"Q_{rank}"]).max()
        res, orth = cb.cacqr.validate(A, qa, qt)
        ok &= er < 1e-12 and eq < 1e-12 and res < 1e-14 and orth < 1e-15
        msgs.append(f"cacqr golden: dR={er:.1e} dQ={eq:.1e} res={res:.1e} orth={orth:.1e}")
    m, n = (1 << 13, 64) if small else (1 << 17, 128)
    A = cb.matrix(n, m, 1, world).distribute_random(qt, rank)
    qa = cb.cacqr.info(2, cb.cholinv.info(0, 1, 0, "U"))
    cb.cacqr.factor(A, qa, qt)
    res, orth = cb.cacqr.validate(A, qa, qt)
    ok &= res < 1e-13 and orth < 1e-14
    msgs.append(f"cacqr m={m} n={n} P={world}: res={res:.1e} orth={orth:.1e}")
    msgs.append(f"peer flag waits: {qt.context().peer_wait_mode()}")
    flag = torch.tensor([0 if ok else 1], device="cuda")
    dist.all_reduce(flag)
    if rank == 0:
        print(("MP_OK " if flag.item() == 0 else "MP_FAIL ") + " | ".join(msgs), flush=True)
    dist.barrier()
    cb.topo.release_contexts()
    dist.destroy_process_group()
    sys.exit(0 if flag.item() == 0 else 1)


if __name__ == "__main__":
    main()
