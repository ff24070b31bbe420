"""Parity of the distributed CholInv schedule across its knob sets (run under torch.distributed.run, every rank on cuda:0).

Runs the GPU cases of tests/dist_cases.py for the grid of WORLD_SIZE ranks -- taken from the table whose every row the CPU replay of
the flag protocol checks (test_dist_protocol.py) -- and checks, per case:
  * R and R^-1 elementwise against the numpy restatement (oracle/capital_oracle.py), 2e-13 of the largest entry, and the residual;
  * zeros on the local diagonal slots of ranks below the global diagonal (y > x);
  * every knob set gives the bits of the default knob set.  The knobs change launch partitioning, stream placement and issue order
    only: inside a GEMM tile every output element accumulates its k range in the same order whatever the tile size or the column
    window (k tiles a triangular operand skips hold exact zeros), and the depth reduction adds the partials in layer order;
  * the depth replicas (same x, y; every z) hold the same bits;
  * a second default call on the same context gives the same bits (the first call of each ragged size follows a power-of-two size,
    so it is the first call on a new arena layout).
Rank 0 prints DV_OK or DV_FAIL and the failures; the exit code is non-zero on any failure."""
import os, sys, time
import numpy as np
import torch
import torch.distributed as dist

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import capital_b200 as cb
from oracle import capital_oracle as co
import dist_cases


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(0)
    dist.init_process_group("gloo")
    c, d = dist_cases.GRIDS[world]
    topo = cb.topo.square(world, rank, c)
    x, y, z = topo.x, topo.y, topo.z
    # the depth replicas of each (x, y): every rank creates every group, in the same order
    groups = {}
    for r in range(world):
        key = (r % (d * c)) // c, r // (d * c)  # (x, y) of rank r (topology.h)
        groups.setdefault(key, []).append(r)
    my_group = None
    for key in sorted(groups):
        g = dist.new_group(groups[key])
        if rank in groups[key]:
            my_group, my_members = g, groups[key]
    fails, timing = [], {}
    mats, oracles, first = {}, {}, {}
    t0 = time.time()

    def run(case):
        dist_cases.set_knobs(case.knobs)
        dist.barrier()  # every rank has the same knobs before any of them enters the schedule
        if case.n not in mats:
            mats.clear()
            mats[case.n] = cb.matrix(case.n, case.n, d, d).distribute_symmetric(topo)
        A = mats[case.n]
        args = cb.cholinv.info(case.ci, case.split, case.bcm, "U")
        t = time.time()
        cb.cholinv.factor(A, args, topo)
        torch.cuda.synchronize()
        timing[case.knobs] = timing.get(case.knobs, 0.0) + time.time() - t
        R, Ri = cb.cholinv.construct_R(args).cpu(), cb.cholinv.construct_Rinv(args).cpu()
        return R, Ri, cb.cholinv.residual(A, args, topo)

    for case in dist_cases.gpu_cases(world):
        name = f"p{world} n={case.n} ci={case.ci} split={case.split} {case.knobs}"
        R, Ri, res = run(case)
        key = (case.n, case.ci, case.split)
        if key not in oracles:
            L = case.n // d
            r_o, ri_o = co.cholinv(co.spd_global(case.n), bool(case.ci), case.split, co.bc_dimension(L, c, d, case.bcm), d=d)
            oracles.clear()
            oracles[key] = (np.triu(co.cyclic_local(r_o, d, d, x, y)), np.triu(co.cyclic_local(ri_o, d, d, x, y)),
                            np.abs(r_o).max(), np.abs(ri_o).max())
        ro, rio, rmax, rimax = oracles[key]
        er = np.abs(R.numpy() - ro).max() / rmax
        ei = np.abs(Ri.numpy() - rio).max() / rimax
        if not (er < 2e-13 and ei < 2e-13 and res <= 1e-12):
            fails.append(f"{name} rank {rank}: dR={er:.1e} dRinv={ei:.1e} res={res:.1e}")
        if y > x and not (torch.all(torch.diagonal(R) == 0) and torch.all(torch.diagonal(Ri) == 0)):
            fails.append(f"{name} rank {rank}: nonzero local diagonal below the global one")
        if case.knobs == "default":
            first[key] = (R, Ri)
        elif not (torch.equal(R, first[key][0]) and torch.equal(Ri, first[key][1])):
            fails.append(f"{name} rank {rank}: differs from the default knob set")
        if len(my_members) > 1:
            reps = [None] * len(my_members)
            dist.all_gather_object(reps, (z, R, Ri), group=my_group)
            if not all(torch.equal(R, rr) and torch.equal(Ri, rri) for _, rr, rri in reps):
                fails.append(f"{name} rank {rank}: replicas z = {[zz for zz, _, _ in reps]} are not bit-identical")
        if case.knobs == list(dist_cases.KNOBS)[-1]:
            # a second default call on this context, after every other knob set
            R2, Ri2, _ = run(case._replace(knobs="default"))
            if not (torch.equal(R2, first[key][0]) and torch.equal(Ri2, first[key][1])):
                fails.append(f"{name} rank {rank}: a second default call differs from the first")
    dist_cases.set_knobs("default")
    allf = [None] * world
    dist.all_gather_object(allf, fails)
    bad = [f for fl in allf for f in fl]
    if rank == 0:
        tm = " ".join(f"{k}={v:.1f}s" for k, v in timing.items())
        ncase = len(dist_cases.gpu_cases(world))
        print(("DV_OK" if not bad else "DV_FAIL") + f" p{world}: {ncase} cases in {time.time() - t0:.0f} s (factor time by knob set: {tm})",
              flush=True)
        for f in bad[:40]:
            print("  " + f, flush=True)
    dist.barrier()
    cb.topo.release_contexts()
    dist.destroy_process_group()
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
