#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path: FP64 CholInv (cholesky::cholinv::factor) on synthetic SPD input.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--n SIZE] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A "step" is one cholinv::factor of the workload below on a resident (HBM) copy of the reference's own generator matrix
(structure.hpp:69-103).  Rank 0 prints ONE JSON line.
  value        whole-job n^3/3 / time ("Cholesky TFLOP/s", the BASELINE.json metric), CUDA events, max over ranks
  e2e          the same through the public Python API with pinned HOST buffers (H2D of A and D2H of R, Rinv inside the timed region)
  roofline     the dominant kernel (128x128 DMMA GEMM) timed with CUDA events on its own stream, against the FP64 tensor-pipe
               peak MEASURED IN THIS RUN (capital_probe_dmma_f64) with the clocks sampled during it
  parity       (N > 1) the distributed result against the reference's own per-rank dumps (tests/golden, 8 ranks) and against the
               single-GPU factorization of the same matrix, before the timed region
  cacqr        CholeskyQR2 (qr::cacqr::factor, 1D grid) on m = 2^17 rows per GPU x 256 columns: BASELINE config 4 at N = 8
  strong       cholinv at a FIXED n = 32768 on the same N GPUs (the headline sizes grow with N)
  cpu_baseline / --impl reference   the reference's own CPU implementation (oracle/_ref, built from /root/reference by
               oracle/build_ref.sh) on this box's host cores.
Workloads (BASELINE.json configs): N=1 n=16384 b=512 | N=8 n=65536 b=1024 on the reference's 2x2x2 grid; N=2 / N=4 are not valid
reference grids (summa.hpp:16-31 needs c == d) and run the library's own 2x1x1 / 1x2x2 grids.
"""
from __future__ import annotations
import argparse, json, os, subprocess, sys, threading, time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NOMINAL_DMMA_TFLOPS = 37.2  # 148 SMs x 64 FMA/clk x 1.965 GHz; only used when the in-run probe fails (said so in the line)
HBM_GBS_FALLBACK = 6570.0
WORKLOADS = {  # n_gpus -> (n, c, bc_mult_dim)  ; base-case size b = 512 (N=1) / 1024 (N=8) as in BASELINE.json configs
    1: (16384, 1, -5),
    2: (24576, 2, -5),
    4: (32768, 1, -5),
    8: (65536, 2, -4),
}
STRONG_N = 32768
STRONG_BCM = {1: -6, 2: -5, 4: -5, 8: -3}  # base case 512 global (1024 on the 2x2x2 grid, as in BASELINE config 3)
DUMP_SAMPLES = 1 << 21  # per output, shared by all ranks: R and Rinv in FP64 come to 32 MB


def sample_outputs(torch, np, pack, world, rank):
    """--dump-outputs: the packed-upper R and Rinv that the last timed cholinv::factor returned, at positions drawn from a fixed seed
    (all of them when an output is small), so that two builds can be compared entry for entry."""
    out = {}
    for name in ("R", "Rinv"):
        t = getattr(pack, name)
        k = min(t.numel(), DUMP_SAMPLES // world)
        idx = np.sort(np.random.default_rng(rank).choice(t.numel(), k, replace=False))
        key = name if world == 1 else f"{name}_rank{rank}"
        out[key] = t[torch.from_numpy(idx).to(t.device)].cpu().numpy()
    return out


def clocks_sampler(stop: threading.Event, out: list, gpu_index: int):
    q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    while not stop.is_set():
        try:
            r = subprocess.run(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                               capture_output=True, text=True, timeout=5)
            f = [x.strip() for x in r.stdout.strip().split(",")]
            if len(f) >= 7:
                out.append(f)
        except Exception:
            pass
        stop.wait(0.2)


def summarize_clocks(samples: list) -> dict:
    if not samples:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no nvidia-smi samples"]}
    sm = sorted(float(s[0]) for s in samples)
    reasons = []
    for idx, name in ((3, "hw_slowdown"), (4, "hw_thermal_slowdown"), (5, "sw_thermal_slowdown"), (6, "sw_power_cap")):
        if any(s[idx].lower().startswith("active") for s in samples):
            reasons.append(name)
    return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(samples[0][1]), "power_w_max": max(float(s[2]) for s in samples),
            "samples": len(samples), "reasons": reasons}


def ref_binary(name="ref_cholinv"):
    p = os.path.join(ROOT, "oracle", "_ref", name)
    return p if os.path.exists(p) else None


def run_reference_cholinv(n: int, bc_mult: int, ranks: int, iters: int, timeout: float):
    """Time the reference's own cholinv::factor on host cores (bench/cholesky/cholinv.cpp protocol). Returns dict or None."""
    exe = ref_binary()
    if exe is None:
        return None
    cores = os.cpu_count() or 1
    threads = max(1, cores // ranks)
    env = dict(os.environ, MINIMPI_NP=str(ranks), OPENBLAS_NUM_THREADS=str(threads), OMP_NUM_THREADS=str(threads))
    policy = 2 if ranks == 1 else 0  # benchmarked NoReplication policy is only valid at P == 1 (SURVEY section 0)
    try:
        r = subprocess.run([exe, str(n), "0", "1", str(bc_mult), str(policy), str(iters)], env=env, capture_output=True,
                           text=True, timeout=timeout)
        line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
        d = json.loads(line)
        d["threads_per_rank"] = threads
        d["cores"] = min(cores, threads * ranks)
        return d
    except Exception as e:  # noqa
        return {"error": repr(e)[:200]}


def reference_arm(args):
    """--impl reference: the reference's CPU path on this box's host cores, same metric/unit keys.  The reference allocates ~30x the
    matrix (SURVEY 8d), so the step is a BOUNDED SAMPLE: `config.n` is the size that actually ran, `config.full_workload_n` the size of
    the GPU arm's workload at this N."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    n_full, c, bcm = WORKLOADS[args.gpus]
    if args.n:
        n_full = args.n
    ranks = 1 if args.gpus == 1 else 8
    n = min(n_full, 16384 if ranks == 1 else 8192)
    t0 = time.time()
    iters = min(max(1, args.steps), 3)  # one reference factorization of the n=16384 sample takes ~10 s on 128 cores
    d = run_reference_cholinv(n, bcm, ranks, iters, timeout=1500)
    if not d or "time_mean_s" not in d:
        print(json.dumps({"impl": "reference", "unavailable": f"oracle/_ref/ref_cholinv missing or failed: {d}"}))
        return 0
    t = d["time_mean_s"]
    val = n ** 3 / 3 / t / 1e12
    sample = (f"n={n} (GPU arm workload at this N: n={n_full}); {ranks} rank(s) x {d['threads_per_rank']} OpenBLAS threads; {iters} timed "
              f"factorizations after one warm-up (bench/cholesky/cholinv.cpp protocol); reference validator residual {d['residual']:.2e}")
    cfg = workload_config(ranks if ranks == 8 else 1, n, 2 if ranks == 8 else 1, bcm)
    cfg["workload"] = "REFERENCE CPU SAMPLE: " + cfg["workload"]
    cfg["full_workload_n"] = n_full
    cfg["sample_n"] = n
    out = {
        "impl": "reference", "metric": "cholesky_tflops_fp64", "value": val, "unit": "TFLOP/s", "n_gpus": args.gpus, "steps": iters,
        "steps_requested": args.steps, "warmup": 1, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": val, "unit": "TFLOP/s", "cores": d["cores"], "kind": "reference", "sample": sample},
        "e2e": {"value": val, "unit": "TFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": time.time() - t0,
    }
    print(json.dumps(out))
    return 0


def workload_config(n_gpus, n, c, bcm):
    d = {1: 1, 2: 1, 4: 2, 8: 2}[n_gpus]
    L = n // d
    bc = (L // min(L, (c * d) << (-bcm))) * d
    return {"workload": f"cholinv::factor n={n} FP64 SPD (distribute_symmetric, diagonally dominant), complete_inv=0 split=1 "
                        f"bc_mult_dim={bcm} (base case {bc}), grid c={c} d={d} ({n_gpus} GPU)",
            "n": n, "grid": f"{c}x{d}x{d}", "base_case": bc, "l2": "inputs larger than L2 (no flush needed)"}


def parity_block(cb, torch, np, world, rank, c):
    """Distributed results before anything is timed: the reference's own per-rank dumps (8 ranks) and the single-GPU factorization
    of the same matrix (the generator is grid-independent).  Returns (max relative error, case list); all-reduced by the caller."""
    gold = os.path.join(ROOT, "tests", "golden")
    worst, cases = 0.0, []

    def load(name):
        z = np.load(os.path.join(gold, name + ".npz"))
        return json.loads(str(z["meta"])), z

    topo = cb.topo.square(world, rank, c)
    d = topo.d
    if world == 8:
        for name in ("cholinv_p8_n128_ci0", "cholinv_p8_n192_ci1"):
            meta, z = load(name)
            n = meta["n"]
            A = cb.matrix(n, n, 2, 2).distribute_symmetric(topo)
            a = cb.cholinv.info(meta["complete_inv"], meta["split"], meta["bc_mult_dim"], "U")
            cb.cholinv.factor(A, a, topo)
            e = max(np.abs(a.R.cpu().numpy() - z[f"R_{rank}"]).max() / np.abs(z[f"R_{rank}"]).max(),
                    np.abs(a.Rinv.cpu().numpy() - z[f"Rinv_{rank}"]).max() / np.abs(z[f"Rinv_{rank}"]).max())
            if not np.array_equal(a.Rinv.cpu().numpy() == 0, z[f"Rinv_{rank}"] == 0):
                e = 1.0
            worst = max(worst, float(e)); cases.append(name)
        t3 = cb.topo.rect(8, rank, 2)
        meta, z = load("cacqr_p8_3d_m256_n64")
        A = cb.matrix(meta["n"], meta["m"], 2, 2).distribute_random(t3, rank // 2)
        qa = cb.cacqr.info(2, cb.cholinv.info(1, 1, -1, "U"))
        cb.cacqr.factor(A, qa, t3)
        worst = max(worst, float(np.abs(qa.Q.cpu().numpy() - z[f"Q_{rank}"]).max())); cases.append("cacqr_p8_3d_m256_n64")
        meta, z = load("cacqr_p8_3d_m256_n64_ci0")  # complete_inv = 0: the reference's block `solve` path (cacqr.hpp:46-71)
        qa = cb.cacqr.info(2, cb.cholinv.info(0, 1, -1, "U"))
        cb.cacqr.factor(A, qa, t3)
        worst = max(worst, float(np.abs(qa.Q.cpu().numpy() - z[f"Q_{rank}"]).max())); cases.append("cacqr_p8_3d_m256_n64_ci0")
        qt = cb.topo.rect(8, rank, 1)
        meta, z = load("cacqr_p8_1d_m1024_n32")
        A = cb.matrix(meta["n"], meta["m"], 1, 8).distribute_random(qt, rank)
        qa = cb.cacqr.info(2, cb.cholinv.info(0, 1, 0, "U"))
        cb.cacqr.factor(A, qa, qt)
        e = max(np.abs(qa.R.cpu().numpy() - z[f"R_{rank}"]).max() / np.abs(z[f"R_{rank}"]).max(), np.abs(qa.Q.cpu().numpy() - z[f"Q_{rank}"]).max())
        worst = max(worst, float(e)); cases.append("cacqr_p8_1d_m1024_n32")
    # distributed vs single GPU, a size with several distributed levels and 128-wide tiles
    n = 4096 if world < 8 else 8192
    bcm = -3
    A = cb.matrix(n, n, d, d).distribute_symmetric(topo)
    a = cb.cholinv.info(0, 1, bcm, "U")
    cb.cholinv.factor(A, a, topo)
    t1 = cb.topo.square(1, 0, 1)
    A1 = cb.matrix(n, n, 1, 1).distribute_symmetric(t1)
    a1 = cb.cholinv.info(0, 1, bcm, "U", serialize=False)
    cb.cholinv.factor(A1, a1, t1)
    R1, Ri1 = cb.cholinv.construct_R(a1), cb.cholinv.construct_Rinv(a1)
    R, Ri = cb.cholinv.construct_R(a), cb.cholinv.construct_Rinv(a)
    sel = (slice(topo.y, None, d), slice(topo.x, None, d))
    e = max(((R - torch.triu(R1[sel])).abs().max() / R1.abs().max()).item(), ((Ri - torch.triu(Ri1[sel])).abs().max() / Ri1.abs().max()).item())
    worst = max(worst, float(e)); cases.append(f"cholinv n={n} on {world} GPUs vs 1 GPU (elementwise R, Rinv)")
    t1.context().release_workspace()
    del A, a, A1, a1, R1, Ri1, R, Ri
    torch.cuda.empty_cache()
    return worst, cases


def cacqr_record(cb, torch, dist, world, rank, peak_tf, hbm_gbs, steps):
    """CholeskyQR2 (BASELINE config 4 at N = 8): m = 2^17 rows per GPU, n = 256, 1D row-partitioned grid, num_iter = 2."""
    m, n = (1 << 17) * world, 256
    qt = cb.topo.rect(world, rank, 1)
    A = cb.matrix(n, m, 1, world).distribute_random(qt, rank)
    qa = cb.cacqr.info(2, cb.cholinv.info(0, 1, 0, "U"))
    for _ in range(3):
        cb.cacqr.factor(A, qa, qt)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        cb.cacqr.factor(A, qa, qt)
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = t.item() / steps
    res, orth = cb.cacqr.validate(A, qa, qt)
    flops = 4.0 * m * n * n + 5.0 * n ** 3 / 3
    tf = flops / (ms * 1e-3) / 1e12
    bytes_alg = 2 * 3 * 8.0 * (m // world) * n  # per GPU: 2 sweeps x (2 reads + 1 write) of the local panel (SURVEY 8d)
    rec = {"workload": f"cacqr::factor (CholeskyQR2) m={m} n={n} 1D grid 1x{world}, num_iter=2", "ms": ms, "tflops": tf,
           "tflops_per_gpu": tf / world, "frac_of_dmma_peak": tf / world / peak_tf if peak_tf else None,
           "hbm_gbs_per_gpu_algorithmic": bytes_alg / (ms * 1e-3) / 1e9, "frac_of_hbm_peak": bytes_alg / (ms * 1e-3) / 1e9 / hbm_gbs,
           "residual": res, "orthogonality": orth, "steps": steps}
    qt.context().release_workspace()
    return rec


def ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import capital_b200 as cb

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    n, c, bcm = WORKLOADS[args.gpus]
    if args.n:
        n = args.n
    topo = cb.topo.square(world, rank, c)
    ctx = topo.context()
    dgrid = topo.d

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    # ---- parity of the distributed path, before anything is timed ----
    parity = None
    if world > 1 and not args.no_parity:
        try:
            worst, cases = parity_block(cb, torch, np, world, rank, c)
            worst = reduce_max(worst)
            parity = {"max_rel_err": worst, "cases": cases, "ok": bool(worst < 2e-13),
                      "against": "tests/golden/*_p8_* (per-rank dumps of the reference run by oracle/_ref) and the single-GPU factorization"}
        except Exception as ex:  # noqa
            parity = {"max_rel_err": None, "ok": False, "error": repr(ex)[:300]}

    A = cb.matrix(n, n, dgrid, dgrid).distribute_symmetric(topo)
    pack = cb.cholinv.info(0, 1, bcm, "U")
    for _ in range(args.warmup):
        cb.cholinv.factor(A, pack, topo)
    # ---- FP64 tensor-pipe peak of this device, now, with the clocks watched ----
    samples, stop = [], threading.Event()
    th = threading.Thread(target=clocks_sampler, args=(stop, samples, local_rank), daemon=True)
    barrier()
    if rank == 0:
        th.start()
    try:
        peak_tf, peak_ms = ctx.probe_dmma()
        peak_src = f"DMMA.8x8x4 register loop on all SMs, {peak_ms:.1f} ms, CUDA events, measured in this run right before the timed steps (capital_probe_dmma_f64)"
    except Exception as ex:  # noqa
        peak_tf, peak_src = NOMINAL_DMMA_TFLOPS, f"NOMINAL 148 SM x 64 FMA/clk x 1.965 GHz (in-run probe failed: {ex!r})"
    hbm_gbs = HBM_GBS_FALLBACK
    try:
        hbm_gbs = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        pass
    # ---- timed region: resident inputs ----
    ctx.reset_counters()
    ctx.profile_begin()  # events around the dominant kernel's launches only: negligible perturbation
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        cb.cholinv.factor(A, pack, topo)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    stop.set()
    k_ms, k_flops, k_launches = ctx.profile_end()
    cnt = ctx.counters()
    dumped = sample_outputs(torch, np, pack, world, rank) if args.dump_outputs else None  # before later steps reuse `pack`
    # The timed steps overlap kernels on two streams, which stretches event-bracketed launch durations.  The roofline
    # number is therefore taken from one extra step with the deferred stream disabled (same kernels, same launches).
    ctx.set_overlap(False)
    cb.cholinv.factor(A, pack, topo)
    ctx.profile_begin()
    barrier()
    e0.record()
    cb.cholinv.factor(A, pack, topo)
    e1.record()
    barrier()
    s_ms_step = e0.elapsed_time(e1)
    s_ms, s_flops, s_launches = ctx.profile_end()
    ctx.set_overlap(True)
    ms_step = reduce_max(ms) / args.steps
    value = n ** 3 / 3 / (ms_step * 1e-3) / 1e12
    residual = cb.cholinv.residual(A, pack, topo)
    # optional: one more step with CUDA events around every launch (the image has no nsys), summarised into the line and saved per rank
    timeline = None
    if os.environ.get("CAPITAL_BENCH_TIMELINE"):
        try:
            cb.cholinv.factor(A, pack, topo)
            barrier()
            ctx.timeline_begin()
            cb.cholinv.factor(A, pack, topo)
            tl = ctx.timeline_end()
            os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
            np.save(os.path.join(ROOT, "gpurun_out", f"timeline_n{world}_r{rank}.npy"), tl)

            def union(iv):
                iv = sorted(iv)
                tot, (cs, ce) = 0.0, iv[0]
                for a, b in iv[1:]:
                    if a > ce:
                        tot += ce - cs; cs, ce = a, b
                    else:
                        ce = max(ce, b)
                return tot + ce - cs
            big = tl[tl[:, 1] == 1]
            ch = tl[tl[:, 0] == 1]
            w = ch[ch[:, 1] == 5]
            chs = ch[np.argsort(ch[:, 2])]
            gaps = chs[1:, 2] - chs[:-1, 3]
            timeline = {"span_ms": float(tl[:, 3].max() - tl[:, 2].min()), "launches": int(len(tl)),
                        "big_gemm_union_ms": float(union([(a, b) for a, b in big[:, 2:4]])) if len(big) else 0.0,
                        "chain_busy_ms": float((ch[:, 3] - ch[:, 2]).sum()), "chain_flag_wait_ms": float((w[:, 3] - w[:, 2]).sum()) if len(w) else 0.0,
                        "chain_gaps_over_1ms": [float(g) for g in np.sort(gaps[gaps > 1.0])[-6:]],
                        "note": "rank 0, one extra step with events around every launch (slower than the timed steps)"}
        except Exception as ex:  # noqa
            timeline = {"error": repr(ex)[:200]}

    # ---- end to end: pinned host buffers through the same public call ----
    e2e = None
    try:
        hostA = cb.matrix(n, n, dgrid, dgrid, data=A.data.cpu().pin_memory())
        hpack = cb.cholinv.info(0, 1, bcm, "U")
        cb.cholinv.factor(hostA, hpack, topo)  # warm-up: allocates pinned outputs + staging
        steps_e = max(1, min(args.steps, 3))
        ctx.reset_counters()
        barrier()
        e0.record()
        for _ in range(steps_e):
            cb.cholinv.factor(hostA, hpack, topo)
        e1.record()
        barrier()
        c2 = ctx.counters()
        ms_e = reduce_max(e0.elapsed_time(e1)) / steps_e
        e2e = {"value": n ** 3 / 3 / (ms_e * 1e-3) / 1e12, "unit": "TFLOP/s", "ms_per_step": ms_e, "steps": steps_e,
               "h2d_bytes_per_step": c2.h2d_bytes // steps_e, "d2h_bytes_per_step": c2.d2h_bytes // steps_e,
               "note": "per rank; pinned host A in, pinned host R and Rinv (packed upper) out"}
        del hostA, hpack
    except Exception as ex:  # noqa
        e2e = {"value": None, "unit": "TFLOP/s", "error": repr(ex)[:200], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    del A, pack
    torch.cuda.empty_cache()

    # ---- fixed-size row: the same n on every N ----
    strong = None
    if not args.no_extra and not args.n:
        try:
            sb = STRONG_BCM[world]
            As = cb.matrix(STRONG_N, STRONG_N, dgrid, dgrid).distribute_symmetric(topo)
            sp = cb.cholinv.info(0, 1, sb, "U")
            for _ in range(2):
                cb.cholinv.factor(As, sp, topo)
            barrier()
            e0.record()
            for _ in range(2):
                cb.cholinv.factor(As, sp, topo)
            e1.record()
            barrier()
            ms_s = reduce_max(e0.elapsed_time(e1)) / 2
            strong = {"n": STRONG_N, "bc_mult_dim": sb, "ms_per_step": ms_s, "tflops": STRONG_N ** 3 / 3 / (ms_s * 1e-3) / 1e12,
                      "residual": cb.cholinv.residual(As, sp, topo), "note": "same n at every N: strong scaling of cholinv::factor"}
            del As, sp
        except Exception as ex:  # noqa
            strong = {"n": STRONG_N, "error": repr(ex)[:200]}
        ctx.release_workspace()
        torch.cuda.empty_cache()
    # ---- CholeskyQR2 ----
    cacqr = None
    if not args.no_extra:
        try:
            cacqr = cacqr_record(cb, torch, dist, world, rank, peak_tf, hbm_gbs, max(3, args.steps))
        except Exception as ex:  # noqa
            cacqr = {"error": repr(ex)[:300]}

    # ---- the same two records with the OTHER flag-wait flavour (same box, same context; nothing above depends on it) ----
    # Default: acquire-spin wait kernels (or flushed memory-op waits where the device can flush).  "memop" = unflushed
    # cuStreamWaitValue64, what the round-2 profiles were measured with and what showed 1e-10-level residuals at n = 32768 over
    # NVLink (DESIGN.md section 5).  Timing and residual of both, side by side.
    wait_modes = None
    if world > 1 and not args.no_extra and not args.n:
        mode0 = ctx.peer_wait_mode()
        try:
            other = "memop" if mode0 != "memop" else "kernel"
            ctx.set_peer_wait_mode(other)
            wait_modes = {"default": mode0, "other": other}
            for label, nn, bb in (("headline", n, bcm), ("strong", STRONG_N, STRONG_BCM[world])):
                Aa = cb.matrix(nn, nn, dgrid, dgrid).distribute_symmetric(topo)
                pp = cb.cholinv.info(0, 1, bb, "U")
                for _ in range(2):
                    cb.cholinv.factor(Aa, pp, topo)
                barrier()
                e0.record()
                for _ in range(3):
                    cb.cholinv.factor(Aa, pp, topo)
                e1.record()
                barrier()
                ms_o = reduce_max(e0.elapsed_time(e1)) / 3
                wait_modes[label + "_with_other"] = {"n": nn, "ms_per_step": ms_o, "tflops": nn ** 3 / 3 / (ms_o * 1e-3) / 1e12,
                                                     "residual": cb.cholinv.residual(Aa, pp, topo), "steps": 3}
                del Aa, pp
                ctx.release_workspace()
                torch.cuda.empty_cache()
        except Exception as ex:  # noqa
            wait_modes = {"default": mode0, "error": repr(ex)[:300]}
        finally:
            try:
                ctx.set_peer_wait_mode(mode0)
            except Exception:  # noqa
                pass

    # ---- EXPERIMENTAL (BASELINE config 5, off by default in the library): trailing updates on the TF32 tensor cores ----
    # Child process: the tcgen05 kernel was written without GPU access and has its own CUDA context here, so that nothing it does can
    # touch the numbers above.  Single GPU only in the bench; the c = 1 grids take the same path through dist.cu.
    tf32 = None
    if world == 1 and not args.no_extra and not args.n:
        try:
            r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "tf32_worker.py"), "bench", str(n), str(bcm), "3"],
                               capture_output=True, text=True, timeout=240)
            if r.returncode == 0:
                tf32 = json.loads(r.stdout.strip().splitlines()[-1])
                tf32["dtype"] = "tf32 (tcgen05.mma.kind::tf32, FP32 accumulation in TMEM) for A22 -= R12^T R12 with k >= 256; everything else f64"
                tf32["status"] = "experimental: first executed by whoever runs this; see tests/test_gpu_zz_late.py for the parity gates"
            else:
                tf32 = {"error": r.stderr[-300:]}
        except Exception as ex:  # noqa
            tf32 = {"error": repr(ex)[:300]}

    # DRAM traffic of the dominant kernel: only from an `ncu --set full` capture of THIS kernel source (hash-checked), else null
    traffic, traffic_src = None, "no ncu --set full capture of this build of gemm_tn.cu travels with the repo"
    try:
        import hashlib
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_gemm_traffic.json")))
        sha = hashlib.sha256(open(os.path.join(ROOT, "capital_b200", "csrc", "gemm_tn.cu"), "rb").read()).hexdigest()[:16]
        if tj.get("gemm_tn_cu_sha256_16") == sha and world == 1:
            traffic = tj["traffic_bytes_per_launch_mean"]
            traffic_src = "profiles/r02_gemm_traffic.json (dram__bytes_read.sum + dram__bytes_write.sum, mean of 3 launches, same gemm_tn.cu hash): " + tj["source"]
    except Exception:
        pass
    if rank == 0:
        ach = s_flops / (s_ms * 1e-3) / 1e12 if s_ms > 0 else None
        ach_ov = k_flops / (k_ms * 1e-3) / 1e12 if k_ms > 0 else None
        out = {
            "metric": "cholesky_tflops_fp64", "value": value, "unit": "TFLOP/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "scaling_note": "sizes are BASELINE.json's per-N configs (n = 16384 / 24576 / 32768 / 65536: per-GPU work is NOT constant); "
                            "`strong` repeats the measurement at one fixed n",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(world, n, c, bcm),
            "work_tflops": 5 * n ** 3 / 12 / (ms_step * 1e-3) / 1e12,  # CholInv with complete_inv=0 does 5n^3/12 flops
            "work_frac_of_peak": 5 * n ** 3 / 12 / (ms_step * 1e-3) / 1e12 / (peak_tf * world),
            "residual": residual,
            "roofline": {"bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": (ach / peak_tf) if ach else None,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "gemm_tn_kernel<128,128,64,32,5> (DMMA.8x8x4 + TMA" + (", depth exchange fused in the epilogue)" if world > 1 else ")"),
                         "launches": s_launches,
                         "kernel_share_of_step": s_ms / s_ms_step if s_ms_step else None,
                         "measured_in": (f"one extra step after the timed region with the deferred stream disabled (single-stream step {s_ms_step:.2f} ms); "
                                         f"inside the overlapped timed region the same launches read {ach_ov:.2f} TF/s because concurrent kernels share SMs")
                                        if ach_ov else None,
                         "peak_source": peak_src},
            "e2e": e2e, "gpu_launches": int(cnt.kernel_launches), "clocks": summarize_clocks(samples),
        }
        if world > 1:
            out["config"]["peer_flag_wait"] = ctx.peer_wait_mode()
        if timeline is not None:
            out["timeline"] = timeline
        if parity is not None:
            out["parity"] = parity
        if strong is not None:
            out["strong"] = strong
        if tf32 is not None:
            out["mixed_precision_tf32"] = tf32
        if wait_modes is not None:
            out["flag_wait_modes"] = wait_modes
        if cacqr is not None:
            out["cacqr"] = cacqr
        if world == 1 and not args.no_cpu:
            d = run_reference_cholinv(min(n, 16384), bcm, 1, 1, timeout=600)
            if d and "time_mean_s" in d:
                ns = min(n, 16384)
                out["cpu_baseline"] = {"value": ns ** 3 / 3 / d["time_mean_s"] / 1e12, "unit": "TFLOP/s", "cores": d["cores"], "kind": "reference",
                                       "sample": f"reference cholinv::factor n={ns} same args, 1 rank x {d['threads_per_rank']} OpenBLAS threads, "
                                                 f"{d['time_mean_s']:.3f} s, residual {d['residual']:.2e}"}
            else:
                out["cpu_baseline"] = {"value": None, "unit": "TFLOP/s", "cores": os.cpu_count(), "kind": "reference", "sample": f"failed: {d}"}
        print(json.dumps(out))
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    if world > 1:
        dist.barrier()
        cb.topo.release_contexts()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=0, help="override the matrix size (debug)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-parity", action="store_true", help="skip the N > 1 parity block")
    ap.add_argument("--no-extra", action="store_true", help="skip the strong-scaling and CholeskyQR2 records")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write a seeded sample of the last step's R and Rinv "
                                                          "to DIR/<name>.npy (FP64, 32 MB)")
    args = ap.parse_args()
    if args.gpus not in WORKLOADS:
        raise SystemExit("--gpus must be one of 1, 2, 4, 8")
    if args.steps < 1:
        raise SystemExit("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        raise SystemExit("--dump-outputs needs --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    return reference_arm(args) if args.impl == "reference" else ours(args)


if __name__ == "__main__":
    sys.exit(main())
