"""CPU check of the multi-GPU flag protocol of capital_b200/csrc/dist.cu (no GPU, no mirror implementation).

`capital_dist_trace_cholinv` dry-runs the REAL schedule code of one rank: every flag wait / signal, fused product, event
record / wait, peer DMA and arena window access it would enqueue for two consecutive cholinv::factor calls.  The traces of all
ranks of a grid are replayed here under CUDA's ordering rules (streams are FIFO; an event wait waits for the record that preceded
it; a flag wait stalls the stream until the flag reaches the value) and checked for
  * deadlock freedom: the replay must drain every stream of every rank;
  * data races: two accesses to overlapping windows of the same rank's arena, at least one a write, must be ordered by
    happens-before (vector clocks) -- i.e. every operand a product reads from a mirror slot was pushed AND waited for, and
    nothing of the next factorization overwrites what the previous one may still be reading;
  * scratch conflicts: a product whose operand starts on an odd row first copies it into an alignment scratch of its stream
    (gemm_tn.cu); two uses of one scratch must be ordered too.
"""
import ctypes as C
import numpy as np
import pytest
import capital_b200 as cb
from capital_b200 import _lib
import dist_cases

T_WAIT, T_SIGNAL, T_PRODUCT, T_EVREC, T_EVWAIT, T_DMA, T_KERNEL, T_READ, T_WRITE, T_MAT = range(1, 11)
NSTREAM = 12


def trace(size, rank, c, n, ci, bcm, split=1):
    g = cb.topo.square(size, rank, c).grid
    args = _lib.CholinvArgs(ci, split, bcm, b"U")
    cnt = C.c_int64()
    L = _lib.lib()
    st = L.capital_dist_trace_cholinv(C.byref(g), n, C.byref(args), None, 0, C.byref(cnt))
    assert st == 0
    buf = np.zeros((cnt.value, 8), dtype=np.int64)
    st = L.capital_dist_trace_cholinv(C.byref(g), n, C.byref(args), buf.ctypes.data_as(C.POINTER(C.c_int64)), cnt.value, C.byref(cnt))
    assert st == 0
    return buf


class Replay:
    def __init__(self, traces):
        self.P = len(traces)
        self.nclk = self.P * NSTREAM
        self.streams = [[[] for _ in range(NSTREAM)] for _ in range(self.P)]
        self.mats = [[] for _ in range(self.P)]
        self.recorded = [set() for _ in range(self.P)]  # events each rank records somewhere in its trace
        for r, tr in enumerate(traces):
            for rec in tr:
                if rec[0] == T_MAT:
                    self.mats[r].append((int(rec[2]), int(rec[3]), int(rec[4])))
                else:
                    self.streams[r][int(rec[1])].append(tuple(int(v) for v in rec))
                    if rec[0] == T_EVREC:
                        self.recorded[r].add(int(rec[2]))
        self.head = [[0] * NSTREAM for _ in range(self.P)]
        self.clock = [[np.zeros(self.nclk, dtype=np.int64) for _ in range(NSTREAM)] for _ in range(self.P)]
        self.flags = {}      # (rank, word) -> (value, clock)
        self.events = {}     # (rank, ev) -> clock
        self.started = {}    # (rank, q, seq) -> clock at kernel start
        self.accesses = []   # (rank_of_memory, off, ld, rows, cols, is_write, group, clock, who)
        self.pending_acc = [[[] for _ in range(NSTREAM)] for _ in range(self.P)]

    def tick(self, r, s):
        c = self.clock[r][s].copy()
        c[r * NSTREAM + s] += 1
        self.clock[r][s] = c
        return c

    def partners(self, r, grid):
        c, d = grid
        z = r % c
        return [r - z + l for l in range(c) if l != z]

    def try_op(self, r, s, grid):
        q = self.streams[r][s]
        i = self.head[r][s]
        if i >= len(q):
            return False
        op = q[i]
        kind = op[0]
        clk = self.clock[r][s]
        if kind == T_WAIT:
            f = self.flags.get((r, op[2]))
            if f is None or f[0] < op[3]:
                return False
            self.clock[r][s] = np.maximum(clk, f[1])
            self.tick(r, s)
        elif kind == T_SIGNAL:
            c = self.tick(r, s)
            key = (op[2], op[3])
            old = self.flags.get(key)
            assert old is None or old[0] < op[4], f"flag {key} goes backwards: {old[0]} -> {op[4]}"
            self.flags[key] = (op[4], c if old is None else np.maximum(c, old[1]))
        elif kind == T_EVREC:
            c = self.tick(r, s)
            self.events[(r, op[2])] = c
        elif kind == T_EVWAIT:
            e = self.events.get((r, op[2]))
            if e is None:
                # CUDA: waiting for an event that was never recorded is a no-op -- but the schedule never does that on purpose
                assert op[2] in self.recorded[r], f"rank {r}: wait for event {op[2]} that is never recorded"
                return False
            self.clock[r][s] = np.maximum(clk, e)
            self.tick(r, s)
        elif kind == T_PRODUCT:
            # a GEMM launch: it needs nothing from other ranks while it runs (partials / final tiles are stored into the partners'
            # buffers, the handshake that follows is explicit flag traffic)
            self.tick(r, s)
            self.flush_accesses(r, s)
        elif kind in (T_READ, T_WRITE):
            self.pending_acc[r][s].append(op)
        else:  # T_DMA, T_KERNEL
            self.tick(r, s)
            self.flush_accesses(r, s)
        self.head[r][s] = i + 1
        return True

    def flush_accesses(self, r, s, start=None):
        end = self.clock[r][s]
        start = end if start is None else start
        for op in self.pending_acc[r][s]:
            self.accesses.append((op[2], op[3], op[4], op[5], op[6], op[0] == T_WRITE, op[7] if op[0] == T_WRITE else 0, start, (r, s), end))
        self.pending_acc[r][s] = []

    def run(self, grid):
        progress = True
        while progress:
            progress = False
            for r in range(self.P):
                for s in range(NSTREAM):
                    while self.try_op(r, s, grid):
                        progress = True
        stuck = [(r, s, self.streams[r][s][self.head[r][s]]) for r in range(self.P) for s in range(NSTREAM)
                 if self.head[r][s] < len(self.streams[r][s])]
        return stuck

    # ---- race detection ----
    def slot_of(self, rank, off):
        for base, ld, cols in self.mats[rank]:
            if base <= off < base + ld * cols * 8:
                return base, ld
        return None

    def races(self):
        """Unordered conflicting pairs: (key, rect, R/W, (rank, stream), rect, R/W, (rank, stream)).  key[1] == "scratch" marks a
        conflict on a GEMM's operand-alignment scratch (a buffer of the rank's context, outside the arena) rather than in the arena."""
        buckets = {}
        for a in self.accesses:
            rank, off, ld, rows, cols = a[:5]
            if off < 0:  # scratch slot -off - 1 of the rank's context: every use overlaps every other
                key, rect = (rank, "scratch", -off - 1), (0, 1, 0, 1)
            elif (sl := self.slot_of(rank, off)) is None or sl[1] != ld:
                key = (rank, "raw")   # 1-D buffers (gather slots): byte ranges
                rect = (off, off + rows * cols * 8, 0, 1)
            else:
                e = (off - sl[0]) // 8
                c0, r0 = divmod(e, ld)
                rect = (r0, r0 + rows, c0, c0 + cols)
                key = (rank, sl[0])
            buckets.setdefault(key, []).append((rect, a))
        bad = []
        for key, lst in buckets.items():
            rect = np.array([r for r, _ in lst], dtype=np.int64).reshape(-1, 4)
            wr = np.array([a[5] for _, a in lst], dtype=bool)
            grp = np.array([a[6] for _, a in lst], dtype=np.int64)
            who = np.array([a[8][0] * NSTREAM + a[8][1] for _, a in lst], dtype=np.int64)
            start = np.array([a[7] for _, a in lst], dtype=np.int64).reshape(len(lst), -1)
            end = np.array([a[9] for _, a in lst], dtype=np.int64).reshape(len(lst), -1)
            end_own = end[np.arange(len(lst)), who]
            idx = np.arange(len(lst))
            for i in np.nonzero(wr)[0]:  # every conflicting pair has a write: pair it with every later access and every earlier read
                m = (idx > i) | ~wr
                if grp[i]:
                    m &= ~(wr & (grp == grp[i]))  # cooperating writers of one fused product (disjoint tiles)
                m &= (rect[:, 0] < rect[i, 1]) & (rect[i, 0] < rect[:, 1]) & (rect[:, 2] < rect[i, 3]) & (rect[i, 2] < rect[:, 3])
                m[i] = False
                m &= end_own[i] > start[:, who[i]]     # not: the write's end happens-before the other's start
                m &= end_own > start[i, who]           # not: the other's end happens-before the write's start
                for j in np.nonzero(m)[0]:
                    (ra, a), (rb, b) = lst[min(i, j)], lst[max(i, j)]
                    bad.append((key, ra, "W" if a[5] else "R", a[8], rb, "W" if b[5] else "R", b[8]))
        return bad


GRIDS = {2: (2, 1), 4: (1, 2), 8: (2, 2)}


@pytest.mark.parametrize("size,n,ci,bcm", [
    (2, 1024, 0, -3), (2, 1024, 1, -2),
    (4, 1024, 0, -2), (4, 2048, 1, -3),
    (8, 1024, 1, -2), (8, 2048, 0, -3), (8, 4096, 1, -3),
])
def test_flag_protocol_is_deadlock_free_and_race_free(size, n, ci, bcm, monkeypatch):
    # small nodes must exercise the deferred class too
    monkeypatch.setenv("CAPITAL_DIST_FAR_MIN", "64")
    monkeypatch.setenv("CAPITAL_DIST_SIDE_MIN", "32")
    monkeypatch.setenv("CAPITAL_DIST_CHUNK_MIN", "256")  # ... and the chunked, pushed products
    c, d = GRIDS[size]
    traces = [trace(size, r, c, n, ci, bcm) for r in range(size)]
    rp = Replay(traces)
    stuck = rp.run((c, d))
    assert not stuck, f"deadlock: {len(stuck)} streams blocked, e.g. {stuck[:4]}"
    kinds = np.concatenate(traces)[:, 0]
    if size > 1:
        assert (kinds == T_PRODUCT).sum() > 0
    if d > 1:
        assert (kinds == T_DMA).sum() > 0 and (kinds == T_WAIT).sum() > 0
    bad = rp.races()
    assert not bad, f"{len(bad)} unordered conflicting accesses, e.g. {bad[:3]}"


@pytest.mark.parametrize("size,n,ci", [(8, 2048, 1), (8, 2048, 0), (4, 2048, 1), (2, 1024, 0)])
def test_uneven_split_is_clean_too(size, n, ci, monkeypatch):
    """split = 2 (cholinv.hpp:92,107: the left child gets a quarter): node sizes stop being powers of two, every window offset changes"""
    monkeypatch.setenv("CAPITAL_DIST_FAR_MIN", "64")
    monkeypatch.setenv("CAPITAL_DIST_SIDE_MIN", "32")
    monkeypatch.setenv("CAPITAL_DIST_CHUNK_MIN", "256")
    c, d = GRIDS[size]
    traces = [trace(size, r, c, n, ci, -3, split=2) for r in range(size)]
    rp = Replay(traces)
    assert not rp.run((c, d))
    assert not rp.races()


def test_pipelined_chunked_products_are_clean_too(monkeypatch):
    """opt-in CAPITAL_DIST_PIPELINE=1: chunk j + 1 is issued before chunk j is added up (three rotating exchange sets + the
    'reduced' flag keep a partner from overwriting a set that is still being read)"""
    monkeypatch.setenv("CAPITAL_DIST_PIPELINE", "1")
    monkeypatch.setenv("CAPITAL_DIST_CHUNK_MIN", "256")
    monkeypatch.setenv("CAPITAL_DIST_FAR_MIN", "64")
    monkeypatch.setenv("CAPITAL_DIST_SIDE_MIN", "32")
    traces = [trace(8, r, 2, 2048, 1, -3) for r in range(8)]
    rp = Replay(traces)
    assert not rp.run((2, 2))
    assert not rp.races()
    # and the flag that protects the rotating sets is load-bearing: without its waits the replay finds the race
    CTRL_RED_LO, CTRL_RED_HI = 192, 272
    mut = [tr[~((tr[:, 0] == T_WAIT) & (tr[:, 2] >= CTRL_RED_LO) & (tr[:, 2] < CTRL_RED_HI))] for tr in traces]
    rp2 = Replay(mut)
    assert not rp2.run((2, 2))
    assert rp2.races()


def test_single_stream_schedule_also_clean(monkeypatch):
    monkeypatch.setenv("CAPITAL_DIST_TWO_STREAM", "0")
    traces = [trace(8, r, 2, 1024, 1, -2) for r in range(8)]
    rp = Replay(traces)
    assert not rp.run((2, 2))
    assert not rp.races()


def replay_case(case):
    traces = [trace(case.size, r, case.c, case.n, case.ci, case.bcm, case.split) for r in range(case.size)]
    rp = Replay(traces)
    stuck = rp.run((case.c, case.d))
    bad = rp.races()
    arena = [b for b in bad if b[0][1] != "scratch"]
    scratch = [b for b in bad if b[0][1] == "scratch"]
    return rp, stuck, arena, scratch


@pytest.mark.parametrize("case", dist_cases.all_cases(), ids=lambda c: f"p{c.size}-n{c.n}-ci{c.ci}-split{c.split}-{c.knobs}")
def test_schedule_table_drains_without_races_or_scratch_conflicts(case, monkeypatch):
    """Every configuration the GPU parity worker runs (tests/dist_cases.py).  Odd split points make every GEMM copy its misaligned
    operands into its stream's alignment scratch first; the chain and the deferred streams of depths 1 and 2 run such products at
    the same time, so one scratch shared between them is overwritten while another stream's GEMM still reads it."""
    for v in dist_cases.KNOB_VARS:
        monkeypatch.delenv(v, raising=False)
    for k, v in dist_cases.KNOBS[case.knobs].items():
        monkeypatch.setenv(k, v)
    rp, stuck, arena, scratch = replay_case(case)
    assert not stuck, f"deadlock: {len(stuck)} streams blocked, e.g. {stuck[:4]}"
    assert not arena, f"{len(arena)} unordered conflicting arena accesses, e.g. {arena[:3]}"
    assert not scratch, f"{len(scratch)} unordered uses of one alignment scratch, e.g. {scratch[:3]}"
    if dist_cases.ragged(case):  # the pseudo-accesses of the scratch must be in the trace
        assert sum(1 for a in rp.accesses if a[1] < 0) > 0


def test_scratch_uses_of_different_streams_are_unordered():
    """The scratch check has teeth: merged onto one scratch slot per rank (as when every stream shared one buffer), the uses of
    the chain and of the deferred streams in a ragged row of the table are unordered."""
    case = next(c for c in dist_cases.all_cases() if c.size == 8 and c.n == 2052 and c.split == 1 and c.knobs == "deferred")
    with pytest.MonkeyPatch.context() as mp:
        for k, v in dist_cases.KNOBS[case.knobs].items():
            mp.setenv(k, v)
        traces = [trace(case.size, r, case.c, case.n, case.ci, case.bcm, case.split) for r in range(case.size)]
    merged = []
    for tr in traces:
        tr = tr.copy()
        scr = (tr[:, 0] == T_WRITE) & (tr[:, 3] < 0)
        assert scr.any()
        tr[scr, 3] = -1
        merged.append(tr)
    rp = Replay(merged)
    assert not rp.run((case.c, case.d))
    bad = rp.races()
    assert bad and all(b[0][1] == "scratch" for b in bad)
    assert {b[3][1] for b in bad} | {b[6][1] for b in bad} >= {1, 3, 4}  # chain, deferred depth 1, deferred depth 2


@pytest.mark.parametrize("size", sorted(dist_cases.GRIDS))
@pytest.mark.parametrize("split", [1, 2, 3])
@pytest.mark.parametrize("bcm", [0, -3, -5, -8])
def test_base_case_windows_fit_their_buffers(size, split, bcm, monkeypatch):
    """Local size 256: bc_mult_dim -8 leaves a local base case of 1, where a split = 2 (3) node still stops at up to 7 (23) rows.
    base_case refuses any window wider than what the gather buffers and the dense block were sized for, in the dry run too, so a
    trace with status 0 proves that every window of the recursion fits."""
    for v in dist_cases.KNOB_VARS:
        monkeypatch.delenv(v, raising=False)
    c, d = dist_cases.GRIDS[size]
    n = 256 * d
    traces = [trace(size, r, c, n, 1, bcm, split) for r in range(size)]
    assert not Replay(traces).run((c, d))
