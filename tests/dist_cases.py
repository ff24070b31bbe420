"""Configurations of the distributed CholInv schedule (capital_b200/csrc/dist.cu) that both the CPU replay of its flag protocol
(test_dist_protocol.py) and the GPU parity worker (dist_variants_worker.py, ranks sharing one GPU) run, so that the GPU never runs a
configuration the replay has not checked.

A knob set is the CAPITAL_DIST_* environment that dist_setup reads on every call.  The knobs only change how the same products are
partitioned into launches, which stream runs them and in which order they are issued; with the lowered thresholds the small sizes
below take every deferred class (one per recursion depth 0 .. 2) and column-chunked, pushed products, as n = 65536 on eight GPUs
does with the defaults.

Sizes: n = 2048 gives power-of-two split points; n = 2052 (local size 1026) and n = 3076 (1538) split on odd rows at every level, so
operand windows start on 8-byte boundaries and every GEMM copies them to its stream's alignment scratch first.  bc_mult_dim = -2
keeps the local base case at 64 or more.

The GPU runs the ragged sizes under every knob set and the power-of-two size under the default one only (gpu_cases): with all ranks
time-slicing one GPU a factorization costs seconds at these sizes, whatever n.
"""
import os
from collections import namedtuple

KNOB_VARS = ("CAPITAL_DIST_TWO_STREAM", "CAPITAL_DIST_FAR_MIN", "CAPITAL_DIST_SIDE_MIN", "CAPITAL_DIST_CHUNK_MIN",
             "CAPITAL_DIST_CHUNKS", "CAPITAL_DIST_BULK", "CAPITAL_DIST_PIPELINE", "CAPITAL_DIST_FLUSH_READS")
_DEFERRED = {"CAPITAL_DIST_FAR_MIN": "64", "CAPITAL_DIST_SIDE_MIN": "32"}
_CHUNKED4 = {**_DEFERRED, "CAPITAL_DIST_CHUNK_MIN": "256", "CAPITAL_DIST_CHUNKS": "4"}
KNOBS = {
    "default": {},
    "deferred": _DEFERRED,
    "chunked4": _CHUNKED4,
    "chunked3": {**_CHUNKED4, "CAPITAL_DIST_CHUNKS": "3"},  # ragged last chunk unless s2 is a multiple of 384
    "pipelined": {**_CHUNKED4, "CAPITAL_DIST_PIPELINE": "1"},
    "single_stream": {"CAPITAL_DIST_TWO_STREAM": "0"},
    "no_bulk": {"CAPITAL_DIST_BULK": "0"},
}

GRIDS = {2: (2, 1), 4: (1, 2), 8: (2, 2)}  # ranks -> (c, d): 2x1x1, 1x2x2, 2x2x2
SIZES = {2: (1024, 1026), 4: (2048, 2052, 3076), 8: (2048, 2052, 3076)}
BC_MULT_DIM = -2

Case = namedtuple("Case", "size c d n ci split bcm knobs")


def cases(size):
    """Every case of one grid, in run order: per (n, complete_inv, split) the default knob set first, then the others.  A ragged size
    follows a power-of-two one, so its first call changes the arena layout of the context."""
    c, d = GRIDS[size]
    for n in SIZES[size]:
        for ci in (0, 1):
            for split in (1, 2):
                for k in KNOBS:
                    yield Case(size, c, d, n, ci, split, BC_MULT_DIM, k)


def all_cases():
    return [cs for size in GRIDS for cs in cases(size)]


def ragged(case):
    L = case.n // case.d
    return L & (L - 1) != 0


def gpu_cases(size):
    return [cs for cs in cases(size) if ragged(cs) or cs.knobs == "default"]


def set_knobs(name, environ=None):
    """Make `environ` (default os.environ) hold exactly the knob set `name` among the CAPITAL_DIST_* variables."""
    env = os.environ if environ is None else environ
    for v in KNOB_VARS:
        env.pop(v, None)
    env.update(KNOBS[name])
