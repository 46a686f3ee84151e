"""A CPU model of the cull walk of the shared-memory-table kernel (render_kernel<false>, rtclj_render_body.cuh): which
blocks each round culls, which half blocks it records in the lane's survivor list, and where the next round starts
after the list filled up (a "flush").  The tests use it to show that a scene reaches the path it was built for.

The walk, per ray.  The table is cut into 16-pair blocks (32 spheres) and, if n is not a multiple of 32, one trailing
8-pair half block (the "tail").  One list entry is one 16-sphere half block with at least one survivor.  A round
starts with an empty list and culls blocks, shared-memory ones first (those below S), then global ones; the
survivors of a block are recorded one block late (the "pending" block), so a block is culled only while the list has
room for the pending block and the one culled next (`cnt <= kListCap - 4`).  When that loop stops, the pending block
is recorded.  The tail is culled once every block is, and only if one entry is still free; otherwise it is left for
the next round.  The rounds go on until every block and the tail are done."""
from __future__ import annotations

import os
import re
from dataclasses import dataclass
from typing import Dict, Iterable, List, Tuple

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "raytracing-clj_b200", "csrc")

# (file, pattern, names of the groups): the constants of the walk and of the shared-memory split, from the source
_PATTERNS = (
    ("rtclj_kernels.cuh", r"constexpr int kListCap = (\d+);", ("kListCap",)),
    ("rtclj_kernels.cuh", r"constexpr int kBlockPairs = (\d+);", ("kBlockPairs",)),
    ("rtclj_kernels.cuh", r"#define RTCLJ_THREADS_SMEM (\d+)", ("RTCLJ_THREADS_SMEM",)),
    ("rtclj_abi.cu", r"const size_t fixed = \(size_t\)kListCap \* threads_of\(false\) \* (\d+) \+ (\d+) \+ "
                     r"\(size_t\)threads_of\(false\) \* (\d+);",
     ("list_entry_bytes", "barrier_bytes", "sum_bytes_per_thread")),
    ("rtclj_abi.cu", r"return smem_optin > fixed \? \(int\)\(\(smem_optin - fixed\) / (\d+)\) : 0;", ("block_bytes",)),
    ("rtclj_abi.cu", r"bool use_const_table\(int nhalf\) \{ return nhalf \* 16 <= (\d+); \}", ("const_table_max",)),
    ("rtclj_abi.cu", r"if \(n > (\d+)\) return fail\(RTCLJ_E_TOO_LARGE,", ("max_spheres",)),
)


def source_constants() -> Dict[str, int]:
    """The constants above, parsed from the library's source.  A pattern that no longer matches is an error: the
    tests built on it would otherwise stop reaching the paths they were written for without noticing."""
    out = {}
    for path, pattern, names in _PATTERNS:
        text = open(os.path.join(CSRC, path)).read()
        found = re.findall(pattern, text)
        if len(found) != 1:
            raise AssertionError(f"{path}: expected one match of {pattern!r}, found {len(found)}")
        values = found[0] if isinstance(found[0], tuple) else (found[0],)
        out.update({name: int(v) for name, v in zip(names, values)})
    return out


C = source_constants()
LIST_CAP = C["kListCap"]        # survivor entries per lane
BLOCK_PAIRS = C["kBlockPairs"]  # a block is 2 * BLOCK_PAIRS spheres, two half blocks
BLOCK_SPHERES = 2 * BLOCK_PAIRS
HALF_SPHERES = BLOCK_PAIRS


def smem_table_blocks(smem_optin: int) -> int:
    """S: the blocks of the table that fit in shared memory next to the lists, the barrier and the unit sums
    (smem_table_blocks in rtclj_abi.cu)."""
    threads = C["RTCLJ_THREADS_SMEM"]
    fixed = LIST_CAP * threads * C["list_entry_bytes"] + C["barrier_bytes"] + threads * C["sum_bytes_per_thread"]
    return (smem_optin - fixed) // C["block_bytes"] if smem_optin > fixed else 0


@dataclass(frozen=True)
class Round:
    start: int                 # the first block the round culls (== nblocks: a round that culls the tail only)
    stop: int                  # one past the last block it culls
    halves: Tuple[int, ...]    # half blocks recorded, in list order
    tail: bool                 # the round culls the tail half block
    global_blocks: Tuple[int, ...]  # blocks it reads from global memory (the tail not included)


def layout(n: int) -> Tuple[int, int]:
    """(nblocks, tail8) of a scene of n spheres, as rtclj_ctx_render sets them."""
    nhalf = -(-n // HALF_SPHERES)
    return nhalf // 2, nhalf & 1


def tail_is_global(n: int, smem_blocks: int) -> bool:
    nblocks, tail8 = layout(n)
    return bool(tail8) and not nblocks < smem_blocks


def walk(n: int, smem_blocks: int, survivors: Iterable[int], cap: int = LIST_CAP) -> List[Round]:
    """Replays the two `while` loops, the pending record, the tail rule and the outer loop of the walk for one ray
    whose surviving half blocks are `survivors` (indices 0 .. ceil(n / 16) - 1)."""
    nblocks, tail8 = layout(n)
    surv = set(survivors)
    assert all(0 <= h < 2 * nblocks + tail8 for h in surv), "half block out of range"
    rounds = []
    blk, tail_done = 0, tail8 == 0
    while True:
        start, cnt, halves, glob, tail = blk, 0, [], [], False
        pending = None

        def record(b):
            nonlocal cnt
            for h in (2 * b, 2 * b + 1):
                if h in surv:
                    halves.append(h)
                    cnt += 1

        smem_end = min(nblocks, smem_blocks)
        while blk < smem_end and cnt <= cap - 4:
            if pending is not None:
                record(pending)
            pending = blk
            blk += 1
        while smem_end <= blk < nblocks and cnt <= cap - 4:
            if pending is not None:
                record(pending)
            glob.append(blk)
            pending = blk
            blk += 1
        if pending is not None:
            record(pending)
        if blk == nblocks and not tail_done and cnt <= cap - 1:
            tail, tail_done = True, True
            if 2 * nblocks in surv:
                halves.append(2 * nblocks)
                cnt += 1
        assert cnt <= cap, "the list overran"  # the walk's invariant
        rounds.append(Round(start, blk, tuple(halves), tail, tuple(glob)))
        if blk == nblocks and tail_done:
            return rounds


def round_of_half(rounds: List[Round], half: int) -> int:
    """The round in which half block `half` is resolved."""
    return next(k for k, r in enumerate(rounds) if half in r.halves)
