"""The CPU model of the shared-memory-table kernel's cull walk (tests/cull_walk_model.py) on cases worked out by hand,
and the source constants it and tests/test_gpu_large_scenes.py are built on."""
import pytest

import cull_walk_model as M


def test_source_constants_parse():
    c = M.source_constants()
    # the values the hand-worked cases below assume; a change in the source has to revisit them
    assert (c["kListCap"], c["kBlockPairs"], c["RTCLJ_THREADS_SMEM"]) == (16, 16, 512)
    assert c["block_bytes"] == 2 * c["kBlockPairs"] * 16  # a block: 16 pairs of {cx, cy, cz, Ws} x 2 fp32
    assert c["const_table_max"] == 512 and c["max_spheres"] == 65532
    # 65 532 spheres end in half block 4095: the largest index a 16-bit list entry holds
    assert (c["max_spheres"] - 1) // 16 == 4095


def test_shared_memory_blocks_formula():
    # 16 x 512 x 4 B of lists, a 16 B barrier and 512 x 24 B of unit sums: 45 072 B
    assert M.smem_table_blocks(45072) == 0 and M.smem_table_blocks(45072 + 511) == 0
    assert M.smem_table_blocks(45072 + 512) == 1
    assert M.smem_table_blocks(227 * 1024) == 365  # the B200's opt-in: 11 680 spheres
    assert M.smem_table_blocks(0) == 0


def test_layout():
    assert M.layout(0) == (0, 0)
    assert M.layout(1) == (0, 1) and M.layout(16) == (0, 1) and M.layout(17) == (1, 0)
    assert M.layout(32 * 365 - 16) == (364, 1) and M.layout(32 * 365) == (365, 0)
    assert M.layout(32 * 365 + 1) == (365, 1) and M.layout(32 * 365 + 17) == (366, 0)
    assert M.layout(65520) == (2047, 1) and M.layout(65532) == (2048, 0)
    assert M.tail_is_global(32 * 365 + 1, 365) and not M.tail_is_global(32 * 365 - 16, 365)


def test_survivors_in_every_half_block_give_eight_blocks_per_round():
    rounds = M.walk(32 * 24, 100, range(48))
    assert [(r.start, r.stop) for r in rounds] == [(0, 8), (8, 16), (16, 24)]
    assert all(r.halves == tuple(range(2 * r.start, 2 * r.stop)) for r in rounds)
    assert not any(r.global_blocks for r in rounds)


def test_no_survivors_is_one_round():
    rounds = M.walk(32 * 24 + 5, 100, [])
    assert rounds == [M.Round(0, 24, (), True, ())]
    assert M.walk(0, 100, []) == [M.Round(0, 0, (), False, ())]


def test_one_entry_per_block_gives_fourteen_blocks_per_round():
    # block b is culled while the list holds <= 12 entries: b - 1 entries before block b, so blocks 0 .. 13, and
    # the pending block 13 makes 14
    rounds = M.walk(32 * 30, 100, range(0, 60, 2))
    assert [(r.start, r.stop, len(r.halves)) for r in rounds] == [(0, 14, 14), (14, 28, 14), (28, 30, 2)]


def test_a_full_list_leaves_the_tail_for_a_round_of_its_own():
    n = 32 * 8 + 16  # 8 blocks and the tail (half block 16)
    rounds = M.walk(n, 100, range(17))
    assert rounds == [M.Round(0, 8, tuple(range(16)), False, ()), M.Round(8, 8, (16,), True, ())]
    # one entry fewer: the tail fits into the first round
    rounds = M.walk(n, 100, range(1, 17))
    assert rounds == [M.Round(0, 8, tuple(range(1, 17)), True, ())]
    # a tail without survivors still takes its round when the list is full
    assert M.walk(n, 100, range(16))[1] == M.Round(8, 8, (), True, ())


def test_a_round_that_ends_at_the_shared_memory_boundary():
    # S = 10 of 12 blocks; survivors in blocks 2 .. 9 fill the list exactly at block 10
    rounds = M.walk(32 * 12, 10, range(4, 20))
    assert rounds[0] == M.Round(0, 10, tuple(range(4, 20)), False, ())
    assert rounds[1] == M.Round(10, 12, (), False, (10, 11))
    # without the flush, one round crosses from shared to global memory
    assert M.walk(32 * 12, 10, [3, 21]) == [M.Round(0, 12, (3, 21), False, (10, 11))]


def test_global_tail():
    n = 32 * 10 + 3  # 10 blocks, S = 10: no global block, a global tail
    assert M.tail_is_global(n, 10)
    rounds = M.walk(n, 10, range(21))
    assert [(r.start, r.stop, r.tail, r.global_blocks) for r in rounds] == [(0, 8, False, ()), (8, 10, True, ())]
    assert rounds[1].halves == (16, 17, 18, 19, 20)


def test_round_of_half_and_range_check():
    rounds = M.walk(32 * 24, 100, range(48))
    assert M.round_of_half(rounds, 0) == 0 and M.round_of_half(rounds, 47) == 2
    with pytest.raises(AssertionError):
        M.walk(32, 100, [2])
