"""The sample counts of test_gpu_large_n.py put every kernel in the regime it is there to check, on one B200 (148 SMs):
each block makes at least three tiles, chunks or passes, some block's last one is partial, and the last row of 128
samples is partial.  The exception is the tile kernel's exact size, where nothing is ragged."""
import pytest

import decomposition as dec

SM = 148


@pytest.mark.parametrize('label,N,split,strided', dec.regimes(SM), ids=lambda v: v if isinstance(v, str) else '')
def test_every_block_loops_with_a_ragged_end(label, N, split, strided):
    assert split.loops_min >= 3, (label, N, split)
    if label.startswith('tile_exact'):
        assert not split.partial and N % 128 == 0 and split.loops_min == split.loops_max, (label, N, split)
        return
    assert N % 128 != 0, (label, N)
    if strided and split.unit == 1:          # one-sample passes: the raggedness is in the last sweep over the grid
        assert dec.ragged_sweep(split, N), (label, N, split)
    else:
        assert split.partial, (label, N, split)
    assert split.second > 0, (label, N, split)


def test_helper_restates_known_launches():
    """Figures worked out by hand from the launchers for 148 SMs."""
    s = dec.tile(1_000_000, SM)
    assert (s.grid, s.loops_min, s.loops_max, s.partial) == (296, 14, 14, True)
    assert dec.tile(75_776, SM).loops_max == 1 and dec.tile(75_777, SM).loops_max == 2
    assert dec.tile(10 ** 6, SM, 8).grid == 296                      # the context's setting is clamped to 2
    assert dec.general(10 ** 6, SM, 6, blocks_per_sm=1).grid == 148
    assert dec.general(10 ** 6, SM, 1, blocks_per_sm=1).grid == 592  # only Cfg6 honours it
    assert dec.general(1_212_416, SM, 6).loops_max == 1 and dec.general(1_212_417, SM, 6).loops_max == 2
    assert dec.general(606_208, SM, 6, gram=True).loops_max == 1
    assert dec.gram_chunks(1 << 18).loops_max == 1 and dec.gram_chunks((1 << 18) + 1).loops_max == 2
    assert dec.sep_eval(1_212_416, SM).loops_max == 1 and dec.sep_eval(1_212_417, SM).loops_max == 2
    assert dec.sepobj(151_552, SM).loops_max == 1 and dec.sepobj(151_553, SM).loops_max == 2
    assert dec.sepobj(151_553, SM, nact=4).grid == 296
    assert [s.unit for s in dec.colstats(1000, 257, SM)] == [1, 256]
    assert [s.unit for s in dec.colstats(1000, 3, SM)] == [85]
