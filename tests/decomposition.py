"""How each reducing or grid-stride kernel splits the samples among its thread blocks, restated from its launcher.

Every function takes the sample count N and the device's SM count and returns a `Split`: per block, how many tiles,
chunks or passes it makes, whether some block's last one is partial, and the first sample of a block's second one.
The large-N GPU tests (test_gpu_large_n.py) pick N with these so that every block loops, whatever the SM count, and
test_decomposition_regimes.py pins the regimes for 148 SMs.  If a launcher changes its grid, change it here too.
"""
from dataclasses import dataclass

import numpy as np

MAX_GRID = 160 * 8      # ttm_api.cu:33, ObjArgs::max_grid of every objective launch
ROW = 128               # samples per row of the general, separable and inverse kernels (T_OBJ, T_SEP, T_INV)


@dataclass(frozen=True)
class Split:
    grid: int
    unit: int            # samples in one full tile, chunk or pass of a block
    loops_min: int       # fewest tiles / chunks / passes any block makes
    loops_max: int
    partial: bool        # the last tile / chunk / pass of some block holds fewer than `unit` samples
    second: int          # first sample of block 0's second tile / chunk / pass (-1: it has none)


def _contiguous(lo, hi, unit, grid):
    """Blocks own the contiguous sample ranges [lo_b, hi_b) and walk them `unit` samples at a time."""
    lo, hi = np.asarray(lo, dtype=np.int64), np.asarray(hi, dtype=np.int64)
    n = hi - lo
    loops = -(-n // unit)
    return Split(grid, unit, int(loops.min()), int(loops.max()), bool(np.any(n % unit != 0)),
                 int(lo[0] + unit) if loops[0] > 1 else -1)


def _strided(N, unit, grid):
    """Block b handles units b, b + grid, b + 2 grid, ... of `unit` consecutive samples."""
    units = -(-N // unit)
    return Split(grid, unit, units // grid, -(-units // grid), N % unit != 0, grid * unit if units > grid else -1)


def tile(N, sm_count, blocks_per_sm=0):
    """K-objgrad tile kernel: ttm_objgrad_tile.cu:544-549 (grid), :333-338 (block ranges in 32-sample units, tiles
    of TB = 256 samples).  The context's blocks per SM is clamped to 2."""
    tiles = -(-N // 256)
    bps = min(blocks_per_sm, 2) if blocks_per_sm > 0 else 2
    grid = max(1, min(sm_count * bps, tiles, MAX_GRID))
    units = -(-N // 32)
    b = np.arange(grid, dtype=np.int64)
    lo = units * b // grid * 32
    hi = np.minimum(units * (b + 1) // grid * 32, N)
    return _contiguous(lo, hi, 256, grid)


# ttm_objgrad_impl.cuh:563-571: resident blocks per SM of Cfg1..Cfg6
GENERAL_BPS = {1: 4, 2: 3, 3: 3, 4: 3, 5: 2, 6: 4}


def general(N, sm_count, cfg, gram=False, blocks_per_sm=0):
    """K-objgrad general kernel, instantiation Cfg<cfg>: ttm_objgrad_impl.cuh:574-579 (grid; only Cfg6 honours the
    context's blocks per SM, ttm_objgrad.cu:19-20), :172-173 (block row ranges, rows of 128 samples) and :183
    (chunks of ch_rows rows: 16 in the two-sweep form, 8 in Gram mode, ttm_objgrad.cu:18)."""
    rows = -(-N // ROW)
    bps = blocks_per_sm if (cfg == 6 and blocks_per_sm > 0) else GENERAL_BPS[cfg]
    grid = max(1, min(sm_count * bps, rows, MAX_GRID))
    b = np.arange(grid, dtype=np.int64)
    lo, hi = rows * b // grid * ROW, np.minimum(rows * (b + 1) // grid * ROW, N)
    return _contiguous(lo, hi, (8 if gram else 16) * ROW, grid)


def gram_chunks(N):
    """K-gram: ttm_gram.cu:119-133, the host loop over chunks of 2^18 samples (transport_map._gram sizes the scratch
    for a full chunk); every chunk after the first accumulates into the split partials."""
    return _contiguous([0], [N], 1 << 18, 1)


def sep_eval(N, sm_count):
    """K-sep-eval, inverse table and bisection kernels (one launch per component over all samples): ttm_sep.cu:201-203,
    ttm_inverse.cu:235-237 (inv_launch, both inverse kernels: grid <= 16 SM blocks), grid-stride over groups of
    R_OBJ = 4 rows (ttm_sep.cu:31, ttm_inverse.cu:108, :136)."""
    rows = -(-N // ROW)
    grid = max(1, min(-(-rows // 4), sm_count * 16))
    return _strided(N, 4 * ROW, grid)


def sepobj(N, sm_count, nact=1):
    """K-sepobj: ttm_sep.cu:218-221 (single, grid <= 8 SM), :237-241 (batched: 8 SM / nact blocks per component),
    grid-stride over rows of T_SEP = 128 samples (ttm_sep.cu:103)."""
    share = sm_count * 8 if nact == 1 else sm_count * 8 // nact
    grid = max(1, min(-(-N // ROW), share, MAX_GRID))
    return _strided(N, ROW, grid)


def colstats(N, D, sm_count):
    """K-std column statistics, one Split per column block of 256 columns: ttm_prep.cu:253-258 (grid <= 4 SM,
    lanes = 256 / Dc rows in flight per block), grid-stride over groups of `lanes` rows (ttm_prep.cu:24).  With one
    lane a pass is one sample, so no pass is partial; what stays ragged is the last sweep over the grid."""
    out = []
    for c0 in range(0, D, 256):
        lanes = 256 // min(256, D - c0)
        out.append(_strided(N, lanes, max(1, min(-(-N // lanes), sm_count * 4))))
    return out


def ragged_sweep(s, N):
    """Some blocks of a grid-stride split make one pass fewer than others."""
    return -(-N // s.unit) % s.grid != 0


def ragged_n(at_least):
    """The first N >= at_least whose last row of 128 samples and last 32-sample unit are partial: N = 2048 t + 1061
    (1061 = 8 * 128 + 37)."""
    t = max(0, -(-(at_least - 1061) // 2048))
    return 2048 * t + 1061


def n_for_loops(split_fn, loops, lo=1 << 12, hi=1 << 26):
    """Smallest ragged N (ragged_n) at which every block of split_fn(N) makes at least `loops` tiles/chunks/passes."""
    while lo < hi:
        mid = (lo + hi) // 2
        if split_fn(ragged_n(mid)).loops_min >= loops:
            hi = mid
        else:
            lo = mid + 1
    return ragged_n(lo)


STD_DS = (3, 129, 257)
SEP_FIT_D = 3           # components of the lockstep separable fit (up to 3 K-sepobj launches batched together)


def sizes(sm_count):
    """The sample counts of test_gpu_large_n.py: every block loops at least 3 times in every form a test runs."""
    sm = sm_count
    std_split = lambda D: lambda n: min(colstats(n, D, sm), key=lambda s: s.loops_min)
    return {
        'tile': n_for_loops(lambda n: tile(n, sm), 3),
        'tile_exact': 256 * 2 * sm * 4,          # no ragged edge: 4 full tiles per block (8 at one block per SM)
        'general': {cfg: n_for_loops(lambda n, cfg=cfg: general(n, sm, cfg), 3) for cfg in range(1, 6)},
        'cfg6': n_for_loops(lambda n: general(n, sm, 6, False, 8), 3),
        'gram': n_for_loops(gram_chunks, 3),
        'sep': max(n_for_loops(lambda n: sep_eval(n, sm), 3), n_for_loops(lambda n: sepobj(n, sm), 3)),
        # at least the headline's 10^6 samples (2.5M where the ensemble stays below 3 GB): accumulation error at
        # production N is what the large-offset columns are there to show
        'std': {D: max(n_for_loops(std_split(D), 3), ragged_n(2_500_000 if D < 256 else 1_000_000)) for D in STD_DS},
    }


def regimes(sm_count):
    """(label, N, Split, grid_stride) of every kernel and form the GPU tests run, at sizes(sm_count)."""
    sm, z = sm_count, sizes(sm_count)
    out = []
    for which in ('tile', 'tile_exact'):
        for bps in (0, 1):
            out.append(('%s bps=%d' % (which, bps), z[which], tile(z[which], sm, bps), False))
    for cfg, N in z['general'].items():
        for gram in (False, True):
            out.append(('cfg%d gram=%d' % (cfg, gram), N, general(N, sm, cfg, gram), False))
    for gram, bps in [(False, b) for b in (0, 1, 2, 8)] + [(True, b) for b in (0, 1, 8)]:
        out.append(('cfg6 gram=%d bps=%d' % (gram, bps), z['cfg6'], general(z['cfg6'], sm, 6, gram, bps), False))
    out.append(('gram', z['gram'], gram_chunks(z['gram']), False))
    out.append(('sep-eval', z['sep'], sep_eval(z['sep'], sm), True))
    out.append(('sepobj', z['sep'], sepobj(z['sep'], sm), True))
    for nact in range(1, SEP_FIT_D + 1):                     # the lockstep fit's batched launches
        out.append(('sepobj batch nact=%d' % nact, z['sep'], sepobj(z['sep'], sm, nact), True))
    for D, N in z['std'].items():
        for j, s in enumerate(colstats(N, D, sm)):
            out.append(('colstats D=%d block %d' % (D, j), N, s, True))
    return out
