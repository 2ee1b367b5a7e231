"""CPU: the tile sequence of the matrix passes (csrc/stream_pass.cuh, TileWalk) through the host-only hook
bioen_b200_selftest_tilewalk -- the code the kernel runs, compiled for the host.  For both passes in the contiguous
order and the column pass in the interleaved order: every tile is visited exactly once, a CTA accumulates over one run
at a time, and the (run, slot) pairs it writes are exactly the ones the readers of the partial sums will add up
(pass_num_slots).  The row pass has no interleaved order: the hook refuses it.  No GPU involved."""
import ctypes as C

import numpy as np
import pytest

from bioen_b200 import _lib

ROW, COL = 0, 1
SMS = 148


def geometry(M, N, sms=SMS):
    """As Context's constructor does (csrc/context.cuh)."""
    nRT, nCB = (M + 31) // 32, (N + 127) // 128
    T = nRT * nCB
    ncta = min(T, sms)
    chunk = (T + ncta - 1) // ncta
    grid = (T + chunk - 1) // chunk
    return nRT, nCB, T, chunk, grid


def walk(lib, mode, nRT, nCB, grid, chunk, interleave, cta):
    cap = nRT * nCB // max(grid, 1) + nRT + nCB + 8
    rt = (C.c_int * cap)()
    cb = (C.c_int * cap)()
    slot = (C.c_longlong * cap)()
    closes = (C.c_int * cap)()
    n = lib.bioen_b200_selftest_tilewalk(mode, nRT, nCB, grid, chunk, interleave, cta, cap, rt, cb, slot, closes)
    assert n <= cap
    return [(rt[i], cb[i], slot[i], closes[i]) for i in range(n)]


@pytest.mark.parametrize("M,N", [(1, 1), (7, 33), (37, 5001), (100, 20000), (300, 3003), (1000, 100000), (1000, 777),
                                 (500, 100000), (5000, 40000), (28, 50001), (33, 80000), (100, 200000),
                                 (1000, 1000000)])
@pytest.mark.parametrize("interleave", [0, 1])
def test_every_tile_once_and_slots_match_the_readers(M, N, interleave):
    lib = _lib.load()
    nRT, nCB, T, chunk, grid = geometry(M, N)
    if interleave and nCB < 4 * grid:
        pytest.skip("the interleaved order is only selected when nCB >= 4 * grid")
    for mode in (ROW, COL):
        if interleave and mode == ROW:
            assert lib.bioen_b200_selftest_tilewalk(mode, nRT, nCB, grid, chunk, 1, 0, 0, None, None, None, None) == -1
            continue
        L = nCB if mode == ROW else nRT
        nruns = nRT if mode == ROW else nCB
        reader_chunk = nRT if interleave else chunk
        seen = np.zeros((nRT, nCB), dtype=np.int32)
        written = {}
        for cta in range(grid):
            seq = walk(lib, mode, nRT, nCB, grid, chunk, interleave, cta)
            current = None
            for (rt, cb, slot, closes) in seq:
                assert 0 <= rt < nRT and 0 <= cb < nCB
                seen[rt, cb] += 1
                run = rt if mode == ROW else cb
                assert current in (None, run), "a CTA accumulates over one run at a time"
                current = run
                if closes:
                    assert (run, slot) not in written, "each partial-sum slot is written once"
                    written[(run, slot)] = cta
                    current = None
            assert current is None, "the last tile of a CTA closes its run"
        assert (seen == 1).all()
        for run in range(nruns):
            ns = lib.bioen_b200_selftest_num_slots(run, L, reader_chunk)
            assert sorted(s for (r, s) in written if r == run) == list(range(ns)), (mode, run, ns)
        assert len(written) == sum(lib.bioen_b200_selftest_num_slots(r, L, reader_chunk) for r in range(nruns))


def test_load_balance():
    """contiguous: +-1 tile; interleaved column pass: +-1 run."""
    lib = _lib.load()
    nRT, nCB, T, chunk, grid = geometry(1000, 1000000)
    for interleave in (0, 1):
        for mode in (ROW, COL):
            if interleave and mode == ROW:
                continue   # refused, see test_every_tile_once_and_slots_match_the_readers
            # count only: max_tiles = 0 makes the hook return the number of tiles without filling the arrays
            counts = [lib.bioen_b200_selftest_tilewalk(mode, nRT, nCB, grid, chunk, interleave, cta, 0, None, None,
                                                       None, None) for cta in range(grid)]
            assert sum(counts) == T
            slack = nRT if interleave else chunk - (T - chunk * (grid - 1))
            assert max(counts) - min(counts) <= max(1, slack), (interleave, mode, max(counts), min(counts))
