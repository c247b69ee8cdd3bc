"""The EP sweep's delayed flush in pairs of blocks (gp_algos_b200/csrc/gpk_ep.cu: ep_sweep_sites / ep_pair_flush) as a
bookkeeping model: every tile of Sigma0 that a later step reads must have received the update of
every earlier block EXACTLY once by then -- whatever the number of blocks or padded size.  The piece list below restates
ep_pair_flush (same order, same bounds; fold=False); the model executes it in program order (it checks coverage, not the
stream dependencies) and counts, per 64 x 64 tile, which blocks' updates have been applied.

What reads what (EpParameterEstimator.scala:44-61 in delayed-update form): apply(b) reads the CROSS of block b -- tile row b left
of the diagonal and tile column b below it -- as of block b-1.  fold=True models the folded schedule, which was measured no
faster and removed from the library (DESIGN.md 7a): there the site kernel of block b read tile (b, b-1) as of block b-2 and
that tile's block b-1 update arrived late, behind it."""
import itertools

import numpy as np
import pytest

EB = 64


def pieces_after_apply(b, nblk, N, late_tile):
    """(row_lo, rows, col_lo, cols, lower_only, blocks) of every flush piece ep_pair_flush issues behind apply(b)."""
    c0, c1 = (b + 1) * EB, (b + 2) * EB
    out = []
    if b % 2 == 0:
        out.append((c0, EB, 0, (c0 - EB) if late_tile else c1, False, (b,)))                 # tile row b+1
        out.append((c1, N - c1, c0, EB, False, (b,)))                                        # tile column b+1
    else:
        cb, r3 = b * EB, min(c1 + EB, N)
        pair = (b - 1, b)
        out.append((c0, r3 - c0, 0, cb, False, pair))                                        # rows b+1, b+2 x columns < b
        out.append(((c1, r3 - c1) if late_tile else (c0, r3 - c0)) + (cb, EB, False, (b,)))  #              x column b
        out.append((c0, r3 - c0, c0, r3 - c0, False, pair))                                  #              x columns b+1, b+2
        out.append((r3, N - r3, c0, r3 - c0, False, pair))                                   # rows >= b+3 x columns b+1, b+2
        if b + 3 < nblk:
            out.append((r3, N - r3, 0, cb, False, pair))                                     # rows >= b+3 x columns < b
            out.append((r3, N - r3, cb, EB, False, (b,)))                                    #              x column b
            out.append((r3, N - r3, r3, N - r3, True, pair))                                 #              trailing triangle
    return [p for p in out if p[1] > 0 and p[3] > 0]


@pytest.mark.parametrize("n,fold", list(itertools.product([1, 64, 65, 128, 130, 200, 300, 448, 700, 1000, 4096], [False, True])))
def test_every_tile_gets_every_earlier_block_exactly_once_before_it_is_read(n, fold):
    nblk = (n + EB - 1) // EB
    N = ((n + 127) // 128) * 128
    nt = N // EB
    applied = np.zeros((nt, nt, nblk), dtype=int)        # applied[tile row, tile column, block]

    def flush(piece):
        row_lo, rows, col_lo, cols, lower_only, blocks = piece
        assert row_lo % EB == 0 and rows % EB == 0 and col_lo % EB == 0 and cols % EB == 0
        assert 0 <= row_lo and row_lo + rows <= N and 0 <= col_lo and col_lo + cols <= N
        for r in range(row_lo // EB, (row_lo + rows) // EB):
            for c in range(col_lo // EB, (col_lo + cols) // EB):
                if lower_only and c > r:
                    continue
                for k in blocks:
                    applied[r, c, k] += 1

    def current(r, c, upto):          # tile (r, c) holds exactly the updates of blocks 0 .. upto-1
        return np.array_equal(applied[r, c, :upto], np.ones(upto, dtype=int)) and not applied[r, c, upto:].any()

    for b in range(nblk):
        if fold and b > 0:
            assert current(b, b - 1, b - 1)              # the site kernel's prologue: tile (b, b-1) as of block b-2
            flush((b * EB, EB, (b - 1) * EB, EB, False, (b - 1,)))      # ep_late_tile, in front of apply(b)
        for c in range(b):                               # apply(b): tile row b left of the diagonal ...
            assert current(b, c, b), (n, fold, b, c)
        for r in range(b + 1, nblk):                     # ... and tile column b below it (rows of sites still to come)
            assert current(r, b, b), (n, fold, b, r)
        if b + 1 < nblk:
            for piece in pieces_after_apply(b, nblk, N, fold):
                flush(piece)
    # nothing is ever applied twice to a tile that is read, and no update of a block reaches the rows of that block or above
    for r, c in itertools.product(range(nblk), range(nblk)):
        if c < r:
            assert applied[r, c].max() <= 1
            assert not applied[r, c, r:].any()
