"""GPU: the dense partition works on tiles of 8192 text positions (k_part_scatter in scan.cuh) and rebuilds every record
from the text words of its tile.  Texts of one or two tiles and a position more or less, N runs across the tile edges,
scan windows that start and end inside a tile, and records formed ahead of the match call (real_gpu_prepare_scan), each
against the oracle: match.hpp:335-416 through AllMatcher::match."""
import numpy as np
import pytest

from oracle import oracle_py as O
from real_b200 import lib as rlib
from real_b200 import synth
from util import canon_hits

pytestmark = pytest.mark.gpu

TILE = 8192
KW = dict(seedl=32, seedkmax=2, totalkmax=4, scores=False)


def _text(seed, n):
    """Random text of n bases with N runs across the tile edges inside it."""
    sym = synth.make_text(seed, n).symbols.copy()
    for edge in range(TILE, n, TILE):
        sym[edge - 3:edge + 2] = 4
    sym[max(0, n - 40):n - 37] = 4
    text = synth.Text(sym, [(" random_%d" % n, 0)])
    reads = synth.make_reads(text, seed + 1, 3000, 60, 0.01, fastq=False)
    return text, reads


def _handle():
    return rlib.Handle(seedl=KW["seedl"], seedkmax=KW["seedkmax"], totalkmax=KW["totalkmax"], scores=False,
                       filter_mult=O.filter_mult(KW["totalkmax"]))


def _same(got, ref):
    a, b = canon_hits(got, with_score=False), canon_hits(ref, with_score=False)
    assert len(b) > 1000
    assert a.shape == b.shape and np.array_equal(a, b)


@pytest.mark.parametrize("prepared", [False, True])
@pytest.mark.parametrize("n", [TILE - 1, TILE, TILE + 1, 2 * TILE - 1, 2 * TILE + 1])
def test_tile_edge_lengths(n, prepared):
    text, reads = _text(700 + n, n)
    ref = O.match_all(text, reads, **KW)
    w, m = text.packed()
    h = _handle()
    try:
        if prepared:
            h.set_text(w, m, text.n, text.record_starts)
            h.prepare_scan(60)
            h.set_reads(reads.mapped, reads.offsets, None)
        else:
            h.set_reads(reads.mapped, reads.offsets, None)
            h.set_text(w, m, text.n, text.record_starts)
        got = h.match_all()
    finally:
        h.close()
    _same(got, ref)


def test_windows_inside_tiles():
    """Two text shards cut inside the fourth tile: the first shard's scan window ends inside a tile, the second's starts
    inside one (its local text begins on the mask word in front of the cut)."""
    n = 6 * TILE + 777
    text, reads = _text(901, n)
    cut = 3 * TILE + 1000
    sb = (cut // 64) * 64
    shards = [(0, cut, 0, min(n, cut + 60)), (cut, n, sb, n - sb)]
    ref = O.match_all(text, reads, **KW)
    w, m = text.packed()
    h = _handle()
    out = []
    try:
        h.set_reads(reads.mapped, reads.offsets, None)
        for ob, oe, s0, sl in shards:
            h.set_text(np.ascontiguousarray(w[s0 // 32:(s0 + sl + 31) // 32]), np.ascontiguousarray(m[s0 // 64:(s0 + sl + 63) // 64]),
                       text.n, text.record_starts, 0, shard_begin=s0, shard_len=sl, own_begin=ob, own_end=oe)
            out.append(h.match_all())
    finally:
        h.close()
    _same(np.concatenate(out), ref)
