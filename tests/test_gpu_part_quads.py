"""GPU: the dense partition (k_part_scatter in scan.cuh) rebuilds every record from one 16-byte quad of its tile -- the 64
bases around a 16-base half-word.  N runs and record ends on the first and last half-word of a tile (quads 0 and 511 read
the halo words), with reads planted on every offset of those half-words, formed by the scan and ahead of the match call,
against the oracle: match.hpp:335-416 through AllMatcher::match."""
import numpy as np
import pytest

from oracle import oracle_py as O
from real_b200 import lib as rlib
from real_b200 import synth
from util import canon_hits

pytestmark = pytest.mark.gpu

TILE = 8192
HALF = 16
KW = dict(seedl=32, seedkmax=2, totalkmax=4, scores=False)


def _handle():
    return rlib.Handle(seedl=KW["seedl"], seedkmax=KW["seedkmax"], totalkmax=KW["totalkmax"], scores=False,
                       filter_mult=O.filter_mult(KW["totalkmax"]))


def _same(got, ref, least):
    a, b = canon_hits(got, with_score=False), canon_hits(ref, with_score=False)
    assert len(b) > least
    assert a.shape == b.shape and np.array_equal(a, b)


def _half_word_text(seed):
    """Four tiles and a bit: N runs exactly on the first half-word of tile 1 and the last of tile 2, single Ns on the last
    base of a first half-word and the first base of a last one, records that start on the first and last half-word of
    tiles; reads planted at every offset of the first and last half-words of every tile."""
    n = 4 * TILE + 100
    sym = synth.make_text(seed, n).symbols.copy()
    sym[TILE:TILE + HALF] = 4
    sym[3 * TILE - HALF:3 * TILE] = 4
    sym[2 * TILE + HALF - 1] = 4
    sym[4 * TILE - HALF] = 4
    starts = [0, TILE + HALF, 2 * TILE, 3 * TILE - HALF, 4 * TILE - 1]
    text = synth.Text(sym, [(" rec_%d" % s, s) for s in starts])
    L = 60
    seqs = []
    for t in range(4):
        for p in list(range(t * TILE - L, t * TILE + 2 * HALF)) + list(range((t + 1) * TILE - 2 * HALF - L, (t + 1) * TILE - HALF + 1)):
            if 0 <= p and p + L <= n:
                s = sym[p:p + L].copy()
                s[L // 2] = (s[L // 2] + 1) & 3 if s[L // 2] < 4 else s[L // 2]        # one substitution behind the seeds
                seqs.append(s)
    planted = synth.reads_from_list(seqs)
    reads = synth.concat_reads([planted, synth.make_reads(text, seed + 1, 2000, L, 0.01, fastq=False)])
    return text, reads


@pytest.mark.parametrize("prepared", [False, True])
def test_half_word_tile_edges(prepared):
    text, reads = _half_word_text(1201)
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
    _same(got, ref, 1000)

