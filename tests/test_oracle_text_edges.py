"""The oracle's text-side predicates -- no N in the window, inside one record, the valid seed windows that place the text
blocks -- on a text whose N runs and records sit at every offset mod 64, against a brute force that tests every window.
The reference's goldens never had such a text, so the brute force is the only independent check here."""
import numpy as np
import pytest

from oracle import oracle_py as O
import util
from util import brute_match_all, canon_hits, edge_case


def small_case(seedl):
    return edge_case(11 + seedl, seedl=seedl, lengths=(60, 100, 120, 0) if seedl < 60 else (100, 120, 0))


def test_edge_case_covers_every_offset():
    """The generator does what its tests rely on: N runs start and end at every residue mod 64, records start at every
    residue, records of every special length and empty ones in a row exist, and every boundary kind has planted reads on
    both strands that must match and that must not."""
    for full in (False, True):
        c = edge_case(3, full=full)
        st = c.text.record_starts.astype(np.int64)
        ends = c.runs[:, 0] + c.runs[:, 1] - 1
        assert set((c.runs[:, 0] % 64).tolist()) == set(range(64)) and set((ends % 64).tolist()) == set(range(64))
        assert set((st[:-1] % 64).tolist()) == set(range(64))
        assert st[0] == 0 and st[-2] == st[-1] == c.text.n and c.text.symbols[0] == 4 and c.text.symbols[-1] == 4
        lens = np.diff(st)
        seedl, L = c.seedl, 100
        assert {0, 1, seedl - 1, seedl, seedl + 1, L - 1, L, L + 1, 2 * L + seedl - 1, 2 * L + seedl, 2 * L + seedl + 1} <= set(lens.tolist())
        empty_runs = np.diff(np.concatenate([[0], (lens == 0).astype(np.int8), [0]]))
        assert (np.nonzero(empty_runs == -1)[0] - np.nonzero(empty_runs == 1)[0]).max() >= 3
        for k in range(len(util.EDGE_KINDS)):
            sel = c.plan[c.plan["kind"] == k]
            for inv in (0, 1):
                for expect in (False, True):
                    assert ((sel["inv"] == inv) & (sel["expect"] == expect)).sum() > 0, (full, util.EDGE_KINDS[k], inv, expect)
        if full:
            assert len(c.text.records) >= 3000 and 1_000_000 <= c.text.n <= 2_500_000
            single = c.runs[c.runs[:, 1] == 1, 0]
            assert set((single % 64).tolist()) == set(range(64))
            for ln in util.EDGE_NRUN_LENS:
                assert set((c.runs[c.runs[:, 1] == ln, 0] % 64).tolist()) == set(range(64)), ln


@pytest.mark.parametrize("seedl,s", [(32, 2), (20, 1), (64, 2)])
def test_oracle_edge_text_vs_brute_force(seedl, s):
    c = small_case(seedl)
    e = 5
    ll = O.build_ll()
    got = canon_hits(O.match_all(c.text, c.reads, seedl=seedl, seedkmax=s, totalkmax=e, scores=True, ll=ll))
    want = brute_match_all(c.text, c.reads, seedl, s, e, ll)
    assert got.shape == want.shape and np.array_equal(got, want)
    # every planted read matches exactly where its window is valid, at its own position and strand, and nowhere else
    hit = {(int(r), int(p), int(inv)) for r, p, inv in got[:, [0, 2, 5]]}
    matched = set(got[:, 0].tolist())
    for x in c.plan:
        if x["expect"]:
            assert (int(x["read"]), int(x["p"]), int(x["inv"])) in hit, x
        else:
            assert int(x["read"]) not in matched, x
    # the codes stored under N change nothing
    got_r = canon_hits(O.match_all(c.text_random, c.reads, seedl=seedl, seedkmax=s, totalkmax=e, scores=True, ll=ll))
    assert np.array_equal(got_r, got)


def test_oracle_window_count_vs_brute_force():
    """oracle_count_windows (a window is emitted iff its seedl bases hold no N) on prefixes of the edge text that end at
    every residue mod 64 and on texts shorter than the seed."""
    c = edge_case(21)
    sym = c.text.symbols
    lib = O.lib()
    for seedl in range(4, 68, 4):
        for n in [0, 1, seedl - 1, seedl, 63, 64, 65] + [20_000 + 37 * k for k in range(8)] + [sym.size]:
            _, nmask = util.synth.pack_text(sym[:n])
            nmask = np.concatenate([nmask, np.zeros(2, np.uint64)])
            want = util.valid_window_starts(sym[:n], seedl).size
            assert lib.oracle_count_windows(nmask.ctypes.data, n, seedl) == want, (seedl, n)
