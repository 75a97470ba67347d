"""GPU: BASELINE.json's FULL sizes, checked through size-independent properties (the oracle is not run at these sizes).

For every configuration the inputs are generated on the device by the counter-based generators (the same formulas as
real_b200/synth.py), the hot path runs once through the C ABI, and the results are checked on the device with plain
torch integer arithmetic:

  * every reported placement re-verifies: the Hamming distance between the read strand and the text under it, counted
    directly from the unpacked text, equals the reported error count and is within the budget; the window holds no
    wildcard and lies inside one record;
  * the planted truth: a read cut from position p on strand s with k substitutions, k <= e and at most 2 of them
    inside the seed, must be reported -- matchAll lists (p, s, k); matchUnique holds err <= k, and if it holds a
    unique hit with err == k it is (p, s);
  * reads that contain a wildcard never match (Pattern.hpp / matchAllImplementation.cpp:275);
  * matchUnique: the state merged from 4 bucket shards (real_gpu_set_bucket_shard + the min/tie fold of
    real_b200.dist.unique_exchange) is the state of the single-handle run, word for word in canonical form.
"""
import numpy as np
import pytest

from real_b200 import lib as rlib
from real_b200 import matcher
from util import need_big_gpu as _need_big_gpu

pytestmark = pytest.mark.gpu

SEED = 0x5EA1


def _record_starts(n, nrec):
    from real_b200 import synth
    if nrec <= 1:
        return np.asarray([0, n], dtype=np.uint64)
    cuts = sorted(set(int(x % np.uint64(n)) for x in synth.splitmix64(np.arange(nrec - 1, dtype=np.uint64) ^ synth.stream(SEED, 3))))
    return np.asarray([0] + [c for c in cuts if c > 0] + [n], dtype=np.uint64)


def _unpack_symbols(words, nmask, n):
    from real_b200 import devsynth
    return devsynth.unpack_symbols(words, nmask, n)


class _Checker:
    def __init__(self, sym, rec, mapped, L, e, seedl=32, seedkmax=2):
        import torch
        self.t = torch
        self.sym, self.L, self.e, self.seedl, self.seedkmax = sym, L, e, seedl, seedkmax
        self.rec = torch.as_tensor(rec.astype(np.int64), device=sym.device)
        self.mapped = mapped.view(-1, L)
        self.ar = torch.arange(L, device=sym.device, dtype=torch.int64)

    def strand_reads(self, rows, strand):
        """The reads `rows` as laid over the text: '+' as they are, '-' reverse complemented."""
        t = self.t
        rd = self.mapped[rows]
        rc = rd.flip(1)
        rc = t.where(rc < 4, 3 - rc, rc)
        return t.where(strand[:, None], rc, rd)

    def distance(self, rows, pos, strand):
        """(k over the whole read, k inside the seed window, window is wildcard free and inside one record)."""
        t = self.t
        tx = self.sym[pos[:, None] + self.ar[None, :]]
        rd = self.strand_reads(rows, strand)
        diff = tx != rd
        k = diff.sum(1)
        ks_plus = diff[:, : self.seedl].sum(1)
        ks_minus = diff[:, self.L - self.seedl:].sum(1)
        ks = t.where(strand, ks_minus, ks_plus)
        clean = (tx < 4).all(1)
        r0 = t.searchsorted(self.rec, pos, right=True)
        r1 = t.searchsorted(self.rec, pos + self.L - 1, right=True)
        return k, ks, clean & (r0 == r1)


def _plan(seed, nreads, span, dev):
    from real_b200 import devsynth
    return devsynth.read_plan_device(seed, nreads, span, dev)


def _unique_fields(info):
    st = (info >> 61) & 7
    pos = info & ((1 << 35) - 1)
    err = (info >> 41) & 15
    return st, pos, err


def _check_unique(chk, info, ppos, pstrand, batch):
    import torch
    R = info.numel()
    st, pos, err = _unique_fields(info)
    stats = dict(matched=0, findable=0, planted_hit=0, nonunique=0)
    for r0 in range(0, R, batch):
        r1 = min(R, r0 + batch)
        rows = torch.arange(r0, r1, device=info.device)
        usable = (chk.mapped[rows] < 4).all(1)
        k, ks, ok = chk.distance(rows, ppos[r0:r1], pstrand[r0:r1])
        findable = usable & ok & (k <= chk.e) & (ks <= chk.seedkmax)
        s, p, er = st[r0:r1], pos[r0:r1], err[r0:r1]
        assert bool((s[~usable] == 0).all()), "a read with a wildcard matched"
        assert bool((s[findable] != 0).all()), "a planted placement was not found"
        assert bool((er[findable] <= k[findable]).all()), "a planted placement was beaten by a worse one"
        uniq = (s == 1) | (s == 2)
        at_planted = findable & uniq & (er == k)
        assert bool((p[at_planted] == ppos[r0:r1][at_planted]).all()) and bool(((s[at_planted] == 2) == pstrand[r0:r1][at_planted]).all()), \
            "a unique hit at the planted error count is not the planted placement"
        # every unique hit re-verifies
        ur = rows[uniq]
        if ur.numel():
            k2, ks2, ok2 = chk.distance(ur, p[uniq], s[uniq] == 2)
            assert bool((k2 == er[uniq]).all()) and bool((k2 <= chk.e).all()) and bool(ok2.all()) and bool((ks2 <= chk.seedkmax).all()), \
                "a reported unique hit does not re-verify"
        stats["matched"] += int((s != 0).sum()); stats["findable"] += int(findable.sum())
        stats["planted_hit"] += int(at_planted.sum()); stats["nonunique"] += int((s == 4).sum())
    return stats


def test_c3_full_size_match_unique():
    """C3: 3.1 Gbp (24 records, 0.1 % N), 50 M x 100 bp, matchUnique -e 4, one handle and 4 bucket shards."""
    _need_big_gpu(150)
    import torch
    from real_b200 import devsynth
    n, R, L, e = 3_100_000_000, 50_000_000, 100, 4
    dev = torch.device("cuda", 0)
    words, nmask = devsynth.text_device(SEED, n, n_per_million=1000)
    mapped, _, offs = devsynth.reads_device(SEED + 1, words, nmask, n, R, L, 0.01)
    rs = _record_starts(n, 24)

    def run(shard=None):
        h = rlib.Handle(seedl=32, seedkmax=2, totalkmax=e, scores=False)
        if shard is not None:
            h.set_bucket_shard(*shard)
        h.set_reads_device(mapped.data_ptr(), offs.data_ptr(), R, R * L, L)
        h.set_text_device(words.data_ptr(), nmask.data_ptr(), n, rs)
        h.match_unique()
        return h

    h = run()
    info = torch.as_tensor(h.get_unique()[0].view(np.int64), device=dev)
    h.close()

    sym = _unpack_symbols(words, nmask, n)
    chk = _Checker(sym, rs, mapped, L, e)
    ppos, pstrand = _plan(SEED + 1, R, n - L + 1, dev)
    stats = _check_unique(chk, info, ppos, pstrand, batch=1 << 20)
    assert stats["findable"] > 0.95 * R and stats["planted_hit"] > 0.9 * R and stats["matched"] >= stats["findable"]
    del sym, chk

    # the same job as 4 bucket shards, folded like real_b200.dist.unique_exchange does (MIN of the keys, SUM of the ties).
    # The shards run one after the other here (four resident handles of this size do not fit one GPU), so every shard
    # runs twice: once for its keys, once more for its ties against the minimum.
    nsh = 4
    keys = torch.empty(R, dtype=torch.int64, device=dev)
    kmin = None
    for r in range(nsh):
        hh = run((r, nsh))
        hh.unique_export_keys(keys.data_ptr())
        kmin = keys.clone() if kmin is None else torch.minimum(kmin, keys)
        hh.close()
    tsum = torch.zeros(R, dtype=torch.uint8, device=dev)
    ties = torch.empty(R, dtype=torch.uint8, device=dev)
    merged = None
    for r in range(nsh):
        hh = run((r, nsh))
        hh.unique_export_ties(kmin.data_ptr(), ties.data_ptr())
        tsum += ties
        if r == nsh - 1:
            torch.cuda.synchronize()
            hh.unique_import(kmin.data_ptr(), tsum.data_ptr())
            merged = hh.get_unique()[0]
        hh.close()
    want = matcher.canonical_unique(info.cpu().numpy().view(np.uint64))
    assert np.array_equal(matcher.canonical_unique(merged), want)


def _check_all(chk, hits, ppos, pstrand, R, batch, scores_ll=None, qual=None):
    """matchAll rows (real_gpu_hit records): every row re-verifies; every findable planted placement is listed once."""
    import torch
    dev = ppos.device
    pat = torch.as_tensor(hits["patid"].astype(np.int64), device=dev)
    pos = torch.as_tensor(hits["pos"].astype(np.int64), device=dev)
    inv = torch.as_tensor(hits["inverted"].astype(bool), device=dev)
    kk = torch.as_tensor(hits["k"].astype(np.int64), device=dev)
    H = pat.numel()
    for h0 in range(0, H, batch):
        h1 = min(H, h0 + batch)
        k2, ks2, ok2 = chk.distance(pat[h0:h1], pos[h0:h1], inv[h0:h1])
        assert bool((k2 == kk[h0:h1]).all()) and bool((k2 <= chk.e).all()) and bool(ok2.all()) and bool((ks2 <= chk.seedkmax).all()), \
            "a reported row does not re-verify"
    # rows are sorted by read; no duplicates
    key = (pat << 37) | (pos << 1) | inv.to(torch.int64)
    assert bool((pat[1:] >= pat[:-1]).all())
    assert torch.unique(key).numel() == H, "a placement is listed twice"
    # planted truth
    keyset = torch.sort(key).values
    found = 0
    findable_n = 0
    for r0 in range(0, R, batch):
        r1 = min(R, r0 + batch)
        rows = torch.arange(r0, r1, device=dev)
        usable = (chk.mapped[rows] < 4).all(1)
        k, ks, ok = chk.distance(rows, ppos[r0:r1], pstrand[r0:r1])
        findable = usable & ok & (k <= chk.e) & (ks <= chk.seedkmax)
        want = (rows << 37) | (ppos[r0:r1] << 1) | pstrand[r0:r1].to(torch.int64)
        at = torch.searchsorted(keyset, want).clamp(max=H - 1)
        present = keyset[at] == want
        assert bool(present[findable].all()), "a planted placement is missing from the list"
        assert not bool(present[~usable].any())
        found += int(present.sum()); findable_n += int(findable.sum())
    return findable_n, found


def test_c2_full_size_match_all_scores():
    """C2: 250 Mbp, 10 M x 100 bp FastQ, matchAll -e 4 with ComputeScore."""
    _need_big_gpu(60)
    import torch
    from real_b200 import devsynth
    n, R, L, e = 250_000_000, 10_000_000, 100, 4
    dev = torch.device("cuda", 0)
    words, nmask = devsynth.text_device(SEED, n)
    mapped, qual, offs = devsynth.reads_device(SEED + 1, words, None, n, R, L, 0.01, quality=True)
    rs = _record_starts(n, 1)
    ll = matcher.scoring_table()
    h = rlib.Handle(seedl=32, seedkmax=2, totalkmax=e, scores=True, ll_table=ll)
    try:
        h.set_reads_device(mapped.data_ptr(), offs.data_ptr(), R, R * L, L, d_quality=qual.data_ptr())
        h.set_text_device(words.data_ptr(), nmask.data_ptr(), n, rs)
        hits = h.match_all()
    finally:
        h.close()
    sym = _unpack_symbols(words, nmask, n)
    chk = _Checker(sym, rs, mapped, L, e)
    ppos, pstrand = _plan(SEED + 1, R, n - L + 1, dev)
    findable, found = _check_all(chk, hits, ppos, pstrand, R, batch=1 << 20)
    assert findable > 0.97 * R and found >= findable
    # ComputeScore (ComputeScore.hpp:50-190): 1.0 + sum of LL[ref][read][q] over the read; bit-exactness is pinned against
    # the oracle at small sizes, here every row is recomputed in fp64 with torch's own summation order
    llt = torch.as_tensor(np.asarray(ll, dtype=np.float64).reshape(4, 4, -1), device=dev)
    sel = torch.arange(0, len(hits), 7, device=dev)[: 1 << 20]
    pat = torch.as_tensor(hits["patid"].astype(np.int64), device=dev)[sel]
    pos = torch.as_tensor(hits["pos"].astype(np.int64), device=dev)[sel]
    inv = torch.as_tensor(hits["inverted"].astype(bool), device=dev)[sel]
    sc = torch.as_tensor(hits["score"].astype(np.float64), device=dev)[sel]
    tx = sym[pos[:, None] + chk.ar[None, :]].to(torch.int64)
    rd = chk.strand_reads(pat, inv).to(torch.int64)
    q = qual.view(-1, L)[pat].to(torch.int64)
    q = torch.where(inv[:, None], q.flip(1), q)
    want = 1.0 + llt[tx, rd, q].sum(1)
    assert bool(((sc - want).abs() <= 1e-4 * want.abs().clamp(min=1.0)).all())


def test_c5_full_size_match_all_long_reads():
    """C5: 3.1 Gbp (24 records, 0.1 % N), 20 M x 250 bp, matchAll -e 8."""
    _need_big_gpu(150)
    import torch
    from real_b200 import devsynth
    n, R, L, e = 3_100_000_000, 20_000_000, 250, 8
    dev = torch.device("cuda", 0)
    words, nmask = devsynth.text_device(SEED, n, n_per_million=1000)
    mapped, _, offs = devsynth.reads_device(SEED + 1, words, nmask, n, R, L, 0.01)
    rs = _record_starts(n, 24)
    h = rlib.Handle(seedl=32, seedkmax=2, totalkmax=e, scores=False)
    try:
        h.set_reads_device(mapped.data_ptr(), offs.data_ptr(), R, R * L, L)
        h.set_text_device(words.data_ptr(), nmask.data_ptr(), n, rs)
        hits = h.match_all()
    finally:
        h.close()
    sym = _unpack_symbols(words, nmask, n)
    chk = _Checker(sym, rs, mapped, L, e)
    ppos, pstrand = _plan(SEED + 1, R, n - L + 1, dev)
    findable, found = _check_all(chk, hits, ppos, pstrand, R, batch=1 << 19)
    assert findable > 0.9 * R and found >= findable


def test_c4_full_size_gapped_pass():
    """C4: 250 Mbp, 5 M x 150 bp FastQ, matchUnique with scores then the gapped extension pass (matchGaps).  30 % of
    the reads carry one planted deletion of 1..3 bases behind the seed.  Properties: reads matched by the Hamming pass
    are left alone by the gapped pass; a GapInfo entry implies the gapped state and a gap of at most 3; the seed position
    of a gapped read re-verifies (seed errors <= 2); of the '+' strand reads with a planted deletion and an
    error-free seed, practically all are rescued at the planted position; a second run reproduces every word."""
    _need_big_gpu(60)
    import torch
    from real_b200 import devsynth
    n, R, L, e = 250_000_000, 5_000_000, 150, 3
    dev = torch.device("cuda", 0)
    words, nmask = devsynth.text_device(SEED, n)
    mapped, qual, offs = devsynth.reads_device(SEED + 1, words, None, n, R, L, 0.01, quality=True)
    rs = _record_starts(n, 1)
    sym = _unpack_symbols(words, nmask, n)
    ppos, pstrand = _plan(SEED + 1, R, n - L + 1, dev)

    # plant the deletions: read[off+g:] moves up, the tail is refilled from the text behind the window
    planted = devsynth.plant_deletions(mapped, sym, ppos, pstrand, n, L)
    m2 = mapped.view(R, L)

    def run():
        h = rlib.Handle(seedl=32, seedkmax=2, totalkmax=e, scores=True, ll_table=matcher.scoring_table())
        try:
            h.set_reads_device(mapped.data_ptr(), offs.data_ptr(), R, R * L, L, d_quality=qual.data_ptr())
            h.set_text_device(words.data_ptr(), nmask.data_ptr(), n, rs)
            h.match_unique()
            before = h.get_unique()[0].copy()
            h.match_gaps(0)
            after, sc = h.get_unique()
            return before, after.copy(), sc.copy(), h.get_gaps().copy()
        finally:
            h.close()

    before, after, sc, gaps = run()
    st0, st1 = matcher.umi_state(before), matcher.umi_state(after)
    keep = (st0 != 0) & (st0 != 3)
    assert np.array_equal(before[keep], after[keep])                     # the gapped pass only touches unmatched reads
    gapped = st1 == 3
    present = gaps["present"] != 0
    assert gapped.sum() > 0 and gapped[present].all()                    # (a second equally good placement erases the GapInfo but keeps the state)
    assert present.sum() > 0.9 * gapped.sum() and (gaps["mingap"][present] <= 3).all()
    # the seed of a gapped hit re-verifies ('+' strand only: match.hpp:477-499)
    gr = torch.as_tensor(np.nonzero(gapped)[0], device=dev)
    gp = torch.as_tensor(matcher.umi_pos(after)[gapped], device=dev)
    tx = sym[gp[:, None] + torch.arange(32, device=dev)[None, :]]
    ks = (tx != m2[gr][:, :32]).sum(1)
    assert bool((ks <= 2).all())
    # planted deletions with a clean seed are rescued where they were planted
    pl = planted.cpu().numpy()
    seed_clean = ((sym[ppos[:, None] + torch.arange(32, device=dev)[None, :]] != m2[:, :32]).sum(1) == 0).cpu().numpy()
    cand = pl & seed_clean & (st0 == 0)
    rescued = cand & gapped & (matcher.umi_pos(after) == ppos.cpu().numpy())
    assert cand.sum() > 0.08 * R and rescued.sum() > 0.99 * cand.sum(), (int(cand.sum()), int(rescued.sum()))
    b2, a2, sc2, gaps2 = run()
    assert np.array_equal(after, a2) and np.array_equal(sc.view(np.uint32), sc2.view(np.uint32)) and np.array_equal(gaps, gaps2)
