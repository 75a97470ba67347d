"""GPU: a text longer than one scan chunk, with positions above 2^32, bit for bit against the oracle.

The oracle cannot run on a text of 4.6 Gbp, but it does not have to: matching is local.  A small text T_small (about
1.2 Mbp) is a row of "islands", each walled off by N runs longer than any read, seed window or gapped band reaches.
T_long (n = 2 * 16384 * 140001 = 4,587,552,768 bases) is random background with the same islands copied in, in the
same order, at the places where the scan of a long text can go wrong:

  * position 0 and the very end of the text;
  * every chunk boundary the scan would cut at for 2, 3 and 4 chunks (plan_scan, real_b200/csrc/real_gpu.cu).  n is
    larger than SC_MAX_CHUNK, so the scan takes at least 2 chunks; how many depends on the free device memory when it
    is planned, so the islands cover all three cuts.  With 2 chunks the cut falls on an odd multiple of 16384, off the
    32768-position tiles of k_own_list;
  * across 2^32, where the 35-bit position fields of the hit rows, the hit16 rows, the unique state words and the
    fold keys carry their top bits; the first record start after 0 lies above 2^32, so record 0 spans 2^32 too.

Every hit of T_long is then an oracle hit of T_small shifted by its island's offset (a hit on the background, which is
practically impossible for reads within a few errors, is reported as such).  The translation is monotone, so it keeps
records, frag indices, error counts, strands, scores and the visiting order that decides score ties.
"""
import functools

import numpy as np
import pytest

from oracle import oracle_py as O
from real_b200 import lib as rlib
from real_b200 import matcher, synth
from util import canon_hits, line, need_big_gpu, read_bases, unify_order_ok

pytestmark = pytest.mark.gpu

SEED = 0x10A6
TILE = 16384                       # SC_TILE_POS (csrc/scan.cuh): chunks are cut at multiples of it
MAX_CHUNK = 0xFFF00000             # SC_MAX_CHUNK (csrc/scan.cuh)
N_LONG = 2 * TILE * 140001         # > MAX_CHUNK; half of it is an odd multiple of TILE
TWO32 = 1 << 32
CUT = TWO32 + 32768                # text shards: shard 1 starts here
WALL = 2048                        # N run at either end of an island: > 2 * 150 + 64, the reach of any window or band
MARGIN = 70_016                    # island bases on either side of the point it is placed over
L1, L2 = 100, 150                  # read lengths: substitutions only / FASTQ for the gapped pass
POS_MASK = np.uint64((1 << 35) - 1)
# Free device memory the module asks for.  The most it had in use, sampled between the library calls with the handle
# alive, was about 47 GB on a B200 (180 GB, 1000 W); the scans of T_long took 2 chunks there (at 80 GB free or more
# plan_scan always takes 2: its record room, 0.6 x free / 16 B positions, is more than n / 2).  80 leaves a margin
# for what the library holds only inside a call.
FREE_GB = 80


def chunk_cuts(x_begin, x_end, nchunks):
    """Where plan_scan (real_b200/csrc/real_gpu.cu) cuts the window range [x_begin, x_end) into `nchunks` equal chunks:
    the span in whole tiles, divided evenly and rounded up to whole tiles."""
    span = -(-(x_end - x_begin) // TILE) * TILE
    chunk = max(TILE, -(-(-(-span // nchunks)) // TILE) * TILE)
    return [x_begin + i * chunk for i in range(1, nchunks) if i * chunk < x_end - x_begin]


def _r64(x, up=False):
    return (x + 63) // 64 * 64 if up else x // 64 * 64


def _island_layout():
    """(long offsets, lengths) of the islands, in text order; both multiples of 64."""
    x_end = N_LONG - 32 + 1 + 16                # last window start + 1 + 2 F of a 32-base seed (fill_scan_params)
    points = sorted(set([TWO32, CUT] + [c for k in (2, 3, 4) for c in chunk_cuts(0, x_end, k)]))
    groups = []
    for p in points:                             # points closer than an island is long share one
        if groups and p - groups[-1][-1] < 2 * MARGIN:
            groups[-1].append(p)
        else:
            groups.append([p])
    spans = [(0, 2 * MARGIN)] + [(_r64(g[0] - MARGIN), _r64(g[-1] + MARGIN, up=True)) for g in groups] + [(N_LONG - 2 * MARGIN, N_LONG)]
    for (a0, a1), (b0, b1) in zip(spans, spans[1:]):
        assert a1 < b0
    return np.asarray([a for a, _ in spans], np.int64), np.asarray([b - a for a, b in spans], np.int64)


class LongText:
    """T_small, the island table, the read sets and (lazily) the oracle's results on T_small; T_long on the device."""

    def __init__(self):
        rng = np.random.RandomState(SEED)
        self.long_off, self.isl_len = _island_layout()
        self.small_off = np.concatenate([[0], np.cumsum(self.isl_len)[:-1]]).astype(np.int64)
        n_small = int(self.isl_len.sum())
        sym = np.full(n_small, 4, np.uint8)
        for i, (so, ln) in enumerate(zip(self.small_off, self.isl_len)):
            body = synth.make_text(SEED + 10 + i, int(ln) - 2 * WALL, n_per_million=1500 if i % 2 else 0).symbols
            sym[so + WALL:so + ln - WALL] = body
        # a tandem repeat behind the first 3-chunk cut (an even multiple of 16384): reads with ~1500 placements each.  The
        # other cuts keep plain text on both sides, where a position scanned twice or not at all changes a unique hit.
        c3 = chunk_cuts(0, N_LONG - 15, 3)[0]
        t0 = self.small(c3 + 4000)
        unit = rng.randint(0, 4, 40).astype(np.uint8)
        sym[t0:t0 + 40 * 1500] = np.tile(unit, 1500)
        self.tandem = (t0, t0 + 40 * 1500)
        # near-identical copies of one piece of island 0 over the other placed points (a few substitutions each):
        # a read of that piece has hits in several islands, in every chunk
        src = sym[WALL + 5000:WALL + 8000].copy()
        for p in sorted(set([TWO32, CUT] + [c for k in (2, 3, 4) for c in chunk_cuts(0, N_LONG - 15, k)])):
            s = self.small(p - 1500)
            if s + 3000 <= self.tandem[0] or s >= self.tandem[1]:
                seg = src.copy()
                at = rng.randint(0, 3000, 8)
                seg[at] = (seg[at] + 1) % 4
                sym[s:s + 3000] = seg
        # island 0's positions [16384, 20096) again at 2^32 above them: a record formed for one of the first positions but
        # placed 2^32 too high (a relative position that wrapped) would verify there (test_text_shards_cut_above_2_32)
        sym[self.small(TWO32 + 16384):self.small(TWO32 + 20096)] = sym[16384:20096]
        # records: none before the island over 2^32, several above 2^32 (in-record positions above 2^32 in record 0)
        rs_long = [0, TWO32 + 45_000, TWO32 + 80_000, TWO32 + 91_000, N_LONG - 120_000, N_LONG - 60_000, N_LONG - 1000]
        self.small_text = synth.Text(sym, [("rec%d" % j, self.small(p)) for j, p in enumerate(rs_long)])
        self.rs_long = np.asarray(rs_long + [N_LONG], np.uint64)
        assert np.array_equal(self.to_long(self.small_text.record_starts[:-1]), self.rs_long[:-1])
        self.words_small, self.nmask_small = self.small_text.packed()

        # reads: drawn from T_small (make_reads), reads of the tandem repeat, and reads placed across every cut and 2^32
        straddle = sorted(set([TWO32, CUT] + [c for k in (2, 3, 4) for c in chunk_cuts(0, N_LONG - 15, k)]))
        self.reads1 = synth.concat_reads([synth.make_reads(self.small_text, SEED + 1, 12_000, L1, 0.012, fastq=True),
                                          self._explicit(rng, [rng.randint(self.tandem[0], self.tandem[1] - L1) for _ in range(30)], L1),
                                          self._straddling(rng, straddle, L1)])
        r2 = synth.make_reads(self.small_text, SEED + 2, 6000, L2, 0.02, fastq=True)
        synth.plant_deletions(self.small_text, r2, SEED + 2, L2)
        self.reads2 = synth.concat_reads([r2, self._straddling(rng, straddle, L2)])
        self.ll = O.build_ll()
        self.words = self.nmask = None

    # ---- the island table
    def small(self, p):
        """T_long position inside an island -> T_small position (scalar)."""
        i = int(np.searchsorted(self.long_off, p, side="right")) - 1
        assert i >= 0 and p < self.long_off[i] + self.isl_len[i], p
        return int(self.small_off[i] + p - self.long_off[i])

    def to_long(self, p):
        p = np.asarray(p, np.int64)
        i = np.searchsorted(self.small_off, p, side="right") - 1
        return (self.long_off[i] + p - self.small_off[i]).astype(np.uint64)

    def to_small(self, p, what="hit"):
        """T_long positions -> T_small positions; a position outside every island fails the test by name."""
        p = np.asarray(p, np.int64)
        i = np.searchsorted(self.long_off, p, side="right") - 1
        ic = np.maximum(i, 0)
        ok = (i >= 0) & (p < self.long_off[ic] + self.isl_len[ic])
        if not ok.all():
            bad = np.nonzero(~ok)[0]
            raise AssertionError("%d %s(s) on the background of T_long, outside every island (first at %s: T_long position %d)"
                                 % (bad.size, what, bad[0], p[bad[0]]))
        return self.small_off[ic] + p - self.long_off[ic]

    def _explicit(self, rng, starts, L, sub=0.01):
        seqs, quals = [], []
        for k, p in enumerate(starts):
            s = self.small_text.symbols[p:p + L].copy()
            assert (s < 4).all()
            q = np.full(L, 35, np.uint8)
            for j in np.nonzero(rng.rand(L) < sub)[0]:
                s[j] = (s[j] + 1 + rng.randint(0, 3)) & 3
                q[j] = 9
            if k % 2:                                 # '-' strand
                s, q = synth.revcomp_mapped(s), q[::-1].copy()
            seqs.append(s)
            quals.append(q)
        return synth.reads_from_list(seqs, quals, ["x%d" % k for k in range(len(seqs))])

    def _straddling(self, rng, points, L):
        """Reads whose windows hold the position `p` of T_long at their first, last and several inner bases, on both
        strands (the seed window is the read's start on '+', its end on '-')."""
        starts = []
        for p in points:
            for d in (1, 2, 16, 31, 32, 33, 50, L - 33, L - 32, L - 31, L - 2, L - 1, L):
                starts += [self.small(p - d)] * 2      # one read per strand (_explicit alternates)
        return self._explicit(rng, starts, L)

    # ---- the oracle on T_small
    @functools.cached_property
    def ref_all(self):
        return O.match_all(self.small_text, self.reads1, seedl=32, seedkmax=2, totalkmax=4, scores=True, ll=self.ll)

    @functools.cached_property
    def ref_all48(self):
        return O.match_all(self.small_text, self.reads1, seedl=48, seedkmax=2, totalkmax=4, scores=False)

    @functools.cached_property
    def ref_unique_plain(self):
        info, _ = O.unique_init(self.reads1.nreads, False)
        O.match_unique(self.small_text, self.reads1, info, None, seedl=32, seedkmax=2, totalkmax=4, scores=False)
        return info

    @functools.cached_property
    def ref_gapped(self):
        """(words, scores) after matchUnique with scores, the same after the gapped pass, GapInfo rows."""
        kw = dict(seedl=32, seedkmax=2, totalkmax=2, scores=True, ll=self.ll)
        info, sc = O.unique_init(self.reads2.nreads, True)
        O.match_unique(self.small_text, self.reads2, info, sc, **kw)
        before = (info.copy(), sc.copy())
        gaps = np.zeros(self.reads2.nreads, dtype=O.GAP_DTYPE)
        O.match_gaps(self.small_text, self.reads2, info, sc, gaps, **kw)
        return before, (info, sc), gaps

    # ---- T_long
    def build_long(self):
        import torch
        from real_b200 import devsynth
        words, nmask = devsynth.text_device(SEED, N_LONG)
        ws, ms = torch.as_tensor(self.words_small.view(np.int64)).cuda(), torch.as_tensor(self.nmask_small.view(np.int64)).cuda()
        for so, lo, ln in zip(self.small_off, self.long_off, self.isl_len):
            words[lo // 32:(lo + ln) // 32] = ws[so // 32:(so + ln) // 32]
            nmask[lo // 64:(lo + ln) // 64] = ms[so // 64:(so + ln) // 64]
        torch.cuda.synchronize()
        self.words, self.nmask = words, nmask

    def handle(self, reads=None, packed=False, shard=None, **kw):
        """A handle with a read set and T_long (or, with shard = (own_begin, own_end, shard_begin, shard_len), a part of it)."""
        h = rlib.Handle(**kw)
        try:
            if shard is not None and len(shard) == 2:
                h.set_bucket_shard(*shard)
                shard = None
            reads = self.reads1 if reads is None else reads
            if packed:
                pk, _, _, flags = synth.pack_reads_2bit(reads)
                h.set_reads_packed(pk, reads.nreads, uniform_length=L1, wildcard_flags=flags, quality=reads.quality)
            else:
                h.set_reads(reads.mapped, reads.offsets, reads.quality)
            self.set_long(h, shard)
        except BaseException:
            h.close()
            raise
        return h

    def set_long(self, h, shard=None):
        if shard is None:
            h.set_text_device(self.words.data_ptr(), self.nmask.data_ptr(), N_LONG, self.rs_long)
        else:
            ob, oe, sb, sl = shard
            h.set_text_device(self.words.data_ptr() + 8 * (sb // 32), self.nmask.data_ptr() + 8 * (sb // 64), N_LONG, self.rs_long,
                              shard_begin=sb, shard_len=sl, own_begin=ob, own_end=oe)

    # ---- comparisons
    def rows_small(self, rows):
        out = np.array(rows, copy=True)
        out["pos"] = self.to_small(rows["pos"]).astype(np.uint64)
        return out

    def info_small(self, info):
        """Unique state words of T_long with the position field of states 1..4 moved to T_small."""
        info = np.asarray(info, np.uint64).copy()
        sel = matcher.umi_state(info) != 0
        info[sel] = (info[sel] & ~POS_MASK) | self.to_small(matcher.umi_pos(info[sel]), "unique hit").astype(np.uint64)
        return info


@pytest.fixture(scope="module")
def lt():
    need_big_gpu(150, FREE_GB)
    fx = LongText()
    fx.build_long()
    yield fx
    fx.words = fx.nmask = None
    import torch
    torch.cuda.empty_cache()


def _chunks(h, scans=1):
    """Chunks the last match call scanned in: run_scan counts 4 launches per chunk (histogram or kept-position list,
    bucket offsets, scatter, probe), `scans` times when the hit buffer overflowed and the scan ran again."""
    n = h.stats()["scan_launches"]
    assert n % (4 * scans) == 0, n
    return n // (4 * scans)


_PEAK = [0]


def _note_memory():
    """Samples the device memory in use (call it while a handle holds its buffers); the module's maximum is kept."""
    import torch
    free, total = torch.cuda.mem_get_info(0)
    _PEAK[0] = max(_PEAK[0], total - free)


def _report(case, chunks):
    print("\n[long text] %s: %s chunk(s); most device memory in use so far %.1f GB" % (case, chunks, _PEAK[0] / 2**30))


def _same_rows(lt, rows, ref, with_score=True):
    got = canon_hits(lt.rows_small(rows), with_score=with_score)
    want = canon_hits(ref, with_score=with_score)
    assert got.shape == want.shape, (got.shape, want.shape)
    assert np.array_equal(got, want)


def test_match_all_scores_multi_chunk(lt):
    """matchAll, seed 32, -e 4, scores, byte reads: the first call overflows the hit buffer and scans again; the second
    one (hit16 rows) scans once, in two chunks or more."""
    ref = lt.ref_all
    nreads = lt.reads1.nreads
    assert len(ref) > max(1 << 16, 2 * nreads)
    h = lt.handle(seedl=32, seedkmax=2, totalkmax=4, scores=True, ll_table=lt.ll, filter_mult=O.filter_mult(4))
    try:
        rows = h.match_all()
        st = h.stats()
        assert st["n_hits"] == len(rows) > max(1 << 16, 2 * nreads)          # the regrowth rescan ran
        assert unify_order_ok(rows)
        _same_rows(lt, rows, ref)
        assert (rows["pos"] >= TWO32).sum() > 100 and (rows["frag"] > 0).sum() > 100
        rows16 = h.match_all_packed()
        _note_memory()
        k = _chunks(h)
        assert k >= 2
        for f in ("patid", "pos", "frag", "k", "inverted"):
            assert np.array_equal(rows16[f], rows[f]), f
        assert np.array_equal(rows16["score"].view(np.uint32), rows["score"].view(np.uint32))
        _report("matchAll -l 32 -e 4 scores", k)
    finally:
        h.close()


def test_match_all_seed48_packed_reads(lt):
    """matchAll, seed 48 (k_bucket_probe<true, true>: wide seeds out of 2-bit reads)."""
    h = lt.handle(packed=True, seedl=48, seedkmax=2, totalkmax=4, scores=False, filter_mult=O.filter_mult(4))
    try:
        rows = h.match_all()
        h.match_all_count()                       # the buffer fits now: one scan
        _note_memory()
        k = _chunks(h)
        assert k >= 2
        _same_rows(lt, rows, lt.ref_all48, with_score=False)
        _report("matchAll -l 48 packed reads", k)
    finally:
        h.close()


def test_match_unique_scores_then_gaps(lt):
    """matchUnique with scores (order faithful), then the gapped pass: words, scores and GapInfo rows."""
    (info0, sc0), (info1, sc1), gaps_ref = lt.ref_gapped
    assert (matcher.umi_state(info1) == 3).sum() > 100 and (matcher.umi_state(info0) == 4).sum() > 10
    h = lt.handle(reads=lt.reads2, seedl=32, seedkmax=2, totalkmax=2, scores=True, ll_table=lt.ll, filter_mult=O.filter_mult(2))
    try:
        h.match_unique()
        k = _chunks(h, 2) if h.stats()["n_hits"] > max(1 << 16, 2 * lt.reads2.nreads) else _chunks(h)
        info, sc = h.get_unique()
        assert np.array_equal(lt.info_small(info), info0)
        assert np.array_equal(sc.view(np.uint32), sc0.view(np.uint32))
        h.match_gaps(0)
        _note_memory()
        kg = _chunks(h)
        info, sc = h.get_unique()
        gaps = h.get_gaps()
    finally:
        h.close()
    assert k >= 2 and kg >= 2
    assert np.array_equal(lt.info_small(info), info1)
    assert np.array_equal(sc.view(np.uint32), sc1.view(np.uint32))
    got, want = gaps[gaps["present"] == 1], gaps_ref[gaps_ref["present"] == 1]
    assert len(got) == len(want) > 100
    for f in ("patid", "mingap", "where", "start", "gap_pos"):
        assert np.array_equal(got[f], want[f]), f
    _report("matchUnique scores / matchGaps", "%d / %d" % (k, kg))


@pytest.mark.parametrize("nsh", [2, 4])
def test_bucket_shards_fold(lt, nsh):
    """matchUnique without scores as 2 bucket shards (filter path) and 4 (k_own_list path), folded through the export
    keys, the ties and the import; the ranks run one after the other.  Every probed position is kept by exactly one
    rank (the stats count the positions a bucket shard formed records of)."""
    import torch
    R = lt.reads1.nreads
    dev = torch.device("cuda", 0)
    kw = dict(seedl=32, seedkmax=2, totalkmax=4, scores=False, filter_mult=O.filter_mult(4))
    keys = torch.empty(R, dtype=torch.int64, device=dev)
    kmin, chunks, kept = None, [], []
    for r in range(nsh):
        h = lt.handle(shard=(r, nsh), **kw)
        try:
            h.match_unique()
            _note_memory()
            chunks.append(_chunks(h))
            kept.append(h.stats()["n_windows"])
            h.unique_export_keys(keys.data_ptr())
            kmin = keys.clone() if kmin is None else torch.minimum(kmin, keys)
        finally:
            h.close()
    tsum = torch.zeros(R, dtype=torch.uint8, device=dev)
    ties = torch.empty(R, dtype=torch.uint8, device=dev)
    for r in range(nsh):
        h = lt.handle(shard=(r, nsh), **kw)
        try:
            h.match_unique()
            h.unique_export_ties(kmin.data_ptr(), ties.data_ptr())
            tsum += ties
            if r == nsh - 1:
                torch.cuda.synchronize()
                h.unique_import(kmin.data_ptr(), tsum.data_ptr())
                merged = h.get_unique()[0]
        finally:
            h.close()
    assert min(chunks) >= 2
    assert sum(kept) == N_LONG - 32 + 1 + 2 * 8 and min(kept) > 0          # seed windows + two fragments, each kept once
    want = matcher.canonical_unique(lt.ref_unique_plain)
    assert (matcher.umi_state(want) == 4).sum() > 100
    assert np.array_equal(matcher.canonical_unique(lt.info_small(merged)), want)
    _report("bucket shards x%d" % nsh, chunks)


def test_text_shards_cut_above_2_32(lt):
    """Text shards cut at CUT > 2^32: the shard that ends there ([0, CUT) plus its read-length halo) is itself longer
    than one chunk, and it owns the positions from `split` on only: its windows start off the partition tiles, so the
    first tile of every chunk is clipped (an unclipped one forms records of positions in front of the chunk, whose
    positions relative to the chunk wrap to 2^32 above them -- where the text repeats them).  The next shard starts
    above 2^32.  The union of their rows is the oracle's."""
    split = 20_032                             # inside island 0, not a multiple of the scatter tile
    shards = [(0, split, 0, split + L1 + 64), (split, CUT, 0, CUT + L1 + 64), (CUT, N_LONG, CUT, N_LONG - CUT)]
    h = lt.handle(shard=shards[0], seedl=32, seedkmax=2, totalkmax=4, scores=True, ll_table=lt.ll, filter_mult=O.filter_mult(4))
    try:
        parts, chunks = [], []
        for i, sh in enumerate(shards):
            if i:
                lt.set_long(h, sh)
            rows = h.match_all()
            _note_memory()
            assert (rows["pos"] >= sh[0]).all() and (rows["pos"] < sh[1]).all()
            parts.append(rows)
            h.match_all_count()             # (a shard scanned in one chunk keeps its records: this scan only probes)
            chunks.append(h.stats()["scan_launches"])
    finally:
        h.close()
    assert min(len(p) for p in parts) > 10
    _same_rows(lt, np.concatenate(parts), lt.ref_all)         # the shards own disjoint ranges: no row twice
    assert chunks[1] % 4 == 0 and chunks[1] // 4 >= 2
    _report("text shards at 2^32 + 32768 (scan launches of a second call)", chunks)


def test_one_handle_long_small_long(lt):
    """One handle, three texts in turn: T_long (several chunks: no records kept), T_small (one chunk: its records are
    kept), T_long again (the kept records belong to another text)."""
    h = lt.handle(seedl=32, seedkmax=2, totalkmax=4, scores=True, ll_table=lt.ll, filter_mult=O.filter_mult(4))
    try:
        _same_rows(lt, h.match_all(), lt.ref_all)
        st = lt.small_text
        h.set_text(lt.words_small, lt.nmask_small, st.n, st.record_starts)
        got = h.match_all()
        a, b = canon_hits(got), canon_hits(lt.ref_all)
        assert a.shape == b.shape and np.array_equal(a, b)
        lt.set_long(h)
        _same_rows(lt, h.match_all(), lt.ref_all)
        _same_rows(lt, h.match_all(), lt.ref_all)
        k = _chunks(h)
    finally:
        h.close()
    assert k >= 2


def _render_fasta(words, nmask, rs, names, line_len=80):
    """T_long as the bytes of a FASTA file, rendered on the device: one header per record, `line_len` bases per line."""
    import torch
    from real_b200 import devsynth
    n = int(rs[-1])
    sym = devsynth.unpack_symbols(words, nmask, n)
    lut = torch.as_tensor(np.frombuffer(b"ACGTN", np.uint8).copy(), device=sym.device)
    step = 1 << 28
    for a in range(0, n, step):
        sym[a:a + step] = lut[sym[a:a + step].long()]
    heads = [b">" + nm + b"\n" for nm in names]
    lens = [int(rs[r + 1] - rs[r]) for r in range(len(names))]
    total = sum(len(hd) + ln + -(-ln // line_len) for hd, ln in zip(heads, lens))
    out = torch.empty(total, dtype=torch.uint8, device=sym.device)
    off = 0
    lines = step // line_len
    for r, (hd, ln) in enumerate(zip(heads, lens)):
        out[off:off + len(hd)] = torch.as_tensor(np.frombuffer(hd, np.uint8).copy(), device=sym.device)
        off += len(hd)
        s0, full = int(rs[r]), ln // line_len
        for l0 in range(0, full, lines):
            l1 = min(full, l0 + lines)
            dst = out[off + l0 * (line_len + 1):off + l1 * (line_len + 1)].view(l1 - l0, line_len + 1)
            dst[:, :line_len] = sym[s0 + l0 * line_len:s0 + l1 * line_len].view(l1 - l0, line_len)
            dst[:, line_len] = 10
        off += full * (line_len + 1)
        tail = ln - full * line_len
        if tail:
            out[off:off + tail] = sym[s0 + full * line_len:s0 + ln]
            out[off + tail] = 10
            off += tail + 1
    assert off == total
    _note_memory()
    del sym
    return out


def test_fasta_above_4gib(lt):
    """K0 on a FASTA file of 4.65 GB (80-column lines): the packed text, the wildcard mask and the record starts are
    T_long's, and matchUnique with scores on the loaded text gives the oracle's words."""
    import torch
    names = [b"rec%d long text record" % r for r in range(len(lt.rs_long) - 1)]
    fa = _render_fasta(lt.words, lt.nmask, lt.rs_long, names)
    total_bytes = fa.numel()
    assert total_bytes > (1 << 32) + (1 << 28)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    (info0, sc0), _, _ = lt.ref_gapped
    h = rlib.Handle(seedl=32, seedkmax=2, totalkmax=2, scores=True, ll_table=lt.ll, filter_mult=O.filter_mult(2))
    try:
        h.set_reads(lt.reads2.mapped, lt.reads2.offsets, lt.reads2.quality)
        n, nrec = h.set_text_fasta(None, device_ptr=fa.data_ptr(), nbytes=fa.numel())
        assert (n, nrec) == (N_LONG, len(names))
        starts, _ = h.get_text_records()
        assert np.array_equal(starts, lt.rs_long)
        w, m = h.get_text_packed(N_LONG)
        assert np.array_equal(w, lt.words[:w.size].cpu().numpy().view(np.uint64))
        assert np.array_equal(m, lt.nmask[:m.size].cpu().numpy().view(np.uint64))
        del w, m
        _note_memory()
        del fa
        torch.cuda.empty_cache()
        h.match_unique()
        _note_memory()
        info, sc = h.get_unique()
    finally:
        h.close()
    assert np.array_equal(lt.info_small(info), info0)
    assert np.array_equal(sc.view(np.uint32), sc0.view(np.uint32))
    _report("FASTA file of %d bytes, matchUnique scores" % total_bytes, "-")


def test_format_all_above_2_32(lt):
    """Output lines of matchAll rows above 2^32: in-record positions above 2^32 (record 0) and records past the first."""
    reads = lt.reads1
    ids = [("read%d" % i).encode() for i in range(reads.nreads)]
    names = [b"rec%d" % r for r in range(len(lt.rs_long) - 1)]
    h = lt.handle(seedl=32, seedkmax=2, totalkmax=4, scores=True, ll_table=lt.ll, filter_mult=O.filter_mult(4))
    try:
        rows = h.match_all()
        h.set_read_ids(ids)
        h.set_record_names(names, lt.rs_long[:-1])
        high = np.nonzero(rows["pos"] >= TWO32)[0]
        rec0 = high[rows["frag"][high] == 0]
        later = high[rows["frag"][high] > 0]
        assert rec0.size > 20 and later.size > 20

        def want(i):
            x = rows[i]
            r, f = int(x["patid"]), int(x["frag"])
            return line(ids[r], read_bases(reads, r, bool(x["inverted"])), x["score"], L1, bool(x["inverted"]), names[f],
                        int(x["pos"]) - int(lt.rs_long[f]) + 1, int(x["k"]))

        for i in sorted(set(rec0[:: max(1, rec0.size // 40)].tolist() + later[:: max(1, later.size // 40)].tolist())):
            assert h.format_all(i, 1) == want(i), i
        for a in (int(rec0[0]), int(later[0])):                       # and a block of rows from there on
            assert h.format_all(a, 300) == b"".join(want(i) for i in range(a, a + 300))
    finally:
        h.close()
