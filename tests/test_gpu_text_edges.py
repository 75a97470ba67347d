"""GPU: the text-side predicates -- no N in a window (wildcard_free), inside one record, the valid seed windows that
place the reference's text blocks (k_window_counts) -- on the edge text of tests/util.py, whose N runs and records sit
at every offset mod 64, bit for bit against the oracle; and the record-count limits of matchUnique (65535 records) and
of a hit's record index (2^24)."""
import numpy as np
import pytest

from oracle import oracle_py as O
from real_b200 import lib as rlib
from real_b200 import dist as rdist
from real_b200 import matcher, synth
from test_gpu_option_range import _load_reads, oracle_run, same_gaps, same_rows, same_unique
from util import block_bounds_ref, edge_case, line, read_bases

pytestmark = pytest.mark.gpu

E = 5
_cases = {}


def case(seedl, uniform=False):
    key = (seedl, uniform)
    if key not in _cases:
        lengths = (100,) if uniform else ((60, 100, 120, 0) if seedl < 60 else (100, 120, 0))
        _cases[key] = edge_case(300 + seedl, full=True, seedl=seedl, lengths=lengths)
    return _cases[key]


def handle(seedl=32, e=E, scores=True, ll=None, **kw):
    return rlib.Handle(seedl=seedl, seedkmax=2, totalkmax=e, scores=scores, filter_mult=O.filter_mult(e), ll_table=ll, **kw)


def gpu_all(c, text, seedl, how, ll):
    h = handle(seedl, ll=ll)
    try:
        _load_reads(h, c.reads, how)
        w, m = text.packed()
        h.set_text(w, m, text.n, text.record_starts)
        rows = h.match_all()
        rows16 = h.match_all_packed()
    finally:
        h.close()
    return rows, rows16


def same_packed_rows(rows16, rows):
    for f in ("patid", "pos", "k", "inverted", "frag"):
        assert np.array_equal(rows16[f], rows[f]), f
    assert np.array_equal(rows16["score"].view(np.uint32), rows["score"].view(np.uint32))


def gpu_unique(c, text, seedl, scores, ll, n_list, gaps=False, e=E):
    h = handle(seedl, e=e, scores=scores, ll=ll)
    try:
        h.set_reads(c.reads.mapped, c.reads.offsets, c.reads.quality)
        h.set_block_windows(n_list)
        w, m = text.packed()
        h.set_text(w, m, text.n, text.record_starts)
        h.match_unique()
        g = None
        if gaps:
            h.match_gaps(n_list)
            g = h.get_gaps()
        info, sc = h.get_unique()
    finally:
        h.close()
    return (info, sc, g) if gaps else (info, sc)


# ------------------------------------------------------------------ 1. matchAll

@pytest.mark.parametrize("how", ["bytes", "packed", "uniform"])
@pytest.mark.parametrize("seedl", [32, 20, 64])
def test_edge_text_match_all(seedl, how):
    """Byte reads and 2 bit/base reads (both verification branches), 16-byte rows too."""
    c = case(seedl, uniform=(how == "uniform"))
    ll = O.build_ll()
    ref = oracle_run("all", [c.text], c.reads, seedl=seedl, e=E, ll=ll)
    rows, rows16 = gpu_all(c, c.text, seedl, how, ll)
    same_rows(rows, ref, int(c.plan["expect"].sum()))
    same_packed_rows(rows16, rows)


def test_codes_under_n_do_not_matter():
    """Random codes under the N positions give the same rows and unique words, on the GPU and in the oracle."""
    c = case(32)
    ll = O.build_ll()
    ref = oracle_run("all", [c.text], c.reads, e=E, ll=ll)
    same_rows(oracle_run("all", [c.text_random], c.reads, e=E, ll=ll), ref, 1000)
    same_rows(gpu_all(c, c.text_random, 32, "bytes", ll)[0], ref, 1000)
    same_rows(gpu_all(c, c.text_random, 32, "packed", ll)[0], ref, 1000)
    a = gpu_unique(c, c.text, 32, True, ll, 997)
    b = gpu_unique(c, c.text_random, 32, True, ll, 997)
    same_unique(b, a, True)
    same_unique(a, oracle_run("unique", [c.text_random], c.reads, e=E, ll=ll, n_list=997), True)


# ------------------------------------------------------------------ 2. shards

def test_text_shards_cut_at_n_runs():
    """Two text shards: the second starts on the mask word that holds the start of a 33-base N run, the first owns the
    positions up to the run's end, where a read planted flush against the run starts."""
    c = case(32)
    t = c.text
    a, ln = next((int(a), int(ln)) for a, ln in c.runs if ln == 33 and a % 64 not in (0, 31) and a > 100_000)
    cut = a + ln
    assert ((c.plan["kind"] == 1) & (c.plan["p"] == cut) & c.plan["expect"]).any()
    sb1 = (a // 64) * 64
    lmax = int(np.diff(c.reads.offsets.astype(np.int64)).max())
    shards = [(0, cut, 0, min(t.n, cut + lmax)), (cut, t.n, sb1, t.n - sb1)]
    ll = O.build_ll()
    w, m = t.packed()
    h = handle(32, ll=ll)
    out = []
    try:
        h.set_reads(c.reads.mapped, c.reads.offsets, c.reads.quality)
        for ob, oe, sb, sl in shards:
            h.set_text(np.ascontiguousarray(w[sb // 32:(sb + sl + 31) // 32]), np.ascontiguousarray(m[sb // 64:(sb + sl + 63) // 64]),
                       t.n, t.record_starts, 0, shard_begin=sb, shard_len=sl, own_begin=ob, own_end=oe)
            out.append(h.match_all())
    finally:
        h.close()
    ref = oracle_run("all", [t], c.reads, e=E, ll=ll)
    same_rows(np.concatenate(out), ref, int(c.plan["expect"].sum()))
    assert (ref["pos"] == cut).any()


@pytest.mark.parametrize("nranks", [2, 4])
def test_bucket_shards_fold_group_unique(nranks):
    c = case(32)
    t = c.text
    R = c.reads.nreads
    hs = [handle(32, scores=False) for _ in range(nranks)]
    try:
        for r, h in enumerate(hs):
            h.set_bucket_shard(r, nranks)
            h.fold_init(r, nranks, R + 5)
        for h in hs:
            h.fold_connect_local(hs)
        w, m = t.packed()
        for h in hs:
            h.set_reads(c.reads.mapped, c.reads.offsets)
            h.set_text(w, m, t.n, t.record_starts)
            h.match_unique()
        rlib.Handle.fold_unique_group(hs)
        got = np.zeros(R, np.uint64)
        for r, h in enumerate(hs):
            lo, hi = rdist.own_read_range(R, r, nranks)
            got[lo:hi] = h.get_unique(first=lo, count=hi - lo)[0]
    finally:
        for h in hs:
            h.close()
    ref = oracle_run("unique", [t], c.reads, e=E, scores=False)
    same_unique((got, None), ref, False)


# ------------------------------------------------------------------ 3. matchUnique, 4. gapped pass

@pytest.mark.parametrize("seedl", [32, 20])
def test_edge_text_match_unique(seedl):
    c = case(seedl)
    ll = O.build_ll()
    same_unique(gpu_unique(c, c.text, seedl, False, None, 0), oracle_run("unique", [c.text], c.reads, seedl=seedl, e=E, scores=False), False)
    for n_list in (0, 997, 5000):
        ref = oracle_run("unique", [c.text], c.reads, seedl=seedl, e=E, ll=ll, n_list=n_list)
        same_unique(gpu_unique(c, c.text, seedl, True, ll, n_list), ref, True)
        st = matcher.umi_state(ref[0])
        assert ((st == 1) | (st == 2)).sum() > 5000


@pytest.mark.parametrize("n_list", [0, 4000])
def test_edge_text_gapped_pass(n_list):
    """-e 2 leaves the gapped-pass reads NoMatch; their DP windows end at record ends (n = 0..2L) or hold an N."""
    c = case(32)
    ll = O.build_ll()
    ref = oracle_run("gaps", [c.text], c.reads, e=2, ll=ll, n_list=n_list)
    got = gpu_unique(c, c.text, 32, True, ll, n_list, gaps=True, e=2)
    same_unique(got, ref, True)
    same_gaps(got[2], ref[2], 5)
    gp = c.gap_plan
    st = matcher.umi_state(ref[0])[gp["read"]]
    rescued = st == 3
    assert rescued.any() and (~rescued).any()
    assert not rescued[gp["n"] == 0].any()                           # n = 0: never a DP
    inside = (gp["nat"] >= 0) & (gp["nat"] < gp["n"])
    assert not rescued[inside].any() and rescued[(gp["nat"] >= gp["n"])].any()


# ------------------------------------------------------------------ 5. block bounds

def _bb_texts(rng):
    """Masks with partial runs at every offset, all-N words and isolated Ns; lengths off the 64 grid and below the seed."""
    out = []
    for n in (10, 63, 64, 65, 1000, 4097, 70_001):
        sym = rng.randint(0, 4, n).astype(np.uint8)
        if n > 1000:
            for s in range(0, n - 200, 97):
                sym[s:s + 1 + (s // 97) % 70] = 4
            sym[1024:1152] = 4
            sym[rng.randint(0, n, n // 300)] = 4
        elif n >= 64:
            sym[rng.randint(0, n, 3)] = 4
        out.append(sym)
    c = case(32)
    out.append(c.text.symbols[:300_001])
    return out


def test_block_bounds_vs_numpy():
    rng = np.random.RandomState(77)
    texts = _bb_texts(rng)
    for seedl in range(4, 68, 4):
        h = handle(seedl, scores=False)
        try:
            for sym in texts:
                w, m = synth.pack_text(sym)
                starts = np.asarray([0, sym.size], np.uint64)
                for async_copy in (False, True):
                    h.set_text(w, m, sym.size, starts, async_copy=async_copy)
                    for n_list in (1, 2, 63, 64, 65, 1000):
                        want = block_bounds_ref(sym, seedl, n_list)
                        got = h.get_block_bounds(n_list, cap=max(1, want.size) + 8)
                        assert np.array_equal(got, want), (seedl, sym.size, n_list, async_copy)
                    assert h.get_block_bounds(0).tolist() == [0]
        finally:
            h.close()


# ------------------------------------------------------------------ 7. text first

def test_text_first_async_prepare_packed_reads():
    c = case(32, uniform=True)
    t = c.text
    ll = O.build_ll()
    ref = oracle_run("all", [t], c.reads, e=E, ll=ll)
    w, m = t.packed()
    import torch
    pw = torch.from_numpy(w.view(np.int64)).pin_memory().numpy().view(np.uint64)
    pm = torch.from_numpy(m.view(np.int64)).pin_memory().numpy().view(np.uint64)
    pk, boffs, lens, flags = synth.pack_reads_2bit(c.reads)
    h = handle(32, ll=ll)
    try:
        h.set_text(pw, pm, t.n, t.record_starts, async_copy=True)
        h.prepare_scan(100)
        h.set_reads_packed(pk, c.reads.nreads, uniform_length=100, wildcard_flags=flags, quality=c.reads.quality)
        rows = h.match_all()
        h.set_block_windows(997)
        h.set_text(pw, pm, t.n, t.record_starts, async_copy=True)
        h.match_unique()
        info, sc = h.get_unique()
    finally:
        h.close()
    same_rows(rows, ref, int(c.plan["expect"].sum()))
    same_unique((info, sc), oracle_run("unique", [t], c.reads, e=E, ll=ll, n_list=997), True)


# ------------------------------------------------------------------ 8. K0 and K8

def edge_fasta(t):
    """61-base lines, empty records as consecutive header lines, a final header with no bases."""
    out = []
    st = t.record_starts.astype(np.int64)
    for i, (name, s) in enumerate(t.records):
        out.append(b">" + name.encode() + b"\n")
        seq = synth.BASES[t.symbols[st[i]:st[i + 1]]].tobytes()
        for j in range(0, len(seq), 61):
            out.append(seq[j:j + 61] + b"\n")
    return b"".join(out)


def test_fasta_text_match_all_and_format_all():
    c = case(32)
    t = c.text
    fa = edge_fasta(t)
    sym, names, starts = O.fasta_text(fa)
    assert np.array_equal(sym, t.symbols) and np.array_equal(starts, t.record_starts)
    ww, mm = synth.pack_text(sym)
    ll = O.build_ll()
    ids = [("e%d" % i).encode() for i in range(c.reads.nreads)]
    h = handle(32, ll=ll)
    try:
        h.set_reads(c.reads.mapped, c.reads.offsets, c.reads.quality)
        assert h.set_text_fasta(fa) == (t.n, len(t.records))
        w, m = h.get_text_packed(t.n)
        rs, _ = h.get_text_records()
        rows = h.match_all()
        h.set_read_ids(ids)
        h.set_record_names(names, starts[:-1])
        text_out = h.format_all(0, len(rows))
    finally:
        h.close()
    assert np.array_equal(w, ww) and np.array_equal(m, mm) and np.array_equal(rs, starts)
    ref = oracle_run("all", [t], c.reads, e=E, ll=ll)
    same_rows(rows, ref, int(c.plan["expect"].sum()))
    lens = np.diff(c.reads.offsets.astype(np.int64))
    want = b"".join(line(ids[int(x["patid"])], read_bases(c.reads, int(x["patid"]), bool(x["inverted"])), x["score"],
                         int(lens[int(x["patid"])]), bool(x["inverted"]), names[int(x["frag"])],
                         int(x["pos"]) - int(starts[int(x["frag"])]) + 1, int(x["k"])) for x in rows)
    assert text_out == want


# ------------------------------------------------------------------ 9. record-count limits

def many_records(seed, nrec, nlong=40, long_len=3000, nreads=2000):
    """nrec records: tiny and empty ones (lengths 0, 1, 2, 5 in turn) in front, then nlong long ones; reads drawn from the
    long records (some segments copied into a second long record: NonUnique reads)."""
    rng = np.random.RandomState(seed)
    ntiny = nrec - nlong
    tiny = np.array([0, 1, 2, 5])[np.arange(ntiny) % 4]
    lens = np.concatenate([tiny, np.full(nlong, long_len)])
    starts = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int64)
    n = int(lens.sum())
    sym = rng.randint(0, 4, n).astype(np.uint8)
    first_long = int(starts[ntiny])
    sym[first_long + 100:first_long + 400] = sym[n - 2000:n - 1700]      # a copy of part of the last record
    text = synth.Text(sym, [(" r%d" % i, int(s)) for i, s in enumerate(starts)])
    seqs, quals = [], []
    for i in range(nreads):
        rec = ntiny + (i % nlong if i % 3 else nlong - 1)
        p = int(starts[rec]) + rng.randint(0, long_len - 100)
        r = sym[p:p + 100].copy()
        j = rng.choice(np.arange(32, 100), i % 3, replace=False)
        r[j] = (r[j] + 1) & 3
        seqs.append(synth.revcomp_mapped(r) if i % 2 else r)
        quals.append(rng.randint(2, 42, 100).astype(np.uint8))
    return text, synth.reads_from_list(seqs, quals)


def test_65535_records_match_unique_and_format():
    text, reads = many_records(1, 65535)
    ll = O.build_ll()
    ref0 = oracle_run("unique", [text], reads, e=E, scores=False)
    ref1 = oracle_run("unique", [text], reads, e=E, ll=ll, n_list=20_000)
    names = [("r%d" % i).encode() for i in range(65535)]
    h = handle(32, scores=False)
    try:
        h.set_reads(reads.mapped, reads.offsets)
        w, m = text.packed()
        h.set_text(w, m, text.n, text.record_starts)
        h.match_unique()
        got0 = h.get_unique()
        h.set_read_ids([x.encode() for x in reads.ids])
        h.set_record_names(names, text.record_starts[:-1])
        out, nl = h.format_unique()
    finally:
        h.close()
    same_unique(got0, ref0, False)
    same_unique(gpu_unique_text(text, reads, ll, 20_000), ref1, True)
    st, fr = matcher.umi_state(ref0[0]), matcher.umi_frag(ref0[0])
    one = (st == 1) | (st == 2)
    assert (one & (fr == 65534)).sum() > 50 and (st == 4).sum() > 0
    assert nl == one.sum() and out.count(b"\tr65534\t") == (one & (fr == 65534)).sum()


def gpu_unique_text(text, reads, ll, n_list):
    h = handle(32, ll=ll)
    try:
        h.set_reads(reads.mapped, reads.offsets, reads.quality)
        h.set_block_windows(n_list)
        w, m = text.packed()
        h.set_text(w, m, text.n, text.record_starts)
        h.match_unique()
        return h.get_unique()
    finally:
        h.close()


def test_65536_records_are_skipped_by_match_unique_and_gaps():
    """A file of 65536 records leaves the unique state and the gap records as the file before left them."""
    t0 = synth.make_text(5, 300_000, nrecords=4)
    t1, reads = many_records(2, 65536)
    sym = t1.symbols.copy()
    sym[-3000:] = t0.symbols[10_000:13_000]                   # reads of file 0 also match file 1
    t1 = synth.Text(sym, t1.records)
    reads = synth.concat_reads([reads, synth.make_reads(t0, 6, 1000, 100, 0.01, fastq=True)])
    reads = synth.Reads(reads.mapped, reads.offsets, np.full(reads.mapped.size, 30, np.uint8), reads.ids)
    ll = O.build_ll()
    for scores in (False, True):
        ref = oracle_run("gaps" if scores else "unique", [t0, t1], reads, e=2, ll=ll, scores=scores)
        ref0 = oracle_run("gaps" if scores else "unique", [t0], reads, e=2, ll=ll, scores=scores)
        same_unique(ref, ref0, scores)
        h = handle(32, e=2, scores=scores, ll=ll)
        try:
            h.set_reads(reads.mapped, reads.offsets, reads.quality)
            states = []
            for fi, t in enumerate((t0, t1)):
                w, m = t.packed()
                h.set_text(w, m, t.n, t.record_starts, fi)
                h.match_unique()
                if scores:
                    h.match_gaps(0)
                states.append((h.get_unique(), h.get_gaps() if scores else None))
        finally:
            h.close()
        (u0, g0), (u1, g1) = states
        assert np.array_equal(u0[0], u1[0])
        if scores:
            assert np.array_equal(u0[1].view(np.uint32), u1[1].view(np.uint32)) and np.array_equal(g0, g1)
            same_gaps(g1, ref[2], 0)
        same_unique(u1, ref, scores)


def test_match_all_record_index_above_16_bits():
    """2^17 + 5 records: rows with record indices above 65535 in both row forms, and their output lines."""
    text, reads = many_records(3, (1 << 17) + 5, nreads=600)
    ll = O.build_ll()
    ref = oracle_run("all", [text], reads, e=E, ll=ll)
    assert (ref["frag"] > 65535).sum() > 300
    names = [("r%d" % i).encode() for i in range(len(text.records))]
    ids = [x.encode() for x in reads.ids]
    h = handle(32, ll=ll)
    try:
        h.set_reads(reads.mapped, reads.offsets, reads.quality)
        w, m = text.packed()
        h.set_text(w, m, text.n, text.record_starts)
        rows = h.match_all()
        rows16 = h.match_all_packed()
        h.set_read_ids(ids)
        h.set_record_names(names, text.record_starts[:-1])
        out = h.format_all(0, len(rows))
    finally:
        h.close()
    same_rows(rows, ref, 500)
    same_packed_rows(rows16, rows)
    st = text.record_starts.astype(np.int64)
    want = b"".join(line(ids[int(x["patid"])], read_bases(reads, int(x["patid"]), bool(x["inverted"])), x["score"], 100,
                         bool(x["inverted"]), names[int(x["frag"])], int(x["pos"]) - int(st[int(x["frag"])]) + 1, int(x["k"])) for x in rows)
    assert out == want


def test_2p24_records_limit():
    """2^24 - 1 records (2^24 - 3 empty ones in front) carry record index 2^24 - 2 in both row forms; 2^24 records are
    refused by set_text and set_text_fasta, and the handle then matches a valid text normally."""
    rng = np.random.RandomState(9)
    n = 40_000
    sym = rng.randint(0, 4, n).astype(np.uint8)
    nrec = (1 << 24) - 1
    starts = np.zeros(nrec + 1, np.uint64)
    starts[-2] = 20_000
    starts[-1] = n
    seqs = [sym[21_000 + 150 * i:21_100 + 150 * i] for i in range(20)] + [sym[1_000:1_100]]
    reads = synth.reads_from_list(seqs)
    h = handle(32, scores=False)
    try:
        h.set_reads(reads.mapped, reads.offsets)
        w, m = synth.pack_text(sym)
        h.set_text(w, m, n, starts)
        rows = h.match_all()
        rows16 = h.match_all_packed()
        assert len(rows) == 21 and set(rows["frag"].tolist()) == {nrec - 2, nrec - 1}
        assert int((rows["frag"] == nrec - 1).sum()) == 20
        same_packed_rows(rows16, rows)
        big = np.zeros((1 << 24) + 1, np.uint64)
        big[-1] = n
        with pytest.raises(rlib.RealGpuError) as ei:
            h.set_text(w, m, n, big)
        assert ei.value.code == rlib.REAL_GPU_E_LIMIT
        with pytest.raises(rlib.RealGpuError) as ei:
            h.set_text_fasta(b">\n" * (1 << 24) + b"ACGT\n")
        assert ei.value.code == rlib.REAL_GPU_E_LIMIT
        text = synth.Text(sym, [(" a", 0), (" b", 20_000)])
        h.set_text(w, m, n, text.record_starts)
        rows = h.match_all()
    finally:
        h.close()
    same_rows(rows, oracle_run("all", [text], reads, e=E, scores=False), 21)
