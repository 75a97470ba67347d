"""GPU: the whole accepted range of the options and of the reads against the oracle -- every seed length 4..64 with
seedkmax 0..2, error budgets 0..15 (also below the seed's), folded index tables, file ids 62 and 63, reads of 32..65535
bases on every packing path, and quality strings that vary along the read and are not tied to the substitutions."""
import numpy as np
import pytest

from oracle import oracle_py as O
from real_b200 import lib as rlib
from real_b200 import matcher, synth
from util import canon_hits, fresh, line, read_bases, unify_order_ok

pytestmark = pytest.mark.gpu

GAP_FIELDS = ("patid", "mingap", "where", "start", "gap_pos")


# ------------------------------------------------------------------ runners

def _load_reads(h, reads, how):
    """Hands the reads to handle h as bytes, as 2 bit/base data (byte offsets or uniform length) or from device memory;
    returns what has to stay alive until the handle is closed."""
    if how == "bytes":
        h.set_reads(reads.mapped, reads.offsets, reads.quality)
        return None
    if how in ("packed", "uniform"):
        pk, boffs, lens, flags = synth.pack_reads_2bit(reads)
        if how == "uniform":
            assert (lens == lens[0]).all()
            h.set_reads_packed(pk, reads.nreads, uniform_length=int(lens[0]), wildcard_flags=flags, quality=reads.quality)
        else:
            h.set_reads_packed(pk, reads.nreads, byte_offsets=boffs, lengths=lens, wildcard_flags=flags, quality=reads.quality)
        return None
    assert how == "device"
    import torch
    dev = torch.device("cuda", 0)
    dm = torch.from_numpy(reads.mapped.copy()).to(dev)
    dq = torch.from_numpy(reads.quality.copy()).to(dev)
    doff = torch.from_numpy(reads.offsets.astype(np.int64)).to(dev)
    maxlen = int(np.diff(reads.offsets.astype(np.int64)).max())
    h.set_reads_device(dm.data_ptr(), doff.data_ptr(), reads.nreads, int(reads.offsets[-1]), maxlen, d_quality=dq.data_ptr())
    return dm, dq, doff


def _set_text(h, t, fileid, shard, words, nmask):
    if shard is None:
        h.set_text(words, nmask, t.n, t.record_starts, fileid)
        return
    ob, oe, sb, sl = shard
    h.set_text(np.ascontiguousarray(words[sb // 32:(sb + sl + 31) // 32]), np.ascontiguousarray(nmask[sb // 64:(sb + sl + 63) // 64]),
               t.n, t.record_starts, fileid, shard_begin=sb, shard_len=sl, own_begin=ob, own_end=oe)


def gpu_run(mode, texts, reads, seedl=32, s=2, e=5, scores=True, ll=None, how="bytes", table_bits=0, nshards=1, n_list=0,
            filter_level=2, fileids=None):
    """mode "all": matchAll rows; "unique": (info, scores); "gaps": (info, scores, GapInfo records) of matchUnique and
    the gapped pass.  Each text is file fileids[i] (default i), cut into nshards text shards for matchAll."""
    fileids = list(range(len(texts))) if fileids is None else fileids
    h = rlib.Handle(seedl=seedl, seedkmax=s, totalkmax=e, scores=scores, filter_mult=O.filter_mult(e, filter_level),
                    ll_table=ll, table_bits=table_bits)
    try:
        keep = _load_reads(h, reads, how)
        maxlen = int(np.diff(reads.offsets.astype(np.int64)).max())
        packed = [t.packed() for t in texts]
        if mode == "all":
            out = []
            for t, fi, (w, m) in zip(texts, fileids, packed):
                for sh in (matcher.shard_ranges(t.n, nshards, maxlen) if nshards > 1 else [None]):
                    _set_text(h, t, fi, sh, w, m)
                    rows = h.match_all()
                    assert unify_order_ok(rows)
                    out.append(rows)
            return np.concatenate(out)
        h.set_block_windows(n_list)
        for t, fi, (w, m) in zip(texts, fileids, packed):
            _set_text(h, t, fi, None, w, m)
            h.match_unique()
        gaps = None
        if mode == "gaps":
            for t, fi, (w, m) in zip(texts, fileids, packed):
                _set_text(h, t, fi, None, w, m)
                h.match_gaps(n_list)
            gaps = h.get_gaps()
        info, sc = h.get_unique()
        del keep
        return (info, sc) if mode == "unique" else (info, sc, gaps)
    finally:
        h.close()


def oracle_run(mode, texts, reads, seedl=32, s=2, e=5, scores=True, ll=None, n_list=0, filter_level=2, fileids=None):
    fileids = list(range(len(texts))) if fileids is None else fileids
    kw = dict(seedl=seedl, seedkmax=s, totalkmax=e, scores=scores, ll=ll, n_list=n_list, filter_level=filter_level)
    if mode == "all":
        return np.concatenate([O.match_all(t, reads, fileid=fi, **kw) for t, fi in zip(texts, fileids)])
    info, sc = O.unique_init(reads.nreads, scores)
    for t, fi in zip(texts, fileids):
        O.match_unique(t, reads, info, sc, fileid=fi, **kw)
    if mode == "unique":
        return info, sc
    gaps = np.zeros(reads.nreads, dtype=O.GAP_DTYPE)
    for t, fi in zip(texts, fileids):
        O.match_gaps(t, reads, info, sc, gaps, fileid=fi, **kw)
    return info, sc, gaps


def same_rows(got, ref, min_rows):
    a, b = canon_hits(got), canon_hits(ref)
    assert len(b) >= min_rows, len(b)
    assert a.shape == b.shape and np.array_equal(a, b)


def same_unique(got, ref, scores):
    if scores:          # order-faithful: words and float scores bit for bit
        assert np.array_equal(got[0], ref[0])
        assert np.array_equal(got[1].view(np.uint32), ref[1].view(np.uint32))
    else:
        assert np.array_equal(matcher.canonical_unique(got[0]), matcher.canonical_unique(ref[0]))


def same_gaps(got, ref, min_present):
    g, r = got[got["present"] == 1], ref[ref["present"] == 1]
    assert len(r) >= min_present and len(g) == len(r), (len(g), len(r))
    for f in GAP_FIELDS:
        assert np.array_equal(g[f], r[f]), f


# ------------------------------------------------------------------ inputs

def seed_case(seedl, seed):
    """Inputs the oracle finishes in well under a second: seeds of at most 12 bases put most text windows into the
    candidate lists, so their texts and reads are small."""
    if seedl == 4:
        text = synth.make_text(seed, 4_000, nrecords=2)
        return text, synth.make_reads(text, seed + 1, 200, 24, 0.03, fastq=True), 2
    if seedl == 8:
        text = synth.make_text(seed, 20_000, nrecords=2, n_per_million=2000)
        return text, synth.make_reads(text, seed + 1, 500, 30, 0.03, fastq=True), 3
    if seedl == 12:
        text = synth.make_text(seed, 50_000, nrecords=3, n_per_million=2000)
        return text, synth.make_reads(text, seed + 1, 1000, 40, 0.03, fastq=True), 3
    text, reads = fresh(seed, n=150_000, nreads=3000, L=max(80, seedl + 16), nrec=3)
    return text, reads, 4


def repeat_rich_text(seed, n=300_000, copies=12, seglen=4000):
    """Near-identical repeats (a few substitutions apart): many reads have several hits within epsilon of each other."""
    text = synth.make_text(seed, n, nrecords=3, n_per_million=1500)
    sym = text.symbols.copy()
    rng = np.random.RandomState(seed)
    for _ in range(copies):
        a, b = rng.randint(0, n - n // 6, 2)
        seg = sym[a:a + seglen].copy()
        pos = rng.randint(0, seglen, 25)
        seg[pos] = (seg[pos] + 1) % 4
        sym[b:b + seglen] = seg
    return synth.Text(sym, text.records)


def illumina_quality(rng, L):
    """Runs of 1..12 bases around a level that drifts down along the read, values 2..41."""
    q = np.empty(L, np.int64)
    i, level = 0, rng.randint(30, 42)
    while i < L:
        run = rng.randint(1, 13)
        q[i:i + run] = level + rng.randint(-3, 4)
        level = max(2, level - rng.randint(0, 3)) if rng.rand() < 0.8 else rng.randint(2, 42)
        i += run
    return np.clip(q, 2, 41).astype(np.uint8)


def with_qualities(reads, kind, seed):
    """The same reads with a quality per base drawn independently of the substitutions: "illumina" (2..41 in runs),
    "phred93" (0..93), "bytes" (0..93 with a fifth of the bytes in 94..255)."""
    rng = np.random.RandomState(seed)
    qs = []
    for r in range(reads.nreads):
        L = int(reads.offsets[r + 1] - reads.offsets[r])
        if kind == "illumina":
            q = illumina_quality(rng, L)
        else:
            q = rng.randint(0, 94, L).astype(np.uint8)
            if kind == "bytes":
                hi = rng.rand(L) < 0.2
                q[hi] = rng.randint(94, 256, int(hi.sum()))
        qs.append(q)
    return synth.Reads(reads.mapped, reads.offsets, np.concatenate(qs).astype(np.uint8), reads.ids)


def quality_case(seed, kind, nper=1500, sub=0.02):
    """Repeat-rich text, reads of 81, 90, 103, 117, 122 and 151 bases (lengths 1, 2 and 3 mod 4: the quality of a read
    starts off a 4-byte boundary) on both strands."""
    text = repeat_rich_text(seed)
    parts = [synth.make_reads(text, seed + L, nper, L, sub, fastq=True) for L in (81, 90, 103, 117, 122, 151)]
    return text, with_qualities(synth.concat_reads(parts), kind, seed + 7)


def long_read_case(seed, e, seedl=32):
    """Ragged reads whose lengths straddle every boundary of the read side: the seed alone and one rest base, the
    four-word verification loop (127..129), W = 64 | 65 words (2047..2049), 2080/2081, 10000 and 65535 bases.  Each
    read is a text window with a planted number of substitutions outside the seed, on either strand, with Illumina-like
    qualities.  Reads of 2047 bases and more carry at most e substitutions -- the gapped pass never extends them -- except
    one 2049-base read with e + 1 and one 10000-base read with 3 in the seed (no seed candidate at all)."""
    rng = np.random.RandomState(seed)
    text = synth.make_text(seed, 220_000, nrecords=1)
    sym = text.symbols.copy()
    sym[150_000:150_128] = 4
    text = synth.Text(sym, [(" chrA first", 0), (" chrB", 100_000), (" chrC", 180_000)])
    clean = np.where(sym > 3, 0, sym).astype(np.uint8)
    plan = [(seedl, 8), (seedl + 1, 8), (127, 8), (128, 8), (129, 8), (2047, 4), (2048, 4), (2049, 4), (2080, 3), (2081, 3),
            (10_000, 3), (65_535, 2)]
    seqs, quals = [], []
    for L, cnt in plan:
        for i in range(cnt):
            rec0, rec1 = (0, 100_000) if L > 20_000 or i % 2 == 0 else (100_000, 150_000)
            p = rng.randint(rec0, rec1 - L)
            r = clean[p:p + L].copy()
            inv = (i + L) % 2
            seed_at = L - seedl if inv else 0
            nsub, in_seed = (rng.randint(0, e + 3), int(rng.rand() < 0.2)) if L < 2047 else (rng.randint(0, e + 1), 0)
            if L == 2049 and i == 0:
                nsub = e + 1
            if L == 10_000 and i == 2:
                in_seed = 3
            rest = np.setdiff1d(np.arange(L), np.arange(seed_at, seed_at + seedl))
            where = list(rng.choice(rest, min(nsub, rest.size), replace=False)) + list(seed_at + rng.choice(seedl, in_seed, replace=False))
            for j in where:
                r[j] = (r[j] + 1 + rng.randint(0, 3)) & 3
            seqs.append(synth.revcomp_mapped(r) if inv else r)
            quals.append(illumina_quality(rng, L))
    return text, synth.reads_from_list(seqs, quals)


# ------------------------------------------------------------------ 1. seed geometries

@pytest.mark.parametrize("s", [0, 1, 2])
@pytest.mark.parametrize("seedl", list(range(4, 68, 4)))
def test_every_seed_length_match_all(seedl, s):
    """Seeds of 4..12 bases have presence tables of 2^4..2^12 slots (no partition depth) and scan buckets of 2..6 bits;
    seeds above 32 bases are indexed on 32 and verified on the whole seed."""
    text, reads, e = seed_case(seedl, 1000 + 3 * seedl + s)
    ll = O.build_ll()
    ref = oracle_run("all", [text], reads, seedl=seedl, s=s, e=e, ll=ll)
    got = gpu_run("all", [text], reads, seedl=seedl, s=s, e=e, ll=ll)
    same_rows(got, ref, reads.nreads // 2)


@pytest.mark.parametrize("variant", ["key_width_table", "text_shards"])
@pytest.mark.parametrize("seedl", [4, 8, 12])
def test_short_seeds_direct_tables_and_text_shards(seedl, variant):
    text, reads, e = seed_case(seedl, 1100 + seedl)
    ll = O.build_ll()
    ref = oracle_run("all", [text], reads, seedl=seedl, s=2, e=e, ll=ll)
    if variant == "key_width_table":
        got = gpu_run("all", [text], reads, seedl=seedl, s=2, e=e, ll=ll, table_bits=seedl)
    else:
        got = gpu_run("all", [text], reads, seedl=seedl, s=2, e=e, ll=ll, nshards=3)
    same_rows(got, ref, reads.nreads // 2)


@pytest.mark.parametrize("seedl", [8, 12, 52, 56])
def test_seed_lengths_match_unique_and_gaps(seedl):
    if seedl == 8:
        text = repeat_rich_text(seedl, n=20_000, copies=3, seglen=1000)
        reads = synth.make_reads(text, seedl + 1, 600, 40, 0.04, fastq=True)
    elif seedl == 12:
        text = repeat_rich_text(seedl, n=50_000, copies=4, seglen=2000)
        reads = synth.make_reads(text, seedl + 1, 1000, 60, 0.04, fastq=True)
    else:
        text = repeat_rich_text(seedl, n=200_000, copies=8)
        reads = synth.make_reads(text, seedl + 1, 4000, 120, 0.03, fastq=True)
    reads = with_qualities(reads, "illumina", seedl)
    ll = O.build_ll()
    ref = oracle_run("unique", [text], reads, seedl=seedl, e=4, scores=False)
    got = gpu_run("unique", [text], reads, seedl=seedl, e=4, scores=False)
    same_unique(got, ref, False)
    st = matcher.umi_state(ref[0])
    assert (st == 1).sum() + (st == 2).sum() > reads.nreads // 3 and (st == 4).sum() > 0
    ref = oracle_run("gaps", [text], reads, seedl=seedl, e=2, ll=ll, n_list=text.n // 3)
    got = gpu_run("gaps", [text], reads, seedl=seedl, e=2, ll=ll, n_list=text.n // 3)
    same_unique(got, ref, True)
    same_gaps(got[2], ref[2], 5)


@pytest.mark.parametrize("which", ["bucket_shard", "comm_init"])
def test_shards_refuse_seeds_shorter_than_16(which):
    """Bucket shards and sharded tables split the 256 scan buckets; a 12-base seed has 64.  The call is refused and the
    handle goes on matching as a single handle."""
    text, reads, e = seed_case(12, 1212)
    h = rlib.Handle(seedl=12, totalkmax=e)
    try:
        with pytest.raises(rlib.RealGpuError) as ei:
            if which == "bucket_shard":
                h.set_bucket_shard(0, 2)
            else:
                h.comm_init(0, 2)
        assert ei.value.code == -1                          # REAL_GPU_E_ARG
        h.set_reads(reads.mapped, reads.offsets)
        w, m = text.packed()
        h.set_text(w, m, text.n, text.record_starts)
        got = h.match_all()
    finally:
        h.close()
    same_rows(got, oracle_run("all", [text], reads, seedl=12, e=e, scores=False), reads.nreads // 2)
    h = rlib.Handle(seedl=16)
    try:
        h.set_bucket_shard(0, 2)                            # 16 bases: accepted
    finally:
        h.close()


# ------------------------------------------------------------------ 2. error budgets

@pytest.mark.parametrize("scores", [False, True])
@pytest.mark.parametrize("e", [0, 1, 9, 12, 15])
def test_error_budgets_match_all(e, scores):
    """k of 9..15 fills the 4-bit k fields; -e 0 / 1 lies below -s 2, so the whole-read test rejects what the seed test
    admits."""
    text = synth.make_text(300 + e, 200_000, nrecords=3, n_per_million=1000)
    reads = synth.make_reads(text, 301 + e, 3000, 150, 0.06 if e >= 9 else 0.004, fastq=True)
    reads = with_qualities(reads, "illumina", e)
    ll = O.build_ll() if scores else None
    ref = oracle_run("all", [text], reads, e=e, scores=scores, ll=ll)
    got = gpu_run("all", [text], reads, e=e, scores=scores, ll=ll)
    same_rows(got, ref, reads.nreads // 3)
    if e >= 9:
        assert (ref["k"] >= 9).sum() > 250 and (ref["k"] == e).sum() > 5
    if e == 15:
        # the 16-byte rows carry the same k, strand and record
        h = rlib.Handle(totalkmax=15, scores=scores, ll_table=ll)
        try:
            h.set_reads(reads.mapped, reads.offsets, reads.quality)
            w, m = text.packed()
            h.set_text(w, m, text.n, text.record_starts)
            full = h.match_all()
            rows16 = h.match_all_packed()
        finally:
            h.close()
        for f in ("patid", "pos", "k", "inverted", "frag"):
            assert np.array_equal(rows16[f], full[f]), f
        assert np.array_equal(rows16["score"].view(np.uint32), full["score"].view(np.uint32))


def test_unique_e15_files_62_63_text_shards_exchange():
    """matchUnique at -e 15 over files 62 and 63, each cut into 3 text shards on 3 handles and folded through the exported
    keys (MIN, then SUM of ties): file 63 and k = 15 make the largest keys short of UNIQUE_KEY_NONE."""
    import torch
    t0 = repeat_rich_text(62, n=250_000, copies=6)
    t1 = repeat_rich_text(63, n=200_000, copies=6)
    sym = t1.symbols.copy()
    sym[5000:45000] = t0.symbols[30000:70000]             # cross-file repeats
    t1 = synth.Text(sym, t1.records)
    reads = synth.concat_reads([synth.make_reads(t0, 64, 2500, 150, 0.06, fastq=False),
                                synth.make_reads(t1, 65, 2000, 150, 0.06, fastq=False)])
    files = (62, 63)
    ref = oracle_run("unique", [t0, t1], reads, e=15, scores=False, fileids=list(files))[0]
    G = 3
    hs = [rlib.Handle(totalkmax=15) for _ in range(G)]
    try:
        for h in hs:
            h.set_reads(reads.mapped, reads.offsets)
        dev = torch.device("cuda", 0)
        for fi, t in zip(files, (t0, t1)):
            w, m = t.packed()
            shards = matcher.shard_ranges(t.n, G, 150)
            keys = [torch.empty(reads.nreads, dtype=torch.int64, device=dev) for _ in range(G)]
            ties = [torch.empty(reads.nreads, dtype=torch.uint8, device=dev) for _ in range(G)]
            for g, h in enumerate(hs):
                _set_text(h, t, fi, shards[g], w, m)
                h.match_unique()
                h.unique_export_keys(keys[g].data_ptr())
            kmin = torch.stack(keys).min(dim=0).values.contiguous()
            for g, h in enumerate(hs):
                h.unique_export_ties(kmin.data_ptr(), ties[g].data_ptr())
            tsum = torch.stack(ties).sum(dim=0).to(torch.uint8).contiguous()
            torch.cuda.synchronize()
            for h in hs:
                h.unique_import(kmin.data_ptr(), tsum.data_ptr())
        infos = [h.get_unique()[0] for h in hs]
    finally:
        for h in hs:
            h.close()
    st, fl, k = matcher.umi_state(ref), matcher.umi_file(ref), matcher.umi_err(ref)
    one = (st == 1) | (st == 2)
    assert (one & (fl == 62)).sum() > 500 and (one & (fl == 63)).sum() > 500 and (st == 4).sum() > 20
    assert (one & (fl == 63) & (k >= 12)).sum() > 5
    want = matcher.canonical_unique(ref)
    for info in infos:
        assert np.array_equal(matcher.canonical_unique(info), want)


# ------------------------------------------------------------------ 3. folded tables

@pytest.mark.parametrize("seedl,table_bits", [(32, 12), (32, 13), (32, 16), (20, 32)])
def test_folded_tables(seedl, table_bits):
    """20000 reads put ~120000 entries into 2^12..2^16 slots (long entry chains); 32 slot bits for a 20-bit key is wider
    than the key."""
    text = repeat_rich_text(400 + table_bits, n=300_000, copies=8)
    reads = with_qualities(synth.make_reads(text, 401 + table_bits, 20_000, 80, 0.02, fastq=True), "illumina", table_bits)
    ll = O.build_ll()
    ref = oracle_run("all", [text], reads, seedl=seedl, e=4, ll=ll)
    got = gpu_run("all", [text], reads, seedl=seedl, e=4, ll=ll, table_bits=table_bits)
    same_rows(got, ref, reads.nreads // 2)
    ref = oracle_run("unique", [text], reads, seedl=seedl, e=4, ll=ll)
    got = gpu_run("unique", [text], reads, seedl=seedl, e=4, ll=ll, table_bits=table_bits)
    same_unique(got, ref, True)
    assert (matcher.umi_state(ref[0]) == 4).sum() > 100


# ------------------------------------------------------------------ 4. read lengths

@pytest.mark.parametrize("how", ["bytes", "packed", "device"])
def test_read_lengths_straddling_every_boundary(how):
    """Byte reads of more than 2048 bases are packed by k_pack_reads + k_read_seeds instead of k_pack_both; verification
    and scoring loop over up to 2047 words; 2 bit/base reads are read in place."""
    e = 6
    text, reads = long_read_case(500, e)
    lens = np.diff(reads.offsets.astype(np.int64))
    ll = O.build_ll()
    ref = oracle_run("all", [text], reads, e=e, ll=ll)
    got = gpu_run("all", [text], reads, e=e, ll=ll, how=how)
    same_rows(got, ref, reads.nreads // 3)
    for L in (2049, 10_000, 65_535):                       # long reads on both strands reach the rows
        assert {int(x) for x in ref["inverted"][lens[ref["patid"].astype(np.int64)] == L]} == {0, 1}, L
    ref = oracle_run("gaps", [text], reads, e=e, ll=ll)
    got = gpu_run("gaps", [text], reads, e=e, ll=ll, how=how)
    same_unique(got, ref, True)
    same_gaps(got[2], ref[2], 0)
    st = matcher.umi_state(ref[0])
    assert ((st == 1) | (st == 2))[lens >= 2047].sum() >= 20


@pytest.mark.parametrize("L", [2048, 2049, 65_535])
def test_uniform_long_reads_2bit(L):
    """2 bit/base reads of one length (uniform_length), matchAll with scores and scored matchUnique."""
    rng = np.random.RandomState(L)
    text = synth.make_text(L, 150_000, nrecords=1)
    seqs, quals = [], []
    for i in range(6):
        p = rng.randint(0, text.n - L)
        r = text.symbols[p:p + L].copy()
        j = rng.choice(np.arange(32, L - 32), 1 + i, replace=False)
        r[j] = (r[j] + 1) & 3
        seqs.append(synth.revcomp_mapped(r) if i % 2 else r)
        quals.append(illumina_quality(rng, L))
    reads = synth.reads_from_list(seqs, quals)
    ll = O.build_ll()
    ref = oracle_run("all", [text], reads, e=6, ll=ll)
    same_rows(gpu_run("all", [text], reads, e=6, ll=ll, how="uniform"), ref, 6)
    ref = oracle_run("unique", [text], reads, e=6, ll=ll)
    same_unique(gpu_run("unique", [text], reads, e=6, ll=ll, how="uniform"), ref, True)


def test_byte_reads_longer_than_2048_bases_take_the_two_kernel_path():
    """Reads of 2049 bases (65 words) are packed by k_pack_reads, then k_read_seeds: one launch more than k_pack_both."""
    text = synth.make_text(77, 50_000)
    launches = {}
    for L in (2047, 2048, 2049):
        reads = synth.reads_from_list([text.symbols[100 * i:100 * i + L] for i in range(8)])
        h = rlib.Handle()
        try:
            h.set_reads(reads.mapped, reads.offsets)
            launches[L] = h.stats()["total_launches"]
        finally:
            h.close()
    assert launches[2047] == launches[2048] and launches[2049] == launches[2048] + 1, launches


def test_read_of_65536_bases_is_refused():
    import torch
    text = synth.make_text(78, 140_000)
    long = synth.reads_from_list([text.symbols[:65_536]])
    h = rlib.Handle()
    try:
        for how in ("bytes", "packed"):
            with pytest.raises(rlib.RealGpuError) as ei:
                _load_reads(h, long, how)
            assert ei.value.code == -4, how                  # REAL_GPU_E_LIMIT
        pk = np.zeros(16_384, np.uint8)
        with pytest.raises(rlib.RealGpuError) as ei:
            h.set_reads_packed(pk, 1, uniform_length=65_536)
        assert ei.value.code == -4
        dm = torch.from_numpy(long.mapped.copy()).cuda()
        doff = torch.from_numpy(long.offsets.astype(np.int64)).cuda()
        with pytest.raises(rlib.RealGpuError) as ei:
            h.set_reads_device(dm.data_ptr(), doff.data_ptr(), 1, 65_536, 65_536)
        assert ei.value.code == -4
        # 65535 bases are accepted and the handle still matches
        ok = synth.reads_from_list([text.symbols[1000:1000 + 65_535]])
        h.set_reads(ok.mapped, ok.offsets)
        w, m = text.packed()
        h.set_text(w, m, text.n, text.record_starts)
        rows = h.match_all()
        assert len(rows) == 1 and int(rows["pos"][0]) == 1000 and int(rows["k"][0]) == 0
    finally:
        h.close()


def test_format_all_long_read_lines():
    e = 6
    text, reads = long_read_case(501, e)
    ll = O.build_ll()
    ids = [("long_%d" % i).encode() for i in range(reads.nreads)]
    names = [b"chrA first", b"chrB", b"chrC"]
    h = rlib.Handle(totalkmax=e, scores=True, ll_table=ll)
    try:
        h.set_reads(reads.mapped, reads.offsets, reads.quality)
        w, m = text.packed()
        h.set_text(w, m, text.n, text.record_starts)
        rows = h.match_all()
        h.set_read_ids(ids)
        h.set_record_names(names, text.record_starts[:-1])
        first = len(rows) - 4                               # the rows of the longest reads come last
        got = h.format_all(first, 4)
    finally:
        h.close()
    lens = np.diff(reads.offsets.astype(np.int64))
    sel = rows[first:]
    assert lens[sel["patid"].astype(np.int64)].min() >= 10_000
    want = b"".join(line(ids[int(x["patid"])], read_bases(reads, int(x["patid"]), bool(x["inverted"])), x["score"],
                         int(lens[int(x["patid"])]), bool(x["inverted"]), names[int(x["frag"])],
                         int(x["pos"]) - int(text.record_starts[int(x["frag"])]) + 1, int(x["k"])) for x in sel)
    assert got == want


# ------------------------------------------------------------------ 5. quality strings

@pytest.mark.parametrize("kind", ["illumina", "phred93", "bytes"])
def test_quality_strings_match_all_scores(kind):
    text, reads = quality_case(600, kind, nper=800)
    ll = O.build_ll()
    ref = oracle_run("all", [text], reads, e=5, ll=ll)
    same_rows(gpu_run("all", [text], reads, e=5, ll=ll), ref, reads.nreads // 2)
    assert (ref["inverted"] == 1).sum() > 1000 and (ref["inverted"] == 0).sum() > 1000


@pytest.mark.parametrize("kind,filter_level,n_list", [("illumina", 1, 0), ("illumina", 2, 33_333), ("illumina", 3, 0),
                                                      ("illumina", 4, 70_000), ("phred93", 2, 0), ("phred93", 4, 45_000),
                                                      ("bytes", 1, 50_000), ("bytes", 3, 0)])
def test_quality_strings_scored_unique(kind, filter_level, n_list):
    """Scores that take many values: the epsilon test of the scored fold meets near-ties (NonUnique reads)."""
    text, reads = quality_case(610 + filter_level, kind)
    ll = O.build_ll()
    ref = oracle_run("unique", [text], reads, e=5, ll=ll, n_list=n_list, filter_level=filter_level)
    got = gpu_run("unique", [text], reads, e=5, ll=ll, n_list=n_list, filter_level=filter_level)
    assert (matcher.umi_state(ref[0]) == 4).sum() > 100
    same_unique(got, ref, True)


@pytest.mark.parametrize("kind,how", [("illumina", "bytes"), ("illumina", "packed"), ("bytes", "packed"), ("phred93", "bytes")])
def test_quality_strings_gapped_pass(kind, how):
    text, reads = quality_case(620, kind, nper=1000, sub=0.03)
    ll = O.build_ll()
    ref = oracle_run("gaps", [text], reads, e=2, ll=ll, n_list=60_000)
    got = gpu_run("gaps", [text], reads, e=2, ll=ll, n_list=60_000, how=how)
    assert (matcher.umi_state(ref[0]) == 3).sum() > 100
    same_unique(got, ref, True)
    same_gaps(got[2], ref[2], 100)
