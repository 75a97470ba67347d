"""Shared helpers of the test-suite: golden fixture loading and canonical forms."""
from __future__ import annotations

import dataclasses
import glob
import gzip
import json
import os

import numpy as np

from real_b200 import synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden_cases(prefix: str):
    return sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, prefix + "*.npz")))


class Case:
    def __init__(self, name: str):
        z = np.load(os.path.join(GOLDEN, name + ".npz"))
        self.name = name
        self.params = json.loads(str(z["params"]))
        nt = int(z["ntexts"])
        texts = []
        for i in range(nt):
            starts = z["text%d_starts" % i]
            sym = z["text%d_symbols" % i]
            texts.append(synth.Text(symbols=sym, records=[("rec%d" % j, int(s)) for j, s in enumerate(starts[:-1])]))
        # texts in the order the reference visited them; fileid = index in that order
        self.texts = [texts[i] for i in z["file_order"]]
        q = z["quality"] if int(z["has_quality"]) else None
        off = z["offsets"]
        self.reads = synth.Reads(mapped=z["mapped"], offsets=off, quality=q, ids=["r%d" % i for i in range(off.size - 1)])
        self.ref_hits = z["ref_hits"] if "ref_hits" in z.files else None
        self.ref_unique = z["ref_unique"] if "ref_unique" in z.files else None
        self.ref_gaps = z["ref_gaps"] if "ref_gaps" in z.files else None

    @property
    def match_args(self):
        p = self.params
        return dict(seedl=p["seedl"], seedkmax=p["seedkmax"], totalkmax=p["totalkmax"], scores=p["scores"])


def load_kat(name: str):
    with gzip.open(os.path.join(GOLDEN, name + ".json.gz"), "rt") as f:
        return json.load(f)


def canon_hits(h, with_block=False, with_score=True):
    """Rows (patid, [block], k, pos, file, frag, inverted, score bits), lexicographically sorted."""
    cols = [h["patid"].astype(np.int64)]
    if with_block:
        cols.append(h["block"].astype(np.int64))
    cols += [h["k"].astype(np.int64), h["pos"].astype(np.int64), h["file"].astype(np.int64), h["frag"].astype(np.int64),
             h["inverted"].astype(np.int64)]
    if with_score:
        cols.append(np.ascontiguousarray(h["score"]).view(np.uint32).astype(np.int64))
    a = np.stack(cols, 1) if len(h) else np.zeros((0, len(cols)), np.int64)
    return a[np.lexsort(a.T[::-1])]


def unify_order_ok(h) -> bool:
    """Rows of one read must come in (k,pos,file,frag,score,inverted) order (matchAllImplementation.cpp:122-136)."""
    if len(h) < 2:
        return True
    key = np.stack([h["patid"].astype(np.float64), h["k"].astype(np.float64), h["pos"].astype(np.float64), h["file"].astype(np.float64),
                    h["frag"].astype(np.float64), h["score"].astype(np.float64), h["inverted"].astype(np.float64)], 1)
    for i in range(1, len(key)):
        a, b = tuple(key[i - 1]), tuple(key[i])
        if a > b:
            return False
    return True


def fresh(seed, n=1_500_000, nreads=40_000, L=100, nrec=7, npm=1500, sub=0.012, fastq=True):
    """A random text with a 20 kbp repeat (reads with several hits) and genpat reads drawn from it."""
    text = synth.make_text(seed, n, nrecords=nrec, n_per_million=npm)
    sym = text.symbols.copy()
    sym[n // 2:n // 2 + 20000] = sym[1000:21000]          # a repeat => multi-hit reads
    text = synth.Text(sym, text.records)
    reads = synth.make_reads(text, seed + 1, nreads, L, sub, fastq=fastq)
    return text, reads


def need_big_gpu(gb, free_gb=0):
    """Skips the calling test unless device 0 has `gb` GB in all and, when given, `free_gb` GB free right now."""
    import pytest
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    if torch.cuda.get_device_properties(0).total_memory < gb * (1 << 30):
        pytest.skip("needs a GPU with %d GB" % gb)
    if free_gb and torch.cuda.mem_get_info(0)[0] < free_gb * (1 << 30):
        pytest.skip("needs %d GB of free device memory" % free_gb)


def line(idb, bases, score, L, inverted, name, pos1, k):
    """One output line of a hit as the reference prints it (read id, bases on the hit's strand, score, record name,
    1-based position in the record, errors)."""
    s = idb + b"\t" + bases + b"\t" + (("%g" % float(score)).encode() if score is not None else b"") + b"\t1\ta\t" + str(L).encode()
    return s + (b"\t-\t" if inverted else b"\t+\t") + name + b"\t" + str(pos1).encode() + b"\t\t" + str(k).encode() + b"\n"


def read_bases(reads, r, inverted):
    """The bases of read r as ACGTN text, reverse complemented for a '-' hit."""
    m = reads.read(r)
    if inverted:
        m = synth.revcomp_mapped(m)
    return bytes(b"ACGTN"[int(x)] for x in m)


def text_quirk_cases():
    """[(name, fasta bytes, symbols, starts incl. terminal, [names])] of tests/golden/text_quirks.npz (the reference's own getText)."""
    z = np.load(os.path.join(GOLDEN, "text_quirks.npz"))
    out = []
    for name in bytes(z["cases"]).decode().split("\n"):
        nrec = int(z[name + "_nrecords"])
        names = bytes(z[name + "_names"]).split(b"\n") if nrec else []
        assert len(names) == nrec
        out.append((name, bytes(z[name + "_fasta"]), z[name + "_symbols"], z[name + "_starts"], names))
    return out


# ------------------------------------------------------------------ brute force and the edge text

def record_index(starts, p):
    """Record of text position p (the last record start <= p); -1 in front of the first record."""
    return int(np.searchsorted(np.asarray(starts, np.int64), p, "right")) - 1


def window_ok(sym, starts, p, L):
    """[p, p+L) lies inside one record and holds no N."""
    starts = np.asarray(starts, np.int64)
    if p < starts[0] or p + L > sym.size:
        return False
    rec = record_index(starts, p)
    return p + L <= starts[rec + 1] and not (sym[p:p + L] > 3).any()


def brute_match_all(text, reads, seedl, s, e, ll):
    """matchAll restated over every window of the text: a seed of at most s mismatches, the whole read of at most e, inside
    one record (never in front of the first one) and free of N.  The seed mismatches of all windows come from one matrix
    product of one-hot codes (an N matches nothing).  Scores are added in float64 in window order, then cast to float32.
    Rows as util.canon_hits makes them (file 0)."""
    sym = text.symbols
    n = text.n
    starts = text.record_starts.astype(np.int64)
    cum_n = np.concatenate([[0], np.cumsum(sym > 3)])
    onehot = np.zeros((n, 4), np.float32)
    ok = sym < 4
    onehot[np.nonzero(ok)[0], sym[ok]] = 1
    rows = []
    if n < seedl:
        return np.zeros((0, 7), np.int64)
    win = np.lib.stride_tricks.sliding_window_view(onehot, (seedl, 4)).reshape(n - seedl + 1, seedl * 4)
    cands = []                                            # (read, strand, fwd bases, seed offset in the window)
    for r in range(reads.nreads):
        rd = reads.read(r)
        if len(rd) < seedl or len(rd) > n or (rd > 3).any():
            continue
        for inv in (0, 1):
            fwd = synth.revcomp_mapped(rd) if inv else rd
            cands.append((r, inv, fwd, len(rd) - seedl if inv else 0))
    for c0 in range(0, len(cands), 512):
        part = cands[c0:c0 + 512]
        q = np.zeros((len(part), seedl, 4), np.float32)
        for i, (_, _, fwd, sa) in enumerate(part):
            q[i, np.arange(seedl), fwd[sa:sa + seedl]] = 1
        seedk = seedl - np.rint(win @ q.reshape(len(part), -1).T).astype(np.int32)   # (seed window, candidate)
        for ws, i in zip(*np.nonzero(seedk <= s)):
            r, inv, fwd, sa = part[i]
            L = len(fwd)
            p = int(ws) - sa
            if p < starts[0] or p + L > n or cum_n[p + L] != cum_n[p]:
                continue
            rec = record_index(starts, p)
            if p + L > starts[rec + 1]:
                continue
            w = sym[p:p + L]
            k = int((w != fwd).sum())
            if k > e:
                continue
            qq = reads.qual(r)[::-1] if inv else reads.qual(r)
            idx = ((w.astype(np.int64) << 8) | (fwd.astype(np.int64) << 6) | qq) & 1023
            raw = 1.0
            for v in ll[idx].tolist():                    # in window order, as the reference adds them
                raw += v
            rows.append((r, k, p, 0, rec, inv, int(np.float32(raw).view(np.uint32))))
    a = np.asarray(rows, dtype=np.int64).reshape(-1, 7)
    return a[np.lexsort(a.T[::-1])]


def valid_window_starts(sym, seedl):
    """Every start p of a seed window [p, p+seedl) inside the text and free of N, by testing each window."""
    if sym.size < seedl:
        return np.zeros(0, np.int64)
    bad = np.lib.stride_tricks.sliding_window_view(sym > 3, seedl).any(axis=1)
    return np.nonzero(~bad)[0].astype(np.int64)


def block_bounds_ref(sym, seedl, n_list):
    """First window position of every reference text block of n_list windows (block 0 starts at 0)."""
    w = valid_window_starts(sym, seedl)
    nb = -(-w.size // n_list) if (n_list and w.size) else 1
    if nb <= 1:
        return np.zeros(1, np.uint64)
    b = w[np.arange(nb) * n_list]
    b[0] = 0
    return b.astype(np.uint64)


@dataclasses.dataclass
class CodedText(synth.Text):
    """A text that stores the given 2-bit code under every base, under its N positions too."""
    codes: np.ndarray = None

    def packed(self):
        words, _ = synth.pack_text(self.codes)
        _, nmask = synth.pack_text(self.symbols)
        return words, nmask


EDGE_NRUN_LENS = (1, 2, 3, 31, 32, 33, 63, 64, 65, 127, 128, 129)
EDGE_KINDS = ("nrun_start", "nrun_end", "rec_end", "rec_start")
PLAN_DTYPE = np.dtype([("read", "<i8"), ("kind", "<i4"), ("b", "<i8"), ("p", "<i8"), ("L", "<i4"), ("inv", "<i4"),
                       ("nsub", "<i4"), ("expect", "?")])
GAP_PLAN_DTYPE = np.dtype([("read", "<i8"), ("p", "<i8"), ("n", "<i8"), ("nat", "<i8")])


@dataclasses.dataclass
class EdgeCase:
    text: synth.Text              # N stored as A, like AutoTextArray
    text_random: CodedText        # the same text with random codes under its N
    reads: synth.Reads            # boundary reads, then the gapped-pass reads
    plan: np.ndarray              # PLAN_DTYPE, one row per boundary read
    gap_plan: np.ndarray          # GAP_PLAN_DTYPE: seed window p, DP length n, N at p+seedl+nat (-1: none)
    runs: np.ndarray              # (start, length) of every N run
    seedl: int
    gap_len: int


def illumina_like(rng, L):
    return rng.randint(2, 42, L).astype(np.uint8)


def edge_case(seed, full=False, seedl=32, lengths=(60, 100, 120, 0), gap_len=100):
    """A text whose N runs and records sit at every offset, and reads planted against every boundary.

    - N runs: `full` has single Ns at all 64 residues mod 64 and runs of every length of EDGE_NRUN_LENS starting at every
      residue; otherwise 128 runs of the lengths of EDGE_NRUN_LENS in turn, 64 of them starting at every residue and 64
      ending at every residue.  Runs are more than twice the longest read apart.  The text starts and ends with N, and
      N runs touch record starts and ends.
    - Records: lengths 0, 1, seedl-1, seedl, seedl+1, L-1, L, L+1, 2L+seedl-1, 2L+seedl, 2L+seedl+1 (L = 100) between
      random ones whose lengths put record starts at every residue; runs of 2 and 3 empty records; an empty last record.
      About 3300 records with `full`, 380 without.
    - Boundary reads: for every N run start a, windows whose last base is a-1, a, a+1; for every run end b (first base
      after the run) and record start b, windows that start at b-1, b, b+1; for every record end b, windows whose last
      base is b-1, b, b+1.  Each is planted with 0..2 substitutions outside the seed, on both strands with `full`,
      else on one in turn; read lengths cycle through `lengths` (0 = random in seedl..150, seedl..120 without `full`),
      with a quality per base.
    - Gapped-pass reads (forward strand, gap_len bases): a 1..3 base deletion seedl+4.. bases into the read, seed window
      at p with the DP window [p+seedl, p+seedl+n) ending at a record end (n = 0..4, m-4..m+4, 2L-1, 2L, and more than
      2L) or with n = 2L and an N at p+seedl+nat (nat = 0, 1, 2, 63, 64, 2L-2, 2L-1: inside; 2L, 2L+1: outside)."""
    rng = np.random.RandomState(seed)
    L = 100
    lmax = max(max(lengths), gap_len, 150 if full else 120)
    spacing = 2 * lmax + 8
    codes, isn, starts, runs = [], [], [], []
    pos = [0]

    def put(k, n_run=False):
        codes.append(rng.randint(0, 4, k).astype(np.uint8))
        isn.append(np.full(k, n_run))
        if n_run and k:
            runs.append((pos[0], k))
        pos[0] += k

    def pad_to(res, extra):
        put(extra + (res - (pos[0] + extra)) % 64)

    # part A: the N runs, in one record that starts with N
    starts.append(0)
    put(3, True)
    specs = ([(1, r) for r in range(64)] + [(ln, r) for ln in EDGE_NRUN_LENS for r in range(64)]) if full else \
        [(EDGE_NRUN_LENS[i % 12], i) for i in range(64)] + [(EDGE_NRUN_LENS[i % 12], i - EDGE_NRUN_LENS[i % 12] + 1) for i in range(64)]
    for ln, r in specs:
        pad_to(r % 64, spacing + rng.randint(0, 64))
        put(ln, True)
    put(spacing)

    # part C: records that end the gapped pass's DP window, or hold an N in it
    m = gap_len - seedl
    gaps = []
    for nn in [0, 1, 2, 3, 4] + list(range(m - 4, m + 5)) + [2 * gap_len - 1, 2 * gap_len, 2 * gap_len + 1, 2 * gap_len + 9]:
        starts.append(pos[0])
        put(150 + rng.randint(0, 64))
        gaps.append((pos[0], min(nn, 2 * gap_len), -1))
        put(seedl + nn)
    for nat in (0, 1, 2, 63, 64, 2 * gap_len - 2, 2 * gap_len - 1, 2 * gap_len, 2 * gap_len + 1):
        starts.append(pos[0])
        put(150 + rng.randint(0, 64))
        gaps.append((pos[0], 2 * gap_len, nat))
        put(seedl + nat)
        put(1, True)
        put(2 * gap_len + 40 - nat)

    # part B: records of every length, starts at every residue
    special = [0, 1, seedl - 1, seedl, seedl + 1, L - 1, L, L + 1, 2 * L + seedl - 1, 2 * L + seedl, 2 * L + seedl + 1]
    nunits = 600 if full else 64
    rmax = 4000 if full else 300
    for u in range(nunits):
        starts.append(pos[0])
        if u % 4 == 1:
            put((1, 33, 64, 2, 65)[u % 5], True)                  # N run at the record's first base
        pad_to(u % 64, rng.randint(200, rmax))
        if u % 4 == 3:
            put((1, 33, 64, 2, 65)[u % 5], True)                  # N run at the record's last base
        for j in range(4):
            starts.append(pos[0])
            put(special[(4 * u + j) % len(special)])
        if u % 7 == 3:
            starts += [pos[0]] * (2 + u % 2)                     # 2 or 3 empty records in a row
            starts.append(pos[0])
            put(rng.randint(300, 600))
    starts.append(pos[0])
    put(300)
    put(5, True)                                                  # the last base is N
    starts.append(pos[0])                                         # an empty last record
    cod = np.concatenate(codes)
    nflag = np.concatenate(isn)
    sym = np.where(nflag, 4, cod).astype(np.uint8)
    n = sym.size
    clean = np.where(nflag, 0, cod).astype(np.uint8)              # what a packed text stores under N
    recs = [(" edge_rec%d" % i, int(s)) for i, s in enumerate(starts)]
    text = synth.Text(sym, recs)
    text_random = CodedText(sym, recs, codes=cod)
    st = np.asarray(starts + [n], np.int64)

    # boundary reads
    seqs, quals, plan = [], [], []
    cnt = [0]

    def plant(kind, b, start=None, last=None):
        """one window [p, p+Lr) that starts at `start` or has its last base at `last`, on both strands"""
        Lr = lengths[cnt[0] % len(lengths)] or rng.randint(seedl, lmax + 1)
        cnt[0] += 1
        p = start if start is not None else last - Lr + 1
        if p < 0 or p + Lr > n:
            return
        for inv in ((0, 1) if full else ((cnt[0] // 2) % 2,)):
            w = clean[p:p + Lr].copy()
            nsub = min((cnt[0] + inv) % 3, Lr - seedl)
            sa = Lr - seedl if inv else 0
            rest = np.setdiff1d(np.arange(Lr), np.arange(sa, sa + seedl))
            for j in rng.choice(rest, nsub, replace=False):
                w[j] = (w[j] + 1 + rng.randint(0, 3)) & 3
            seqs.append(synth.revcomp_mapped(w) if inv else w)
            quals.append(illumina_like(rng, Lr))
            plan.append((len(seqs) - 1, kind, b, p, Lr, inv, nsub, Lr >= seedl and window_ok(sym, st, p, Lr)))

    for a, ln in runs:
        for d in (-1, 0, 1):
            plant(0, a, last=a + d)
            plant(1, a + ln, start=a + ln + d)
    for b in np.unique(st[1:]):
        for d in (-1, 0, 1):
            plant(2, int(b), last=int(b) + d)
            plant(3, int(b), start=int(b) + d)

    # gapped-pass reads
    gplan = []
    for i, (p, nn, nat) in enumerate(gaps):
        off, g = seedl + 4 + i % 20, 1 + i % 3
        r = np.concatenate([clean[p:p + off], clean[p + off + g:p + gap_len + g]])
        seqs.append(r)
        quals.append(illumina_like(rng, gap_len))
        gplan.append((len(seqs) - 1, p, nn, nat))
    reads = synth.reads_from_list(seqs, quals)
    return EdgeCase(text=text, text_random=text_random, reads=reads, plan=np.array(plan, dtype=PLAN_DTYPE),
                    gap_plan=np.array(gplan, dtype=GAP_PLAN_DTYPE), runs=np.asarray(runs, np.int64).reshape(-1, 2),
                    seedl=seedl, gap_len=gap_len)
