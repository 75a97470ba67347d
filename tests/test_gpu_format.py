"""K8, the output lines formatted on the device (csrc/format.cuh), through the C ABI: the bytes of real_gpu_format_all /
real_gpu_format_unique against lines assembled here from the rows / state words the same handle reports (which the
parity tests pin to the reference), and the score formatter against printf's %g."""
import numpy as np
import pytest

from real_b200 import lib as rlib, matcher, synth
from util import line as _line, read_bases as _bases

pytestmark = pytest.mark.gpu


def test_score_formatter_equals_printf_g():
    rng = np.random.default_rng(7)
    bits = rng.integers(0, 2**32, size=400_000, dtype=np.uint64).astype(np.uint32)
    vals = [bits.view(np.float32)]
    vals.append((rng.random(200_000) * 700 - 600).astype(np.float32))                   # where scores live
    e = np.arange(-45, 39)
    p10 = (10.0 ** e.astype(np.float64))
    for f in (1.0, 9.999995, 9.9999949, 1.2345650, 1.2345649, 0.99999949, 0.9999995):
        vals.append((p10 * f).astype(np.float32))
    vals.append(np.asarray([0.0, -0.0, np.inf, -np.inf, 1.0, -1.0, 100000.0, 999999.0, 1000000.0, 999999.5, 0.0001, 0.00001, 123456.5, 1e-45], dtype=np.float32))
    v = np.concatenate(vals)
    v = v[~np.isnan(v)]
    got = rlib.selftest_format_scores(v)
    want = [("%g" % float(x)).encode() for x in v]
    bad = [(float(x), g, w) for x, g, w in zip(v, got, want) if g != w]
    assert not bad, bad[:10]


@pytest.mark.parametrize("scores", [False, True])
def test_format_all_lines(scores):
    text = synth.make_text(11, 300_000, nrecords=5, n_per_million=500)
    reads = synth.make_reads(text, 12, 6000, 75, 0.02, fastq=scores)
    ids = [("read_%d/x y" % (i * 7919 % 100003)).encode() + b"#" * (i % 41) for i in range(reads.nreads)]
    names = [("chr%d some description %s" % (i, "z" * (i * 13))).encode() for i in range(len(text.record_starts) - 1)]
    ll = matcher.scoring_table()
    h = rlib.Handle(totalkmax=4, scores=scores, ll_table=ll if scores else None)
    try:
        h.set_reads(reads.mapped, reads.offsets, reads.quality if scores else None)
        words, nmask = text.packed()
        h.set_text(words, nmask, text.n, text.record_starts)
        rows = h.match_all()
        assert len(rows) > 4000
        # the compact rows are the same rows
        rows16 = h.match_all_packed()
        for f in ("patid", "pos", "frag", "k", "inverted"):
            assert np.array_equal(rows16[f], rows[f]), f
        assert np.array_equal(rows16["score"].view(np.uint32), rows["score"].view(np.uint32))
        h.set_read_ids(ids)
        h.set_record_names(names, text.record_starts[:-1])
        want = [_line(ids[int(x["patid"])], _bases(reads, int(x["patid"]), bool(x["inverted"])), x["score"] if scores else None, 75, bool(x["inverted"]),
                      names[int(x["frag"])], int(x["pos"]) - int(text.record_starts[int(x["frag"])]) + 1, int(x["k"])) for x in rows]
        got = b"".join(h.format_all(a, min(1500, len(rows) - a)) for a in range(0, len(rows), 1500))
        assert got == b"".join(want)
        assert h.format_all(len(rows), 0) == b""
    finally:
        h.close()


@pytest.mark.parametrize("scores", [False, True])
def test_format_unique_lines(scores):
    texts = [synth.make_text(21 + f, 150_000 + 1000 * f, nrecords=3 + f, n_per_million=300) for f in range(2)]
    parts = [synth.make_reads(t, 30 + f, 2500, 60 + 20 * f, 0.01, fastq=scores) for f, t in enumerate(texts)]
    reads = synth.concat_reads(parts)
    ids = [("q%d" % i).encode() for i in range(reads.nreads)]
    ll = matcher.scoring_table()
    h = rlib.Handle(totalkmax=3, scores=scores, ll_table=ll if scores else None)
    try:
        h.set_reads(reads.mapped, reads.offsets, reads.quality if scores else None)
        names = []
        for f, t in enumerate(texts):
            w, m = t.packed()
            h.set_text(w, m, t.n, t.record_starts, fileid=f)
            h.match_unique()
            names.append([("f%d_r%d" % (f, i)).encode() for i in range(len(t.record_starts) - 1)])
            h.set_record_names(names[f], t.record_starts[:-1], fileid=f)
        info = np.zeros(reads.nreads, dtype=np.uint64)
        sc = np.zeros(reads.nreads, dtype=np.float32)
        h._check(h.L.real_gpu_get_unique(h.h, info.ctypes.data, sc.ctypes.data))
        h.set_read_ids(ids)
        want, nl = [], 0
        for r in range(reads.nreads):
            d = int(info[r]); st = d >> 61
            if st not in (1, 2):
                continue
            f, frag, k, pos = (d >> 35) & 63, (d >> 45) & 0xFFFF, (d >> 41) & 15, d & ((1 << 35) - 1)
            L = int(reads.offsets[r + 1] - reads.offsets[r])
            want.append(_line(ids[r], _bases(reads, r, st == 2), sc[r] if scores else None, L, st == 2, names[f][frag], pos - int(texts[f].record_starts[frag]) + 1, k))
            nl += 1
        assert nl > 3000
        got, gl = h.format_unique()
        assert gl == nl and got == b"".join(want)
        # a sub-range, with only its ids set
        h.set_read_ids(ids[1000:3000], first=1000)
        got2, _ = h.format_unique(1000, 2000)
        assert got2 in got and len(got2) > 0
        with pytest.raises(rlib.RealGpuError):
            h.format_unique(0, 10)
    finally:
        h.close()
