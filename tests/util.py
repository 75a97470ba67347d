"""Shared helpers of the test-suite: golden fixture loading and canonical forms."""
from __future__ import annotations

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
