#!/usr/bin/env python
"""Benchmark of the matching hot path (BASELINE.json): reads/s and text Gbp/s.

    python bench.py --gpus N --steps K --warmup W [--workload c3|c2|c1|tiny] [--impl reference] [--dump-outputs DIR]

A step = one pass of the hot path over the synthetic workload: read packing + read-side signature
index build (K1+K2), text scan with probe/verify (K3), result reduction (and, for N>1, the one
cross-shard exchange of matchUnique).  N>1 (default --parallel buckets): the signature space is
sharded -- every rank indexes and probes 1/N of the scan buckets against the whole text, no record
exchange (DESIGN.md 5); total work is fixed as N grows ("strong").

`value`  : whole-job reads/s with inputs resident in HBM (device pointers through the C ABI).
`e2e`    : the same from pinned host buffers (H2D of text + 2-bit reads and D2H of the per-read
           results inside the timed region); N=1 through the host-pointer C ABI, N>1 every rank
           uploads 1/N of the bytes and NCCL all-gathers the rest over NVLink.
`roofline`: the text-scan kernels against the measured HBM peak, algorithmic bytes per SURVEY 8(d);
           `traffic` = DRAM bytes of the committed ncu capture (profiles/r02_kernels_c3.json), `hbm_traffic_frac` what
           that is of the HBM peak over the measured scan time, `l1tex` the bound the probe kernel runs against
           (scattered loads out of L2), `kernels` the per-kernel table of the capture.
`cpu_baseline` / --impl reference: the reference's own CPU code (oracle/_ref/ref_harness, compiled
from the reference sources) on a bounded sample, extrapolated linearly to the workload.
`ingest` : (N=1, an extra outside the timed step) K0, the FASTA text loader on the device, on a 260 MB
           file held in HBM: device time, file GB/s, HBM fraction, parity of the packed words.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: text bases, reads, read length, -e, mode, scores, substitution rate, records, N per million
    "c3": dict(n=3_100_000_000, reads=50_000_000, L=100, e=4, mode="unique", scores=False, sub=0.01, nrec=24, npm=1000,
               desc="C3: synthetic 3.1 Gbp genome (24 records, 0.1% N), 50M x 100bp reads, matchUnique -s 2 -e 4 -l 32 -q 0"),
    "c2": dict(n=250_000_000, reads=10_000_000, L=100, e=4, mode="all", scores=True, sub=0.01, nrec=1, npm=0,
               desc="C2: synthetic 250 Mbp chromosome, 10M x 100bp FastQ reads, matchAll -e 4 with ComputeScore"),
    "c1": dict(n=10_000_000, reads=1_000_000, L=36, e=2, mode="all", scores=False, sub=0.02, nrec=1, npm=0,
               desc="C1: 10 Mbp text, 1M x 36bp reads, matchAll -e 2, no scores"),
    "c5": dict(n=3_100_000_000, reads=20_000_000, L=250, e=8, mode="all", scores=False, sub=0.01, nrec=24, npm=1000,
               desc="C5: 3.1 Gbp genome, 20M x 250bp reads, matchAll -e 8"),
    "c4": dict(n=250_000_000, reads=5_000_000, L=150, e=3, mode="gaps", scores=True, sub=0.01, nrec=1, npm=0,
               desc="C4: synthetic 250 Mbp text, 5M x 150bp FastQ reads (30% of the '+' reads with one planted 1-3 base deletion), "
                    "matchUnique -e 3 with scores, then the gapped extension pass (matchGaps, MAXgap 3)"),
    "tiny": dict(n=20_000_000, reads=500_000, L=100, e=4, mode="unique", scores=False, sub=0.01, nrec=3, npm=1000,
                 desc="tiny: 20 Mbp, 500k x 100bp reads, matchUnique -e 4 (smoke-size)"),
}
SEED = 0x5EA1

# Digest of the result of one step, per workload, as the single-GPU run produces it (real_gpu_unique_checksum of the
# canonical unique state / matcher.hits_checksum of the matchAll rows).  The single-GPU run is gated on the reference
# (parity_checked) and property-checked at full size (tests/test_gpu_fullsize.py); a multi-GPU run must reproduce the digest.
EXPECTED_DIGEST = {
    "c3": 0xf32fdc56b7229760,
    "tiny": 0x70668eb87d6ea3c8,
}


def workload_config(wl: dict) -> dict:
    """The `config` object of the bench line: the same for both arms."""
    return {"workload": wl["desc"], "text_bases": wl["n"], "reads": wl["reads"], "read_len": wl["L"], "mode": wl["mode"], "scores": wl["scores"],
            "l2": "no flush between steps: every step streams inputs and tables far larger than the 126 MB L2 (text %.0f MB 2 bit/base, read set %.0f MB, "
                  "index tables and window records of several GB)" % (wl["n"] / 4 / 1e6, wl["reads"] * ((wl["L"] + 3) // 4) / 1e6)}


def record_starts(n: int, nrec: int):
    import numpy as np
    from real_b200 import synth
    if nrec <= 1:
        return np.asarray([0, n], dtype=np.uint64)
    cuts = sorted(set(int(x % np.uint64(n)) for x in synth.splitmix64(np.arange(nrec - 1, dtype=np.uint64) ^ synth.stream(SEED, 3))))
    return np.asarray([0] + [c for c in cuts if c > 0] + [n], dtype=np.uint64)


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------

class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        exe = shutil.which("nvidia-smi")
        if not exe:
            return
        try:
            self.proc = subprocess.Popen([exe, "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU reference leg
# ------------------------------------------------------------------------------------------------

_REF_SAMPLE = {}     # the sample's input files, written once per process and reused by every step of the reference arm


def cpu_reference(wl: dict, sample_text: int, sample_reads: int, threads: int) -> dict:
    """Times the reference's own CPU path (oracle/_ref/ref_harness: its index build per text block and its
    OpenMP matching region) on a bounded sample of the workload, and extrapolates linearly: index time
    with the text length, match time with reads x text blocks (one block assumed at full scale, which
    favours the CPU).  Falls back to the oracle port when the harness binary is absent."""
    import numpy as np
    from real_b200 import synth
    from oracle import oracle_py as O
    n_s = min(sample_text, wl["n"])
    r_s = min(sample_reads, wl["reads"])
    fastq = bool(wl["scores"])
    key = (wl["desc"], n_s, r_s)
    if key not in _REF_SAMPLE:
        text = synth.make_text(SEED, n_s, nrecords=min(wl["nrec"], 4), n_per_million=wl["npm"])
        if n_s >= 1_000_000:
            # a planted 20 kb repeat: reads with two placements (NonUnique words, multi-row reads) are part of what the gate compares
            sym = text.symbols.copy()
            sym[n_s // 2:n_s // 2 + 20_000] = sym[5000:25_000]
            text = synth.Text(sym, text.records)
        reads = synth.make_reads(text, SEED + 1, r_s, wl["L"], wl["sub"], fastq=fastq)
        if wl["mode"] == "gaps":
            synth.plant_deletions(text, reads, SEED + 1, wl["L"])
        work = None
        if O.have_ref():
            import atexit
            work = tempfile.mkdtemp(prefix="bench_ref_")
            atexit.register(shutil.rmtree, work, ignore_errors=True)
            synth.write_fasta(os.path.join(work, "t.fa"), text)
            synth.write_reads(os.path.join(work, "r.fq" if fastq else "r.fa"), reads, fastq)
        _REF_SAMPLE[key] = (text, reads, work)
    text, reads, work = _REF_SAMPLE[key]
    gaps = wl["mode"] == "gaps"
    unique = wl["mode"] != "all"
    result = {}
    if work is not None:
        if gaps:
            threads = 1            # the reference's gapped pass races on its gapinfos map with more than one thread (SURVEY 8d)
        rf = os.path.join(work, "r.fq" if fastq else "r.fa")
        args = ["-t", os.path.join(work, "t.fa"), "-p", rf, "-o", "x", "-u", "1" if unique else "0", "-R", "0",
                "-s", "2", "-e", str(wl["e"]), "-l", "32", "-q", "1" if wl["scores"] else "0", "-T", str(threads)]
        if fastq:
            args += ["-Q", "33"]
        if gaps:
            args += ["-g", "1"]
        # one reference text block for the sample (with scores the unique fold depends on the block boundaries)
        timing, dump, gdump = O.run_ref("unique" if unique else "all", work, args, gap_dump=gaps, env={"REAL_HARNESS_NLIST": str(n_s)}, threads=threads)
        index_s, match_s, kind = timing["index_s"], timing["match_s"], "reference"
        if unique:
            result["unique"] = np.fromfile(dump, dtype=O.UNIQUE_DTYPE)
            if gaps:
                result["gaps"] = np.fromfile(gdump, dtype=O.GAP_DTYPE)
                # the restatement on the same sample: it tells which reads the reference's gapped pass has no defined result for
                ll = O.build_ll()
                pi, ps = O.unique_init(reads.nreads, wl["scores"])
                O.match_unique(text, reads, pi, ps, totalkmax=wl["e"], scores=wl["scores"], ll=ll)
                pg = np.zeros(reads.nreads, dtype=O.GAP_DTYPE)
                und = np.zeros(reads.nreads, dtype=np.uint8)
                O.match_gaps(text, reads, pi, ps, pg, totalkmax=wl["e"], scores=wl["scores"], ll=ll, undefined=und)
                result["undefined"] = und
                result["port"] = {"data": pi, "score": ps, "gaps": pg[pg["present"] == 1]}
        else:
            result["hits"] = np.fromfile(dump, dtype=O.HIT_DTYPE)
    else:
        O.lib()
        t0 = time.perf_counter()
        if unique:
            info, sc = O.unique_init(reads.nreads, wl["scores"])
            O.match_unique(text, reads, info, sc, totalkmax=wl["e"], scores=wl["scores"])
            if gaps:
                g = np.zeros(reads.nreads, dtype=O.GAP_DTYPE)
                O.match_gaps(text, reads, info, sc, g, totalkmax=wl["e"], scores=wl["scores"])
                result["gaps"] = g[g["present"] == 1]
            u = np.zeros(reads.nreads, dtype=O.UNIQUE_DTYPE)
            u["data"] = info
            if sc is not None:
                u["score"] = sc
            result["unique"] = u
        else:
            result["hits"] = O.match_all(text, reads, totalkmax=wl["e"], scores=wl["scores"])
        index_s, match_s, kind, threads = 0.0, time.perf_counter() - t0, "port", 1
    full_s = index_s * (wl["n"] / n_s) + match_s * (wl["reads"] / r_s)
    return {"value": wl["reads"] / full_s, "unit": "reads/s", "cores": threads, "kind": kind, "_sample": (text, reads), "_result": result,
            "text_gbp_per_s": wl["n"] / full_s / 1e9,
            "sample": "%d bp text + %d reads of the workload: index build %.2f s, OpenMP matching region %.2f s; extrapolated linearly "
                      "(index x text length, matching x reads, one text block at full scale)" % (n_s, r_s, index_s, match_s),
            "sample_index_s": index_s, "sample_match_s": match_s, "extrapolated_full_s": full_s}


def table_bits_of(wl: dict) -> int:
    """log2 of the slots the library gives the presence tables of the FULL workload (about 32 slots per entry of the largest
    table, 2^20 .. 2^32): the gate runs its sample with the same geometry, so that it takes the same kernels as the timed step."""
    want = max(1, wl["reads"] * 2 * 3) * 32
    b = 20
    while b < 32 and (1 << b) < want:
        b += 1
    return b


def parity_gate(wl: dict, sample, result: dict) -> dict:
    """BASELINE.md 3: "match sets bit-exact vs the oracle harness on the same inputs before any timing counts".  Runs the GPU
    path on the very sample the CPU reference leg was timed on and compares with what the reference produced there:
    matchAll rows field for field (scores by bit pattern); matchUnique words -- Straight/Reverse words whole, NonUnique words
    by state and error count (the position a NonUnique word keeps is the first one the reference happened to visit; this
    path keeps the smallest) -- and with scores the words and score bits whole; gapped pass: words, score bits, GapInfo rows."""
    import numpy as np
    from real_b200 import matcher
    text, reads = sample
    gaps = wl["mode"] == "gaps"
    opts = matcher.RealOptions(totalkmax=wl["e"], scores=wl["scores"])
    opts.gaps = gaps
    words, nmask = text.packed()
    out = {"reads": int(reads.nreads), "text_bases": int(text.n), "table_bits": table_bits_of(wl)}
    if wl["mode"] == "all":
        m = matcher.AllMatcher(opts, table_bits=table_bits_of(wl))
        try:
            m.set_reads(reads.mapped, reads.offsets, reads.quality if wl["scores"] else None)
            m.set_text(words, nmask, text.n, text.record_starts)
            got = m.match()
        finally:
            m.close()
        ref = result["hits"]

        def canon(h):
            a = np.stack([h["patid"].astype(np.int64), h["k"].astype(np.int64), h["pos"].astype(np.int64), h["frag"].astype(np.int64),
                          h["inverted"].astype(np.int64), np.ascontiguousarray(h["score"]).view(np.uint32).astype(np.int64)], 1)
            return a[np.lexsort(a.T[::-1])]
        a, b = canon(got), canon(ref)
        out.update(rows=int(len(b)), ok=bool(a.shape == b.shape and np.array_equal(a, b)))
        return out
    m = matcher.UniqueMatcher(opts, table_bits=table_bits_of(wl))
    try:
        m.set_reads(reads.mapped, reads.offsets, reads.quality if wl["scores"] else None)
        m.handle.set_block_windows(0)
        m.set_text(words, nmask, text.n, text.record_starts)
        m.match()
        if gaps:
            m.matchGaps(0)
        info, sc = m.info()
        grows = m.gaps() if gaps else None
    finally:
        m.close()
    ref = result["unique"]
    defined = np.ones(reads.nreads, dtype=bool)
    if gaps and "undefined" in result:
        # The reference's gapped pass reads uninitialised locals when a seed candidate's band never reaches MINscore
        # (match.hpp:518-522; oracle/real_oracle.c gapped_dp): its result for such a read depends on what its stack held.
        # Those reads are compared with the restatement (which treats the candidate as "no gap found"), all others with
        # the reference itself.
        defined = result["undefined"] == 0
        out["reference_undefined_reads"] = int((~defined).sum())
        port = result["port"]
        port_ok = np.array_equal(info, port["data"]) and np.array_equal(sc.view(np.uint32), port["score"].view(np.uint32))
        pg = port["gaps"]
        gg = grows[grows["present"] == 1]
        port_ok = port_ok and len(gg) == len(pg) and all(np.array_equal(gg[f], pg[f]) for f in ("patid", "mingap", "where", "start", "gap_pos"))
        out["restatement_ok"] = bool(port_ok)
    if wl["scores"]:
        ok = np.array_equal(info[defined], ref["data"][defined]) and np.array_equal(sc.view(np.uint32)[defined], ref["score"].view(np.uint32)[defined])
    else:
        ok = np.array_equal(matcher.canonical_unique(info), matcher.canonical_unique(ref["data"]))
    st = matcher.umi_state(ref["data"])
    out.update(placed=int((st != 0).sum()), nonunique=int((st == 4).sum()), gapped=int((st == 3).sum()))
    if gaps:
        g, r = grows[grows["present"] == 1], result["gaps"]          # the harness dumps only the rows that exist (its last field is padding)
        out["words_ok"] = bool(ok)
        g = g[defined[g["patid"]]]
        r = r[defined[r["patid"]]]
        ok = ok and len(g) == len(r) and all(np.array_equal(g[f], r[f]) for f in ("patid", "mingap", "where", "start", "gap_pos"))
        out["gapinfo_rows"] = int(len(r))
        if "restatement_ok" in out:
            ok = ok and out["restatement_ok"]
    out["ok"] = bool(ok)
    return out


def run_reference_arm(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    # every execution runs the identical bounded sample from scratch (6-7 s): at most one warm-up and three timed
    # executions are made however large --steps is, and their mean is the line's value
    n_warm, n_timed = min(args.warmup, 1), max(1, min(args.steps, 3))
    vals = []
    last = None
    for i in range(n_warm + n_timed):
        last = cpu_reference(wl, args.ref_text, args.ref_reads, threads)
        if i >= n_warm:
            vals.append(last)
    v = statistics.mean(x["value"] for x in vals)
    full_s = statistics.mean(x["extrapolated_full_s"] for x in vals)
    line = {"impl": "reference", "metric": "matching-path reads/s", "value": v, "unit": "reads/s", "n_gpus": args.gpus, "steps": n_timed,
            "warmup": n_warm, "ms_per_step": full_s * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "u64", "data": "synthetic", "config": workload_config(wl),
            "executions": {"warmup": n_warm, "timed": n_timed, "note": "the sample is run from scratch each time; more repetitions would only repeat it"},
            "text_gbp_per_s": wl["n"] / full_s / 1e9,
            "cpu_baseline": {k: last[k] for k in ("kind", "cores", "sample")} | {"value": v, "unit": "reads/s"},
            "e2e": {"value": v, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


def kernel_table(workload: str, world: int, as_rank: str):
    """The committed per-kernel summary of an `ncu --set full` capture of one step of this workload on one GPU
    (profiles/r02_kernels_<workload>.json, made by tools/kernel_table.py; falls back to the round-1 traffic file), or None."""
    if world != 1 or as_rank:
        return None
    for name in ("r02_kernels_%s.json", "r01_traffic_%s.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name % workload)) as f:
                d = json.load(f)
            d["file"] = "profiles/" + name % workload
            return d
        except Exception:
            continue
    return None


# scattered loads served by L2: one distinct 128-byte line per cycle and SM through the L1TEX tag stage -- 277-281 G lines/s on
# this pool's B200 for resident sets up to ~96 MB (tools/l2_resident_bench.cu, profiles/r01_l2_resident_bench.txt)
L1TEX_LINES_PER_S = 280e9


DUMP_READS = 1 << 19          # --dump-outputs: reads of the fixed sample whose results are written
DUMP_BYTES = 60 << 20         # --dump-outputs: at most this many bytes of array data in all (below 64 MB with the file headers)


def dump_outputs(out_dir: str, h, R: int, unique: bool, gaps: bool) -> dict:
    """--dump-outputs: what the last timed step computed, as the caller of the matching path receives it, for the reads of a
    fixed seeded sample (the same for every run of a workload), so that two builds can be compared output for output.
    One field per file DIR/<name>.npy; integers as float64 (exact below 2^53), scores as float32.
    matchUnique: the UniqueMatchInfo fields of each sampled read (unique_*), the score with scores, the GapInfo rows of the
    sampled reads after the gapped pass (gaps_*).  matchAll: the real_gpu_hit16 rows the last step received for the sampled
    reads (hits_*), in the library's order, cut to the byte budget."""
    import numpy as np
    from real_b200 import matcher
    reads = np.sort(np.random.default_rng(SEED).choice(R, size=min(R, DUMP_READS), replace=False))
    f64 = lambda a: np.asarray(a).astype(np.float64)
    out = {}
    if unique:
        info, sc = h.get_unique()
        info = info[reads]
        out.update(unique_read=f64(reads), unique_state=f64(matcher.umi_state(info)), unique_pos=f64(matcher.umi_pos(info)),
                   unique_file=f64(matcher.umi_file(info)), unique_err=f64(matcher.umi_err(info)), unique_frag=f64(matcher.umi_frag(info)))
        if sc is not None:
            out["unique_score"] = sc[reads].astype(np.float32)
        if gaps:
            g = h.get_gaps()
            g = g[(g["present"] == 1) & np.isin(g["patid"], reads)]
            out.update({"gaps_" + k: f64(g[k]) for k in ("patid", "mingap", "where", "start", "gap_pos")})
    else:
        rows = h.last_rows_packed()
        rows = rows[np.isin(rows["patid"], reads)]
        fields = ("patid", "pos", "frag", "k", "inverted")         # a real_gpu_hit16 row has no file: the one the call matched against
        rows = rows[:DUMP_BYTES // (8 * len(fields) + 4)]
        out.update({"hits_" + k: f64(rows[k]) for k in fields})
        out["hits_score"] = np.ascontiguousarray(rows["score"]).astype(np.float32)
    nbytes = sum(a.nbytes for a in out.values())
    assert nbytes <= DUMP_BYTES, nbytes
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return {"dir": out_dir, "sampled_reads": int(reads.size), "files": len(out), "bytes": int(nbytes)}


def ingest_probe(torch, rlib, peak_gbs: float) -> dict:
    """K0, the FASTA text loader on the device (csrc/ingest.cuh), on a bounded synthetic file held in HBM: 256 Mbp in one record,
    60-column lines.  Device time of real_gpu_set_text_fasta_device (summary + scan + clear + pack, CUDA events on the library's
    stream), and the packed words it produced against the symbols the file was written from.  An extra of the bench line,
    not part of the timed step; tools/ingest_bench.py is the full-size measurement (profiles/r01_ingest_bench.txt)."""
    import numpy as np
    n = 480 * 533_333                                   # a multiple of the 60-column lines and of the 32-base words
    g = torch.Generator(device="cuda")
    g.manual_seed(SEED)
    sym = torch.randint(0, 4, (n,), device="cuda", dtype=torch.uint8, generator=g)
    lut = torch.tensor([65, 67, 71, 84], dtype=torch.uint8, device="cuda")
    rows = torch.empty((n // 60, 61), dtype=torch.uint8, device="cuda")
    rows[:, :60] = lut[sym.long()].reshape(-1, 60)
    rows[:, 60] = 10
    data = torch.cat([torch.frombuffer(bytearray(b"> bench_ingest\n"), dtype=torch.uint8).cuda(), rows.reshape(-1)])
    del rows
    h = rlib.Handle(seedl=32, seedkmax=2, totalkmax=4)
    try:
        ms = []
        for _ in range(5):
            nb, nrec = h.set_text_fasta(None, device_ptr=data.data_ptr(), nbytes=data.numel())
            ms.append(h.stats()["h2d_text_ms"])
        words, _ = h.get_text_packed(nb)
        starts, _ = h.get_text_records()
    finally:
        h.close()
    sh = 62 - 2 * torch.arange(32, device="cuda", dtype=torch.int64)
    want = (sym.long().reshape(-1, 32) << sh).sum(1).cpu().numpy()
    t = float(np.median(ms[2:]))
    alg = data.numel() + n * 3 / 8.0
    return {"kernel": "K0 text ingest: k_fa_summary + k_fa_scan + k_fa_pack", "file_bytes": int(data.numel()), "bases": int(nb), "records": int(nrec),
            "device_ms": t, "file_GBps": data.numel() / t / 1e6, "gbp_per_s": n / t / 1e6,
            "roofline": {"bound": "hbm", "achieved": alg / t / 1e6, "peak": peak_gbs, "unit": "GB/s", "frac": alg / t / 1e6 / peak_gbs,
                         "note": "algorithmic bytes = file bytes read once + 3/8 byte written per kept base; the kernels read the file twice"},
            "parity": bool(nb == n and nrec == 1 and list(starts) == [0, n] and np.array_equal(words.view(np.int64), want))}


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------

def bind_to_gpu_numa(torch, local: int) -> dict:
    """One process per GPU: run (and first-touch the pinned host buffers) on the CPUs of the NUMA node the GPU hangs on, so that
    the host<->device copies of the end-to-end leg do not cross the socket interconnect -- with eight ranks pulling their slices out
    of host memory at once that interconnect, not PCIe, was the bound.  Reads the GPU's PCI address from torch and its
    local_cpulist from sysfs; does nothing when either is not there."""
    info = {"bound": False}
    try:
        p = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        base = "/sys/bus/pci/devices/" + bdf
        with open(base + "/local_cpulist") as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(","):
            if not part:
                continue
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        node = None
        try:
            with open(base + "/numa_node") as f:
                node = int(f.read().strip())
        except Exception:
            pass
        info.update(pci=bdf, numa_node=node, cpus=len(cpus), allowed=len(allowed))
        if cpus and len(cpus) < len(allowed):
            os.sched_setaffinity(0, cpus)
            info["bound"] = True
    except Exception as e:          # no sysfs, no such property: stay where the launcher put us
        info["error"] = "%s: %s" % (type(e).__name__, e)
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--table-bits", type=int, default=0)
    ap.add_argument("--parallel", default="buckets", choices=["buckets", "tables", "text"],
                    help="N>1: 'buckets' = signature tables sharded by scan bucket, every rank reads the whole text and keeps the positions "
                         "of its own buckets, no record exchange (default); 'tables' = the same sharding with the window records exchanged "
                         "through peer memory; 'text' = text sharded with a read-length halo, index replicated on every rank")
    ap.add_argument("--round-mpos", type=int, default=0, help="sharded tables: text positions per round in units of 2^20 (0 = 2^30 positions)")
    ap.add_argument("--as-rank", default="", help="development: R/N = run on ONE GPU the work rank R of an N-rank bucket-sharded job does "
                                                  "(no exchange; for profiling a rank's kernels under ncu; not a reportable number)")
    ap.add_argument("--reads-format", default="packed", choices=["packed", "bytes"],
                    help="layout of the HBM-resident read set of the timed step: 'packed' = 2 bit/base, the reference's rewritten pattern file "
                         "(TemporaryFile.hpp:231-268; verified in place, only the seeds are extracted); 'bytes' = one mapped byte per base "
                         "(Pattern::mapped; packed into both strands by K1)")
    ap.add_argument("--fold", default="peer", choices=["peer", "nccl"],
                    help="N>1, matchUnique: 'peer' = the fold as one exchange over NVLink peer memory (real_gpu_fold_unique, reduce-scatter "
                         "form: every rank ends up with the merged state of its own 1/N of the reads); 'nccl' = MIN + SUM all-reduce "
                         "(real_b200.dist.unique_exchange: every rank ends up with the whole merged state)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-order", choices=["text-first", "reads-first"], default="text-first",
                    help="end-to-end leg: text-first = set_text_async, prepare_scan, set_reads, match (the partition of the text runs while "
                         "the reads cross PCIe); reads-first = set_reads, set_text_async, match")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true", help="N>1: do not bind the rank to the CPUs of its GPU's NUMA node")
    ap.add_argument("--no-ingest", action="store_true", help="skip the K0 (device text loader) extra of the bench line")
    ap.add_argument("--ref-text", type=int, default=32_000_000, help="reference arm: text bases of the sample")
    ap.add_argument("--ref-reads", type=int, default=500_000, help="reference arm: reads of the sample")
    ap.add_argument("--cpu-text", type=int, default=16_000_000)
    ap.add_argument("--cpu-reads", type=int, default=250_000)
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="one GPU: after the timed steps, write what the last step computed to DIR/<name>.npy (the results of a fixed "
                         "seeded sample of %d reads, at most %d MiB in all), for comparing two builds output for output"
                         % (DUMP_READS, DUMP_BYTES >> 20))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    wl = WORKLOADS[args.workload]
    if args.warmup < 3 and args.impl == "ours":
        print("note: fewer than 3 warm-up steps; not a reportable number", file=sys.stderr)

    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes what the GPU path computed: not with --impl reference")
        return run_reference_arm(args, wl)

    import numpy as np
    import torch
    import torch.distributed as dist
    from real_b200 import devsynth, matcher
    from real_b200 import dist as rdist
    from real_b200 import lib as rlib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the matching path has no CPU fallback")
    if args.dump_outputs and (world > 1 or args.as_rank):
        raise SystemExit("--dump-outputs: one GPU running the whole job only")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    affinity = bind_to_gpu_numa(torch, local) if (world > 1 and not args.no_numa_bind) else {"bound": False}
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    if args.gpus != world and rank == 0:
        print("note: --gpus %d but WORLD_SIZE %d; using WORLD_SIZE" % (args.gpus, world), file=sys.stderr)

    n, R, L = wl["n"], wl["reads"], wl["L"]
    unique = wl["mode"] in ("unique", "gaps")
    gaps = wl["mode"] == "gaps"
    if gaps and world > 1:
        raise SystemExit("the gapped pass is order dependent: one handle per job (replicas only, DESIGN.md 5)")
    rs = record_starts(n, wl["nrec"])
    tables_mode = world > 1 and args.parallel == "tables"
    buckets_mode = world > 1 and args.parallel == "buckets"
    ob, oe, sb, sl = (0, n, 0, n) if (tables_mode or buckets_mode or world == 1) else matcher.shard_ranges(n, world, L)[rank]

    # ---- synthetic inputs, generated on the device: this rank's text shard and the whole read set.
    # Reads are cut from the whole text, so they are generated from a transient full copy.
    full_w, full_m = devsynth.text_device(SEED, n, device=local, n_per_million=wl["npm"])
    mapped, qual, offs = devsynth.reads_device(SEED + 1, full_w, full_m if wl["npm"] else None, n, R, L, wl["sub"], device=local,
                                               quality=wl["scores"])
    if gaps:
        sym = devsynth.unpack_symbols(full_w, full_m, n)
        ppos, pstrand = devsynth.read_plan_device(SEED + 1, R, n - L + 1, dev)
        devsynth.plant_deletions(mapped, sym, ppos, pstrand, n, L)
        del sym, ppos, pstrand
    w0, w1 = sb // 32, (sb + sl + 31) // 32
    m0, m1 = sb // 64, (sb + sl + 63) // 64
    sh_w = full_w[w0:w1 + 2].clone()
    sh_m = full_m[m0:m1 + 2].clone()
    del full_w, full_m
    torch.cuda.empty_cache()

    ll = matcher.scoring_table() if (wl["scores"] or gaps) else None
    h = rlib.Handle(seedl=32, seedkmax=2, totalkmax=wl["e"], scores=wl["scores"], ll_table=ll, device=local, table_bits=args.table_bits)
    if tables_mode:
        rdist.connect_sharded_tables(h, dev, round_positions=args.round_mpos << 20)
    if buckets_mode:
        h.set_bucket_shard(rank, world)
    if args.as_rank:
        er, en = (int(x) for x in args.as_rank.split("/"))
        h.set_bucket_shard(er, en)
        print("note: --as-rank %d/%d: one rank's share of a bucket-sharded job; not a reportable number" % (er, en), file=sys.stderr)
    shard = rdist.HandleShard(h, R)
    peer_fold = world > 1 and unique and args.fold == "peer"
    if peer_fold:
        rdist.connect_fold(h, dev, R)
    keys = torch.empty(R, dtype=torch.int64, device=dev) if (unique and world > 1 and not peer_fold) else None
    ties = torch.empty(R, dtype=torch.uint8, device=dev) if (unique and world > 1 and not peer_fold) else None
    r_lo, r_hi = rdist.own_read_range(R, rank, world)

    def exchange():
        """The one cross-GPU step of matchUnique."""
        if peer_fold:
            h.fold_unique()
        else:
            rdist.unique_exchange(shard, keys=keys, ties=ties)
    hstream = torch.cuda.ExternalStream(h.stream(), device=dev)

    phase = {"pack_ms": [], "index_ms": [], "scan_ms": [], "probe_ms": [], "part_ms": [], "post_ms": [], "d2h_ms": [], "h2d_text_ms": [], "exchange_ms": [], "fold_ms": [],
             "gap_scan_ms": [], "gap_post_ms": [],
             "api_set_reads_ms": [], "api_set_text_ms": [], "api_match_ms": []}
    last_stats = {}
    nhits_holder = [0]

    def pack_2bit():
        """The read set 2 bit/base on the device (4 bases per byte, first base in bits 7..6) + per-read wildcard flags."""
        L4 = (L + 3) // 4
        m2 = mapped.view(R, L)
        if L % 4:
            m2 = torch.nn.functional.pad(m2, (0, 4 * L4 - L))
        m2 = (m2 & 3).view(R, L4, 4)
        d_packed = ((m2[:, :, 0] << 6) | (m2[:, :, 1] << 4) | (m2[:, :, 2] << 2) | m2[:, :, 3]).contiguous().view(-1)
        d_flags = (mapped.view(R, L) > 3).any(dim=1).to(torch.uint8)
        return d_packed, d_flags

    d_packed = d_flags = None
    if args.reads_format == "packed" or not args.no_e2e:
        d_packed, d_flags = pack_2bit()
        torch.cuda.synchronize()

    def step_device():
        t0 = time.perf_counter()
        if args.reads_format == "packed":
            h.set_reads_packed_device(d_packed.data_ptr(), R, L, d_wildcard_flags=d_flags.data_ptr(), d_quality=qual.data_ptr() if qual is not None else None)
        else:
            h.set_reads_device(mapped.data_ptr(), offs.data_ptr(), R, R * L, L, d_quality=qual.data_ptr() if qual is not None else None)
        t1 = time.perf_counter()
        h.set_text_device(sh_w.data_ptr(), sh_m.data_ptr(), n, rs, shard_begin=sb, shard_len=sl, own_begin=ob, own_end=oe)
        t2 = time.perf_counter()
        if unique:
            h.match_unique()
            t3 = time.perf_counter()
            st = h.stats()
            if gaps:
                h.match_gaps(0)
                g = h.stats()
                st["gap_scan_ms"], st["gap_post_ms"] = g["scan_ms"], g["post_ms"]
            if world > 1:
                exchange()
                st["fold_ms"] = h.stats()["fold_ms"]
            t4 = time.perf_counter()
        else:
            nhits_holder[0] = h.match_all_count(packed=True)          # rows read back as real_gpu_hit16
            t3 = t4 = time.perf_counter()
            st = h.stats()
        st["exchange_ms"] = (t4 - t3) * 1e3
        st["api_set_reads_ms"] = (t1 - t0) * 1e3
        st["api_set_text_ms"] = (t2 - t1) * 1e3
        st["api_match_ms"] = (t3 - t2) * 1e3
        return st

    def timed(fn, steps, warmup, collect=None):
        for _ in range(warmup):
            fn()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        launches0 = h.stats()["total_launches"]
        e0.record(hstream)
        for _ in range(steps):
            st = fn()
            if collect is not None:
                collect(st)
        e1.record(hstream)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), h.stats()["total_launches"] - launches0

    def collect(st):
        for k in phase:
            phase[k].append(st.get(k, 0.0))
        last_stats.update(st)

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    total_ms, launches = timed(step_device, args.steps, args.warmup, collect)
    clk = clocks.stop() if rank == 0 else {}
    ms_per_step = total_ms / args.steps
    value = R / (ms_per_step * 1e-3)
    # before anything else runs on the handle: it holds the result of the last timed step
    dumped = dump_outputs(args.dump_outputs, h, R, unique, gaps) if args.dump_outputs else None

    # ---- digest of the result of the last step (outside the timed region): must not depend on the number of GPUs
    def result_digest():
        if unique:
            if world > 1 and not peer_fold:
                part = h.unique_checksum(r_lo, r_hi - r_lo)          # every rank holds the whole merged state: digest the own share
            else:
                part = h.unique_checksum(r_lo, r_hi - r_lo) if world > 1 else h.unique_checksum()
        else:
            part = matcher.hits_checksum(h.match_all())
        if world > 1:
            parts = [None] * world
            dist.all_gather_object(parts, int(part))
            return sum(parts) & 0xFFFFFFFFFFFFFFFF
        return part & 0xFFFFFFFFFFFFFFFF

    digest = result_digest()
    expected = EXPECTED_DIGEST.get(args.workload)
    digest_ok = None if (expected is None or args.as_rank) else (digest == expected)

    # ---- roofline of the dominant kernel (K3 text scan), algorithmic bytes per SURVEY.md 8(d)
    # the scan = its partition kernels + its probe kernels.  The library starts the partition of a text as soon as the text is set
    # (on a stream of its own, beside the index build: DESIGN 4.9), so the window the scan call itself measures (scan_ms) may hold
    # the probe only: the roofline is taken on the SUM of the two kernel groups' own durations, which overlap makes longer, not shorter
    scan_call_ms = statistics.mean(phase["scan_ms"])
    scan_ms = max(scan_call_ms, statistics.mean(phase["part_ms"]) + statistics.mean(phase["probe_ms"]))
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    n_text_local = last_stats["n_windows"]
    nwin_tot = torch.tensor([last_stats["n_windows"], last_stats["n_candidates"], last_stats["n_hits"], last_stats["n_seedpass"]],
                            dtype=torch.float64, device=dev)
    alg_bytes = 0.375 * n_text_local + 192.0 * last_stats["n_windows"] + 64.0 * last_stats["n_candidates"] + 16.0 * last_stats["n_hits"]
    design_bytes = 0.375 * n_text_local + 32.0 * last_stats["n_probes"] + 64.0 * last_stats["n_candidates"] + 16.0 * last_stats["n_hits"]
    achieved = alg_bytes / (scan_ms * 1e-3) / 1e9
    ktab = kernel_table(args.workload, world, args.as_rank)
    traffic = float(ktab["scan_dram_bytes_per_step"]) if ktab else None
    probe_ms = statistics.mean(phase["probe_ms"]) if phase["probe_ms"] else 0.0
    # what the probe kernel pushes through the L1TEX tag stage: one line per probe, per entry followed, per 128 bytes of records
    lines = last_stats["n_probes"] + last_stats["n_candidates"] + last_stats["n_windows"] * 16.0 / 128.0
    roofline = {"bound": "hbm", "kernel": "k_bucket_probe (+k_part): text scan", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "peak_source": "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback",
                "traffic": traffic, "alg_bytes_per_launch": alg_bytes, "scan_ms": scan_ms, "scan_call_ms": scan_call_ms,
                "design_bytes_per_launch": design_bytes, "design_frac": design_bytes / (scan_ms * 1e-3) / 1e9 / peak,
                # the physical picture next to the contract's figure: DRAM bytes the scan kernels really moved (ncu) over the
                # measured scan time, as a fraction of the HBM peak
                "hbm_traffic_frac": (traffic / (scan_ms * 1e-3) / 1e9 / peak) if traffic else None,
                # the bound the design runs against: probes are scattered 8-byte loads served by L2
                "l1tex": {"bound": "L1TEX tag stage, one distinct 128-byte line per cycle and SM (scattered loads out of L2)",
                          "lines_per_step": lines, "probe_ms": probe_ms, "partition_ms": scan_ms - probe_ms,
                          "achieved_lines_per_s": (lines / (probe_ms * 1e-3)) if probe_ms else None, "peak_lines_per_s": L1TEX_LINES_PER_S,
                          "frac": (lines / (probe_ms * 1e-3) / L1TEX_LINES_PER_S) if probe_ms else None,
                          "peak_source": "tools/l2_resident_bench.cu on this pool (profiles/r01_l2_resident_bench.txt)"},
                "kernels": ({"file": ktab.get("file"), "source": ktab.get("source"),
                             "table": [{k: a.get(k) for k in ("kernel", "launches", "ms_under_ncu", "dram_read_bytes", "dram_write_bytes", "dram_GBps_under_ncu", "registers",
                                                              "warps_active_pct", "issue_active_pct", "busiest_unit", "unit_pct_of_peak", "l2_hit_rate_pct", "top_stalls")}
                                       for a in ktab.get("kernels", [])[:8]]} if ktab and "kernels" in ktab else None),
                "note": "alg bytes = 0.375*N_text + 6*32*N_win + 64*N_cand + 16*N_hit (SURVEY 8d, six lists); the kernel probes 3 merged "
                        "tables per window out of L2-resident slices (design bytes = 3*32*N_win + ...), so frac exceeds the sector-traffic "
                        "fraction: hbm_traffic_frac is what DRAM really carried, l1tex.frac is the bound the probe kernel runs against"}
    if world > 1:
        dist.all_reduce(nwin_tot, op=dist.ReduceOp.SUM)

    # ---- e2e: host buffers through the host-pointer ABI, H2D + D2H inside the timed region
    e2e = None
    if not args.no_e2e:
        try:
            # reads cross PCIe 2 bit/base, the layout of the reference's own rewritten pattern file (-R 1, the default of
            # matchUnique; TemporaryFile.hpp:231-268); qualities (only with scores) stay 1 byte/base
            L4 = (L + 3) // 4
            h_mapped = torch.empty(R * L4, dtype=torch.uint8).pin_memory()
            h_mapped.copy_(d_packed)
            h_flags = torch.empty(R, dtype=torch.uint8).pin_memory()
            h_flags.copy_(d_flags)
            del d_packed, d_flags
            torch.cuda.empty_cache()
            h_qual = None
            if qual is not None:
                h_qual = torch.empty(R * L, dtype=torch.uint8).pin_memory()
                h_qual.copy_(qual)
            h_w = sh_w.cpu().pin_memory()
            h_m = sh_m.cpu().pin_memory()
            h_info = torch.empty(R, dtype=torch.int64).pin_memory()
            np_w = h_w.numpy().view(np.uint64)
            np_m = h_m.numpy().view(np.uint64)
            np_mapped = h_mapped.numpy()
            np_flags = h_flags.numpy()
            np_qual = h_qual.numpy() if h_qual is not None else None
            np_info = h_info.numpy().view(np.uint64)
            d2h = [0]

            # N > 1 with replicated inputs (bucket shards): every rank uploads 1/N of the input bytes from its pinned host copy and
            # the ranks all-gather them over NVLink, instead of every rank pulling everything through its own PCIe link
            gather = None
            if world > 1 and (buckets_mode or tables_mode):
                sections = [("reads", h_mapped), ("flags", h_flags)]
                if h_qual is not None:
                    sections.append(("qual", h_qual))
                gather = rdist.ShardedUpload(sections, dev)
                gather_text = rdist.ShardedUpload([("words", h_w.view(torch.uint8)), ("nmask", h_m.view(torch.uint8))], dev)
                if args.e2e_order == "text-first":
                    # the words alone in front of the partition; the wildcard mask (read by the probe only) is gathered under the index build
                    gather_text = None
                    gather_words = rdist.ShardedUpload([("words", h_w.view(torch.uint8))], dev)
                    gather_mask = rdist.ShardedUpload([("nmask", h_m.view(torch.uint8))], dev)
                    mask_off, mask_len = gather_mask.offsets["nmask"]
                    d_mask_ptr = gather_mask.d_all[mask_off:mask_off + mask_len].data_ptr()

            e2e_phase = {"h2d_reads_ms": [], "h2d_text_ms": [], "pack_ms": [], "index_ms": [], "scan_ms": [], "part_ms": [], "probe_ms": [], "fold_ms": [], "d2h_ms": [],
                         "api_set_reads_ms": [], "api_set_text_ms": [], "api_match_ms": [], "api_exchange_ms": [], "api_get_ms": []}

            text_first = args.e2e_order == "text-first"

            def step_host():
                t0 = time.perf_counter()
                if gather is not None and text_first:
                    # text first: its records are formed (real_gpu_prepare_scan, a stream of its own) while the reads are uploaded and gathered
                    d = gather_words.run()
                    h.set_text_device(d["words"].data_ptr(), d_mask_ptr, n, rs, shard_begin=sb, shard_len=sl, own_begin=ob, own_end=oe, async_copy=True)
                    h.prepare_scan(L)
                    t1 = time.perf_counter()
                    d = gather.run()
                    h.set_reads_packed_device(d["reads"].data_ptr(), R, L, d_wildcard_flags=d["flags"].data_ptr(),
                                              d_quality=d["qual"].data_ptr() if "qual" in d else None)
                    gather_mask.run()                 # the mask arrives while the index builds; the library reads it when the match call starts
                    t2 = time.perf_counter()
                    t_text, t_reads = t1 - t0, t2 - t1
                elif gather is not None:
                    d = gather.run()
                    h.set_reads_packed_device(d["reads"].data_ptr(), R, L, d_wildcard_flags=d["flags"].data_ptr(),
                                              d_quality=d["qual"].data_ptr() if "qual" in d else None)
                    d = gather_text.run()             # upload + all-gather of the text while the index build runs
                    h.set_text_device(d["words"].data_ptr(), d["nmask"].data_ptr(), n, rs, shard_begin=sb, shard_len=sl, own_begin=ob, own_end=oe)
                    t2 = time.perf_counter()
                    t_text, t_reads = 0.0, t2 - t0
                elif text_first:
                    # text first (real_gpu_set_text_async: the copies are only enqueued; the pinned buffers stay untouched until the match
                    # call has returned): the partition kernels of the scan (real_gpu_prepare_scan) start when the words have arrived and
                    # run while the reads cross PCIe; the wildcard mask, which the probe alone reads, travels behind the reads, under the
                    # index build
                    h.set_text(np_w, np_m, n, rs, shard_begin=sb, shard_len=sl, own_begin=ob, own_end=oe, async_copy=True)
                    h.prepare_scan(L)
                    t1 = time.perf_counter()
                    h.set_reads_packed(np_mapped, R, uniform_length=L, wildcard_flags=np_flags, quality=np_qual)
                    t2 = time.perf_counter()
                    t_text, t_reads = t1 - t0, t2 - t1
                else:
                    h.set_reads_packed(np_mapped, R, uniform_length=L, wildcard_flags=np_flags, quality=np_qual)
                    t1 = time.perf_counter()
                    # the copies of the text are enqueued (real_gpu_set_text_async): the partition of the scan starts when the words have
                    # arrived, the wildcard mask travels meanwhile; the pinned buffers stay untouched until the match call has returned
                    h.set_text(np_w, np_m, n, rs, shard_begin=sb, shard_len=sl, own_begin=ob, own_end=oe, async_copy=True)
                    t2 = time.perf_counter()
                    t_text, t_reads = t2 - t1, t1 - t0
                t4 = t3 = t2
                if unique:
                    h.match_unique()
                    if gaps:
                        h.match_gaps(0)
                    t3 = time.perf_counter()
                    st = h.stats()
                    if world > 1:
                        exchange()
                        st["fold_ms"] = h.stats()["fold_ms"]
                    t4 = time.perf_counter()
                    # after the exchange every rank holds the merged state of (at least) its own 1/N of the reads: it reads that back
                    h.get_unique(out=np_info[r_lo:r_hi], first=r_lo, count=r_hi - r_lo)
                    st["d2h_ms"] = h.stats()["d2h_ms"]
                    d2h[0] = (r_hi - r_lo) * 8
                else:
                    nh = h.match_all_count(packed=True)          # 16-byte rows land in the library's pinned host buffer
                    t4 = t3 = time.perf_counter()
                    st = h.stats()
                    d2h[0] = nh * 16
                t5 = time.perf_counter()
                st.update(api_set_reads_ms=t_reads * 1e3, api_set_text_ms=t_text * 1e3, api_match_ms=(t3 - t2) * 1e3,
                          api_exchange_ms=(t4 - t3) * 1e3, api_get_ms=(t5 - t4) * 1e3)
                return st

            def collect_e2e(st):
                for k in e2e_phase:
                    e2e_phase[k].append(st.get(k, 0.0))

            e_steps = args.steps
            e_ms, _ = timed(step_host, e_steps, 1, collect_e2e)
            # the state the last end-to-end step left on the device must be the one of the device-resident steps
            e2e_digest = result_digest()
            if e2e_digest != digest:
                print("bench: the end-to-end leg produced another result (digest %016x, device-resident %016x)" % (e2e_digest, digest), file=sys.stderr)
                sys.exit(3)
            h2d = R * L4 + R + (R * L if qual is not None else 0) + np_w.nbytes + np_m.nbytes + rs.nbytes
            if gather is not None:
                h2d = gather.chunk + (gather_text.chunk if gather_text is not None else gather_words.chunk + gather_mask.chunk) + rs.nbytes          # per rank; the rest arrives over NVLink
            e2e = {"value": R / (e_ms / e_steps * 1e-3), "unit": "reads/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h[0]),
                   "ms_per_step": e_ms / e_steps, "steps": e_steps, "order": args.e2e_order, "digest_ok": True, "prepared_scans": int(h.stats().get("prepared_scans", 0)),
                   "phases_ms": {k: statistics.mean(v) for k, v in e2e_phase.items() if v},
                   "input": "host buffers: text 2 bit/base + N mask, reads 2 bit/base (the reference's rewritten pattern file layout), "
                            "qualities 1 byte/base when scoring; result read back to pinned host memory"
                            + ("; every rank uploads 1/%d of the bytes, NCCL all-gather over NVLink for the rest (h2d_bytes_per_step is per rank)" % world
                               if gather is not None else "")
                            + ("; every rank reads back the merged result of its own 1/%d of the reads (d2h_bytes_per_step is per rank)" % world if world > 1 and unique else "")}
            del h_mapped, h_qual, h_w, h_m, h_flags
        except Exception as exc:          # the device-resident numbers above stand on their own: the line is printed either way
            import traceback
            traceback.print_exc()
            e2e = {"error": "%s: %s" % (type(exc).__name__, exc)}

    dev_bytes = h.device_bytes()
    h.close()

    ingest = None
    if rank == 0 and world == 1 and not args.no_ingest and not args.as_rank:
        try:
            ingest = ingest_probe(torch, rlib, float(roofline["peak"]))
        except Exception as e:                          # an extra: never in the way of the bench line
            ingest = {"error": "%s: %s" % (type(e).__name__, e)}

    cpu = None
    parity = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_reference(wl, args.cpu_text, args.cpu_reads, os.cpu_count() or 1)
        # the gate: the GPU path on the very sample the reference was just timed on, against what the reference produced there
        parity = parity_gate(wl, cpu.pop("_sample"), cpu.pop("_result"))
        parity["against"] = "oracle/_ref/ref_harness (the reference's own objects)" if cpu["kind"] == "reference" else "oracle/liboracle.so (restatement)"

    if rank == 0:
        tot = nwin_tot.tolist()
        line = {
            "metric": "matching-path reads/s", "value": value, "unit": "reads/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": workload_config(wl),
            "parity_checked": (parity["ok"] if parity is not None else None), "parity": parity,
            "result_digest": "%016x" % digest, "digest_expected": ("%016x" % expected) if expected is not None else None, "digest_ok": digest_ok,
            "setup": {"parallelism": ("signature tables sharded by scan bucket x%d: every rank indexes 1/%d of the signature space, reads the whole text and "
                                       "keeps the positions of its own buckets (no record exchange); reads and text replicated; one fold of the "
                                       "per-read results" % (world, world)) if buckets_mode else
                                      ("signature tables sharded x%d: every rank indexes 1/%d of the buckets, partitions 1/%d of the text positions of a round "
                                       "and stores the window records into the owners' windows (peer memory over NVLink); reads and text replicated"
                                       % (world, world, world)) if tables_mode else
                                      ("text sharded x%d with %d-base halo, read index replicated" % (world, L)) if world > 1 else "one GPU",
                       "fold": ("peer memory, reduce-scatter form (real_gpu_fold_unique)" if peer_fold else "NCCL MIN + SUM all-reduce") if (world > 1 and unique) else None,
                       "table_bits": args.table_bits or 32,
                       "reads_format": "2 bit/base (the reference's rewritten pattern layout), verified in place" if args.reads_format == "packed"
                                       else "1 byte/base (Pattern::mapped)"},
            "text_gbp_per_s": n / (ms_per_step * 1e-3) / 1e9,
            "scan_only": {"ms": scan_ms, "text_gbp_per_s_per_gpu": last_stats["n_windows"] / (scan_ms * 1e-3) / 1e9,
                          "reads_per_s": R / (scan_ms * 1e-3)},
            "phases_ms": {k: statistics.mean(v) for k, v in phase.items()},
            # short texts and bucket shards: real_gpu_set_text* starts the partition of the text beside the index build (DESIGN 4.9);
            # index_ms and part_ms then cover the same stretch of time and scan_ms holds the probe only
            "partition_beside_build": bool(last_stats.get("prepared_scans", 0)),
            "counts": {"windows": tot[0], "candidates": tot[1], "hits": tot[2], "seedpass": tot[3], "matchall_hits": nhits_holder[0]},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clk,
            "device_bytes": dev_bytes, "ingest": ingest, "cpu_affinity": affinity, "dump_outputs": dumped,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    if rank == 0 and parity is not None and not parity["ok"]:
        print("PARITY GATE FAILED: the GPU result differs from the reference on the sample", file=sys.stderr)
        return 3
    if rank == 0 and digest_ok is False:
        print("DIGEST MISMATCH: the result of this run differs from the recorded single-GPU result", file=sys.stderr)
        return 4
    return 0


if __name__ == "__main__":
    sys.exit(main())
