"""ctypes binding of the C ABI in include/real_gpu.h (libreal_gpu.so, sm_100a CUDA).

This is the only way the Python host layer reaches the kernels; there is no CPU path.  Loading
fails loudly when the shared library is missing or exports less than the header declares.
"""
from __future__ import annotations

import ctypes as C
import os
import re
from typing import List

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("REAL_GPU_LIB") or os.path.join(HERE, "libreal_gpu.so")      # REAL_GPU_LIB: a differently tuned build (development)
HEADER_PATH = os.path.join(HERE, "..", "include", "real_gpu.h")

REAL_GPU_OK = 0
REAL_GPU_E_ARG = -1
REAL_GPU_E_CUDA = -2
REAL_GPU_E_STATE = -3
REAL_GPU_E_LIMIT = -4


class Params(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("device", C.c_int32), ("seedl", C.c_uint32), ("seedkmax", C.c_uint32),
                ("totalkmax", C.c_uint32), ("scores", C.c_uint32), ("filter_mult", C.c_double), ("ll_table", C.c_void_p),
                ("table_bits", C.c_uint32), ("reserved", C.c_uint32)]


class Stats(C.Structure):
    _fields_ = [("h2d_text_ms", C.c_float), ("h2d_reads_ms", C.c_float), ("pack_ms", C.c_float), ("index_ms", C.c_float),
                ("scan_ms", C.c_float), ("post_ms", C.c_float), ("d2h_ms", C.c_float),
                ("scan_launches", C.c_uint32), ("total_launches", C.c_uint32),
                ("n_windows", C.c_uint64), ("n_probes", C.c_uint64), ("n_candidates", C.c_uint64),
                ("n_seedpass", C.c_uint64), ("n_hits", C.c_uint64), ("fold_ms", C.c_float), ("probe_ms", C.c_float),
                ("part_ms", C.c_float), ("prepared_scans", C.c_uint32)]

    def asdict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


HIT_DTYPE = np.dtype([("patid", "<u8"), ("pos", "<u8"), ("file", "<u4"), ("frag", "<u4"),
                      ("k", "<u4"), ("inverted", "<u4"), ("score", "<f4"), ("reserved", "<u4")])
HIT16_DTYPE = np.dtype([("pos_k_inv_frag", "<u8"), ("patid", "<u4"), ("score", "<f4")])
GAP_DTYPE = np.dtype([("patid", "<u4"), ("mingap", "<u4"), ("where", "<u4"), ("start", "<u4"),
                      ("gap_pos", "<u4"), ("present", "<u4")])


def declared_symbols() -> List[str]:
    """Every function name include/real_gpu.h declares."""
    with open(HEADER_PATH) as f:
        src = f.read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(real_gpu_[a-z_0-9]+)\s*\(", src)))


class RealGpuError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("real_gpu error %d: %s" % (code, msg))
        self.code = code


_lib = None


def load(build_if_missing: bool = True):
    """Loads libreal_gpu.so; raises if it is absent (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if build_if_missing:
        from . import build as _b
        if _b.needs_build():
            _b.build()
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("libreal_gpu.so is missing: run `python -m real_b200.build` (the CUDA extension is mandatory)")
    L = C.CDLL(LIB_PATH)
    missing = [s for s in declared_symbols() if not hasattr(L, s)]
    if missing:
        raise RuntimeError("libreal_gpu.so does not export: %s" % ", ".join(missing))
    vp, u64, u32, i32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int
    L.real_gpu_abi_version.restype = i32
    L.real_gpu_create.argtypes = [C.POINTER(Params), C.POINTER(vp)]
    L.real_gpu_destroy.argtypes = [vp]
    L.real_gpu_last_error.argtypes = [vp]
    L.real_gpu_last_error.restype = C.c_char_p
    L.real_gpu_set_text.argtypes = [vp, u32, vp, vp, u64, u64, u64, u64, u64, vp, u32]
    L.real_gpu_set_text_device.argtypes = [vp, u32, vp, vp, u64, u64, u64, u64, u64, vp, u32]
    L.real_gpu_set_text_device_async.argtypes = [vp, u32, vp, vp, u64, u64, u64, u64, u64, vp, u32]
    L.real_gpu_set_text_async.argtypes = [vp, u32, vp, vp, u64, u64, u64, u64, u64, vp, u32]
    L.real_gpu_prepare_scan.argtypes = [vp, u32]
    L.real_gpu_set_text_fasta.argtypes = [vp, u32, vp, u64, C.POINTER(u64), C.POINTER(u64)]
    L.real_gpu_set_text_fasta_device.argtypes = [vp, u32, vp, u64, C.POINTER(u64), C.POINTER(u64)]
    L.real_gpu_get_text_records.argtypes = [vp, vp, vp]
    L.real_gpu_get_text_packed.argtypes = [vp, u64, vp, vp]
    L.real_gpu_set_reads.argtypes = [vp, vp, vp, vp, u64]
    L.real_gpu_set_reads_device.argtypes = [vp, vp, vp, vp, u64, u64, u32]
    L.real_gpu_set_reads_packed.argtypes = [vp, vp, vp, vp, u32, vp, vp, u64]
    L.real_gpu_set_reads_fasta.argtypes = [vp, vp, u64, u32, C.POINTER(u64)]
    L.real_gpu_get_read_table.argtypes = [vp, vp, vp]
    L.real_gpu_get_read_ids.argtypes = [vp, vp, vp]
    L.real_gpu_get_reads_packed.argtypes = [vp, vp, vp]
    L.real_gpu_match_all.argtypes = [vp, C.POINTER(vp), C.POINTER(u64)]
    L.real_gpu_match_all_packed.argtypes = [vp, C.POINTER(vp), C.POINTER(u64)]
    L.real_gpu_match_unique.argtypes = [vp]
    L.real_gpu_get_unique.argtypes = [vp, vp, vp]
    L.real_gpu_get_unique_range.argtypes = [vp, u64, u64, vp, vp]
    L.real_gpu_reset_unique.argtypes = [vp]
    L.real_gpu_unique_checksum.argtypes = [vp, u64, u64, C.POINTER(u64)]
    L.real_gpu_set_block_windows.argtypes = [vp, u64]
    L.real_gpu_unique_export_keys.argtypes = [vp, vp]
    L.real_gpu_unique_export_ties.argtypes = [vp, vp, vp]
    L.real_gpu_unique_import.argtypes = [vp, vp, vp]
    L.real_gpu_match_gaps.argtypes = [vp, u64]
    L.real_gpu_get_gaps.argtypes = [vp, vp]
    L.real_gpu_comm_init.argtypes = [vp, u32, u32, u64, vp]
    L.real_gpu_comm_connect.argtypes = [vp, vp]
    L.real_gpu_comm_connect_local.argtypes = [vp, vp]
    L.real_gpu_set_reads_packed_device.argtypes = [vp, vp, u32, vp, vp, u64]
    L.real_gpu_fold_init.argtypes = [vp, u32, u32, u64, vp]
    L.real_gpu_fold_connect.argtypes = [vp, vp]
    L.real_gpu_fold_connect_local.argtypes = [vp, vp]
    L.real_gpu_fold_unique.argtypes = [vp]
    L.real_gpu_fold_unique_group.argtypes = [vp, u32]
    L.real_gpu_set_bucket_shard.argtypes = [vp, u32, u32]
    L.real_gpu_set_read_ids.argtypes = [vp, u64, u64, vp, vp]
    L.real_gpu_set_record_names.argtypes = [vp, u32, u32, vp, vp, vp]
    L.real_gpu_format_unique.argtypes = [vp, u64, u64, C.POINTER(vp), C.POINTER(u64), C.POINTER(u64)]
    L.real_gpu_format_all.argtypes = [vp, u64, u64, C.POINTER(vp), C.POINTER(u64)]
    L.real_gpu_selftest_format_scores.argtypes = [i32, vp, u64, vp]
    L.real_gpu_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.real_gpu_stream.argtypes = [vp]
    L.real_gpu_stream.restype = vp
    L.real_gpu_device_bytes.argtypes = [vp]
    L.real_gpu_device_bytes.restype = u64
    L.real_gpu_synth_text.argtypes = [i32, u64, u64, u64, u32, vp, vp]
    L.real_gpu_synth_reads.argtypes = [i32, u64, vp, vp, u64, u64, u64, u64, u32, u32, vp, vp]
    for name in declared_symbols():
        fn = getattr(L, name)
        if name not in ("real_gpu_last_error", "real_gpu_stream", "real_gpu_device_bytes"):      # (real_gpu_device_count returns a plain int)
            fn.restype = i32
    if L.real_gpu_abi_version() != 1:
        raise RuntimeError("libreal_gpu.so ABI version mismatch")
    _lib = L
    return L


def _np_ptr(a: np.ndarray, dtype) -> int:
    assert a.dtype == np.dtype(dtype) and a.flags["C_CONTIGUOUS"], (a.dtype, dtype)
    return a.ctypes.data


def selftest_format_scores(values: np.ndarray, device: int = 0):
    """The device's score formatter (printf %g) on float32 values; returns a list of byte strings."""
    v = np.ascontiguousarray(values, dtype=np.float32)
    out = np.zeros((v.size, 16), dtype=np.uint8)
    rc = load().real_gpu_selftest_format_scores(device, v.ctypes.data, v.size, out.ctypes.data)
    if rc != 0:
        raise RealGpuError(rc, "selftest_format_scores failed")
    return [bytes(r).split(b"\0", 1)[0] for r in out]


class Handle:
    """Thin RAII wrapper of one real_gpu handle (one CUDA device, single-threaded)."""

    def __init__(self, seedl: int = 32, seedkmax: int = 2, totalkmax: int = 5, scores: bool = False,
                 filter_mult: float = 0.0, ll_table: np.ndarray | None = None, device: int = 0, table_bits: int = 0):
        self.L = load()
        self._ll = None
        if ll_table is not None:
            self._ll = np.ascontiguousarray(ll_table, dtype=np.float64)
            assert self._ll.size == 1024
        P = Params(C.sizeof(Params), device, seedl, seedkmax, totalkmax, 1 if scores else 0, filter_mult,
                   self._ll.ctypes.data if self._ll is not None else None, table_bits, 0)
        h = C.c_void_p()
        rc = self.L.real_gpu_create(C.byref(P), C.byref(h))
        if rc != 0:
            raise RealGpuError(rc, "real_gpu_create failed (see stderr)")
        self.h = h
        self.device = device
        self.nreads = 0
        self.scores = scores

    def close(self):
        if getattr(self, "h", None):
            self.L.real_gpu_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            raise RealGpuError(rc, self.L.real_gpu_last_error(self.h).decode())

    # ---- text
    def set_text(self, words: np.ndarray, nmask: np.ndarray, n_total: int, record_starts: np.ndarray, fileid: int = 0,
                 shard_begin: int = 0, shard_len: int | None = None, own_begin: int | None = None, own_end: int | None = None, async_copy: bool = False):
        """async_copy: real_gpu_set_text_async -- the buffers (pinned) must stay valid until the next match call has returned"""
        shard_len = n_total - shard_begin if shard_len is None else shard_len
        own_begin = shard_begin if own_begin is None else own_begin
        own_end = shard_begin + shard_len if own_end is None else own_end
        rs = np.ascontiguousarray(record_starts, dtype=np.uint64)
        if async_copy:
            self._keep_text = (words, nmask, rs)
            self._check(self.L.real_gpu_set_text_async(self.h, fileid, _np_ptr(words, np.uint64), _np_ptr(nmask, np.uint64), n_total,
                                                       shard_begin, shard_len, own_begin, own_end, rs.ctypes.data, rs.size - 1))
            return
        self._check(self.L.real_gpu_set_text(self.h, fileid, _np_ptr(words, np.uint64), _np_ptr(nmask, np.uint64), n_total,
                                             shard_begin, shard_len, own_begin, own_end, rs.ctypes.data, rs.size - 1))

    def prepare_scan(self, max_read_len: int):
        """real_gpu_prepare_scan: text first, reads second -- the scan's records of the current text are formed now, on a stream of
        their own, while a following set_reads* call moves the reads; the next match call uses them."""
        self._check(self.L.real_gpu_prepare_scan(self.h, max_read_len))

    def set_text_device(self, d_words: int, d_nmask: int, n_total: int, record_starts: np.ndarray, fileid: int = 0,
                        shard_begin: int = 0, shard_len: int | None = None, own_begin: int | None = None, own_end: int | None = None,
                        async_copy: bool = False):
        """async_copy: real_gpu_set_text_device_async -- the words' copy is enqueued, the mask behind d_nmask is read when the next
        match call starts (the caller may complete it until then); both buffers stay valid until that call has returned"""
        shard_len = n_total - shard_begin if shard_len is None else shard_len
        own_begin = shard_begin if own_begin is None else own_begin
        own_end = shard_begin + shard_len if own_end is None else own_end
        rs = np.ascontiguousarray(record_starts, dtype=np.uint64)
        if async_copy:
            self._keep_text = (rs,)
            self._check(self.L.real_gpu_set_text_device_async(self.h, fileid, d_words, d_nmask, n_total, shard_begin, shard_len,
                                                              own_begin, own_end, rs.ctypes.data, rs.size - 1))
            return
        self._check(self.L.real_gpu_set_text_device(self.h, fileid, d_words, d_nmask, n_total, shard_begin, shard_len,
                                                    own_begin, own_end, rs.ctypes.data, rs.size - 1))

    def set_text_fasta(self, data, fileid: int = 0, device_ptr: int | None = None, nbytes: int | None = None):
        """Text straight from the bytes of a FASTA file (K0, on the device).  data = bytes / uint8 array, or device_ptr + nbytes.
        Returns (n_bases, nrecords); no text is set when either is 0."""
        n, r = C.c_uint64(), C.c_uint64()
        if device_ptr is not None:
            self._check(self.L.real_gpu_set_text_fasta_device(self.h, fileid, device_ptr, nbytes, C.byref(n), C.byref(r)))
        else:
            a = np.frombuffer(data, dtype=np.uint8) if isinstance(data, (bytes, bytearray, memoryview)) else np.ascontiguousarray(data, dtype=np.uint8)
            self._check(self.L.real_gpu_set_text_fasta(self.h, fileid, a.ctypes.data if a.size else None, a.size, C.byref(n), C.byref(r)))
        self._text_n, self._text_nrec = int(n.value), int(r.value)
        return self._text_n, self._text_nrec

    def get_text_records(self):
        """(record_starts[nrecords+1], header_ends[nrecords]) of the text set by set_text_fasta."""
        starts = np.zeros(self._text_nrec + 1, dtype=np.uint64)
        ends = np.zeros(max(self._text_nrec, 1), dtype=np.uint64)
        self._check(self.L.real_gpu_get_text_records(self.h, starts.ctypes.data, ends.ctypes.data))
        return starts, ends[:self._text_nrec]

    def get_text_packed(self, n: int):
        """The current text as (words, nmask) in the layout set_text takes; n = its length in bases."""
        words = np.zeros((n + 31) // 32, dtype=np.uint64)
        nmask = np.zeros((n + 63) // 64, dtype=np.uint64)
        self._check(self.L.real_gpu_get_text_packed(self.h, n, words.ctypes.data, nmask.ctypes.data))
        return words, nmask

    # ---- reads
    def set_reads(self, mapped: np.ndarray, offsets: np.ndarray, quality: np.ndarray | None = None):
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        mapped = np.ascontiguousarray(mapped, dtype=np.uint8)
        q = None
        if quality is not None:
            quality = np.ascontiguousarray(quality, dtype=np.uint8)
            q = quality.ctypes.data
        self.nreads = int(offsets.size - 1)
        self._check(self.L.real_gpu_set_reads(self.h, mapped.ctypes.data if mapped.size else None, q, offsets.ctypes.data, self.nreads))

    def set_reads_packed(self, packed: np.ndarray, nreads: int, uniform_length: int = 0, byte_offsets: np.ndarray | None = None,
                         lengths: np.ndarray | None = None, wildcard_flags: np.ndarray | None = None, quality: np.ndarray | None = None):
        self.nreads = nreads
        p = lambda a, dt: (None if a is None else _np_ptr(np.ascontiguousarray(a, dtype=dt), dt))
        keep = [np.ascontiguousarray(a, dtype=dt) if a is not None else None
                for a, dt in ((packed, np.uint8), (byte_offsets, np.uint64), (lengths, np.uint32), (wildcard_flags, np.uint8), (quality, np.uint8))]
        ptrs = [a.ctypes.data if a is not None else None for a in keep]
        self._check(self.L.real_gpu_set_reads_packed(self.h, ptrs[0], ptrs[1], ptrs[2], uniform_length, ptrs[3], ptrs[4], nreads))

    def set_reads_fasta(self, data, rewrite_order: bool = False) -> int:
        """Read set straight from the bytes of a FASTA pattern file (parsed and packed on the device); returns the number of reads."""
        buf = np.frombuffer(bytes(data), dtype=np.uint8) if not isinstance(data, np.ndarray) else np.ascontiguousarray(data, dtype=np.uint8)
        n = C.c_uint64()
        self._check(self.L.real_gpu_set_reads_fasta(self.h, buf.ctypes.data if buf.size else None, buf.size, 1 if rewrite_order else 0, C.byref(n)))
        self.nreads = int(n.value)
        return self.nreads

    def get_read_table(self):
        """(lengths, wildcard flags) of the reads set by set_reads_fasta"""
        ln = np.zeros(max(1, self.nreads), dtype=np.uint32)
        fl = np.zeros(max(1, self.nreads), dtype=np.uint8)
        self._check(self.L.real_gpu_get_read_table(self.h, ln.ctypes.data, fl.ctypes.data))
        return ln[:self.nreads], fl[:self.nreads]

    def get_read_ids(self):
        offs = np.zeros(self.nreads + 1, dtype=np.uint64)
        self._check(self.L.real_gpu_get_read_ids(self.h, None, offs.ctypes.data))
        blob = np.zeros(max(1, int(offs[-1])), dtype=np.uint8)
        self._check(self.L.real_gpu_get_read_ids(self.h, blob.ctypes.data, offs.ctypes.data))
        b = blob.tobytes()
        return [b[int(offs[i]):int(offs[i + 1])] for i in range(self.nreads)]

    def get_reads_mapped(self):
        """The reads of a 2 bit/base read set unpacked to one list of base codes per read (wildcards read as 0)."""
        offs = np.zeros(self.nreads + 1, dtype=np.uint64)
        self._check(self.L.real_gpu_get_reads_packed(self.h, None, offs.ctypes.data))
        blob = np.zeros(max(1, int(offs[-1])), dtype=np.uint8)
        self._check(self.L.real_gpu_get_reads_packed(self.h, blob.ctypes.data, offs.ctypes.data))
        ln, _ = self.get_read_table()
        out = []
        for i in range(self.nreads):
            p = blob[int(offs[i]):int(offs[i + 1])]
            codes = np.stack([(p >> 6) & 3, (p >> 4) & 3, (p >> 2) & 3, p & 3], 1).reshape(-1)[:int(ln[i])]
            out.append(codes)
        return out

    def set_reads_packed_device(self, d_packed: int, nreads: int, uniform_length: int, d_wildcard_flags: int | None = None, d_quality: int | None = None):
        self.nreads = nreads
        self._check(self.L.real_gpu_set_reads_packed_device(self.h, d_packed, uniform_length, d_wildcard_flags, d_quality, nreads))

    def set_reads_device(self, d_mapped: int, d_offsets: int, nreads: int, total_bases: int, maxlen: int, d_quality: int | None = None):
        self.nreads = nreads
        self._check(self.L.real_gpu_set_reads_device(self.h, d_mapped, d_quality, d_offsets, nreads, total_bases, maxlen))

    # ---- matching
    def match_all(self) -> np.ndarray:
        p = C.c_void_p()
        n = C.c_uint64()
        self._check(self.L.real_gpu_match_all(self.h, C.byref(p), C.byref(n)))
        if n.value == 0:
            return np.zeros(0, dtype=HIT_DTYPE)
        buf = (C.c_char * (n.value * HIT_DTYPE.itemsize)).from_address(p.value)
        return np.frombuffer(buf, dtype=HIT_DTYPE).copy()

    def match_all_count(self, packed: bool = False) -> int:
        """match_all without copying the records out of the library's pinned buffer (packed: 16-byte rows)."""
        p = C.c_void_p()
        n = C.c_uint64()
        self._check((self.L.real_gpu_match_all_packed if packed else self.L.real_gpu_match_all)(self.h, C.byref(p), C.byref(n)))
        self._last_packed = (p.value, int(n.value)) if packed else None
        return int(n.value)

    def last_rows_packed(self) -> np.ndarray:
        """The rows the last match_all_count(packed=True) left in the library's pinned buffer, expanded like match_all_packed,
        without matching again; valid until the handle matches again or is closed."""
        if getattr(self, "_last_packed", None) is None:
            raise RuntimeError("last_rows_packed: the last match call was not match_all_count(packed=True)")
        return self._expand_hit16(*self._last_packed)

    def match_all_packed(self) -> np.ndarray:
        """The rows of match_all as real_gpu_hit16, expanded to the fields of HIT_DTYPE."""
        p = C.c_void_p()
        n = C.c_uint64()
        self._check(self.L.real_gpu_match_all_packed(self.h, C.byref(p), C.byref(n)))
        return self._expand_hit16(p.value, n.value)

    @staticmethod
    def _expand_hit16(ptr: int, count: int) -> np.ndarray:
        out = np.zeros(count, dtype=HIT_DTYPE)
        if count:
            buf = (C.c_char * (count * HIT16_DTYPE.itemsize)).from_address(ptr)
            r = np.frombuffer(buf, dtype=HIT16_DTYPE)
            w = r["pos_k_inv_frag"]
            out["patid"] = r["patid"]; out["pos"] = w & np.uint64((1 << 35) - 1); out["k"] = (w >> np.uint64(35)) & np.uint64(15)
            out["inverted"] = (w >> np.uint64(39)) & np.uint64(1); out["frag"] = (w >> np.uint64(40)) & np.uint64(0xFFFFFF); out["score"] = r["score"]
        return out

    def match_unique(self):
        self._check(self.L.real_gpu_match_unique(self.h))

    def get_unique(self, out: np.ndarray | None = None, first: int = 0, count: int | None = None):
        """UniqueMatchInfo words (and scores) of the reads [first, first+count); default: all reads."""
        count = self.nreads - first if count is None else count
        info = out if out is not None else np.zeros(count, dtype=np.uint64)
        sc = np.zeros(count, dtype=np.float32) if self.scores else None
        self._check(self.L.real_gpu_get_unique_range(self.h, first, count, info.ctypes.data, sc.ctypes.data if sc is not None else None))
        return info, sc

    def unique_checksum(self, first: int = 0, count: int | None = None) -> int:
        """Digest of the canonical unique state of the reads [first, first+count) (matcher.unique_checksum is the numpy form)."""
        count = self.nreads - first if count is None else count
        v = C.c_uint64()
        self._check(self.L.real_gpu_unique_checksum(self.h, first, count, C.byref(v)))
        return int(v.value)

    def reset_unique(self):
        self._check(self.L.real_gpu_reset_unique(self.h))

    def set_block_windows(self, n_list: int):
        self._check(self.L.real_gpu_set_block_windows(self.h, n_list))

    def unique_export_keys(self, d_keys: int):
        self._check(self.L.real_gpu_unique_export_keys(self.h, d_keys))

    def unique_export_ties(self, d_min_keys: int, d_ties: int):
        self._check(self.L.real_gpu_unique_export_ties(self.h, d_min_keys, d_ties))

    def unique_import(self, d_min_keys: int, d_tie_sums: int):
        self._check(self.L.real_gpu_unique_import(self.h, d_min_keys, d_tie_sums))

    # ---- sharded tables (one handle per rank)
    def comm_init(self, rank: int, nranks: int, round_positions: int = 0) -> bytes:
        """Allocates this rank's window; returns the 64-byte handle the other ranks connect with."""
        buf = C.create_string_buffer(64)
        self._check(self.L.real_gpu_comm_init(self.h, rank, nranks, round_positions, buf))
        return buf.raw

    def set_bucket_shard(self, rank: int, nranks: int):
        """This handle indexes and probes 1/nranks of the signature space (no peer memory); call before set_reads."""
        self._check(self.L.real_gpu_set_bucket_shard(self.h, rank, nranks))

    def comm_connect(self, all_handles: bytes):
        self._check(self.L.real_gpu_comm_connect(self.h, all_handles))

    def comm_connect_local(self, peers):
        arr = (C.c_void_p * len(peers))(*[p.h for p in peers])
        self._check(self.L.real_gpu_comm_connect_local(self.h, arr))

    # ---- peer-memory fold of the unique state (one handle per rank)
    def fold_init(self, rank: int, nranks: int, max_reads: int) -> bytes:
        buf = C.create_string_buffer(64)
        self._check(self.L.real_gpu_fold_init(self.h, rank, nranks, max_reads, buf))
        return buf.raw

    def fold_connect(self, all_handles: bytes):
        self._check(self.L.real_gpu_fold_connect(self.h, all_handles))

    def fold_connect_local(self, peers):
        arr = (C.c_void_p * len(peers))(*[p.h for p in peers])
        self._check(self.L.real_gpu_fold_connect_local(self.h, arr))

    def fold_unique(self):
        """Collective (one process per GPU): afterwards this rank holds the merged words of its own 1/nranks of the reads."""
        self._check(self.L.real_gpu_fold_unique(self.h))

    @staticmethod
    def fold_unique_group(handles):
        """The ranks of one process: handles[r] = rank r."""
        arr = (C.c_void_p * len(handles))(*[p.h for p in handles])
        rc = handles[0].L.real_gpu_fold_unique_group(arr, len(handles))
        if rc != 0:
            msgs = [p.L.real_gpu_last_error(p.h).decode() for p in handles]
            raise RealGpuError(rc, "; ".join(m for m in msgs if m))

    def match_gaps(self, n_list: int = 0):
        self._check(self.L.real_gpu_match_gaps(self.h, n_list))

    def get_gaps(self) -> np.ndarray:
        g = np.zeros(self.nreads, dtype=GAP_DTYPE)
        self._check(self.L.real_gpu_get_gaps(self.h, g.ctypes.data))
        return g

    # ---- output lines formatted on the device (K8)
    @staticmethod
    def _strings(items):
        """bytes + offsets of a list of byte strings"""
        blob = b"".join(items)
        offs = np.zeros(len(items) + 1, dtype=np.uint64)
        if items:
            offs[1:] = np.cumsum([len(x) for x in items], dtype=np.uint64)
        return blob, offs

    def set_read_ids(self, ids, first: int = 0):
        blob, offs = self._strings([x if isinstance(x, bytes) else x.encode() for x in ids])
        buf = np.frombuffer(blob, dtype=np.uint8) if blob else np.zeros(1, dtype=np.uint8)
        self._check(self.L.real_gpu_set_read_ids(self.h, first, len(ids), buf.ctypes.data, offs.ctypes.data))

    def set_record_names(self, names, record_starts, fileid: int = 0):
        blob, offs = self._strings([x if isinstance(x, bytes) else x.encode() for x in names])
        buf = np.frombuffer(blob, dtype=np.uint8) if blob else np.zeros(1, dtype=np.uint8)
        rs = np.ascontiguousarray(record_starts, dtype=np.uint64)
        assert rs.size >= len(names)
        self._check(self.L.real_gpu_set_record_names(self.h, fileid, len(names), buf.ctypes.data, offs.ctypes.data, rs.ctypes.data))

    def format_unique(self, first: int = 0, count: int | None = None):
        """(bytes of the lines of the reads [first, first+count), number of lines)"""
        count = self.nreads - first if count is None else count
        p, nb, nl = C.c_void_p(), C.c_uint64(), C.c_uint64()
        self._check(self.L.real_gpu_format_unique(self.h, first, count, C.byref(p), C.byref(nb), C.byref(nl)))
        return (C.string_at(p.value, nb.value) if nb.value else b""), int(nl.value)

    def format_all(self, first_row: int, count: int) -> bytes:
        p, nb = C.c_void_p(), C.c_uint64()
        self._check(self.L.real_gpu_format_all(self.h, first_row, count, C.byref(p), C.byref(nb)))
        return C.string_at(p.value, nb.value) if nb.value else b""

    def stats(self) -> dict:
        s = Stats()
        self._check(self.L.real_gpu_get_stats(self.h, C.byref(s)))
        return s.asdict()

    def stream(self) -> int:
        return int(self.L.real_gpu_stream(self.h) or 0)

    def device_bytes(self) -> int:
        return int(self.L.real_gpu_device_bytes(self.h))
