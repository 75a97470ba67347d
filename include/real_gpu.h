/* real_gpu.h -- C ABI of the B200-native REAL matching path (libreal_gpu.so).
 *
 * Drop-in boundary for the hot path of solonas13/REAL v0.0.31.  The reference has no FFI
 * layer; the seams this ABI replaces are the per-read matcher entry points that its run
 * drivers call inside the text-block loop:
 *
 *   AllMatcher::match(pattern, fi, RWB, handled, localmatches)       matchAllImplementation.cpp:261-355
 *     + unifyMatches(localmatches)                                   matchAllImplementation.cpp:150-161
 *   UniqueMatcher::match(pattern, info, fi, RWB, handled)            matchUniqueImplementation.cpp:369-500
 *   UniqueMatcher::matchGaps(pattern, info, RWB, gapinfos, handled)  matchUniqueImplementation.cpp:501-572
 *   ListSetBlockReader::readNextBlock() (index build)                ListSetBlockReader.hpp:24-56
 *
 * Those are per-read calls over a text-side index; here they are batched and the index is on
 * the read side (BASELINE.json north_star): the host hands over one text file (or a shard of
 * it) and the whole read set, and gets back exactly what the per-read calls would have
 * accumulated -- the set of MatchPosAndError rows in unifyMatches order, or the array of
 * UniqueMatchInfo words.
 *
 * Conventions: every entry point is extern "C", takes plain pointers and sizes, returns 0 on
 * success or a negative REAL_GPU_E_* code, never throws.  real_gpu_last_error() gives the text.
 * Host buffers passed in belong to the caller and may be reused as soon as the call returns.
 * Buffers handed out by the library stay valid until the next call on the same handle.
 * A handle is single-threaded and bound to one CUDA device.  There is no CPU fallback: if no
 * device is present real_gpu_create fails with REAL_GPU_E_CUDA.
 */
#ifndef REAL_GPU_H
#define REAL_GPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define REAL_GPU_ABI_VERSION 1

enum
{
        REAL_GPU_OK = 0,
        REAL_GPU_E_ARG = -1,       /* bad argument (also: option outside what RealOptions accepts) */
        REAL_GPU_E_CUDA = -2,      /* CUDA runtime error, no device, out of device memory */
        REAL_GPU_E_STATE = -3,     /* call order: text or reads not set */
        REAL_GPU_E_LIMIT = -4      /* input exceeds a format limit (see real_gpu_set_text / set_reads) */
};

typedef struct real_gpu real_gpu;

/* Run parameters: the subset of RealOptions (RealOptions.hpp:29-77) the hot path reads. */
typedef struct
{
        uint32_t struct_size;   /* sizeof(real_gpu_params), for ABI evolution */
        int32_t device;         /* CUDA device ordinal */
        uint32_t seedl;         /* -l  seed length, multiple of 4, 4..64 (RealOptions.cpp:434-447); above 32 the first 32 bases are
                                   indexed and the whole seed is tested at verification (same match sets, DESIGN.md 6) */
        uint32_t seedkmax;      /* -s  mismatches allowed in the seed, 0..2 (RealOptions.cpp:449-453) */
        uint32_t totalkmax;     /* -e  mismatches allowed in the read, 0..15 (RealOptions.cpp:176-180) */
        uint32_t scores;        /* -q  quality-aware scores on/off */
        double filter_mult;     /* epsilon(patl) = (float)(filter_mult * patl) (RealOptions.hpp:74-77, RealOptions.cpp:455-463) */
        const double * ll_table;/* Scoring::LL, 4*4*64 doubles indexed (ref<<8)|(read<<6)|q (Scoring.hpp:70-73);
                                   required when scores != 0 or for real_gpu_match_gaps; copied */
        uint32_t table_bits;    /* 0 = automatic; else log2 of the slots of each signature presence table */
        uint32_t reserved;
} real_gpu_params;

/* One reported match == MatchPosAndError (matchAllImplementation.cpp:99-120) plus the read ordinal. */
typedef struct
{
        uint64_t patid;         /* 0-based ordinal of the read in the set (Pattern::patid) */
        uint64_t pos;           /* 0-based start in the concatenated text of the file */
        uint32_t file;          /* fileid given to real_gpu_set_text */
        uint32_t frag;          /* FASTA record index, RangeVector::positionToRange(pos) */
        uint32_t k;             /* mismatches over the whole read */
        uint32_t inverted;      /* 0 = '+', 1 = '-' (read reverse complemented) */
        float score;            /* ComputeScore::computeScore; 1.0f when scores are off */
        uint32_t reserved;
} real_gpu_hit;

/* The same row in 16 bytes, for callers that read back many rows (a 40-byte row costs 2.5x the PCIe time): position (bits 0..34),
 * k (35..38), inverted (39) and frag (40..63) share one word; the file is the one the call matched against. */
typedef struct
{
        uint64_t pos_k_inv_frag;
        uint32_t patid;         /* read sets hold fewer than 2^28 reads */
        float score;
} real_gpu_hit16;
#define REAL_GPU_HIT16_POS(w)      ((uint64_t)(w) & ((1ULL << 35) - 1))
#define REAL_GPU_HIT16_K(w)        ((uint32_t)(((uint64_t)(w) >> 35) & 15))
#define REAL_GPU_HIT16_INVERTED(w) ((uint32_t)(((uint64_t)(w) >> 39) & 1))
#define REAL_GPU_HIT16_FRAG(w)     ((uint32_t)(((uint64_t)(w) >> 40) & 0xFFFFFF))

/* GapInfo (match.hpp:420-426) of a read whose state is Gapped and whose entry survived. */
typedef struct
{
        uint32_t patid;
        uint32_t mingap;
        uint32_t where;
        uint32_t start;
        uint32_t gap_pos;
        uint32_t present;
} real_gpu_gapinfo;

/* Device-side phase timings of the last calls, milliseconds, measured with CUDA events on the
 * handle's stream. */
typedef struct
{
        float h2d_text_ms;      /* text transfer; after real_gpu_set_text_fasta*: transfer of the file bytes + the K0 kernels */
        float h2d_reads_ms;
        float pack_ms;          /* K1: read packing + seed extraction */
        float index_ms;         /* K2: the two partition passes over the index items + the sub-bucket build of the tables */
        float scan_ms;          /* K3: text scan (probe + verify), the dominant kernel */
        float post_ms;          /* K4/K6: scoring, per-read ordering */
        float d2h_ms;
        uint32_t scan_launches; /* kernels launched by the last match call */
        uint32_t total_launches;/* kernels launched since create */
        uint64_t n_windows;     /* text positions scanned by the last scan */
        uint64_t n_probes;      /* presence-table probes issued */
        uint64_t n_candidates;  /* signature-equal (window, entry) pairs examined */
        uint64_t n_seedpass;    /* candidates that passed the seed test and the canonical-list rule */
        uint64_t n_hits;        /* hits emitted */
        float fold_ms;          /* real_gpu_fold_unique*: push + hand-over + merge */
        float probe_ms;         /* the probe kernels' part of scan_ms (the rest is the partition of the text positions) */
        float part_ms;          /* the partition kernels of the last scan; part of scan_ms unless real_gpu_prepare_scan ran them ahead */
        uint32_t prepared_scans; /* scans of this handle that found their records formed by real_gpu_prepare_scan */
} real_gpu_stats;

int real_gpu_abi_version(void);
/* CUDA devices visible to the process (0 when there is none or the runtime fails): host drivers that put one handle on
 * every GPU of the box size their team with it. */
int real_gpu_device_count(void);

/* Creates a handle on params->device.  Replaces the construction of SignatureConstruction,
 * Scoring and the matcher object (matchAllImplementation.cpp:381-390,447). */
int real_gpu_create(const real_gpu_params * params, real_gpu ** out);
int real_gpu_destroy(real_gpu * h);
const char * real_gpu_last_error(const real_gpu * h);

/* Text of one file, or a shard of it (replaces getText + AutoTextArray + RangeVector construction,
 * getText.hpp:31-58, and the text side of MatcherBase, MatcherBase.hpp:18-33).
 *   words         2 bit/base, 32 bases per u64, base i of the shard at bits 63-2(i%32).. (AutoTextArray.hpp:27-43)
 *   nmask         1 bit/base, 64 per u64, base i at bit 63-(i%64) (AutoTextArray.hpp:45-61)
 *   n_total       length of the whole file in bases (positions are file-global everywhere)
 *   shard_begin   global position of base 0 of words/nmask; must be a multiple of 64
 *   shard_len     bases present in words/nmask
 *   own_begin/own_end  half-open range of hit START positions this shard reports; the shard must
 *                 contain [own_begin, min(n_total, own_end + maxreadlen)) (read-length halo)
 *   record_starts nrecords+1 global offsets, last == n_total (countReads.cpp:58,81)
 * Limits (REAL_GPU_E_LIMIT): n_total < 2^35, fileid < 64, nrecords <= 65535 for unique matching
 * (UniqueMatchInfo.hpp:29-33). */
int real_gpu_set_text(real_gpu * h, uint32_t fileid,
                      const uint64_t * words, const uint64_t * nmask,
                      uint64_t n_total, uint64_t shard_begin, uint64_t shard_len,
                      uint64_t own_begin, uint64_t own_end,
                      const uint64_t * record_starts, uint32_t nrecords);
/* real_gpu_set_text whose copies are only ENQUEUED when the call returns: words, nmask and record_starts must stay valid and
 * unchanged until the next real_gpu_match_* call on the handle has returned (or another real_gpu_set_text* / real_gpu_get_text*
 * call, which wait for the copies).  The scan then starts partitioning as soon as the text words have arrived -- the wildcard
 * mask (a third of the bytes) is needed by the probe only and travels meanwhile.  Pinned host memory, or the copies block. */
int real_gpu_set_text_async(real_gpu * h, uint32_t fileid,
                            const uint64_t * words, const uint64_t * nmask,
                            uint64_t n_total, uint64_t shard_begin, uint64_t shard_len,
                            uint64_t own_begin, uint64_t own_end,
                            const uint64_t * record_starts, uint32_t nrecords);
/* Text first, reads second: forms the scan's records of the current text NOW -- the partition kernels (K3, step 1) are enqueued
 * on a stream of their own, behind the arrival of the words of a real_gpu_set_text_async, and the call returns at once -- so
 * that they run while a following real_gpu_set_reads* call moves the reads over PCIe (the partition needs the text only; the
 * index build needs all the reads).  max_read_len = the longest read of the set that will be matched (it bounds the last seed
 * window of a text shard).  The next real_gpu_match_* call uses the records if it would form the very same ones (same text,
 * shard, bucket split, window range) and forms its own otherwise: a hint, never a change of the result.  One scan per call;
 * nothing is prepared (and REAL_GPU_OK returned) when the text needs several chunks or the handle exchanges records with
 * peers (real_gpu_comm_*).  The order set_text_async -> prepare_scan -> set_reads* -> match also sends the text's wildcard
 * mask behind the reads (it is read by the probe only). */
int real_gpu_prepare_scan(real_gpu * h, uint32_t max_read_len);
/* real_gpu_set_text_async for a text already in device memory: the copy of the words is enqueued; d_nmask is only REMEMBERED and
 * copied when the next real_gpu_match_* call (or real_gpu_set_text* / real_gpu_get_text*) starts, so the caller may still be
 * completing the mask while it hands over the reads -- ranks that upload 1/N of every input and all-gather the rest send the
 * words, let the partition start (real_gpu_prepare_scan), gather the reads, and gather the mask while the index builds. */
int real_gpu_set_text_device_async(real_gpu * h, uint32_t fileid,
                                   const uint64_t * d_words, const uint64_t * d_nmask,
                                   uint64_t n_total, uint64_t shard_begin, uint64_t shard_len,
                                   uint64_t own_begin, uint64_t own_end,
                                   const uint64_t * record_starts, uint32_t nrecords);
/* Same, with words/nmask already resident in device memory (record_starts stays a host pointer). */
int real_gpu_set_text_device(real_gpu * h, uint32_t fileid,
                             const uint64_t * d_words, const uint64_t * d_nmask,
                             uint64_t n_total, uint64_t shard_begin, uint64_t shard_len,
                             uint64_t own_begin, uint64_t own_end,
                             const uint64_t * record_starts, uint32_t nrecords);

/* Text of one whole file straight from the BYTES of its FASTA file: the library runs the reference's text loader on
 * the device (K0, csrc/ingest.cuh) -- countLength + readFile (countReads.cpp:28-125: '>' opens a header up to the
 * next '\n', wherever it stands; outside headers A C G T N are kept, every other byte is dropped) and the packing of
 * AutoTextArray (AutoTextArray.hpp:27-61) -- and sets the result as the current text, as real_gpu_set_text would with
 * shard = own range = the whole file.  *n_bases = bases kept, *nrecords = headers closed by a '\n'
 * (ranges.size() - 1 of countLength).  When either is 0 the call succeeds but no text is set.
 * Limits as for real_gpu_set_text.  The caller's buffer is free again when the call returns.  A call refused with
 * REAL_GPU_E_ARG changes nothing; after any other failure the handle has no text. */
int real_gpu_set_text_fasta(real_gpu * h, uint32_t fileid, const void * fasta_bytes, uint64_t nbytes,
                            uint64_t * n_bases, uint64_t * nrecords);
/* Same, with the file bytes already in device memory (16-byte aligned; not modified, not kept). */
int real_gpu_set_text_fasta_device(real_gpu * h, uint32_t fileid, const void * d_fasta_bytes, uint64_t nbytes,
                                   uint64_t * n_bases, uint64_t * nrecords);
/* Record table of the text set by real_gpu_set_text_fasta*: record_starts[nrecords+1] (last == n_bases) and, per
 * record, the file offset of the '\n' that closed its header -- the record's name is the bytes between the last '>'
 * in front of that offset and the offset itself (countReads.cpp:44-58).  Either pointer may be NULL. */
int real_gpu_get_text_records(real_gpu * h, uint64_t * record_starts, uint64_t * header_ends);
/* Copies the current text (shard) back in the layout real_gpu_set_text takes: (n_bases+31)/32 words and
 * (n_bases+63)/64 mask words.  n_bases must be the length of the current text (shard), REAL_GPU_E_ARG otherwise:
 * it is what the caller sized its buffers for.  Either pointer may be NULL. */
int real_gpu_get_text_packed(real_gpu * h, uint64_t n_bases, uint64_t * words, uint64_t * nmask);

/* Read set (replaces reader_type::fillPatternBlock + Pattern::computeMapped + RestWordBuffer::setup*
 * + SignatureConstruction::signatureMapped/reverseMappedSignature per read, and the index build
 * ListSet::sort + getLookupTable, here on the read side).
 *   mapped   one byte per base, 0..3 = ACGT, anything >3 = wildcard (Pattern.hpp:105-128)
 *   quality  one byte per base, PHRED minus offset (FastQReader.hpp:168); NULL = constant 30 (Pattern.hpp:42-45)
 *   offsets  nreads+1 byte offsets into mapped/quality
 * Reads shorter than seedl or containing a wildcard are kept but never match
 * (matchAllImplementation.cpp:273-289).  Resets the unique-match state.
 * Limits: nreads < 2^28 per read set (a raw hit carries the read ordinal in 28 bits beside its exact-fragment mask; the
 * reference counts reads in 64 bits -- larger sets are matched in batches of reads, each batch against every file, and their
 * output concatenated: reads are independent of each other), read length <= 65535. */
int real_gpu_set_reads(real_gpu * h, const uint8_t * mapped, const uint8_t * quality,
                       const uint64_t * offsets, uint64_t nreads);
/* Same as real_gpu_set_reads for reads that are already packed 2 bit/base the way the reference's rewritten pattern
 * file stores them (-R 1, TemporaryFile.hpp:231-268 writePatternDontCareFree): 4 bases per byte, first base in bits 7..6,
 * every read starting on a byte boundary.  A quarter of the host-to-device traffic of the byte-per-base form.
 *   byte_offsets   nreads+1 offsets into packed, lengths nreads base counts; both may be NULL when uniform_length != 0
 *                  (all reads have that many bases and are stored back to back, ceil(L/4) bytes each)
 *   wildcard_flags nreads bytes, non-zero = the read contains a wildcard (such reads never match; the reference
 *                  keeps them in a separate 4 bit/base section) or NULL
 *   quality        one byte per BASE, reads back to back (as in real_gpu_set_reads), or NULL */
int real_gpu_set_reads_packed(real_gpu * h, const uint8_t * packed, const uint64_t * byte_offsets, const uint32_t * lengths,
                              uint32_t uniform_length, const uint8_t * wildcard_flags, const uint8_t * quality, uint64_t nreads);
/* Read set straight from the BYTES of a FASTA pattern file: the library runs the reference's pattern reader on the device (K0
 * in pattern-file mode, csrc/ingest.cuh) -- FastAReader::getNextPatternUnlocked (FastAReader.hpp:107-138: everything in front of
 * the first '>' is skipped; a '>' opens an id line that runs to the next '\n'; behind it every byte that is not white space is a
 * base of the read, up to the next '>' or the end of the file; an id line the file ends in without a '\n' opens no read) and
 * Pattern::computeMapped (Pattern.hpp:105-128: A C G T, anything else is a wildcard) -- and sets the result as the current read
 * set, 2 bit/base, as real_gpu_set_reads_packed would.  rewrite_order != 0 numbers the reads in the order of the reference's
 * rewritten pattern file (-R 1: by length, reads without wildcards first, file order inside a group; ReorderFastA.hpp) instead
 * of file order.  The ids (the bytes between '>' and '\n') are kept on the device for real_gpu_format_*; real_gpu_get_read_ids
 * and real_gpu_get_read_table copy ids, lengths and wildcard flags out, real_gpu_get_reads_packed the packed bytes.
 * *nreads = reads found.  Limits as for real_gpu_set_reads, and 2^32 bytes of packed reads / of ids per call. */
int real_gpu_set_reads_fasta(real_gpu * h, const void * fasta_bytes, uint64_t nbytes, uint32_t rewrite_order, uint64_t * nreads);
int real_gpu_get_read_table(real_gpu * h, uint32_t * lengths, uint8_t * wildcard_flags);
int real_gpu_get_read_ids(real_gpu * h, char * bytes, uint64_t * offsets);
int real_gpu_get_reads_packed(real_gpu * h, uint8_t * packed, uint64_t * byte_offsets);
int real_gpu_set_reads_device(real_gpu * h, const uint8_t * d_mapped, const uint8_t * d_quality,
                              const uint64_t * d_offsets, uint64_t nreads, uint64_t total_bases, uint32_t maxlen);
/* real_gpu_set_reads_packed for a read set of uniform length that is already in device memory (all pointers are
 * device pointers): the multi-GPU drivers upload 1/nranks of the reads per GPU and all-gather them over NVLink. */
int real_gpu_set_reads_packed_device(real_gpu * h, const uint8_t * d_packed, uint32_t uniform_length,
                                     const uint8_t * d_wildcard_flags, const uint8_t * d_quality, uint64_t nreads);
/* Device-pointer entry points (real_gpu_set_*_device, real_gpu_unique_export_*, real_gpu_unique_import) read and write
 * the caller's device buffers on the handle's own stream (real_gpu_stream): whatever produced the buffers on another
 * stream must have finished before the call (the caller synchronizes).
 * Asynchrony: the real_gpu_set_reads* calls return as soon as the caller's buffers have been consumed (copied, or for
 * device buffers packed); the index build they started keeps running on the handle's stream and is waited for by the
 * next call that needs it.  real_gpu_set_text* does not wait for it -- the text goes over a second stream -- so calling
 * set_reads, then set_text, then match overlaps the text transfer with the index build.  Every call still returns
 * only when the caller's buffers may be reused; errors of the deferred build are reported by the call that waits. */

/* All matches of every read against the current text: what AllMatcher::match + unifyMatches
 * accumulate over the file, sorted by (patid, k, pos, file, frag, score, inverted)
 * (matchAllImplementation.cpp:122-136).  *hits points to library-owned pinned host memory. */
int real_gpu_match_all(real_gpu * h, const real_gpu_hit ** hits, uint64_t * nhits);
/* The same matches in the same order as compact 16-byte rows (real_gpu_hit16): 2.5x less to read back over PCIe.  The
 * full rows stay on the device for real_gpu_format_all. */
int real_gpu_match_all_packed(real_gpu * h, const real_gpu_hit16 ** rows, uint64_t * nhits);

/* Folds the current text into the per-read unique state (UniqueMatcher::match for every read);
 * call once per file/shard, state persists like the reference's uniqueinfo array
 * (matchUniqueImplementation.cpp:1097).
 * Without scores the fold is order independent and the words equal the reference's bit for bit, with one exception the
 * reference itself leaves to its visiting order: the position / file / record fields of a word whose state is NonUnique
 * (two placements at the lowest error count) hold the placement the reference happened to visit first; here they hold the
 * smallest one (file, then position), which makes the word deterministic.  NonUnique reads are never printed, and tests and
 * gates compare those words by state and error count (matcher.canonical_unique, real_gpu_unique_checksum).
 * With scores (order dependent) the words and score bits equal the reference's exactly, given its text-block size
 * (real_gpu_set_block_windows). */
int real_gpu_match_unique(real_gpu * h);
/* Copies out the state: info[nreads] in UniqueMatchInfo bit layout (UniqueMatchInfo.hpp:26-39:
 * pos 35 | file 6 | err 4 | frag 16 | state 3, low to high), scores[nreads] or NULL. */
int real_gpu_get_unique(real_gpu * h, uint64_t * info, float * scores);
/* The same for the reads [first, first+count) only: after the cross-shard exchange every rank of a multi-GPU job holds
 * the merged state, and each reads back (formats, writes) its own 1/nranks of the reads. */
int real_gpu_get_unique_range(real_gpu * h, uint64_t first, uint64_t count, uint64_t * info, float * scores);
/* Order independent digest of the unique state of the reads [first, first+count), computed on the device: the sum over
 * the reads of splitmix64(canonical word ^ splitmix64(read ordinal)) mod 2^64 -- canonical = what the reference defines
 * independently of its visiting order (the whole word for Straight/Reverse, state and error count for NonUnique, the
 * state alone for NoMatch).  Digests of disjoint ranges add up: the ranks of a multi-GPU job digest their own reads.
 * Benchmarks and tests compare it with the digest of the single-GPU run / of the reference's dump. */
int real_gpu_unique_checksum(real_gpu * h, uint64_t first, uint64_t count, uint64_t * checksum);
/* Clears the unique state (fresh UniqueMatchInfo objects). */
int real_gpu_reset_unique(real_gpu * h);
/* With scores the unique fold is order dependent (UpdateUniqueInfo<true>::update, matchUniqueImplementation.cpp:179-248):
 * the reference visits the hits of a read text block by text block.  n_list = seed windows per reference text block
 * as its memory planner would choose them (matchUniqueImplementation.cpp:1208-1244); 0 = one block per file.
 * Also used by real_gpu_match_gaps.  In this mode the handle must hold the whole file (one shard). */
int real_gpu_set_block_windows(real_gpu * h, uint64_t n_list);
/* Test hook: the reference text blocks the order dependent folds would use on the current text with n_list windows per
 * block.  *nblocks receives their number (1 when n_list is 0 or the text has at most n_list seed windows) and
 * bounds[0 .. min(nblocks, cap)) the position of the first seed window of each block (bounds[0] = 0).  The handle's own
 * n_list (real_gpu_set_block_windows) is left as it was.  Needs the whole file in one shard. */
int real_gpu_get_block_bounds(real_gpu * h, uint64_t n_list, uint64_t * bounds, uint64_t cap, uint64_t * nblocks);

/* Cross-shard exchange for matchUnique without scores (SURVEY.md 8e): the per-read state is
 * exported as an order-preserving u64 key so that a MIN all-reduce followed by a SUM all-reduce of
 * the tie counts reproduces the reference's reduction over disjoint text shards.
 *   step 1: real_gpu_unique_export_keys   -> d_keys[nreads]   (device pointer owned by caller)
 *   step 2: caller all-reduces d_keys with MIN
 *   step 3: real_gpu_unique_export_ties   -> d_ties[nreads] u8: 1 where this shard holds a hit at the winning error count on a DIFFERENT position
 *   step 4: caller all-reduces d_ties with SUM
 *   step 5: real_gpu_unique_import        <- d_keys, d_ties; replaces the state by the merged one */
int real_gpu_unique_export_keys(real_gpu * h, uint64_t * d_keys);
int real_gpu_unique_export_ties(real_gpu * h, const uint64_t * d_min_keys, uint8_t * d_ties);
int real_gpu_unique_import(real_gpu * h, const uint64_t * d_min_keys, const uint8_t * d_tie_sums);

/* The same exchange over peer memory, as ONE step (reduce-scatter form; no collective library on the path): rank r of
 * nranks owns the reads [nreads r / nranks, nreads (r+1) / nranks).  Every rank stores the state words of each owner's
 * reads straight into the owner's staging area (NVLink peer stores, 8 bytes per read and peer), the ranks hand over with
 * release/acquire flags, and each owner folds the nranks words of its reads by the rule above.  Afterwards rank r holds
 * the merged UniqueMatchInfo words of ITS reads (real_gpu_get_unique_range); the words of the other reads keep the
 * rank's own contribution, so further files can be matched and folded again (the fold is idempotent and order
 * independent).  Without scores only.
 *   real_gpu_fold_init           allocates this rank's window for read sets of up to max_reads reads; handle_out receives
 *                                REAL_GPU_COMM_HANDLE_BYTES bytes (a CUDA IPC handle) to pass to the other ranks
 *   real_gpu_fold_connect        all_handles = the nranks handles in rank order (one process per GPU)
 *   real_gpu_fold_connect_local  the same for ranks that live in one process (peers = the nranks handles)
 *   real_gpu_fold_unique         collective over the ranks of a one-process-per-GPU job: call it on every rank after
 *                                real_gpu_match_unique; returns when this rank's reads are merged
 *   real_gpu_fold_unique_group   the ranks of ONE process (handles[r] = rank r), driven by one host thread */
int real_gpu_fold_init(real_gpu * h, uint32_t rank, uint32_t nranks, uint64_t max_reads, void * handle_out);
int real_gpu_fold_connect(real_gpu * h, const void * all_handles);
int real_gpu_fold_connect_local(real_gpu * h, real_gpu * const * peers);
int real_gpu_fold_unique(real_gpu * h);
int real_gpu_fold_unique_group(real_gpu * const * handles, uint32_t n);

/* Sharded tables: the multi-GPU form of the scan (SURVEY.md 8e; BASELINE.json north_star asks for the text to be
 * split over the GPUs of one box).  One handle = one rank = one GPU, at most 8.  Every rank is given the whole read
 * set and the whole text, but builds and keeps the index tables of its own 1/nranks of the signature space only
 * (scan buckets = the first 4 bases of a seed window).  In every round of the scan (round_positions text positions,
 * 0 = 2^30) each rank forms the window records of ITS slice of the positions and its partition kernel stores the
 * records of a bucket straight into the record area of the bucket's owner -- peer memory over NVLink, no staging
 * copy, no collective -- after which each owner probes what it was sent.  Ranks hand over with release/acquire
 * flags in each other's windows.  Every hit is found by exactly one rank; matchAll results are the union of the
 * ranks' results, matchUnique states are merged with the real_gpu_unique_export_* exchange below.
 *   real_gpu_comm_init           allocates this rank's window; call it BEFORE real_gpu_set_reads.  handle_out
 *                                receives REAL_GPU_COMM_HANDLE_BYTES bytes (a CUDA IPC handle) to pass to the others
 *   real_gpu_comm_connect        all_handles = the nranks handles in rank order (one process per GPU)
 *   real_gpu_comm_connect_local  the same for ranks that live in one process (peers = the nranks handles)
 * All ranks must use the same round_positions and make the same sequence of match calls.  Order dependent folds
 * (matchUnique with scores, real_gpu_match_gaps) are not available in this mode.  Seeds of fewer than 16 bases are
 * refused (REAL_GPU_E_ARG, the handle is left as it was): they have fewer than 256 scan buckets to split. */
#define REAL_GPU_COMM_HANDLE_BYTES 64
int real_gpu_comm_init(real_gpu * h, uint32_t rank, uint32_t nranks, uint64_t round_positions, void * handle_out);
int real_gpu_comm_connect(real_gpu * h, const void * all_handles);
int real_gpu_comm_connect_local(real_gpu * h, real_gpu * const * peers);

/* Bucket shards: the multi-GPU form of the scan without any record exchange.  Every rank is given the whole read set
 * and the whole text (the text is 2 bit/base: 0.78 GB for 3.1 Gbp); rank r builds and keeps the index tables of its
 * own 1/nranks of the signature space (the scan buckets [256 r / nranks, 256 (r+1) / nranks) = first 4 bases of a
 * seed window) and its partition kernel keeps only the text positions whose bucket it owns, so a rank does 1/nranks
 * of the index build, of the record traffic and of the probes.  Every hit is found by exactly one rank; matchAll
 * results are the union of the ranks' results, matchUnique states are merged with the real_gpu_unique_export_*
 * exchange above -- the only cross-GPU traffic of the path.  Call before real_gpu_set_reads.  Order dependent folds
 * (matchUnique with scores, real_gpu_match_gaps) are not available in this mode.  Seeds of fewer than 16 bases are
 * refused (REAL_GPU_E_ARG, the handle is left as it was): they have fewer than 256 scan buckets to split. */
int real_gpu_set_bucket_shard(real_gpu * h, uint32_t rank, uint32_t nranks);

/* Gapped extension pass (UniqueMatcher::matchGaps) for reads still NoMatch/Gapped; updates the
 * unique state (state Gapped, score, seed position).  gaps[nreads], present==1 where a GapInfo
 * entry exists. */
int real_gpu_match_gaps(real_gpu * h, uint64_t n_list_windows);
int real_gpu_get_gaps(real_gpu * h, real_gpu_gapinfo * gaps);

/* Output lines formatted on the device (K8, csrc/format.cuh).  Replaces the serial print loops of the reference:
 * matchAllImplementation.cpp:485-510 (one line per MatchPosAndError) and matchUniqueImplementation.cpp:252-321,1455-1486 (one
 * line per read whose state is Straight or Reverse):
 *     id \t bases \t [score] \t1\ta\t L \t +|- \t record name \t 1-based position in the record \t\t k \n
 * bases = toollib::remapString of the read ('-': of its reverse complement); the score is printed like an ostream with default
 * flags does (printf %g, bit-exact incl. rounding: csrc/fmt_g.h); no score column content when scores are off.
 *   real_gpu_set_read_ids      ids (the part of the '>'/'@' line the reference keeps) of the reads [first, first+count):
 *                              bytes + count+1 offsets.  Call after real_gpu_set_reads*; a rank of a multi-GPU job sets the
 *                              ids of the reads it will format (its own share after the fold).
 *   real_gpu_set_record_names  per text file: names of its records (bytes + nrecords+1 offsets) and their start offsets
 *   real_gpu_format_unique     the lines of the reads [first, first+count) from the current unique state (+ scores), in read order;
 *                              *nlines = reads that printed a line
 *   real_gpu_format_all        the lines of the rows [first_row, first_row+count) of the last real_gpu_match_all, in row order
 * *bytes points to library-owned pinned host memory that stays valid until the next-but-one format call (two buffers are
 * handed out in turn, so a writer thread can drain one batch while the next is formatted).  A batch is limited to 4 GiB of
 * output (REAL_GPU_E_LIMIT: format fewer items per call).  For reads given by real_gpu_set_reads_packed_device the caller's
 * device buffer must still be valid. */
int real_gpu_set_read_ids(real_gpu * h, uint64_t first, uint64_t count, const char * bytes, const uint64_t * offsets);
int real_gpu_set_record_names(real_gpu * h, uint32_t fileid, uint32_t nrecords, const char * bytes, const uint64_t * offsets,
                              const uint64_t * record_starts);
int real_gpu_format_unique(real_gpu * h, uint64_t first, uint64_t count, const char ** bytes, uint64_t * nbytes, uint64_t * nlines);
int real_gpu_format_all(real_gpu * h, uint64_t first_row, uint64_t count, const char ** bytes, uint64_t * nbytes);

/* Test hook: the score formatter of the device (csrc/fmt_g.h) on n host floats; out16 receives 16 bytes per value, the
 * characters followed by zero bytes. */
int real_gpu_selftest_format_scores(int device, const float * values, uint64_t n, char * out16);

/* Introspection for benchmarks and tests. */
int real_gpu_get_stats(real_gpu * h, real_gpu_stats * out);
void * real_gpu_stream(real_gpu * h);                  /* cudaStream_t the kernels are launched on */
uint64_t real_gpu_device_bytes(const real_gpu * h);    /* device memory currently held */

/* Counter-based synthetic inputs generated directly in device memory (benchmark tooling; the same
 * formulas as real_b200/synth.py). */
int real_gpu_synth_text(int device, uint64_t seed, uint64_t first_word, uint64_t nwords,
                        uint32_t n_per_million, uint64_t * d_words, uint64_t * d_nmask_or_null);
                        /* first_word must be even when d_nmask_or_null is given; it receives ceil(nwords/2) words */
int real_gpu_synth_reads(int device, uint64_t seed, const uint64_t * d_words, const uint64_t * d_nmask_or_null,
                         uint64_t text_n, uint64_t total_reads, uint64_t first_read, uint64_t nreads,
                         uint32_t length, uint32_t sub_per_16384, uint8_t * d_mapped, uint8_t * d_quality_or_null);

#ifdef __cplusplus
}
#endif
#endif
