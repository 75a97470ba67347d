// libreal_gpu.so -- C ABI (include/real_gpu.h) and host orchestration of the sm_100a kernels.
// No CPU fallback: every entry point that computes runs CUDA kernels on the handle's device.
#include "../../include/real_gpu.h"

#include "common.cuh"
#include "prims.cuh"
#include "index.cuh"
#include "scan.cuh"
#include "post.cuh"
#include "ingest.cuh"
#include "format.cuh"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <thread>
#include <cstring>
#include <cstdlib>
#include <cfloat>
#include <vector>

using namespace realgpu;

namespace
{

struct LimitError : public std::runtime_error
{
        explicit LimitError(std::string const & s) : std::runtime_error(s) {}
};

struct DevBuf
{
        void * p;
        size_t bytes;
        DevBuf() : p(nullptr), bytes(0) {}
};

struct Table
{
        DevBuf bitmap, E;
        uint32_t hb, nlists, nblocks;
        uint64_t nentries, ndistinct;
        size_t bitmap_bytes;
        Table() : hb(0), nlists(0), nblocks(0), nentries(0), ndistinct(0), bitmap_bytes(0) {}
};

} // namespace

struct real_gpu
{
        real_gpu_params prm;
        std::string err;
        cudaStream_t st;               // every kernel of the path
        cudaStream_t st2;              // host<->device copies of the text, so that they overlap the index build on st
        cudaEvent_t ev[8];
        cudaEvent_t evc[2];
        cudaEvent_t ev_words;          // real_gpu_set_text_async: the text words are on the device (the partition may start; the probe waits for evc[1])
        bool text_pending;             // an asynchronous text copy has been enqueued and not yet waited for by the host
        // real_gpu_set_text_async leaves the copy of the wildcard mask to the next call that can place it: behind the reads of a
        // real_gpu_set_reads* call that follows (the index build needs the reads, the mask is read by the probe only) or, at the
        // latest, at the start of the scan
        const uint64_t * mask_src; uint64_t mask_words; bool mask_deferred;
        bool mask_on_device;           // real_gpu_set_text_device_async: mask_src is a device pointer whose contents the caller completes before the match call
        // real_gpu_prepare_scan: the text records formed ahead of the match call, on a stream of their own
        struct Prepared
        {
                bool valid, inflight, ahead;   // ahead: formed by real_gpu_prepare_scan (else: left behind by the last scan)
                uint64_t x_begin, x_end, win_begin, win_end, chunk_cap;
                uint32_t bucket_bits, own_b_lo, own_b_cnt;
                bool own_list;
                const void * recs;             // where the records are: a buffer that has been re-allocated since does not hold them
                cudaEvent_t ev0, done;
                Prepared() : valid(false), inflight(false), ahead(false), x_begin(0), x_end(0), win_begin(0), win_end(0), chunk_cap(0), bucket_bits(0), own_b_lo(0), own_b_cnt(0),
                             own_list(false), recs(nullptr), ev0(nullptr), done(nullptr) {}
        } prep;
        cudaStream_t st3;              // the partition kernels of real_gpu_prepare_scan
        bool auto_prepare;             // real_gpu_set_text* prepares the scan itself when the read set is known (REAL_GPU_AUTO_PREPARE=0 turns it off)
        std::vector<cudaEvent_t> evp;  // pairs around the probe kernel of every chunk of a scan (stats.probe_ms)
        bool fused_build;              // the current tables were built by build_tables_fused (entry arrays in item numbering)
        bool build_pending;            // the index build of the current read set has been enqueued but not yet waited for
        uint64_t held;
        int sm_count;

        // text
        bool have_text;
        DevBuf text, nmask, rec;
        uint64_t n_total, shard_begin, shard_len, own_begin, own_end;
        uint32_t nrec, fileid;
        // text ingest (real_gpu_set_text_fasta*): file bytes, tile summaries and offsets, record table of the last file
        DevBuf fa_raw, fa_sums, fa_tbase, fa_trec, fa_recnl, fa_tot;
        uint64_t * fa_totals;          // [2] pinned host memory: kept bases, records
        std::vector<uint64_t> fa_rec_starts, fa_rec_nl;

        // reads
        bool have_reads;
        DevBuf mapped, qual, offs, rpack, rlen, seeds, usable, usable_rank, bad;
        uint64_t nreads, n_usable, total_bases;
        uint32_t W, maxlen;
        bool qual_present;

        // index
        Table tab[3];
        uint32_t F, keybits;

        // results
        DevBuf rec_win, rec_pos, part_meta, own_list, large_list;
        DevBuf win_valid, win_counts, bounds, gapres, gaps, boffs, flags8;   // reference text blocks (order-faithful replay)
        uint64_t n_list;               // windows per reference text block, 0 = one block per file
        DevBuf ws_k0, ws_v0, ws_k1, ws_v1, ws_flags, ws_hist, ws_stmp;   // index build workspace, kept between calls
        uint32_t * table_counts;       // [6] pinned host memory; per table: entries, distinct slots (copied back asynchronously by the build)
        const uint8_t * src_packed; const uint64_t * src_byte_offsets; uint32_t src_packed_uniform;   // 2-bit input (set_reads_packed)
        const uint32_t * src_len32;    // 2-bit input with per-read lengths instead of base offsets (set_reads_fasta)
        DevBuf rd_raw, rd_sums, rd_tbase, rd_trec, rd_stream, rd_mask, rd_start, rd_nl, rd_open, rd_len, rd_wild, rd_idlen, rd_perm, rd_olen, rd_obytes, rd_oidlen, rd_boff, rd_ioff, rd_misc;   // K0 for pattern files
        const uint8_t * src_mapped;    // device pointer the reads are packed from (caller's buffer or h->mapped)
        DevBuf ll, hits_raw, hits_seg, hits_out, hits_out16, counters, counts, starts, cursor, scantmp, info, scores;
        uint64_t hit_cap;
        real_gpu_hit * host_hits;
        uint64_t host_hits_cap;

        // sharded tables (real_gpu_comm_*): one window per rank = {flags, bucket counts per source, record area}
        struct Comm
        {
                uint32_t nranks, rank, epoch, seg_cap;
                uint64_t round_positions;
                DevBuf window, ptrs, pairs, error;
                size_t meta_off, recs_off;
                char * base[SC_MAX_RANKS];      // window of every rank as mapped into this process
                bool ipc_opened[SC_MAX_RANKS];
                bool connected;
                // ranks that live in one process (real_gpu_comm_connect_local) hand over with CUDA events instead of
                // spinning on the device: kernels of different streams of ONE context may share a hardware queue, and
                // a kernel that spins at the head of such a queue would hold back the very kernels it waits for
                real_gpu * local[SC_MAX_RANKS];
                cudaEvent_t ev[2];
                std::atomic<uint32_t> enqueued[2];      // last round whose signal of slot 0/1 has been recorded on this rank's stream
                uint32_t bucket_lo[SC_MAX_RANKS + 1];
                Comm() : nranks(1), rank(0), epoch(0), seg_cap(0), round_positions(0), meta_off(0), recs_off(0), connected(false)
                { for ( int i = 0; i < SC_MAX_RANKS; ++i ) { base[i] = nullptr; ipc_opened[i] = false; local[i] = nullptr; } for ( int i = 0; i <= SC_MAX_RANKS; ++i ) bucket_lo[i] = 0;
                  ev[0] = ev[1] = nullptr; enqueued[0] = 0; enqueued[1] = 0; }
        } comm;

        // peer-memory fold of the unique state (real_gpu_fold_*): one window per rank = {flags, two staging areas}
        struct Fold
        {
                uint32_t nranks, rank, epoch;
                uint64_t cap, seg;              // reads the window was sized for; words per source in a staging area
                DevBuf window, ptrs, error;
                size_t stage_off;
                char * base[SC_MAX_RANKS];
                bool ipc_opened[SC_MAX_RANKS];
                real_gpu * local[SC_MAX_RANKS];
                bool connected;
                cudaEvent_t ev;                 // ranks of one process: "my words are pushed"
                Fold() : nranks(1), rank(0), epoch(0), cap(0), seg(0), stage_off(4096), connected(false), ev(nullptr)
                { for ( int i = 0; i < SC_MAX_RANKS; ++i ) { base[i] = nullptr; ipc_opened[i] = false; local[i] = nullptr; } }
        } fold;

        // output lines formatted on the device (real_gpu_format_*, csrc/format.cuh)
        struct Format
        {
                DevBuf ids, id_off, names, name_off, rec_start, file_first, len, off, out;
                uint64_t id_first, id_count, id_bytes, max_name;
                std::vector<char> file_names[64];                // per file: the record names back to back
                std::vector<uint64_t> file_name_off[64], file_starts[64];
                bool tables_dirty;
                char * host[2]; size_t host_cap[2]; int flip;    // two pinned buffers handed out in turn
                uint64_t nrows_all;                              // rows of the last real_gpu_match_all
                Format() : id_first(0), id_count(0), id_bytes(0), max_name(0), tables_dirty(true), flip(0), nrows_all(0) { host[0] = host[1] = nullptr; host_cap[0] = host_cap[1] = 0; }
        } fmt;

        // pageable host memory -> device through pinned staging buffers filled by a few host threads (h2d_from_host)
        void * stage_buf[8]; cudaStream_t stage_st[4];

        real_gpu_stats stats;

        real_gpu() : n_list(0), src_packed(nullptr), src_byte_offsets(nullptr), src_packed_uniform(0), src_len32(nullptr), src_mapped(nullptr), fused_build(false), st(nullptr), st2(nullptr), build_pending(false), table_counts(nullptr), fa_totals(nullptr), held(0), sm_count(148), have_text(false), n_total(0), shard_begin(0), shard_len(0), own_begin(0), own_end(0),
                     nrec(0), fileid(0), have_reads(false), nreads(0), n_usable(0), total_bases(0), W(0), maxlen(0), qual_present(false),
                     F(0), keybits(0), hit_cap(0), host_hits(nullptr), host_hits_cap(0)
        {
                memset(&prm, 0, sizeof(prm));
                memset(&stats, 0, sizeof(stats));
                for ( int i = 0; i < 8; ++i ) ev[i] = nullptr;
                evc[0] = evc[1] = nullptr; ev_words = nullptr; text_pending = false;
                mask_src = nullptr; mask_words = 0; mask_deferred = false; mask_on_device = false; st3 = nullptr; auto_prepare = true;
                for ( int i = 0; i < 8; ++i ) stage_buf[i] = nullptr;
                for ( int i = 0; i < 4; ++i ) stage_st[i] = nullptr;
        }
};

namespace
{

void dev_free(real_gpu * h, DevBuf & b)
{
        if ( b.p )
        {
                cudaFree(b.p);
                h->held -= b.bytes;
        }
        b.p = nullptr; b.bytes = 0;
}

void dev_alloc(real_gpu * h, DevBuf & b, size_t bytes)
{
        dev_free(h, b);
        if ( bytes == 0 ) bytes = 16;
        RG_CUDA(cudaMalloc(&b.p, bytes));
        b.bytes = bytes;
        h->held += bytes;
}

// grows only
void dev_reserve(real_gpu * h, DevBuf & b, size_t bytes)
{
        if ( b.bytes < bytes || ! b.p )
                dev_alloc(h, b, bytes);
}

template<typename T> T * ptr(DevBuf const & b) { return reinterpret_cast<T *>(b.p); }

inline unsigned blocks_for(uint64_t n, unsigned threads) { return (unsigned)((n + threads - 1) / threads); }

void launch_count(real_gpu * h, uint32_t n = 1) { h->stats.total_launches += n; }

float elapsed(cudaEvent_t a, cudaEvent_t b)
{
        float ms = 0;
        cudaEventElapsedTime(&ms, a, b);
        return ms;
}

int fail(real_gpu * h, int code, std::string const & msg)
{
        if ( h ) h->err = msg;
        return code;
}

void finish_build(real_gpu * h);
// every entry point first waits for an index build that is still in flight -- except the ones that set the text,
// whose transfer is meant to overlap it
#define RG_API_BEGIN(h)  if ( ! (h) ) return REAL_GPU_E_ARG; try { RG_CUDA(cudaSetDevice((h)->prm.device)); finish_build(h);
#define RG_API_BEGIN_ASYNC(h)  if ( ! (h) ) return REAL_GPU_E_ARG; try { RG_CUDA(cudaSetDevice((h)->prm.device));
#define RG_API_END(h)    } catch ( LimitError const & e ) { return fail((h), REAL_GPU_E_LIMIT, e.what()); } \
                           catch ( realgpu::CudaError const & e ) { return fail((h), REAL_GPU_E_CUDA, e.what()); } \
                           catch ( std::exception const & e ) { return fail((h), REAL_GPU_E_CUDA, e.what()); }


// Host bytes -> device.  Pinned (or registered) memory goes as one asynchronous copy on `st`.  Pageable memory -- the mapped
// bytes of a FASTA file, typically -- would crawl through the driver's single staging path (about 5 GB/s measured: 1.1 s for
// the 5.6 GB pattern file of C3): four host threads copy 16 MB pieces into pinned buffers of their own (two each) and send
// them on streams of their own, so the page-cache reads, the staging copies and the PCIe transfers overlap.  Returns when the
// bytes are on the device (the kernels on `st` may be launched right after).
void h2d_from_host(real_gpu * h, void * dst, const void * src, size_t nbytes, cudaStream_t st)
{
        if ( ! nbytes ) return;
        cudaPointerAttributes attr;
        bool pageable = true;
        if ( cudaPointerGetAttributes(&attr, src) == cudaSuccess ) pageable = attr.type == cudaMemoryTypeUnregistered;
        else cudaGetLastError();
        size_t const piece = 16u << 20;
        if ( ! pageable || nbytes < 4 * piece )
        {
                RG_CUDA(cudaMemcpyAsync(dst, src, nbytes, cudaMemcpyHostToDevice, st));
                RG_CUDA(cudaStreamSynchronize(st));
                return;
        }
        for ( int i = 0; i < 8; ++i ) if ( ! h->stage_buf[i] ) RG_CUDA(cudaMallocHost(&h->stage_buf[i], piece));
        for ( int i = 0; i < 4; ++i ) if ( ! h->stage_st[i] ) RG_CUDA(cudaStreamCreateWithFlags(&h->stage_st[i], cudaStreamNonBlocking));
        RG_CUDA(cudaStreamSynchronize(st));              // whatever was writing dst before
        size_t const npieces = (nbytes + piece - 1) / piece;
        std::atomic<int> failed(0);
        std::vector<std::thread> team;
        for ( int t = 0; t < 4; ++t )
                team.push_back(std::thread([h, t, dst, src, nbytes, piece, npieces, &failed]()
                {
                        if ( cudaSetDevice(h->prm.device) != cudaSuccess ) { failed = 1; return; }
                        cudaEvent_t ev[2] = { nullptr, nullptr };
                        bool used[2] = { false, false };
                        for ( int k = 0; k < 2; ++k ) if ( cudaEventCreateWithFlags(&ev[k], cudaEventDisableTiming) != cudaSuccess ) failed = 1;
                        int k = 0;
                        for ( size_t i = (size_t)t; i < npieces && ! failed; i += 4, k ^= 1 )
                        {
                                size_t const off = i * piece, n = std::min(piece, nbytes - off);
                                if ( used[k] && cudaEventSynchronize(ev[k]) != cudaSuccess ) { failed = 1; break; }
                                memcpy(h->stage_buf[2 * t + k], static_cast<const char *>(src) + off, n);
                                if ( cudaMemcpyAsync(static_cast<char *>(dst) + off, h->stage_buf[2 * t + k], n, cudaMemcpyHostToDevice, h->stage_st[t]) != cudaSuccess
                                     || cudaEventRecord(ev[k], h->stage_st[t]) != cudaSuccess ) { failed = 1; break; }
                                used[k] = true;
                        }
                        if ( cudaStreamSynchronize(h->stage_st[t]) != cudaSuccess ) failed = 1;
                        for ( int q = 0; q < 2; ++q ) if ( ev[q] ) cudaEventDestroy(ev[q]);
                }));
        for ( std::thread & th : team ) th.join();
        if ( failed ) { cudaGetLastError(); throw CudaError("host to device copy through the staging buffers failed"); }
}

// ---------------------------------------------------------------------------------------------
// text
// ---------------------------------------------------------------------------------------------

// enqueues the copy of the wildcard mask real_gpu_set_text_async has left to a later call.  behind_reads: called by a
// real_gpu_set_reads* -- a mask in device memory (real_gpu_set_text_device_async) is not touched yet: its owner may still be
// completing it (it has until the match call)
void flush_mask(real_gpu * h, bool behind_reads = false)
{
        if ( ! h->mask_deferred ) return;
        if ( behind_reads && h->mask_on_device ) return;
        h->mask_deferred = false;
        RG_CUDA(cudaMemcpyAsync(ptr<uint64_t>(h->nmask) + TEXT_PAD_WORDS, h->mask_src, h->mask_words * 8,
                                h->mask_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, h->st2));
        RG_CUDA(cudaEventRecord(h->evc[1], h->st2));
}

// waits (on the host) for a text copy real_gpu_set_text_async has left in flight
void finish_text(real_gpu * h)
{
        if ( ! h->text_pending ) return;
        flush_mask(h);
        h->text_pending = false;
        RG_CUDA(cudaEventSynchronize(h->evc[1]));
        h->stats.h2d_text_ms = elapsed(h->evc[0], h->evc[1]);
}

void auto_prepare_scan(real_gpu * h);

// the records real_gpu_prepare_scan has formed (or is forming) are given up: the text, the shard or the buffers change
void drop_prepared(real_gpu * h)
{
        if ( h->prep.inflight ) cudaEventSynchronize(h->prep.done);
        h->prep.inflight = false;
        h->prep.valid = false;
}

int set_text_common(real_gpu * h, uint32_t fileid, const uint64_t * words, const uint64_t * nmask, bool on_device,
                    uint64_t n_total, uint64_t shard_begin, uint64_t shard_len, uint64_t own_begin, uint64_t own_end,
                    const uint64_t * record_starts, uint32_t nrecords, bool async_copy = false)
{
        finish_text(h);
        drop_prepared(h);
        if ( ! words || ! nmask || ! record_starts || nrecords == 0 )
                return fail(h, REAL_GPU_E_ARG, "set_text: null pointer or no records");
        if ( shard_begin % 64 )
                return fail(h, REAL_GPU_E_ARG, "set_text: shard_begin must be a multiple of 64");
        if ( shard_begin + shard_len > n_total || own_begin > own_end || own_end > n_total || own_begin < shard_begin )
                return fail(h, REAL_GPU_E_ARG, "set_text: inconsistent shard/own ranges");
        if ( n_total >= (1ULL << 35) )
                return fail(h, REAL_GPU_E_LIMIT, "set_text: text longer than 2^35 bases (UniqueMatchInfo.hpp:29-33)");
        if ( fileid >= 64 )
                return fail(h, REAL_GPU_E_LIMIT, "set_text: fileid >= 64 (UniqueMatchInfo.hpp:31)");
        if ( record_starts[nrecords] != n_total )
                return fail(h, REAL_GPU_E_ARG, "set_text: record_starts[nrecords] must equal n_total");

        if ( own_end > shard_begin + shard_len )
                return fail(h, REAL_GPU_E_ARG, "set_text: the own range must lie inside the shard");
        if ( nrecords >= (1u << 24) )
                return fail(h, REAL_GPU_E_LIMIT, "set_text: more than 2^24 records (the record index of a hit has 24 bits)");
        h->have_text = false;          // whatever fails below, the old text is gone

        uint64_t const nw = (shard_len + 31) / 32, nmw = (shard_len + 63) / 64;
        size_t const tail = TEXT_PAD_WORDS + 2 * SC_SMEM_WORDS + SC_TILE_WORDS + 2 * OL_TILE_WORDS;     // the last tile of every kernel stays inside the allocation
        size_t const tbytes = (TEXT_PAD_WORDS + nw + tail) * 8, mbytes = (TEXT_PAD_WORDS + nmw + tail) * 8;

        // The text goes over the copy stream: an index build that real_gpu_set_reads* has left running on the kernel
        // stream (it does not touch the text) overlaps the transfer.  Scans are over when their call returns, so
        // nothing on the kernel stream still reads the old text.
        dev_reserve(h, h->text, tbytes);
        dev_reserve(h, h->nmask, mbytes);
        dev_reserve(h, h->rec, (size_t)(nrecords + 1) * 8);
        RG_CUDA(cudaEventRecord(h->evc[0], h->st2));
        // the padding in front and behind (the words in between are overwritten by the copy)
        RG_CUDA(cudaMemsetAsync(h->text.p, 0, TEXT_PAD_WORDS * 8, h->st2));
        RG_CUDA(cudaMemsetAsync(ptr<uint64_t>(h->text) + TEXT_PAD_WORDS + nw, 0, tail * 8, h->st2));
        RG_CUDA(cudaMemsetAsync(h->nmask.p, 0, TEXT_PAD_WORDS * 8, h->st2));
        RG_CUDA(cudaMemsetAsync(ptr<uint64_t>(h->nmask) + TEXT_PAD_WORDS + nmw, 0, tail * 8, h->st2));
        cudaMemcpyKind const kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
        // the words first: the partition kernels of a scan need nothing else (the wildcard mask is read by the probe only)
        RG_CUDA(cudaMemcpyAsync(h->rec.p, record_starts, (size_t)(nrecords + 1) * 8, cudaMemcpyHostToDevice, h->st2));
        RG_CUDA(cudaMemcpyAsync(ptr<uint64_t>(h->text) + TEXT_PAD_WORDS, words, nw * 8, kind, h->st2));
        RG_CUDA(cudaEventRecord(h->ev_words, h->st2));
        if ( async_copy )
        {
                // the mask is read by the probe only: its copy is placed by flush_mask -- behind the reads of a real_gpu_set_reads*
                // call that comes next (text first, reads second: the partition runs while the reads arrive), else when the scan starts;
                // a mask in device memory is copied when the scan starts (the caller may complete it until then)
                h->mask_src = nmask; h->mask_words = nmw; h->mask_deferred = true; h->mask_on_device = on_device;
        }
        else
        {
                RG_CUDA(cudaMemcpyAsync(ptr<uint64_t>(h->nmask) + TEXT_PAD_WORDS, nmask, nmw * 8, kind, h->st2));
                RG_CUDA(cudaEventRecord(h->evc[1], h->st2));
        }
        if ( async_copy )
                h->text_pending = true;                 // real_gpu_set_text_async: the scan waits on the device, the host at its end
        else
        {
                RG_CUDA(cudaEventSynchronize(h->evc[1]));       // the caller's buffers are free again; later launches on the kernel stream come after
                h->stats.h2d_text_ms = elapsed(h->evc[0], h->evc[1]);
        }

        h->fileid = fileid; h->n_total = n_total; h->shard_begin = shard_begin; h->shard_len = shard_len;
        h->own_begin = own_begin; h->own_end = own_end; h->nrec = nrecords;
        h->fa_rec_starts.clear(); h->fa_rec_nl.clear();
        h->have_text = true;
        auto_prepare_scan(h);
        return REAL_GPU_OK;
}

// K0: the text straight from the bytes of its FASTA file (ingest.cuh).  Everything runs on the copy stream, like the
// transfer of a packed text, so an index build in flight on the kernel stream overlaps it.
int set_text_fasta_common(real_gpu * h, uint32_t fileid, const void * bytes, uint64_t nbytes, bool on_device, uint64_t * n_bases, uint64_t * nrecords)
{
        if ( (! bytes && nbytes) || ! n_bases || ! nrecords )
                return fail(h, REAL_GPU_E_ARG, "set_text_fasta: null pointer");
        if ( on_device && ((uintptr_t)bytes & 15) )
                return fail(h, REAL_GPU_E_ARG, "set_text_fasta_device: the buffer must be 16-byte aligned");
        if ( fileid >= 64 )
                return fail(h, REAL_GPU_E_LIMIT, "set_text: fileid >= 64 (UniqueMatchInfo.hpp:31)");
        uint64_t const ntiles = (nbytes + FA_TILE - 1) / FA_TILE;
        if ( ntiles >= (1ULL << 31) )
                return fail(h, REAL_GPU_E_LIMIT, "set_text_fasta: file longer than 2^43 bytes");
        finish_text(h);
        drop_prepared(h);
        h->have_text = false;
        h->fa_rec_starts.clear(); h->fa_rec_nl.clear();
        *n_bases = 0; *nrecords = 0;

        RG_CUDA(cudaEventRecord(h->evc[0], h->st2));
        const uint8_t * d_raw = static_cast<const uint8_t *>(bytes);
        if ( ! on_device )
        {
                dev_reserve(h, h->fa_raw, nbytes);
                h2d_from_host(h, h->fa_raw.p, bytes, nbytes, h->st2);
                d_raw = ptr<uint8_t>(h->fa_raw);
        }
        dev_reserve(h, h->fa_sums, ntiles * sizeof(FaSum32));
        dev_reserve(h, h->fa_tbase, ntiles * 8);
        dev_reserve(h, h->fa_trec, ntiles * 8);
        dev_reserve(h, h->fa_tot, 16);
        if ( ntiles )
                k_fa_summary<<<(unsigned)ntiles, FA_THREADS, 0, h->st2>>>(d_raw, nbytes, ptr<FaSum32>(h->fa_sums), 0u);
        k_fa_scan<<<1, FA_SCAN_THREADS, 0, h->st2>>>(ptr<FaSum32>(h->fa_sums), ntiles, ptr<uint64_t>(h->fa_tbase), ptr<uint64_t>(h->fa_trec), ptr<uint64_t>(h->fa_tot));
        RG_CUDA(cudaGetLastError());
        launch_count(h, ntiles ? 2 : 1);
        RG_CUDA(cudaMemcpyAsync(h->fa_totals, h->fa_tot.p, 16, cudaMemcpyDeviceToHost, h->st2));
        RG_CUDA(cudaStreamSynchronize(h->st2));                 // the caller's bytes are on the device; the sizes are known
        uint64_t const n = h->fa_totals[0], nrec = h->fa_totals[1];
        *n_bases = n; *nrecords = nrec;
        if ( n >= (1ULL << 35) )
                return fail(h, REAL_GPU_E_LIMIT, "set_text: text longer than 2^35 bases (UniqueMatchInfo.hpp:29-33)");
        if ( nrec >= (1ULL << 24) )
                return fail(h, REAL_GPU_E_LIMIT, "set_text_fasta: more than 2^24 records (the record index of a hit has 24 bits)");
        if ( n == 0 || nrec == 0 )
                return REAL_GPU_OK;                             // nothing to match against; no text is set

        uint64_t const nw = (n + 31) / 32, nmw = (n + 63) / 64;
        size_t const tail = TEXT_PAD_WORDS + 2 * SC_SMEM_WORDS + SC_TILE_WORDS + 2 * OL_TILE_WORDS;
        size_t const tbytes = (TEXT_PAD_WORDS + nw + tail) * 8, mbytes = (TEXT_PAD_WORDS + nmw + tail) * 8;
        dev_reserve(h, h->text, tbytes);
        dev_reserve(h, h->nmask, mbytes);
        dev_reserve(h, h->rec, (size_t)(nrec + 1) * 8);
        dev_reserve(h, h->fa_recnl, (size_t)nrec * 8);
        RG_CUDA(cudaMemsetAsync(h->text.p, 0, tbytes, h->st2));
        RG_CUDA(cudaMemsetAsync(h->nmask.p, 0, mbytes, h->st2));
        k_fa_pack<<<(unsigned)ntiles, FA_THREADS, 0, h->st2>>>(d_raw, nbytes, ptr<uint64_t>(h->fa_tbase), ptr<uint64_t>(h->fa_trec),
                                                               ptr<unsigned long long>(h->text) + TEXT_PAD_WORDS, ptr<unsigned long long>(h->nmask) + TEXT_PAD_WORDS,
                                                               ptr<uint64_t>(h->rec), ptr<uint64_t>(h->fa_recnl), nullptr, 0u);
        RG_CUDA(cudaGetLastError());
        launch_count(h);
        RG_CUDA(cudaMemcpyAsync(ptr<uint64_t>(h->rec) + nrec, h->fa_totals, 8, cudaMemcpyHostToDevice, h->st2));
        RG_CUDA(cudaEventRecord(h->evc[1], h->st2));
        h->fa_rec_starts.resize(nrec + 1); h->fa_rec_nl.resize(nrec);
        RG_CUDA(cudaMemcpyAsync(&h->fa_rec_starts[0], h->rec.p, (size_t)(nrec + 1) * 8, cudaMemcpyDeviceToHost, h->st2));
        RG_CUDA(cudaMemcpyAsync(&h->fa_rec_nl[0], h->fa_recnl.p, (size_t)nrec * 8, cudaMemcpyDeviceToHost, h->st2));
        RG_CUDA(cudaStreamSynchronize(h->st2));
        h->stats.h2d_text_ms = elapsed(h->evc[0], h->evc[1]);   // transfer of the file bytes + the three ingest kernels
        if ( ! on_device && h->fa_raw.bytes > (64u << 20) )
                dev_free(h, h->fa_raw);                         // the file bytes are ~2.7x the packed text: not kept between files

        h->fileid = fileid; h->n_total = n; h->shard_begin = 0; h->shard_len = n;
        h->own_begin = 0; h->own_end = n; h->nrec = (uint32_t)nrec;
        h->have_text = true;
        auto_prepare_scan(h);
        return REAL_GPU_OK;
}

// ---------------------------------------------------------------------------------------------
// reads + index
// ---------------------------------------------------------------------------------------------

// geometry and partition parameters of one table
struct TablePlan
{
        EntryPartParams EP;
        uint32_t e2, nsub, sub_shift, words, first_sub, own_subs;
        uint32_t * d_total, * d_ndist;
        bool empty;
};
static const size_t TABLE_META_WORDS = 1024 + 256 * EP_CURSOR_STRIDE;

// sizes, buffers and the level-1 parameters of table t; meta = its bookkeeping words, cleared here
TablePlan plan_table(real_gpu * h, int t, uint32_t * meta)
{
        TablePlan TP;
        memset(&TP, 0, sizeof(TP));
        Table & T = h->tab[t];
        T.nlists = table_lists(t, h->prm.seedkmax);
        uint64_t const cap_entries = h->nreads * 2 * T.nlists;        // upper bound (unusable reads produce none)
        T.nentries = 0;
        {
                // automatic: about 32 slots per entry of the largest table, at least 2^20, at most the key width / 32 bits
                uint32_t const cap = std::min<uint32_t>(h->keybits, 32);
                uint64_t const want = std::max<uint64_t>(1, h->nreads * 2 * table_lists(0, h->prm.seedkmax)) * 32;
                uint32_t autob = 20;
                while ( autob < cap && (1ULL << autob) < want ) ++autob;
                T.hb = h->prm.table_bits ? std::min<uint32_t>(h->prm.table_bits, cap) : std::min<uint32_t>(autob, cap);
                if ( T.hb < h->keybits && T.hb < SLOT_PREFIX_BITS + 4 ) T.hb = std::min<uint32_t>(cap, SLOT_PREFIX_BITS + 4);
        }
        T.ndistinct = 0;
        // partition depth: sub-buckets of about SUB_TARGET_ENTRIES entries, of at most 2^16 slots, of whole slot words
        uint32_t const pbmin = T.hb > 16 ? T.hb - 16 : 0, pbmax = std::min<uint32_t>(16, T.hb > 5 ? T.hb - 5 : 0);
        uint32_t pb = 0;
        while ( (cap_entries >> pb) > SUB_TARGET_ENTRIES ) ++pb;
        pb = std::min(std::max(pb, pbmin), pbmax);
        uint32_t const e1 = std::min<uint32_t>(8, pb);
        TP.e2 = pb - e1;
        TP.nsub = 1u << pb; TP.sub_shift = T.hb - pb;
        TP.words = TP.sub_shift >= 5 ? (1u << (TP.sub_shift - 5)) : 1u;
        T.nblocks = TP.nsub;
        T.bitmap_bytes = (size_t)TP.nsub * TP.words * sizeof(SlotWord);
        dev_reserve(h, T.bitmap, T.bitmap_bytes);
        EntryPartParams & EP = TP.EP;
        EP.G.F = h->F; EP.G.keybits = h->keybits; EP.G.hb = T.hb; EP.G.nlists = 0; EP.G.table = t;
        if ( T.nlists == 0 || h->nreads == 0 )
        {
                RG_CUDA(cudaMemsetAsync(T.bitmap.p, 0, T.bitmap_bytes, h->st));
                TP.empty = true;
                return TP;
        }
        if ( cap_entries >= 0xFFFFFFFFULL )
                throw CudaError("index: more than 2^32 entries in one table");

        // meta layout (u32): [0,256) bucket counts, [256,513) bucket starts, 520 total, 521 ndistinct, [600,857) level-2 tile starts, [1024, ...) cursors
        EP.seeds = ptr<uint64_t>(h->seeds); EP.usable = ptr<uint32_t>(h->usable); EP.nids = 2 * h->nreads;
        EP.G.nlists = T.nlists;
        EP.ebits = e1; EP.e2bits = TP.e2;
        EP.own_shift = 0; EP.own_lo = 0; EP.own_last = 0xFFFFFFFFu;
        TP.first_sub = 0; TP.own_subs = TP.nsub;
        if ( h->comm.nranks > 1 )
        {
                // this rank owns the slots whose top 8 bits (= top 8 bits of the key = scan bucket) fall into its bucket range
                if ( T.hb < 8 ) throw CudaError("sharded tables need presence tables of at least 2^8 slots");
                EP.own_shift = T.hb - 8; EP.own_lo = h->comm.bucket_lo[h->comm.rank]; EP.own_last = h->comm.bucket_lo[h->comm.rank + 1] - 1;
                if ( pb >= 8 )
                {
                        TP.first_sub = EP.own_lo << (pb - 8);
                        TP.own_subs = (EP.own_last + 1 - EP.own_lo) << (pb - 8);
                }
        }
        EP.ent_seed = ptr<uint64_t>(h->ws_k0); EP.ent_val = ptr<uint32_t>(h->ws_v0);
        EP.ent2_seed = ptr<uint64_t>(h->ws_k1); EP.ent2_val = ptr<uint32_t>(h->ws_v1);
        EP.bucket_count = meta; EP.bucket_start = meta + 256; EP.tile_start = meta + 600; EP.bucket_cursor = meta + 1024;
        uint32_t * sub = ptr<uint32_t>(h->ws_flags);
        EP.sub_count = sub; EP.sub_start = sub + 65600; EP.sub_cursor = sub + 2 * 65600;
        TP.d_total = meta + 520; TP.d_ndist = meta + 521;
        RG_CUDA(cudaMemsetAsync(meta, 0, 1024 * 4, h->st));
        return TP;
}

// one table, its level-1 histogram already counted: group the entries by slot prefix (two levels; the grouped
// entries of the tables share one workspace, so the tables are built one after the other), then build every
// sub-bucket in shared memory
struct Grouped { const uint64_t * seed; const uint32_t * val; const uint32_t * start; };

// the two staged partition passes over the entries (or items) of TP: grouped by the top e1, then by the next e2 bits of the slot
Grouped partition_entries(real_gpu * h, TablePlan const & TP)
{
        EntryPartParams const & EP = TP.EP;
        k_ent_offsets<<<1, EP_MAX_BUCKETS, 0, h->st>>>(EP, TP.d_total);
        RG_KERNEL_CHECK();
        size_t const esmem = sizeof(EntryPartSmem);
        RG_CUDA(cudaFuncSetAttribute(k_ent_scatter, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)esmem));
        RG_CUDA(cudaFuncSetAttribute(k_ent2_scatter, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)esmem));
        int occ = 0, occ2 = 0, occh = 0;
        RG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_ent_scatter, 256, esmem));
        RG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ2, k_ent2_scatter, 256, esmem));
        RG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occh, k_ent2_hist, 256, 0));
        uint64_t const etiles = (EP.nids + EP_TILE_IDS - 1) / EP_TILE_IDS;
        if ( h->comm.nranks > 1 )
        {
                size_t const osmem = sizeof(EntryOwnSmem);
                int occ_o = 0;
                RG_CUDA(cudaFuncSetAttribute(k_ent_scatter_own, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)osmem));
                RG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_o, k_ent_scatter_own, 256, osmem));
                uint64_t const otiles = (EP.nids + EO_TILE_IDS - 1) / EO_TILE_IDS;
                k_ent_scatter_own<<<(unsigned)std::min<uint64_t>(otiles, (uint64_t)h->sm_count * std::max(1, occ_o)), 256, osmem, h->st>>>(EP);
        }
        else
                k_ent_scatter<<<(unsigned)std::min<uint64_t>(etiles, (uint64_t)h->sm_count * std::max(1, occ)), 256, esmem, h->st>>>(EP);
        RG_KERNEL_CHECK();
        launch_count(h, 2);

        const uint64_t * fin_seed = EP.ent_seed; const uint32_t * fin_val = EP.ent_val; const uint32_t * fin_start = EP.bucket_start;
        if ( TP.e2 )
        {
                // one resident wave each: the grid-stride sweeps then pass over the level-1 buckets in order
                RG_CUDA(cudaMemsetAsync(EP.sub_count, 0, (size_t)3 * 65600 * 4, h->st));
                k_ent2_hist<<<(unsigned)(h->sm_count * std::max(1, occh)), 256, 0, h->st>>>(EP);
                RG_KERNEL_CHECK(); launch_count(h);
                uint32_t nl = 0;
                exclusive_scan_u32(EP.sub_count, EP.sub_start, (uint64_t)TP.nsub + 1, ptr<uint32_t>(h->ws_stmp), h->st, &nl);
                launch_count(h, nl);
                k_ent2_scatter<<<(unsigned)(h->sm_count * std::max(1, occ2)), 256, esmem, h->st>>>(EP);
                RG_KERNEL_CHECK(); launch_count(h);
                fin_seed = EP.ent2_seed; fin_val = EP.ent2_val; fin_start = EP.sub_start;
        }
        Grouped G; G.seed = fin_seed; G.val = fin_val; G.start = fin_start;
        return G;
}

void build_table(real_gpu * h, int t, TablePlan const & TP)
{
        if ( TP.empty ) return;
        Table & T = h->tab[t];
        EntryPartParams const & EP = TP.EP;
        Grouped const GR = partition_entries(h, TP);
        const uint64_t * fin_seed = GR.seed; const uint32_t * fin_val = GR.val; const uint32_t * fin_start = GR.start;
        k_build_sub<<<TP.own_subs, 256, (size_t)3 * TP.words * 4, h->st>>>(fin_seed, fin_val, fin_start, EP.G, TP.sub_shift, TP.words, ptr<SlotWord>(T.bitmap), ptr<Entry>(T.E), TP.d_ndist, TP.first_sub);
        RG_KERNEL_CHECK(); launch_count(h);
        RG_CUDA(cudaMemcpyAsync(&h->table_counts[2*t], TP.d_total, 8, cudaMemcpyDeviceToHost, h->st));   // total, ndistinct
}

// The fused build (index.cuh, TABLE_ITEMS): possible when the slots are the keys themselves and the partition depth does not
// exceed a fragment -- then the entries (A,t), (B,t), (C,t) of a strand share their bucket at both partition levels, ITEMS
// (strand, t) are partitioned once for all three tables, and one CTA per sub-bucket builds its piece of each table.
// Returns false when the geometry does not allow it (folded slots: the per-table build runs).
bool build_tables_fused(real_gpu * h, TablePlan * plan)
{
        uint32_t const hb = h->tab[0].hb, fb = 2 * h->F;
        if ( hb != h->keybits || h->nreads == 0 || plan[0].empty ) return false;
        uint32_t const nlA = table_lists(0, h->prm.seedkmax);
        uint64_t const cap_items = h->nreads * 2 * nlA;
        uint32_t const pbmin = hb > 16 ? hb - 16 : 0, pbmax = std::min<uint32_t>(std::min<uint32_t>(16, hb > 5 ? hb - 5 : 0), fb);
        if ( pbmin > pbmax ) return false;
        uint32_t pb = 0;
        while ( (cap_items >> pb) > SUB_TARGET_ENTRIES ) ++pb;
        pb = std::min(std::max(pb, pbmin), pbmax);
        if ( h->comm.nranks > 1 && pb < 8 ) return false;

        TablePlan TP = plan[0];                       // buffers, meta block, ownership of table A's plan
        uint32_t * meta = TP.EP.bucket_count;
        uint32_t const e1 = std::min<uint32_t>(8, pb);
        TP.e2 = pb - e1; TP.nsub = 1u << pb; TP.sub_shift = hb - pb;
        TP.words = TP.sub_shift >= 5 ? (1u << (TP.sub_shift - 5)) : 1u;
        TP.EP.G.table = TABLE_ITEMS; TP.EP.G.nlists = nlA;
        TP.EP.ebits = e1; TP.EP.e2bits = TP.e2;
        TP.first_sub = 0; TP.own_subs = TP.nsub;
        if ( h->comm.nranks > 1 )
        {
                TP.first_sub = TP.EP.own_lo << (pb - 8);
                TP.own_subs = (TP.EP.own_last + 1 - TP.EP.own_lo) << (pb - 8);
        }
        Build3Params B;
        memset(&B, 0, sizeof(B));
        for ( int t = 0; t < 3; ++t )
        {
                Table & T = h->tab[t];
                T.nblocks = TP.nsub;
                T.bitmap_bytes = (size_t)TP.nsub * TP.words * sizeof(SlotWord);
                dev_reserve(h, T.bitmap, T.bitmap_bytes);
                // the entry arrays of all three tables use the item numbering (k_build_sub3)
                dev_reserve(h, T.E, std::max<size_t>(16, cap_items * sizeof(Entry)) + 256);
                if ( plan[t].empty ) RG_CUDA(cudaMemsetAsync(T.bitmap.p, 0, T.bitmap_bytes, h->st));
                B.G[t] = plan[t].EP.G; B.G[t].table = t; B.G[t].nlists = plan[t].empty ? 0 : T.nlists;
                B.slots[t] = ptr<SlotWord>(T.bitmap); B.E[t] = ptr<Entry>(T.E);
                B.ndistinct[t] = meta + 521 + t;
        }
        // level-1 histogram of the items, then the two partition passes
        EntryPartParams3 Q;
        for ( int t = 0; t < 3; ++t ) { Q.P[t] = TP.EP; if ( t ) Q.P[t].G.nlists = 0; }
        k_ent_hist3<<<(unsigned)(h->sm_count * 8), 256, 0, h->st>>>(Q);
        RG_KERNEL_CHECK(); launch_count(h);
        Grouped const GR = partition_entries(h, TP);
        B.item_seed = GR.seed; B.item_val = GR.val; B.sub_start = GR.start;
        B.sub_shift = TP.sub_shift; B.words = TP.words; B.first_sub = TP.first_sub;
        // one CTA per (sub-bucket, table): three times the CTAs with a third of the shared memory each, faster than one CTA
        // building the sub-bucket of all three tables (measured, r02)
        size_t const smem = (size_t)(2 * TP.words + (TP.words + 1) / 2) * 4;
        // -l 32: fragments of 8 bases, direct addressing, sub-buckets of 2^16 slots (sub_local_slot)
        bool const fast = h->F == 8 && hb == 32 && TP.sub_shift == 16;
        typedef void (*build_fn)(const Build3Params);
        build_fn const kb = fast ? (build_fn)k_build_sub3<true> : (build_fn)k_build_sub3<false>;
        RG_CUDA(cudaFuncSetAttribute(kb, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kb<<<TP.own_subs * 3, 256, smem, h->st>>>(B);
        RG_KERNEL_CHECK(); launch_count(h);
        RG_CUDA(cudaMemcpyAsync(&h->table_counts[0], TP.d_total, 16, cudaMemcpyDeviceToHost, h->st));   // items, distinct slots of A, B, C
        h->fused_build = true;
        return true;
}

int build_from_device(real_gpu * h)
{
        // Seeds of more than 32 bases (64-bit signatures in the reference): the index and the scan work on the first 32
        // bases of the seed ('-': the last 32 of the strand, which lie inside the seed too) -- a seed with at most
        // seedkmax <= 2 mismatches has at most that many in any part of it, so this finds a superset of the reference's
        // candidates -- and the verification applies the test to the whole seed (verify_and_report, scan.cuh).
        uint32_t const seedl = std::min<uint32_t>(h->prm.seedl, 32);
        h->F = seedl / 4;
        h->keybits = seedl;                    // two fragments of F bases = 4F bits
        h->W = std::max<uint32_t>(1, (h->maxlen + 31) / 32);
        uint64_t const nreads = h->nreads;

        RG_CUDA(cudaEventRecord(h->ev[2], h->st));
        if ( ! h->src_packed )
                dev_reserve(h, h->rpack, (size_t)nreads * 2 * h->W * 8 + 16);
        dev_reserve(h, h->rlen, (size_t)nreads * 4 + 16);
        dev_reserve(h, h->seeds, (size_t)nreads * 2 * 8 + 16);
        dev_reserve(h, h->usable, (size_t)nreads * 4 + 16);
        dev_reserve(h, h->bad, (size_t)nreads * 4 + 16);
        if ( ! h->src_packed && h->W > PB_MAX_W )
                RG_CUDA(cudaMemsetAsync(h->bad.p, 0, (size_t)nreads * 4 + 16, h->st));
        if ( nreads )
        {
                if ( ! h->src_packed && h->W <= PB_MAX_W )
                {
                        uint32_t const rpb = 256 / h->W;
                        k_pack_both<<<blocks_for(nreads, rpb), 256, 0, h->st>>>(h->src_mapped, ptr<uint64_t>(h->offs), nreads, h->W, seedl, h->prm.seedl, ptr<uint64_t>(h->rpack),
                                                                                ptr<uint32_t>(h->rlen), ptr<uint64_t>(h->seeds), ptr<uint32_t>(h->usable));
                        RG_KERNEL_CHECK(); launch_count(h);
                }
                else if ( h->src_packed )
                {
                        // 2 bit/base input stays as it is (the verification reads it in place): only lengths and seeds
                        k_seeds_packed<<<blocks_for(nreads, 256), 256, 0, h->st>>>(h->src_packed, h->src_byte_offsets,
                                                                                 (h->src_packed_uniform || h->src_len32) ? nullptr : ptr<uint64_t>(h->offs), h->src_len32,
                                                                                 h->src_packed_uniform, nreads, seedl, h->prm.seedl, ptr<uint32_t>(h->bad),
                                                                                 ptr<uint32_t>(h->rlen), ptr<uint64_t>(h->seeds), ptr<uint32_t>(h->usable));
                        RG_KERNEL_CHECK(); launch_count(h);
                }
                else
                {
                        k_pack_reads<<<blocks_for(nreads * 2 * h->W, 256), 256, 0, h->st>>>(h->src_mapped, ptr<uint64_t>(h->offs), nreads, h->W,
                                                                                          ptr<uint64_t>(h->rpack), ptr<uint32_t>(h->bad));
                        RG_KERNEL_CHECK(); launch_count(h);
                        k_read_seeds<<<blocks_for(nreads, 256), 256, 0, h->st>>>(ptr<uint64_t>(h->offs), nreads, h->W, seedl, h->prm.seedl, ptr<uint64_t>(h->rpack),
                                                                               ptr<uint32_t>(h->bad), ptr<uint32_t>(h->rlen), ptr<uint64_t>(h->seeds), ptr<uint32_t>(h->usable));
                        RG_KERNEL_CHECK(); launch_count(h);
                }
        }
        RG_CUDA(cudaEventRecord(h->ev[3], h->st));

        // workspace sized for the largest table (A: up to 3 entries per read strand)
        uint64_t const maxent = std::max<uint64_t>(1, nreads * 2 * table_lists(0, h->prm.seedkmax));
        uint32_t const hbmax = std::min<uint32_t>(h->keybits, 32);
        dev_reserve(h, h->ws_k0, maxent * 8 + 16);           // entries grouped by the first level: seeds
        dev_reserve(h, h->ws_v0, maxent * 4 + 16);           //                                     values
        dev_reserve(h, h->ws_k1, maxent * 8 + 16);           // entries grouped by both levels
        dev_reserve(h, h->ws_v1, maxent * 4 + 16);
        dev_reserve(h, h->ws_flags, (size_t)3 * 65600 * 4);  // sub-bucket counts, starts, cursors
        dev_reserve(h, h->ws_stmp, scan_temp_elems(65600) * 4 + 64);
        dev_reserve(h, h->ws_hist, 3 * TABLE_META_WORDS * 4);
        memset(h->table_counts, 0, 6 * sizeof(uint32_t));
        TablePlan plan[3];
        EntryPartParams3 Q;
        bool any_table = false;
        for ( int t = 0; t < 3; ++t )
        {
                plan[t] = plan_table(h, t, ptr<uint32_t>(h->ws_hist) + (size_t)t * TABLE_META_WORDS);
                Q.P[t] = plan[t].EP;
                any_table = any_table || ! plan[t].empty;
        }
        h->fused_build = false;
        if ( any_table && build_tables_fused(h, plan) )
                any_table = false;             // built
        else
        for ( int t = 0; t < 3 && any_table; ++t )
                if ( ! plan[t].empty )
                {
                        // per-table build: the entry array holds exactly the table's entries
                        Table & T = h->tab[t];
                        dev_reserve(h, T.E, std::max<size_t>(16, h->nreads * 2 * T.nlists * sizeof(Entry)) + 256);
                }
        if ( any_table )
        {
                // the level-1 histograms of the three tables in one pass over the seeds
                for ( int t = 0; t < 3; ++t )
                        if ( plan[t].empty ) { Q.P[t].nids = 2 * nreads; Q.P[t].seeds = ptr<uint64_t>(h->seeds); Q.P[t].usable = ptr<uint32_t>(h->usable); }
                if ( plan[0].empty )
                        for ( int t = 1; t < 3; ++t ) if ( ! plan[t].empty ) { std::swap(Q.P[0], Q.P[t]); break; }       // slot 0 carries the seed pointers
                k_ent_hist3<<<(unsigned)(h->sm_count * 8), 256, 0, h->st>>>(Q);
                RG_KERNEL_CHECK(); launch_count(h);
        }
        for ( int t = 0; t < 3 && any_table; ++t )
                build_table(h, t, plan[t]);
        RG_CUDA(cudaEventRecord(h->ev[4], h->st));

        // fresh unique state (UniqueMatchInfo.hpp:172,190)
        dev_reserve(h, h->info, (size_t)nreads * 8 + 16);
        RG_CUDA(cudaMemsetAsync(h->info.p, 0, (size_t)nreads * 8 + 16, h->st));
        if ( h->ll.p )
        {
                dev_reserve(h, h->gaps, (size_t)nreads * sizeof(real_gpu_gapinfo) + 16);
                RG_CUDA(cudaMemsetAsync(h->gaps.p, 0, (size_t)nreads * sizeof(real_gpu_gapinfo) + 16, h->st));
        }
        if ( h->prm.scores )
        {
                dev_reserve(h, h->scores, (size_t)nreads * 4 + 16);
                k_fill_f32<<<blocks_for(nreads + 1, 256), 256, 0, h->st>>>(ptr<float>(h->scores), nreads, -FLT_MAX);      // UniqueMatchInfo.hpp:190
                RG_KERNEL_CHECK(); launch_count(h);
        }
        if ( h->comm.nranks > 1 && h->hit_cap == 0 )
        {
                // sharded tables: nothing may be allocated or freed between the hand-over kernels of a scan
                uint64_t const cap = std::max<uint64_t>(1u << 16, 4 * h->nreads);
                dev_alloc(h, h->hits_raw, cap * sizeof(RawHit));
                h->hit_cap = cap;
        }
        // Everything above is enqueued; the build is waited for by the next call that needs the index (finish_build),
        // so that a text transfer issued in between overlaps it.
        h->build_pending = true;
        return REAL_GPU_OK;
}

// waits for the index build real_gpu_set_reads* has enqueued and takes over its counts
void finish_build(real_gpu * h)
{
        if ( ! h->build_pending ) return;
        h->build_pending = false;
        RG_CUDA(cudaStreamSynchronize(h->st));
        h->n_usable = 0;
        if ( h->fused_build )
        {
                // table_counts = items, distinct slots of A, B, C; an item (strand, t) is an entry of every table with more than t lists
                uint32_t const nlA = table_lists(0, h->prm.seedkmax);
                uint64_t const strands = nlA ? h->table_counts[0] / nlA : 0;
                for ( int t = 0; t < 3; ++t )
                {
                        h->tab[t].nentries = strands * h->tab[t].nlists;
                        h->tab[t].ndistinct = h->table_counts[1 + t];
                }
        }
        else
        for ( int t = 0; t < 3; ++t )
        {
                h->tab[t].nentries = h->table_counts[2*t];
                h->tab[t].ndistinct = h->table_counts[2*t+1];
        }
        if ( h->tab[0].nlists ) h->n_usable = h->tab[0].nentries / (2 * h->tab[0].nlists);
        h->stats.pack_ms = elapsed(h->ev[2], h->ev[3]);
        h->stats.index_ms = elapsed(h->ev[3], h->ev[4]);
        h->have_reads = true;
}

// ---------------------------------------------------------------------------------------------
// scan
// ---------------------------------------------------------------------------------------------

// where the kernels find the bases of the reads (ReadSrc, common.cuh)
ReadSrc read_src(real_gpu * h)
{
        ReadSrc S;
        memset(&S, 0, sizeof(S));
        if ( h->src_packed )
        {
                S.packed = h->src_packed;
                S.ubytes = h->src_packed_uniform ? (h->src_packed_uniform + 3) / 4 : 0;
                S.boffs = h->src_byte_offsets;
        }
        else
        {
                S.rpack = ptr<uint64_t>(h->rpack);
                S.W = h->W;
        }
        return S;
}

void fill_scan_params(real_gpu * h, ScanParams & P, int mode)
{
        memset(&P, 0, sizeof(P));
        P.text = ptr<uint64_t>(h->text) + TEXT_PAD_WORDS;
        P.nmask = ptr<uint64_t>(h->nmask) + TEXT_PAD_WORDS;
        P.shard_begin = h->shard_begin;
        uint32_t const seedl = std::min<uint32_t>(h->prm.seedl, 32);       // the indexed part of the seed
        // seed windows this shard evaluates: every window whose hit start (p for '+', p-(L-seedl) for '-')
        // may fall into [own_begin, own_end)
        uint64_t gwin_b = h->own_begin;
        uint64_t gwin_e = h->own_end + (h->maxlen > seedl ? h->maxlen - seedl : 0);
        uint64_t const last_window_end = (h->n_total >= seedl) ? (h->n_total - seedl + 1) : 0;
        gwin_e = std::min(gwin_e, last_window_end);
        uint64_t const shard_end = h->shard_begin + h->shard_len;
        if ( gwin_e + seedl > shard_end + 1 )
                gwin_e = (shard_end + 1 >= seedl) ? (shard_end + 1 - seedl) : 0;
        if ( gwin_e < gwin_b ) gwin_e = gwin_b;
        P.win_begin = gwin_b - h->shard_begin;
        P.win_end = gwin_e - h->shard_begin;
        P.x_begin = P.win_begin;
        P.x_end = (P.win_end > P.win_begin) ? std::min<uint64_t>(P.win_end + 2 * h->F, h->shard_len) : P.win_begin;
        P.own_begin = h->own_begin;
        P.own_end = h->own_end;
        for ( int t = 0; t < 3; ++t )
        {
                P.tab[t].slots = ptr<SlotWord>(h->tab[t].bitmap);
                P.tab[t].E = ptr<Entry>(h->tab[t].E);
                P.tab[t].hb = h->tab[t].hb;
                P.tab[t].nlists = h->tab[t].nentries ? h->tab[t].nlists : 0;
        }
        P.seedl = seedl; P.vseedl = h->prm.seedl; P.F = h->F; P.keybits = h->keybits; P.seedkmax = h->prm.seedkmax; P.totalkmax = h->prm.totalkmax;
        P.rs = read_src(h); P.rlen = ptr<uint32_t>(h->rlen);
        P.rec = ptr<uint64_t>(h->rec); P.nrec = h->nrec; P.fileid = h->fileid;
        P.nranks = 1; P.rank = 0; P.bucket_lo[0] = 0; P.bucket_lo[1] = SC_MAX_BUCKETS; P.seg_cap = 0; P.npairs = 0;
        P.own_b_lo = 0; P.own_b_cnt = SC_MAX_BUCKETS;
        P.nprobed = ptr<unsigned long long>(h->counters) + 4;
        P.mode = mode;
        P.hits = ptr<RawHit>(h->hits_raw);
        P.hit_cap = h->hit_cap;
        P.hit_count = ptr<unsigned long long>(h->counters);
        P.stats = ptr<unsigned long long>(h->counters) + 1;
        P.info = ptr<unsigned long long>(h->info);
}

// hand-over between the ranks of a sharded scan: "slot 0 of round e" = my records of round e are delivered,
// "slot 1" = I have consumed what I was sent in round e
void comm_signal(real_gpu * h, uint32_t slot)
{
        real_gpu::Comm & CM = h->comm;
        if ( CM.local[CM.rank] )
        {
                RG_CUDA(cudaEventRecord(CM.ev[slot], h->st));
                CM.enqueued[slot].store(CM.epoch, std::memory_order_release);
                return;
        }
        k_comm_signal<<<1, 32, 0, h->st>>>(ptr<uint32_t *>(CM.ptrs), CM.nranks, CM.rank, slot, CM.epoch);
        RG_KERNEL_CHECK(); launch_count(h);
}

void comm_wait(real_gpu * h, uint32_t slot, uint32_t epoch, long long wait_ms)
{
        real_gpu::Comm & CM = h->comm;
        if ( CM.local[CM.rank] )
        {
                if ( epoch == 0 ) return;
                auto const t0 = std::chrono::steady_clock::now();
                for ( uint32_t r = 0; r < CM.nranks; ++r )
                {
                        if ( r == CM.rank ) continue;
                        real_gpu::Comm & Q = CM.local[r]->comm;
                        while ( (int32_t)(Q.enqueued[slot].load(std::memory_order_acquire) - epoch) < 0 )
                        {
                                if ( std::chrono::duration_cast<std::chrono::milliseconds>(std::chrono::steady_clock::now() - t0).count() > wait_ms )
                                        throw CudaError("sharded tables: timed out waiting for rank " + std::to_string(r));
                                std::this_thread::yield();
                        }
                        RG_CUDA(cudaStreamWaitEvent(h->st, Q.ev[slot], 0));
                }
                return;
        }
        k_comm_wait<<<1, 32, 0, h->st>>>(reinterpret_cast<uint32_t *>(CM.base[CM.rank]), CM.nranks, slot, epoch, wait_ms * 2000000LL, ptr<uint32_t>(CM.error));
        RG_KERNEL_CHECK(); launch_count(h);
}

// What a scan decides before its chunk loop: the windows it evaluates, the bucket bits, the positions per chunk, its buffers
// and the shapes of its kernels.  real_gpu_prepare_scan makes the same plan ahead of the match call (prepare = true: the read
// set is not known yet, the finest bucket split is taken).
static const uint64_t L2_SLICE_BYTES = 48ull << 20;       // table bytes (presence bits + entries) one bucket may touch
static const uint32_t OWN_LIST_MAX_BUCKETS = 64;          // bucket shards: own buckets up to which the kept positions are listed first
struct ScanPlan
{
        ScanParams P;
        uint64_t x_begin, x_end, chunk_cap, ntiles;
        uint32_t * meta;
        bool sharded, own_only, own_list;
        int occ_p, occ_s, occ_b;
        size_t psmem, ssmem, bsmem;
        long long wait_ms;
        typedef void (*probe_fn)(const ScanParams);
        probe_fn probe;
};

void plan_scan(real_gpu * h, int mode, bool prepare, ScanPlan & S)
{
        ScanParams & P = S.P;
        fill_scan_params(h, P, mode);
        uint64_t const first_tile = P.x_begin / SC_TILE_POS, end_tile = (P.x_end + SC_TILE_POS - 1) / SC_TILE_POS;
        S.ntiles = (P.x_end > P.x_begin) ? (end_tile - first_tile) : 0;
        S.x_begin = P.x_begin; S.x_end = P.x_end; S.chunk_cap = 0; S.meta = nullptr;
        S.sharded = S.own_only = S.own_list = false;
        if ( ! S.ntiles ) return;

        // buckets: cut the tables into key-prefix slices that stay resident in L2 while a bucket is probed
        uint64_t table_bytes = 0;
        uint32_t const maxbits = std::min<uint32_t>(SLOT_PREFIX_BITS, 2 * h->F);
        for ( int t = 0; t < 3; ++t )
                if ( P.tab[t].nlists )
                        table_bytes += h->tab[t].bitmap_bytes + h->tab[t].nentries * sizeof(Entry);
        uint32_t bbits = 0;
        if ( prepare || h->build_pending )
                bbits = maxbits;
        else
                while ( bbits < maxbits && (table_bytes >> bbits) > L2_SLICE_BYTES ) ++bbits;
        P.bucket_bits = bbits;

        real_gpu::Comm & CM = h->comm;
        bool const sharded = S.sharded = CM.nranks > 1 && CM.window.p;          // records exchanged through peer memory
        bool const own_only = S.own_only = CM.nranks > 1 && ! CM.window.p;      // bucket shard: this handle keeps the positions of its own buckets
        if ( own_only )
        {
                if ( maxbits < 8 ) throw CudaError("bucket shards need seeds of at least 16 bases");
                if ( h->shard_begin != 0 || h->shard_len != h->n_total || h->own_begin != 0 || h->own_end != h->n_total )
                        throw CudaError("bucket shards: every rank must be given the whole text (the ranks split the signature space, not the text)");
                P.bucket_bits = 8;
                P.own_b_lo = CM.bucket_lo[CM.rank];
                P.own_b_cnt = CM.bucket_lo[CM.rank + 1] - CM.bucket_lo[CM.rank];
        }
        if ( sharded )
        {
                if ( ! CM.connected ) throw CudaError("sharded tables: real_gpu_comm_connect has not been called");
                if ( maxbits < 8 ) throw CudaError("sharded tables need seeds of at least 16 bases");
                if ( h->shard_begin != 0 || h->shard_len != h->n_total || h->own_begin != 0 || h->own_end != h->n_total )
                        throw CudaError("sharded tables: every rank must be given the whole text (the ranks split the positions among themselves)");
                P.bucket_bits = 8;
        }
        uint64_t const x_begin = P.x_begin, x_end = P.x_end;
        // Positions partitioned at a time.  One handle with the whole signature space: as many as fit -- the records of
        // C3's 3.1 G positions take 50 GB of the 180 -- because every chunk walks through all the tables again (three chunks
        // of 2^30 positions read the entries three times over: 105 GB of DRAM traffic instead of 10, 2 ms of the C3 scan).
        // Equal chunks when the text does not fit.  Sharded tables: the rounds the record areas of the windows were sized for.
        // A bucket shard is sized like a single handle -- all positions of a chunk may fall into its buckets -- plus the 4-byte
        // list of the kept positions: one chunk for C3 on every rank too (r02 up to here: rounds of 2^30 positions).
        bool const will_list = own_only && P.own_b_cnt <= OWN_LIST_MAX_BUCKETS;
        uint64_t chunk_max = CM.round_positions;
        if ( ! sharded )
        {
                uint64_t const span = ((x_end - x_begin + SC_TILE_POS - 1) / SC_TILE_POS) * SC_TILE_POS;
                uint64_t const pad = (uint64_t)SC_MAX_BUCKETS * SC_UNIT;
                uint64_t fit = SC_MAX_CHUNK;
                // the memory query costs milliseconds (3.7 ms measured on C1, whose whole scan takes 0.5): it is made only
                // when the buffers already held are too small for the span
                uint64_t const want = std::min<uint64_t>(span, SC_MAX_CHUNK);
                if ( (want + pad) * sizeof(uint4) + 64 > h->rec_win.bytes || (will_list && want * 4 + 64 > h->own_list.bytes) )
                {
                        size_t free_b = 0, total_b = 0;
                        RG_CUDA(cudaMemGetInfo(&free_b, &total_b));
                        // the buffers already held count as room; ahead of the match call the read set and its tables are still to come
                        uint64_t const held = h->rec_win.bytes + (will_list ? h->own_list.bytes : 0);
                        uint64_t const room = (uint64_t)((free_b + held) * (prepare ? 0.4 : 0.6)) / (sizeof(uint4) + (will_list ? 4 : 0));
                        fit = std::max<uint64_t>(SC_TILE_POS, std::min<uint64_t>(SC_MAX_CHUNK, room > pad ? room - pad : 0) / SC_TILE_POS * SC_TILE_POS);
                }
                uint64_t const nchunks = (span + fit - 1) / fit;
                chunk_max = std::max<uint64_t>(SC_TILE_POS, ((span + nchunks - 1) / nchunks + SC_TILE_POS - 1) / SC_TILE_POS * SC_TILE_POS);
        }
        uint64_t const chunk_cap = S.chunk_cap = std::min<uint64_t>(chunk_max, ((x_end - x_begin + SC_TILE_POS - 1) / SC_TILE_POS) * SC_TILE_POS);
        if ( sharded && prepare ) return;                                        // nothing to form ahead: the caller gives up
        // entries are touched about once per chunk and bucket: several chunks stream them past the probed slot words
        // (evict_first); a single chunk re-uses every entry line about nine times while its bucket is probed (evict_normal)
        P.entries_evict_normal = x_end - x_begin <= chunk_cap;
        uint32_t * meta = nullptr;
        if ( sharded )
        {
                // everything was allocated by real_gpu_comm_init: no allocation may happen between the hand-over kernels
                meta = ptr<uint32_t>(h->part_meta);
                P.recs = reinterpret_cast<uint4 *>(CM.base[CM.rank] + CM.recs_off);
                P.nranks = CM.nranks; P.rank = CM.rank; P.seg_cap = CM.seg_cap;
                for ( uint32_t r = 0; r <= CM.nranks; ++r ) P.bucket_lo[r] = CM.bucket_lo[r];
                for ( uint32_t r = 0; r < CM.nranks; ++r )
                {
                        P.peer_recs[r] = reinterpret_cast<uint4 *>(CM.base[r] + CM.recs_off);
                        P.peer_meta[r] = reinterpret_cast<uint32_t *>(CM.base[r] + CM.meta_off);
                }
                P.pair_grab = ptr<uint32_t>(CM.pairs); P.pair_rec = ptr<uint32_t>(CM.pairs) + 1024;
                P.npairs = (CM.bucket_lo[CM.rank + 1] - CM.bucket_lo[CM.rank]) * CM.nranks;
        }
        else
        {
                dev_reserve(h, h->rec_win, (chunk_cap + (uint64_t)SC_MAX_BUCKETS * SC_UNIT) * sizeof(uint4) + 64);
                dev_reserve(h, h->part_meta, (1100 + 256 * SC_CURSOR_STRIDE) * 4);
                meta = ptr<uint32_t>(h->part_meta);
                P.recs = ptr<uint4>(h->rec_win);
                P.peer_recs[0] = P.recs;
        }
        S.meta = meta;
        P.nprobed = reinterpret_cast<unsigned long long *>(meta + 784);          // kept with the records: a scan that re-uses them takes the count over
        P.bucket_count = meta;
        P.bucket_start = meta + 256;
        P.unit_counter = meta + 256 + 520;
        P.bucket_cursor = meta + 1088;

        S.psmem = sizeof(HistSmem); S.ssmem = sizeof(ScatterSmem); S.bsmem = sizeof(ProbeSmem);
        // Bucket shard: with few own buckets (four ranks or more) one light pass lists the kept positions and counts them per
        // bucket, and the staged scatter runs on the list; with many (two ranks: half of all positions are kept) listing
        // costs more than it saves, and the dense kernels run with a filter on the bucket (measured, profiles/r02_*)
        bool const own_list = S.own_list = will_list;
        if ( own_list )
        {
                // the positions of a chunk this rank keeps, 4 bytes each (all of them if the text falls into its buckets only)
                dev_reserve(h, h->own_list, chunk_cap * 4 + 64);
                P.list = ptr<uint32_t>(h->own_list);
                P.list_count = reinterpret_cast<unsigned long long *>(meta + 780);
        }
        RG_CUDA(cudaFuncSetAttribute(k_part_hist, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S.psmem));
        RG_CUDA(cudaFuncSetAttribute(k_part_scatter<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S.ssmem));
        RG_CUDA(cudaFuncSetAttribute(k_part_scatter<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S.ssmem));
        bool const wide = h->prm.seedl > 32;
        typedef ScanPlan::probe_fn probe_fn;
        bool const packed_src = h->src_packed != nullptr;
        S.probe = wide ? (packed_src ? (probe_fn)k_bucket_probe<true, true> : (probe_fn)k_bucket_probe<true, false>)
                       : (packed_src ? (probe_fn)k_bucket_probe<false, true> : (probe_fn)k_bucket_probe<false, false>);
        RG_CUDA(cudaFuncSetAttribute(S.probe, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S.bsmem));
        int occ_p = 0, occ_b = 0, occ_s = 0;
        RG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_p, k_part_hist, SC_THREADS, S.psmem));
        RG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_s, own_list ? k_part_scatter<true> : k_part_scatter<false>, PS_THREADS, S.ssmem));
        RG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_b, S.probe, SC_THREADS, S.bsmem));
        if ( occ_p < 1 ) occ_p = 1;
        if ( occ_s < 1 ) occ_s = 1;
        if ( occ_b < 1 ) occ_b = 1;
        // more than SC_PROBE_MINB CTAs per SM make the probe slower (measured: 87 vs 74 ms scan on C3 with four): the grabs
        // of more warps spread over more of the bucket order and the probed slices lose their place in L2
        if ( occ_b > SC_PROBE_MINB ) occ_b = SC_PROBE_MINB;
        S.occ_p = occ_p; S.occ_s = occ_s; S.occ_b = occ_b;
        S.wait_ms = 30000;             // a peer that never arrives is reported, not waited for forever
        if ( const char * e = getenv("REAL_GPU_COMM_TIMEOUT_MS") ) S.wait_ms = atoll(e);
}

// the partition kernels of one chunk (P.x_begin .. P.x_end) on stream st: bucket histogram (or the kept-position list of a
// bucket shard), bucket offsets, staged scatter of the records.  nprobed: where a bucket shard counts the positions it kept.
void launch_partition(real_gpu * h, ScanPlan const & S, ScanParams const & P, cudaStream_t st)
{
        real_gpu::Comm & CM = h->comm;
        bool const any = P.x_end > P.x_begin;
        uint64_t const ft = P.x_begin / SC_TILE_POS, et = (P.x_end + SC_TILE_POS - 1) / SC_TILE_POS;
        unsigned const pgrid = (unsigned)std::min<uint64_t>(et - ft, (uint64_t)h->sm_count * S.occ_p);
        RG_CUDA(cudaMemsetAsync(S.meta, 0, 256 * 4, st));
        if ( S.own_list ) RG_CUDA(cudaMemsetAsync(P.list_count, 0, 8, st));
        if ( any && S.own_list )
        {
                uint64_t const oft = P.x_begin / OL_TILE_POS, oet = (P.x_end + OL_TILE_POS - 1) / OL_TILE_POS;
                k_own_list<<<(unsigned)std::min<uint64_t>(oet - oft, (uint64_t)h->sm_count * 8), OL_THREADS, 0, st>>>(P);
                RG_KERNEL_CHECK(); launch_count(h); h->stats.scan_launches += 1;
        }
        else if ( any )
        {
                k_part_hist<<<pgrid, SC_THREADS, S.psmem, st>>>(P);
                RG_KERNEL_CHECK(); launch_count(h); h->stats.scan_launches += 1;
        }
        if ( S.sharded )
        {
                // the owners must have consumed the previous round before their record areas are written again
                comm_wait(h, 1, CM.epoch - 1, S.wait_ms);
        }
        k_part_offsets<<<1, SC_MAX_BUCKETS, 0, st>>>(P);
        RG_KERNEL_CHECK();
        if ( any )
        {
                uint64_t const sft = P.x_begin / PS_TILE_POS, set = (P.x_end + PS_TILE_POS - 1) / PS_TILE_POS;
                unsigned const sgrid = (unsigned)std::min<uint64_t>(set - sft, (uint64_t)h->sm_count * S.occ_s);
                if ( S.own_list )
                        k_part_scatter<true><<<(unsigned)(h->sm_count * S.occ_s), PS_THREADS, S.ssmem, st>>>(P);
                else
                        k_part_scatter<false><<<sgrid, PS_THREADS, S.ssmem, st>>>(P);
                RG_KERNEL_CHECK(); launch_count(h); h->stats.scan_launches += 1;
        }
        launch_count(h);               // k_part_offsets
        h->stats.scan_launches += 1;
}

// real_gpu_prepare_scan: the partition of the current text, enqueued on a stream of its own behind the arrival of the words
void prepare_scan(real_gpu * h, uint32_t max_read_len, bool reads_known)
{
        uint32_t const seedl = std::min<uint32_t>(h->prm.seedl, 32);
        h->F = seedl / 4; h->keybits = seedl;
        real_gpu::Prepared & R = h->prep;
        if ( R.valid )
        {
                // records of this text are there already (or on their way: real_gpu_set_text* has started them because a read set
                // was known): they serve if they cover the windows asked for
                uint32_t const kept_maxlen = h->maxlen;
                h->maxlen = max_read_len;
                ScanParams Q;
                fill_scan_params(h, Q, 0);
                h->maxlen = kept_maxlen;
                uint32_t const maxbits = std::min<uint32_t>(SLOT_PREFIX_BITS, 2 * h->F);
                if ( R.x_begin == Q.x_begin && R.x_end == Q.x_end && R.win_begin == Q.win_begin && R.win_end == Q.win_end
                     && (reads_known || R.bucket_bits >= maxbits || h->comm.nranks > 1) )
                        return;
        }
        drop_prepared(h);
        uint32_t const kept_maxlen = h->maxlen;
        h->maxlen = max_read_len;
        ScanPlan S;
        try { plan_scan(h, 0, ! reads_known, S); } catch ( ... ) { h->maxlen = kept_maxlen; throw; }
        h->maxlen = kept_maxlen;
        if ( ! S.ntiles || S.sharded || S.x_end - S.x_begin > S.chunk_cap ) return;         // several chunks, or records that cross NVLink: formed by the scan itself
        if ( ! h->st3 ) RG_CUDA(cudaStreamCreateWithFlags(&h->st3, cudaStreamNonBlocking));
        if ( ! R.ev0 ) { RG_CUDA(cudaEventCreate(&R.ev0)); RG_CUDA(cudaEventCreate(&R.done)); }
        ScanParams & P = S.P;
        P.pos_base = S.x_begin;
        if ( h->text_pending ) RG_CUDA(cudaStreamWaitEvent(h->st3, h->ev_words, 0));
        RG_CUDA(cudaMemsetAsync(P.nprobed, 0, 8, h->st3));
        RG_CUDA(cudaEventRecord(R.ev0, h->st3));
        launch_partition(h, S, P, h->st3);
        RG_CUDA(cudaEventRecord(R.done, h->st3));
        R.x_begin = S.x_begin; R.x_end = S.x_end; R.win_begin = P.win_begin; R.win_end = P.win_end; R.chunk_cap = S.chunk_cap;
        R.bucket_bits = P.bucket_bits; R.own_b_lo = P.own_b_lo; R.own_b_cnt = P.own_b_cnt; R.own_list = S.own_list; R.recs = P.recs;
        R.valid = true; R.inflight = true; R.ahead = true;
}

// real_gpu_set_text* with the read set already known (the usual order: reads, then text file after text file): the partition
// of the new text is enqueued at once, on its own stream -- beside an index build that real_gpu_set_reads* has left running.
// Measured: texts of a few ten Mbp gain (C1, 10 Mbp: 2.09 -> 1.64 ms per step -- short kernels that are bound by latencies
// fill each other's gaps); on C3 the two kernel groups take as long together as one after the other (37.3 against 15.2 + 22.8 ms:
// both live on shared-memory bandwidth), so long texts are left to the scan itself and the phase times stay readable.
static const uint64_t AUTO_PREPARE_MAX_POSITIONS = 1ull << 26;
void auto_prepare_scan(real_gpu * h)
{
        if ( ! h->auto_prepare || ! h->have_text || ! (h->have_reads || h->build_pending) || ! h->maxlen ) return;
        // (a bucket shard keeps a part of the positions of a long text: its filter / list and scatter kernels leave room again --
        // one rank of 2 / 4 / 8 on C3: 51.6 -> 49.0, 28.6 -> 27.4, 15.4 -> 14.9 ms per step)
        bool const light_shard = h->comm.nranks >= 2 && ! h->comm.window.p;
        if ( h->shard_len > AUTO_PREPARE_MAX_POSITIONS && ! light_shard ) return;
        try { prepare_scan(h, h->maxlen, true); }
        catch ( LimitError const & ) { h->prep.valid = false; }
        catch ( CudaError const & ) { cudaGetLastError(); h->prep.valid = false; }          // what is wrong with the set-up is reported by the match call
}

// launches K3 once; returns the number of hits the kernel counted
uint64_t run_scan(real_gpu * h, int mode)
{
        dev_reserve(h, h->counters, 8 * 8);
        RG_CUDA(cudaMemsetAsync(h->counters.p, 0, 8 * 8, h->st));
        ScanPlan S;
        plan_scan(h, mode, false, S);
        ScanParams & P = S.P;
        uint64_t const ntiles = S.ntiles;
        if ( h->text_pending )
        {
                flush_mask(h);                                                  // the wildcard mask follows the words, unless it is on its way already
                RG_CUDA(cudaStreamWaitEvent(h->st, h->ev_words, 0));            // asynchronous text copy: the words must have arrived
        }
        // records formed ahead by real_gpu_prepare_scan serve this scan if it would form the very same ones
        real_gpu::Prepared & R = h->prep;
        bool const use_prep = R.valid && ntiles && ! S.sharded && S.x_end - S.x_begin <= S.chunk_cap
                              && R.x_begin == S.x_begin && R.x_end == S.x_end && R.win_begin == P.win_begin && R.win_end == P.win_end
                              && R.bucket_bits >= P.bucket_bits && R.own_b_lo == P.own_b_lo && R.own_b_cnt == P.own_b_cnt && R.own_list == S.own_list && R.recs == P.recs;
        if ( R.inflight ) RG_CUDA(cudaStreamWaitEvent(h->st, R.done, 0));        // either way: the record buffer is written or read next
        bool const was_ahead = use_prep && R.ahead;
        R.valid = false;
        RG_CUDA(cudaEventRecord(h->ev[5], h->st));
        size_t nprobe_ev = 0;
        if ( ntiles )
        {
                real_gpu::Comm & CM = h->comm;
                bool const sharded = S.sharded, own_only = S.own_only;
                uint64_t const x_begin = S.x_begin, x_end = S.x_end, chunk_cap = S.chunk_cap;
                if ( use_prep )
                {
                        P.bucket_bits = R.bucket_bits;
                        RG_CUDA(cudaMemsetAsync(P.unit_counter, 0, 4, h->st));          // the work counter of the probe (k_part_offsets clears it otherwise)
                }
                else
                        RG_CUDA(cudaMemsetAsync(P.nprobed, 0, 8, h->st));
                h->stats.n_windows = 0;
                for ( uint64_t cb = x_begin; cb < x_end; cb += chunk_cap )
                {
                        if ( nprobe_ev >= 64 ) nprobe_ev = 63;              // (very long texts: the last pairs are re-used)
                        uint64_t const ce = std::min<uint64_t>(x_end, cb + chunk_cap);
                        P.pos_base = cb;
                        P.x_begin = cb; P.x_end = ce;
                        if ( sharded )
                        {
                                // this rank's slice of the round
                                uint64_t const per = (chunk_cap + CM.nranks - 1) / CM.nranks;
                                P.x_begin = std::min<uint64_t>(ce, cb + (uint64_t)CM.rank * per);
                                P.x_end = std::min<uint64_t>(ce, P.x_begin + per);
                                ++CM.epoch;
                        }
                        if ( ! own_only ) h->stats.n_windows += P.x_end - P.x_begin;
                        if ( ! use_prep ) launch_partition(h, S, P, h->st);
                        if ( sharded )
                        {
                                comm_signal(h, 0);
                                comm_wait(h, 0, CM.epoch, S.wait_ms);
                                k_comm_pairs<<<1, SC_PAIR_THREADS, 0, h->st>>>(P, reinterpret_cast<uint32_t *>(CM.base[CM.rank] + CM.meta_off));
                                RG_KERNEL_CHECK(); launch_count(h);
                        }
                        if ( h->evp.size() < 2 * (nprobe_ev + 1) )
                        {
                                cudaEvent_t a, b;
                                RG_CUDA(cudaEventCreate(&a)); RG_CUDA(cudaEventCreate(&b));
                                h->evp.push_back(a); h->evp.push_back(b);
                        }
                        if ( h->text_pending ) RG_CUDA(cudaStreamWaitEvent(h->st, h->evc[1], 0));          // ... and now the wildcard mask
                        RG_CUDA(cudaEventRecord(h->evp[2 * nprobe_ev], h->st));
                        S.probe<<<(unsigned)(h->sm_count * S.occ_b), SC_THREADS, S.bsmem, h->st>>>(P);
                        RG_KERNEL_CHECK();
                        RG_CUDA(cudaEventRecord(h->evp[2 * nprobe_ev + 1], h->st));
                        ++nprobe_ev;
                        if ( sharded )
                        {
                                comm_signal(h, 1);
                        }
                        launch_count(h);
                        h->stats.scan_launches += 1;
                }
                P.x_begin = x_begin; P.x_end = x_end;
                RG_CUDA(cudaMemcpyAsync(ptr<unsigned long long>(h->counters) + 4, P.nprobed, 8, cudaMemcpyDeviceToDevice, h->st));
                // a scan of one chunk leaves the records of the whole text behind: the next scan of the same text (the gapped pass
                // after matchUnique, a second file set against ... the same text) finds them; a new text drops them
                if ( ! sharded && x_end - x_begin <= chunk_cap )
                {
                        R.x_begin = S.x_begin; R.x_end = S.x_end; R.win_begin = P.win_begin; R.win_end = P.win_end; R.chunk_cap = S.chunk_cap;
                        R.bucket_bits = P.bucket_bits; R.own_b_lo = P.own_b_lo; R.own_b_cnt = P.own_b_cnt; R.own_list = S.own_list; R.recs = P.recs;
                        R.valid = true; R.ahead = false;
                }
        }
        RG_CUDA(cudaEventRecord(h->ev[6], h->st));
        unsigned long long c[5] = {0, 0, 0, 0, 0};
        RG_CUDA(cudaMemcpyAsync(c, h->counters.p, sizeof(c), cudaMemcpyDeviceToHost, h->st));
        RG_CUDA(cudaStreamSynchronize(h->st));
        R.inflight = false;
        h->stats.scan_ms = elapsed(h->ev[5], h->ev[6]);
        finish_text(h);
        h->stats.probe_ms = 0;
        for ( size_t i = 0; i < nprobe_ev; ++i ) h->stats.probe_ms += elapsed(h->evp[2*i], h->evp[2*i+1]);
        // the partition kernels' time: part of scan_ms, unless the records were formed ahead (then it ran beside the transfer of the reads)
        h->stats.part_ms = was_ahead ? elapsed(R.ev0, R.done) : (use_prep ? 0.f : h->stats.scan_ms - h->stats.probe_ms);
        h->stats.prepared_scans += was_ahead ? 1 : 0;
        if ( ! ntiles ) h->stats.n_windows = 0;
        else if ( h->comm.nranks > 1 && ! h->comm.window.p ) h->stats.n_windows = c[4];     // bucket shard: the positions this handle kept
        if ( h->comm.nranks > 1 && h->comm.window.p )
        {
                uint32_t cerr = 0;
                RG_CUDA(cudaMemcpy(&cerr, h->comm.error.p, 4, cudaMemcpyDeviceToHost));
                if ( cerr ) throw CudaError("sharded tables: timed out waiting for rank " + std::to_string(cerr - 1));
        }
        uint32_t nt = 0;
        for ( int t = 0; t < 3; ++t ) if ( P.tab[t].nlists ) ++nt;
        h->stats.n_probes = h->stats.n_windows * nt;
        h->stats.n_candidates = c[1];
        h->stats.n_seedpass = c[2];
        h->stats.n_hits = c[3];
        return (mode != 1) ? (uint64_t)c[0] : (uint64_t)c[3];
}

// CUDA loads kernels lazily, and loading one may wait for the device to drain.  With sharded tables a rank's
// kernels wait (on the device) for kernels another rank has yet to launch, so a first-time load in the middle of a
// scan could wait forever: every kernel of this library is loaded when the first handle is created.
void preload_kernels(int device)
{
        static bool done[64] = { false };
        if ( device < 0 || device >= 64 || done[device] ) return;
        cudaFuncAttributes a;
#define RG_PRELOAD(k) RG_CUDA(cudaFuncGetAttributes(&a, k))
        RG_PRELOAD(k_pack_reads); RG_PRELOAD(k_pack_both); RG_PRELOAD(k_seeds_packed); RG_PRELOAD(k_read_seeds); RG_PRELOAD(k_uniform_offsets); RG_PRELOAD(k_flags_to_bad);
        RG_PRELOAD(k_ent_hist3); RG_PRELOAD(k_ent_offsets); RG_PRELOAD(k_ent_scatter); RG_PRELOAD(k_ent_scatter_own); RG_PRELOAD(k_ent2_hist); RG_PRELOAD(k_ent2_scatter); RG_PRELOAD(k_build_sub); RG_PRELOAD(k_build_sub3<true>); RG_PRELOAD(k_build_sub3<false>);
        RG_PRELOAD(k_scan_reduce); RG_PRELOAD(k_scan_apply); RG_PRELOAD(k_fill_f32);
        RG_PRELOAD(k_part_hist); RG_PRELOAD(k_part_offsets); RG_PRELOAD(k_part_scatter<false>); RG_PRELOAD(k_part_scatter<true>); RG_PRELOAD(k_own_list); RG_PRELOAD((k_bucket_probe<false, false>)); RG_PRELOAD((k_bucket_probe<true, false>)); RG_PRELOAD((k_bucket_probe<false, true>)); RG_PRELOAD((k_bucket_probe<true, true>));
        RG_PRELOAD(k_comm_signal); RG_PRELOAD(k_comm_wait); RG_PRELOAD(k_comm_pairs);
        RG_PRELOAD(k_score_hits); RG_PRELOAD(k_hit_count); RG_PRELOAD(k_hit_scatter); RG_PRELOAD(k_hit_order<real_gpu_hit>);
        RG_PRELOAD(k_unique_export); RG_PRELOAD(k_unique_ties); RG_PRELOAD(k_unique_import); RG_PRELOAD(k_unique_replay); RG_PRELOAD(k_fold_push); RG_PRELOAD(k_fold_merge); RG_PRELOAD(k_unique_checksum); RG_PRELOAD(k_mark_large); RG_PRELOAD(k_sort_large<0>); RG_PRELOAD(k_sort_large<1>); RG_PRELOAD(k_sort_large<2>);
        RG_PRELOAD(k_fmt_len<false>); RG_PRELOAD(k_fmt_len<true>); RG_PRELOAD(k_fmt_write<false>); RG_PRELOAD(k_fmt_write<true>);
        RG_PRELOAD(k_fa_summary); RG_PRELOAD(k_rd_table); RG_PRELOAD(k_rd_permute); RG_PRELOAD(k_rd_repack); RG_PRELOAD(k_rd_sums); RG_PRELOAD(k_fa_scan); RG_PRELOAD(k_fa_pack);
        RG_PRELOAD(k_window_counts); RG_PRELOAD(k_block_bounds); RG_PRELOAD(k_gap_dp); RG_PRELOAD(k_gap_replay);
#undef RG_PRELOAD
        done[device] = true;
}

int check_ready(real_gpu * h)
{
        if ( ! h->have_text ) return fail(h, REAL_GPU_E_STATE, "no text set");
        if ( ! h->have_reads ) return fail(h, REAL_GPU_E_STATE, "no reads set");
        if ( std::min<uint64_t>(h->n_total, h->own_end + h->maxlen) > h->shard_begin + h->shard_len )
                return fail(h, REAL_GPU_E_ARG, "the shard does not hold the read-length halo behind its own range (real_gpu_set_text: [own_begin, min(n_total, own_end + maxreadlen)))");
        return REAL_GPU_OK;
}

} // namespace

// =============================================================================================
// C ABI
// =============================================================================================

extern "C" {

int real_gpu_abi_version(void) { return REAL_GPU_ABI_VERSION; }

int real_gpu_device_count(void)
{
        int n = 0;
        if ( cudaGetDeviceCount(&n) != cudaSuccess ) { (void)cudaGetLastError(); return 0; }
        return n;
}

int real_gpu_create(const real_gpu_params * params, real_gpu ** out)
{
        if ( ! params || ! out ) return REAL_GPU_E_ARG;
        *out = nullptr;
        if ( params->struct_size != sizeof(real_gpu_params) ) return REAL_GPU_E_ARG;
        real_gpu * h = new real_gpu();
        h->prm = *params;
        h->prm.ll_table = nullptr;
        int code = REAL_GPU_OK;
        try
        {
                // option domain = what RealOptions lets through (RealOptions.cpp:434-453,176-180)
                if ( params->seedl < 4 || params->seedl > 64 || params->seedl % 4 )
                        throw std::invalid_argument("seed length must be a multiple of 4 in 4..64");
                if ( params->seedkmax > 2 ) throw std::invalid_argument("seedkmax > 2");
                if ( params->totalkmax > 15 ) throw std::invalid_argument("totalkmax > 15");
                if ( params->scores && ! params->ll_table ) throw std::invalid_argument("scores requested without ll_table");
                int ndev = 0;
                RG_CUDA(cudaGetDeviceCount(&ndev));
                if ( params->device < 0 || params->device >= ndev ) throw CudaError("no such CUDA device");
                RG_CUDA(cudaSetDevice(params->device));
                cudaDeviceProp prop;
                RG_CUDA(cudaGetDeviceProperties(&prop, params->device));
                if ( prop.major < 10 ) throw CudaError("device is not sm_100 class; this library only carries sm_100a code");
                h->sm_count = prop.multiProcessorCount;
                preload_kernels(params->device);
                if ( const char * e = getenv("REAL_GPU_AUTO_PREPARE") ) h->auto_prepare = atoi(e) != 0;
                RG_CUDA(cudaStreamCreateWithFlags(&h->st, cudaStreamNonBlocking));
                RG_CUDA(cudaStreamCreateWithFlags(&h->st2, cudaStreamNonBlocking));
                RG_CUDA(cudaMallocHost(&h->table_counts, 6 * sizeof(uint32_t)));
                RG_CUDA(cudaMallocHost(&h->fa_totals, 2 * sizeof(uint64_t)));
                for ( int i = 0; i < 8; ++i ) RG_CUDA(cudaEventCreate(&h->ev[i]));
                for ( int i = 0; i < 2; ++i ) RG_CUDA(cudaEventCreate(&h->evc[i]));
                RG_CUDA(cudaEventCreateWithFlags(&h->ev_words, cudaEventDisableTiming));
                if ( params->ll_table )
                {
                        dev_alloc(h, h->ll, 1024 * 8);
                        RG_CUDA(cudaMemcpyAsync(h->ll.p, params->ll_table, 1024 * 8, cudaMemcpyHostToDevice, h->st));
                        RG_CUDA(cudaStreamSynchronize(h->st));
                }
        }
        catch ( std::invalid_argument const & e ) { h->err = e.what(); code = REAL_GPU_E_ARG; }
        catch ( std::exception const & e ) { h->err = e.what(); code = REAL_GPU_E_CUDA; }
        if ( code != REAL_GPU_OK )
        {
                fprintf(stderr, "real_gpu_create: %s\n", h->err.c_str());
                real_gpu_destroy(h);
                return code;
        }
        *out = h;
        return REAL_GPU_OK;
}

int real_gpu_destroy(real_gpu * h)
{
        if ( ! h ) return REAL_GPU_OK;
        cudaSetDevice(h->prm.device);
        if ( h->text_pending && ! h->mask_deferred ) cudaEventSynchronize(h->evc[1]);
        if ( h->text_pending ) cudaStreamSynchronize(h->st2);
        if ( h->prep.inflight ) cudaEventSynchronize(h->prep.done);
        if ( h->prep.ev0 ) { cudaEventDestroy(h->prep.ev0); cudaEventDestroy(h->prep.done); }
        if ( h->st3 ) cudaStreamDestroy(h->st3);
        DevBuf * all[] = { &h->text, &h->nmask, &h->rec, &h->mapped, &h->qual, &h->offs, &h->rpack, &h->rlen, &h->seeds, &h->usable, &h->usable_rank, &h->bad,
                           &h->rec_win, &h->rec_pos, &h->part_meta, &h->own_list, &h->large_list, &h->win_valid, &h->win_counts, &h->bounds, &h->gapres, &h->gaps, &h->boffs, &h->flags8, &h->ws_k0, &h->ws_v0, &h->ws_k1, &h->ws_v1, &h->ws_flags, &h->ws_hist, &h->ws_stmp, &h->ll, &h->hits_raw, &h->hits_seg, &h->hits_out, &h->hits_out16, &h->counters, &h->counts, &h->starts, &h->cursor, &h->scantmp, &h->info, &h->scores,
                           &h->fa_raw, &h->fa_sums, &h->fa_tbase, &h->fa_trec, &h->fa_recnl, &h->fa_tot,
                           &h->rd_raw, &h->rd_sums, &h->rd_tbase, &h->rd_trec, &h->rd_stream, &h->rd_mask, &h->rd_start, &h->rd_nl, &h->rd_open, &h->rd_len, &h->rd_wild, &h->rd_idlen,
                           &h->rd_perm, &h->rd_olen, &h->rd_obytes, &h->rd_oidlen, &h->rd_boff, &h->rd_ioff, &h->rd_misc };
        for ( DevBuf * b : all ) dev_free(h, *b);
        for ( int t = 0; t < 3; ++t ) { dev_free(h, h->tab[t].bitmap); dev_free(h, h->tab[t].E); }
        for ( int r = 0; r < SC_MAX_RANKS; ++r )
                if ( h->comm.ipc_opened[r] ) { cudaIpcCloseMemHandle(h->comm.base[r]); h->comm.ipc_opened[r] = false; }
        for ( int i = 0; i < 2; ++i ) if ( h->comm.ev[i] ) cudaEventDestroy(h->comm.ev[i]);
        dev_free(h, h->comm.window); dev_free(h, h->comm.ptrs); dev_free(h, h->comm.pairs); dev_free(h, h->comm.error);
        for ( int r = 0; r < SC_MAX_RANKS; ++r )
                if ( h->fold.ipc_opened[r] ) { cudaIpcCloseMemHandle(h->fold.base[r]); h->fold.ipc_opened[r] = false; }
        if ( h->fold.ev ) cudaEventDestroy(h->fold.ev);
        dev_free(h, h->fold.window); dev_free(h, h->fold.ptrs); dev_free(h, h->fold.error);
        if ( h->host_hits ) cudaFreeHost(h->host_hits);
        {
                DevBuf * fb[] = { &h->fmt.ids, &h->fmt.id_off, &h->fmt.names, &h->fmt.name_off, &h->fmt.rec_start, &h->fmt.file_first, &h->fmt.len, &h->fmt.off, &h->fmt.out };
                for ( DevBuf * b : fb ) dev_free(h, *b);
                for ( int i = 0; i < 2; ++i ) if ( h->fmt.host[i] ) cudaFreeHost(h->fmt.host[i]);
        }
        for ( int i = 0; i < 8; ++i ) if ( h->ev[i] ) cudaEventDestroy(h->ev[i]);
        for ( cudaEvent_t e : h->evp ) cudaEventDestroy(e);
        for ( int i = 0; i < 8; ++i ) if ( h->stage_buf[i] ) cudaFreeHost(h->stage_buf[i]);
        for ( int i = 0; i < 4; ++i ) if ( h->stage_st[i] ) cudaStreamDestroy(h->stage_st[i]);
        for ( int i = 0; i < 2; ++i ) if ( h->evc[i] ) cudaEventDestroy(h->evc[i]);
        if ( h->ev_words ) cudaEventDestroy(h->ev_words);
        if ( h->st2 ) cudaStreamDestroy(h->st2);
        if ( h->table_counts ) cudaFreeHost(h->table_counts);
        if ( h->fa_totals ) cudaFreeHost(h->fa_totals);
        if ( h->st ) cudaStreamDestroy(h->st);
        delete h;
        return REAL_GPU_OK;
}

const char * real_gpu_last_error(const real_gpu * h) { return h ? h->err.c_str() : "null handle"; }

int real_gpu_set_text(real_gpu * h, uint32_t fileid, const uint64_t * words, const uint64_t * nmask,
                      uint64_t n_total, uint64_t shard_begin, uint64_t shard_len, uint64_t own_begin, uint64_t own_end,
                      const uint64_t * record_starts, uint32_t nrecords)
{
        RG_API_BEGIN_ASYNC(h)
        return set_text_common(h, fileid, words, nmask, false, n_total, shard_begin, shard_len, own_begin, own_end, record_starts, nrecords);
        RG_API_END(h)
}

int real_gpu_set_text_async(real_gpu * h, uint32_t fileid, const uint64_t * words, const uint64_t * nmask,
                            uint64_t n_total, uint64_t shard_begin, uint64_t shard_len, uint64_t own_begin, uint64_t own_end,
                            const uint64_t * record_starts, uint32_t nrecords)
{
        RG_API_BEGIN_ASYNC(h)
        return set_text_common(h, fileid, words, nmask, false, n_total, shard_begin, shard_len, own_begin, own_end, record_starts, nrecords, true);
        RG_API_END(h)
}

int real_gpu_prepare_scan(real_gpu * h, uint32_t max_read_len)
{
        RG_API_BEGIN_ASYNC(h)
        if ( ! h->have_text ) return fail(h, REAL_GPU_E_STATE, "prepare_scan: no text set");
        prepare_scan(h, max_read_len, false);
        return REAL_GPU_OK;
        RG_API_END(h)
}

int real_gpu_set_text_device(real_gpu * h, uint32_t fileid, const uint64_t * d_words, const uint64_t * d_nmask,
                             uint64_t n_total, uint64_t shard_begin, uint64_t shard_len, uint64_t own_begin, uint64_t own_end,
                             const uint64_t * record_starts, uint32_t nrecords)
{
        RG_API_BEGIN_ASYNC(h)
        return set_text_common(h, fileid, d_words, d_nmask, true, n_total, shard_begin, shard_len, own_begin, own_end, record_starts, nrecords);
        RG_API_END(h)
}

int real_gpu_set_text_device_async(real_gpu * h, uint32_t fileid, const uint64_t * d_words, const uint64_t * d_nmask,
                                   uint64_t n_total, uint64_t shard_begin, uint64_t shard_len, uint64_t own_begin, uint64_t own_end,
                                   const uint64_t * record_starts, uint32_t nrecords)
{
        RG_API_BEGIN_ASYNC(h)
        return set_text_common(h, fileid, d_words, d_nmask, true, n_total, shard_begin, shard_len, own_begin, own_end, record_starts, nrecords, true);
        RG_API_END(h)
}

int real_gpu_set_text_fasta(real_gpu * h, uint32_t fileid, const void * fasta_bytes, uint64_t nbytes, uint64_t * n_bases, uint64_t * nrecords)
{
        RG_API_BEGIN_ASYNC(h)
        return set_text_fasta_common(h, fileid, fasta_bytes, nbytes, false, n_bases, nrecords);
        RG_API_END(h)
}

int real_gpu_set_text_fasta_device(real_gpu * h, uint32_t fileid, const void * d_fasta_bytes, uint64_t nbytes, uint64_t * n_bases, uint64_t * nrecords)
{
        RG_API_BEGIN_ASYNC(h)
        return set_text_fasta_common(h, fileid, d_fasta_bytes, nbytes, true, n_bases, nrecords);
        RG_API_END(h)
}

int real_gpu_get_text_records(real_gpu * h, uint64_t * record_starts, uint64_t * header_ends)
{
        RG_API_BEGIN_ASYNC(h)
        if ( ! h->have_text || h->fa_rec_starts.size() != (size_t)h->nrec + 1 )
                return fail(h, REAL_GPU_E_STATE, "get_text_records: the current text was not set by real_gpu_set_text_fasta");
        if ( record_starts ) memcpy(record_starts, &h->fa_rec_starts[0], h->fa_rec_starts.size() * 8);
        if ( header_ends && h->nrec ) memcpy(header_ends, &h->fa_rec_nl[0], h->fa_rec_nl.size() * 8);
        return REAL_GPU_OK;
        RG_API_END(h)
}

int real_gpu_get_text_packed(real_gpu * h, uint64_t n_bases, uint64_t * words, uint64_t * nmask)
{
        RG_API_BEGIN_ASYNC(h)
        if ( ! h->have_text ) return fail(h, REAL_GPU_E_STATE, "no text set");
        if ( n_bases != h->shard_len ) return fail(h, REAL_GPU_E_ARG, "get_text_packed: n_bases is not the length of the current text (shard)");
        flush_mask(h);                  // a wildcard mask real_gpu_set_text_async has left behind goes first (same stream)
        if ( words ) RG_CUDA(cudaMemcpyAsync(words, ptr<uint64_t>(h->text) + TEXT_PAD_WORDS, (h->shard_len + 31) / 32 * 8, cudaMemcpyDeviceToHost, h->st2));
        if ( nmask ) RG_CUDA(cudaMemcpyAsync(nmask, ptr<uint64_t>(h->nmask) + TEXT_PAD_WORDS, (h->shard_len + 63) / 64 * 8, cudaMemcpyDeviceToHost, h->st2));
        RG_CUDA(cudaStreamSynchronize(h->st2));
        return REAL_GPU_OK;
        RG_API_END(h)
}

int real_gpu_set_reads(real_gpu * h, const uint8_t * mapped, const uint8_t * quality, const uint64_t * offsets, uint64_t nreads)
{
        RG_API_BEGIN(h)
        if ( ! offsets || (nreads && ! mapped) ) return fail(h, REAL_GPU_E_ARG, "set_reads: null pointer");
        if ( nreads >= (1ULL << 28) ) return fail(h, REAL_GPU_E_LIMIT, "set_reads: more than 2^28 reads in one set");
        uint64_t const total = offsets[nreads] - offsets[0];
        uint32_t maxlen = 0;
        for ( uint64_t i = 0; i < nreads; ++i )
        {
                if ( offsets[i+1] < offsets[i] ) return fail(h, REAL_GPU_E_ARG, "set_reads: offsets not ascending");
                uint64_t const L = offsets[i+1] - offsets[i];
                if ( L > 65535 ) return fail(h, REAL_GPU_E_LIMIT, "set_reads: read longer than 65535 bases");
                maxlen = std::max<uint32_t>(maxlen, (uint32_t)L);
        }
        h->have_reads = false;
        h->nreads = nreads; h->total_bases = total; h->maxlen = maxlen;
        if ( h->text_pending ) RG_CUDA(cudaStreamWaitEvent(h->st, h->ev_words, 0));   // one transfer after the other (see real_gpu_set_reads_packed)
        RG_CUDA(cudaEventRecord(h->ev[0], h->st));
        dev_reserve(h, h->mapped, total + 64);
        dev_reserve(h, h->offs, (nreads + 1) * 8);
        h->src_mapped = ptr<uint8_t>(h->mapped); h->src_packed = nullptr; h->src_len32 = nullptr;
        if ( total ) RG_CUDA(cudaMemcpyAsync(h->mapped.p, mapped + offsets[0], total, cudaMemcpyHostToDevice, h->st));
        if ( offsets[0] != 0 )
        {
                std::vector<uint64_t> rel(nreads + 1);
                for ( uint64_t i = 0; i <= nreads; ++i ) rel[i] = offsets[i] - offsets[0];
                RG_CUDA(cudaMemcpyAsync(h->offs.p, rel.data(), (nreads + 1) * 8, cudaMemcpyHostToDevice, h->st));
                RG_CUDA(cudaStreamSynchronize(h->st));
        }
        else
                RG_CUDA(cudaMemcpyAsync(h->offs.p, offsets, (nreads + 1) * 8, cudaMemcpyHostToDevice, h->st));
        h->qual_present = false;
        if ( quality && (h->prm.scores || h->ll.p) )
        {
                dev_reserve(h, h->qual, total + 64);
                if ( total ) RG_CUDA(cudaMemcpyAsync(h->qual.p, quality + offsets[0], total, cudaMemcpyHostToDevice, h->st));
                h->qual_present = true;
        }
        RG_CUDA(cudaEventRecord(h->ev[1], h->st));
        int const brc = build_from_device(h);           // enqueued; waited for by the next call that needs the index
        RG_CUDA(cudaEventSynchronize(h->ev[1]));        // the caller's buffers have been copied
        h->stats.h2d_reads_ms = elapsed(h->ev[0], h->ev[1]);
        flush_mask(h, true);    // a wildcard mask real_gpu_set_text_async has left behind travels now, behind the reads
        return brc;
        RG_API_END(h)
}

int real_gpu_set_reads_device(real_gpu * h, const uint8_t * d_mapped, const uint8_t * d_quality, const uint64_t * d_offsets,
                              uint64_t nreads, uint64_t total_bases, uint32_t maxlen)
{
        RG_API_BEGIN(h)
        if ( ! d_offsets || (nreads && ! d_mapped) ) return fail(h, REAL_GPU_E_ARG, "set_reads_device: null pointer");
        if ( nreads >= (1ULL << 28) ) return fail(h, REAL_GPU_E_LIMIT, "set_reads: more than 2^28 reads in one set");
        if ( maxlen > 65535 ) return fail(h, REAL_GPU_E_LIMIT, "set_reads: read longer than 65535 bases");
        h->have_reads = false;
        h->nreads = nreads; h->total_bases = total_bases; h->maxlen = maxlen;
        dev_reserve(h, h->offs, (nreads + 1) * 8);
        h->src_packed = nullptr; h->src_len32 = nullptr;
        h->src_mapped = d_mapped;          // packed before this call returns; the caller's buffer is not referenced afterwards
        RG_CUDA(cudaMemcpyAsync(h->offs.p, d_offsets, (nreads + 1) * 8, cudaMemcpyDeviceToDevice, h->st));
        h->qual_present = false;
        if ( d_quality && (h->prm.scores || h->ll.p) )
        {
                dev_reserve(h, h->qual, total_bases + 64);
                if ( total_bases ) RG_CUDA(cudaMemcpyAsync(h->qual.p, d_quality, total_bases, cudaMemcpyDeviceToDevice, h->st));
                h->qual_present = true;
        }
        h->stats.h2d_reads_ms = 0;
        int const brc = build_from_device(h);
        RG_CUDA(cudaEventSynchronize(h->ev[3]));        // the reads are packed: the caller's buffers are not referenced any more
        flush_mask(h, true);    // a wildcard mask real_gpu_set_text_async has left behind travels now, behind the reads
        return brc;
        RG_API_END(h)
}

int real_gpu_set_reads_packed(real_gpu * h, const uint8_t * packed, const uint64_t * byte_offsets, const uint32_t * lengths, uint32_t uniform_length,
                              const uint8_t * wildcard_flags, const uint8_t * quality, uint64_t nreads)
{
        RG_API_BEGIN(h)
        if ( nreads && ! packed ) return fail(h, REAL_GPU_E_ARG, "set_reads_packed: null pointer");
        if ( ! uniform_length && (! byte_offsets || ! lengths) ) return fail(h, REAL_GPU_E_ARG, "set_reads_packed: offsets and lengths are needed unless uniform_length is given");
        if ( nreads >= (1ULL << 28) ) return fail(h, REAL_GPU_E_LIMIT, "set_reads: more than 2^28 reads in one set");
        std::vector<uint64_t> boffs, offs;
        uint32_t maxlen = uniform_length;
        uint64_t total = (uint64_t)uniform_length * nreads, total_bytes = (uint64_t)((uniform_length + 3) / 4) * nreads;
        if ( ! uniform_length )
        {
                offs.resize(nreads + 1); offs[0] = 0;
                for ( uint64_t i = 0; i < nreads; ++i )
                {
                        if ( lengths[i] > 65535 ) return fail(h, REAL_GPU_E_LIMIT, "set_reads: read longer than 65535 bases");
                        maxlen = std::max(maxlen, lengths[i]);
                        offs[i+1] = offs[i] + lengths[i];
                }
                total = offs[nreads];
                total_bytes = byte_offsets[nreads] - byte_offsets[0];
                boffs.resize(nreads + 1);
                for ( uint64_t i = 0; i <= nreads; ++i ) boffs[i] = byte_offsets[i] - byte_offsets[0];
        }
        else if ( uniform_length > 65535 ) return fail(h, REAL_GPU_E_LIMIT, "set_reads: read longer than 65535 bases");
        h->have_reads = false;
        h->nreads = nreads; h->total_bases = total; h->maxlen = maxlen;
        // text words still on their way (real_gpu_set_text_async before the reads): one transfer after the other -- the partition
        // of real_gpu_prepare_scan starts when the words are complete and runs while the reads arrive
        if ( h->text_pending ) RG_CUDA(cudaStreamWaitEvent(h->st, h->ev_words, 0));
        RG_CUDA(cudaEventRecord(h->ev[0], h->st));
        dev_reserve(h, h->mapped, total_bytes + 64);
        dev_reserve(h, h->offs, (nreads + 1) * 8);
        dev_reserve(h, h->bad, (size_t)nreads * 4 + 16);
        if ( total_bytes ) RG_CUDA(cudaMemcpyAsync(h->mapped.p, packed + (uniform_length ? 0 : byte_offsets[0]), total_bytes, cudaMemcpyHostToDevice, h->st));
        h->src_packed = ptr<uint8_t>(h->mapped); h->src_mapped = nullptr; h->src_packed_uniform = uniform_length; h->src_byte_offsets = nullptr; h->src_len32 = nullptr;
        if ( uniform_length )
        {
                k_uniform_offsets<<<blocks_for(nreads + 1, 256), 256, 0, h->st>>>(ptr<uint64_t>(h->offs), nreads, uniform_length);
                RG_KERNEL_CHECK(); launch_count(h);
        }
        else
        {
                dev_reserve(h, h->boffs, (nreads + 1) * 8);
                RG_CUDA(cudaMemcpyAsync(h->offs.p, offs.data(), (nreads + 1) * 8, cudaMemcpyHostToDevice, h->st));
                RG_CUDA(cudaMemcpyAsync(h->boffs.p, boffs.data(), (nreads + 1) * 8, cudaMemcpyHostToDevice, h->st));
                h->src_byte_offsets = ptr<uint64_t>(h->boffs);
        }
        if ( wildcard_flags && nreads )
        {
                dev_reserve(h, h->flags8, nreads + 64);
                RG_CUDA(cudaMemcpyAsync(h->flags8.p, wildcard_flags, nreads, cudaMemcpyHostToDevice, h->st));
                k_flags_to_bad<<<blocks_for(nreads, 256), 256, 0, h->st>>>(ptr<uint8_t>(h->flags8), nreads, ptr<uint32_t>(h->bad));
                RG_KERNEL_CHECK(); launch_count(h);
        }
        else
                RG_CUDA(cudaMemsetAsync(h->bad.p, 0, (size_t)nreads * 4 + 16, h->st));
        h->qual_present = false;
        if ( quality && (h->prm.scores || h->ll.p) )
        {
                dev_reserve(h, h->qual, total + 64);
                if ( total ) RG_CUDA(cudaMemcpyAsync(h->qual.p, quality, total, cudaMemcpyHostToDevice, h->st));
                h->qual_present = true;
        }
        RG_CUDA(cudaEventRecord(h->ev[1], h->st));
        int const brc = build_from_device(h);           // enqueued; waited for by the next call that needs the index
        RG_CUDA(cudaEventSynchronize(h->ev[1]));        // the caller's buffers (and the staging vectors above) have been copied
        h->stats.h2d_reads_ms = elapsed(h->ev[0], h->ev[1]);
        flush_mask(h, true);    // a wildcard mask real_gpu_set_text_async has left behind travels now, behind the reads
        return brc;
        RG_API_END(h)
}


int real_gpu_set_reads_fasta(real_gpu * h, const void * fasta_bytes, uint64_t nbytes, uint32_t rewrite_order, uint64_t * nreads_out)
{
        RG_API_BEGIN(h)
        if ( (! fasta_bytes && nbytes) || ! nreads_out ) return fail(h, REAL_GPU_E_ARG, "set_reads_fasta: null pointer");
        *nreads_out = 0;
        uint64_t const ntiles = (nbytes + FA_TILE - 1) / FA_TILE;
        if ( ntiles >= (1ULL << 31) ) return fail(h, REAL_GPU_E_LIMIT, "set_reads_fasta: file longer than 2^43 bytes");
        h->have_reads = false;
        RG_CUDA(cudaEventRecord(h->ev[0], h->st));
        // the bytes of the file, then the three ingest kernels in pattern-file mode
        dev_reserve(h, h->rd_raw, nbytes + 64);
        h2d_from_host(h, h->rd_raw.p, fasta_bytes, nbytes, h->st);
        dev_reserve(h, h->rd_sums, std::max<uint64_t>(1, ntiles) * sizeof(FaSum32));
        dev_reserve(h, h->rd_tbase, std::max<uint64_t>(1, ntiles) * 8);
        dev_reserve(h, h->rd_trec, std::max<uint64_t>(1, ntiles) * 8);
        dev_reserve(h, h->rd_misc, 64);
        RG_CUDA(cudaMemsetAsync(h->rd_misc.p, 0, 64, h->st));
        const uint8_t * d_raw = ptr<uint8_t>(h->rd_raw);
        if ( ntiles )
                k_fa_summary<<<(unsigned)ntiles, FA_THREADS, 0, h->st>>>(d_raw, nbytes, ptr<FaSum32>(h->rd_sums), 1u);
        k_fa_scan<<<1, FA_SCAN_THREADS, 0, h->st>>>(ptr<FaSum32>(h->rd_sums), ntiles, ptr<uint64_t>(h->rd_tbase), ptr<uint64_t>(h->rd_trec), ptr<uint64_t>(h->rd_misc));
        RG_KERNEL_CHECK(); launch_count(h, ntiles ? 2 : 1);
        RG_CUDA(cudaMemcpyAsync(h->fa_totals, h->rd_misc.p, 16, cudaMemcpyDeviceToHost, h->st));
        RG_CUDA(cudaEventRecord(h->ev[1], h->st));
        RG_CUDA(cudaStreamSynchronize(h->st));                  // the caller's bytes are on the device; bases and reads are counted
        h->stats.h2d_reads_ms = elapsed(h->ev[0], h->ev[1]);
        uint64_t const nb = h->fa_totals[0], nreads = h->fa_totals[1];
        if ( nreads >= (1ULL << 28) ) return fail(h, REAL_GPU_E_LIMIT, "set_reads: more than 2^28 reads in one set");
        if ( nb / 4 + nreads >= (1ULL << 32) ) return fail(h, REAL_GPU_E_LIMIT, "set_reads_fasta: more than 2^32 bytes of packed reads; hand the reads over in batches");
        uint64_t const nw = (nb + 31) / 32 + 4, nmw = (nb + 63) / 64 + 4;
        dev_reserve(h, h->rd_stream, nw * 8);
        dev_reserve(h, h->rd_mask, nmw * 8);
        dev_reserve(h, h->rd_start, (nreads + 2) * 8);
        dev_reserve(h, h->rd_nl, (nreads + 2) * 8);
        dev_reserve(h, h->rd_open, (nreads + 2) * 8);
        RG_CUDA(cudaMemsetAsync(h->rd_stream.p, 0, nw * 8, h->st));
        RG_CUDA(cudaMemsetAsync(h->rd_mask.p, 0, nmw * 8, h->st));
        if ( ntiles )
                k_fa_pack<<<(unsigned)ntiles, FA_THREADS, 0, h->st>>>(d_raw, nbytes, ptr<uint64_t>(h->rd_tbase), ptr<uint64_t>(h->rd_trec),
                                                                      ptr<unsigned long long>(h->rd_stream), ptr<unsigned long long>(h->rd_mask),
                                                                      ptr<uint64_t>(h->rd_start), ptr<uint64_t>(h->rd_nl), ptr<uint64_t>(h->rd_open), 1u);
        RG_KERNEL_CHECK(); launch_count(h);
        RG_CUDA(cudaMemcpyAsync(ptr<uint64_t>(h->rd_start) + nreads, h->fa_totals, 8, cudaMemcpyHostToDevice, h->st));      // read_start[nreads] = all bases
        // per read: length, wildcard flag, id length; the longest read and the range of the ordering keys
        dev_reserve(h, h->rd_len, (nreads + 1) * 4);
        dev_reserve(h, h->rd_wild, (nreads + 1) * 4);
        dev_reserve(h, h->rd_idlen, (nreads + 1) * 4);
        unsigned int * d_mx = ptr<unsigned int>(h->rd_misc) + 8;           // [8] max length, [9] min key, [10] max key
        unsigned int const init[3] = { 0u, 0xFFFFFFFFu, 0u };
        RG_CUDA(cudaMemcpyAsync(d_mx, init, 12, cudaMemcpyHostToDevice, h->st));
        if ( nreads )
        {
                k_rd_table<<<blocks_for(nreads, 256), 256, 0, h->st>>>(ptr<uint64_t>(h->rd_start), ptr<uint64_t>(h->rd_mask), ptr<uint64_t>(h->rd_open), ptr<uint64_t>(h->rd_nl),
                                                                       nreads, ptr<uint32_t>(h->rd_len), ptr<uint32_t>(h->rd_wild), ptr<uint32_t>(h->rd_idlen), d_mx);
                RG_KERNEL_CHECK(); launch_count(h);
        }
        unsigned int mx[3] = { 0, 0, 0 };
        RG_CUDA(cudaMemcpyAsync(mx, d_mx, 12, cudaMemcpyDeviceToHost, h->st));
        RG_CUDA(cudaStreamSynchronize(h->st));
        if ( mx[0] > 65535 ) return fail(h, REAL_GPU_E_LIMIT, "set_reads: read longer than 65535 bases");
        // The order of the reference's rewritten pattern file (reorderFastA, ReorderFastA.hpp: by length, reads without wildcards
        // first, file order inside a group).  When all reads share one key -- the usual case -- it is the file order; otherwise the
        // keys (8 bytes per read) go to the host for one stable counting sort and the permutation comes back.
        const uint32_t * d_perm = nullptr;
        if ( rewrite_order && nreads && mx[1] != mx[2] )
        {
                std::vector<uint32_t> len(nreads), wild(nreads), perm(nreads);
                RG_CUDA(cudaMemcpyAsync(len.data(), h->rd_len.p, nreads * 4, cudaMemcpyDeviceToHost, h->st));
                RG_CUDA(cudaMemcpyAsync(wild.data(), h->rd_wild.p, nreads * 4, cudaMemcpyDeviceToHost, h->st));
                RG_CUDA(cudaStreamSynchronize(h->st));
                std::vector<uint64_t> cnt((size_t)2 * (mx[0] + 1) + 1, 0);
                for ( uint64_t r = 0; r < nreads; ++r ) ++cnt[(size_t)2 * len[r] + wild[r] + 1];
                for ( size_t k = 1; k < cnt.size(); ++k ) cnt[k] += cnt[k-1];
                for ( uint64_t r = 0; r < nreads; ++r ) perm[cnt[(size_t)2 * len[r] + wild[r]]++] = (uint32_t)r;
                dev_reserve(h, h->rd_perm, nreads * 4);
                RG_CUDA(cudaMemcpyAsync(h->rd_perm.p, perm.data(), nreads * 4, cudaMemcpyHostToDevice, h->st));
                RG_CUDA(cudaStreamSynchronize(h->st));
                d_perm = ptr<uint32_t>(h->rd_perm);
        }
        // lengths, flags and sizes in output order; byte offsets of the packed reads and of the ids
        dev_reserve(h, h->rd_olen, (nreads + 1) * 4);
        dev_reserve(h, h->flags8, nreads + 64);
        dev_reserve(h, h->rd_obytes, (nreads + 1) * 4);
        dev_reserve(h, h->rd_oidlen, (nreads + 1) * 4);
        dev_reserve(h, h->rd_boff, (nreads + 1) * 4);
        dev_reserve(h, h->rd_ioff, (nreads + 1) * 4);
        dev_reserve(h, h->scantmp, scan_temp_elems(nreads + 1) * 4 + 64);
        unsigned long long tot[2] = { 0, 0 };
        if ( nreads )
        {
                k_rd_permute<<<blocks_for(nreads, 256), 256, 0, h->st>>>(d_perm, nreads, ptr<uint32_t>(h->rd_len), ptr<uint32_t>(h->rd_wild), ptr<uint32_t>(h->rd_idlen),
                                                                         ptr<uint32_t>(h->rd_olen), ptr<uint8_t>(h->flags8), ptr<uint32_t>(h->rd_obytes), ptr<uint32_t>(h->rd_oidlen));
                RG_KERNEL_CHECK(); launch_count(h);
                RG_CUDA(cudaMemsetAsync(h->rd_misc.p, 0, 16, h->st));
                k_rd_sums<<<(unsigned)std::min<uint64_t>(blocks_for(nreads, 256), (uint64_t)h->sm_count * 8), 256, 0, h->st>>>(ptr<uint32_t>(h->rd_obytes), ptr<uint32_t>(h->rd_oidlen), nreads,
                                                                                                                       ptr<unsigned long long>(h->rd_misc));
                RG_KERNEL_CHECK(); launch_count(h);
                RG_CUDA(cudaMemcpyAsync(tot, h->rd_misc.p, 16, cudaMemcpyDeviceToHost, h->st));
                uint32_t nl = 0;
                exclusive_scan_u32(ptr<uint32_t>(h->rd_obytes), ptr<uint32_t>(h->rd_boff), nreads, ptr<uint32_t>(h->scantmp), h->st, &nl);
                exclusive_scan_u32(ptr<uint32_t>(h->rd_oidlen), ptr<uint32_t>(h->rd_ioff), nreads, ptr<uint32_t>(h->scantmp), h->st, &nl);
                launch_count(h, nl);
                RG_CUDA(cudaStreamSynchronize(h->st));
        }
        if ( tot[0] >= (1ULL << 32) || tot[1] >= (1ULL << 32) )
                return fail(h, REAL_GPU_E_LIMIT, "set_reads_fasta: more than 2^32 bytes of packed reads or of ids; hand the reads over in batches");
        // the read set as real_gpu_set_reads_packed leaves it: packed bytes, byte offsets, lengths, flags -- and the ids for K8
        h->nreads = nreads; h->total_bases = nb; h->maxlen = mx[0];
        dev_reserve(h, h->mapped, tot[0] + 64);
        dev_reserve(h, h->boffs, (nreads + 1) * 8);
        dev_reserve(h, h->bad, (size_t)nreads * 4 + 16);
        real_gpu::Format & F = h->fmt;
        dev_reserve(h, F.ids, tot[1] + 16);
        dev_reserve(h, F.id_off, (nreads + 1) * 8);
        k_rd_repack<<<blocks_for(nreads + 1, 256), 256, 0, h->st>>>(d_perm, nreads, ptr<uint64_t>(h->rd_stream), ptr<uint64_t>(h->rd_start), ptr<uint32_t>(h->rd_boff),
                                                                    ptr<uint8_t>(h->mapped), ptr<uint64_t>(h->boffs), d_raw, ptr<uint64_t>(h->rd_open), ptr<uint32_t>(h->rd_oidlen),
                                                                    ptr<uint32_t>(h->rd_ioff), ptr<char>(F.ids), ptr<uint64_t>(F.id_off), tot[0], tot[1]);
        RG_KERNEL_CHECK(); launch_count(h);
        F.id_first = 0; F.id_count = nreads; F.id_bytes = tot[1];
        if ( nreads )
        {
                k_flags_to_bad<<<blocks_for(nreads, 256), 256, 0, h->st>>>(ptr<uint8_t>(h->flags8), nreads, ptr<uint32_t>(h->bad));
                RG_KERNEL_CHECK(); launch_count(h);
        }
        h->src_packed = ptr<uint8_t>(h->mapped); h->src_mapped = nullptr; h->src_packed_uniform = 0;
        h->src_byte_offsets = ptr<uint64_t>(h->boffs); h->src_len32 = ptr<uint32_t>(h->rd_olen);
        h->qual_present = false;
        RG_CUDA(cudaStreamSynchronize(h->st));
        // the file bytes and the intermediate stream are several times the packed reads: released
        DevBuf * rel[] = { &h->rd_raw, &h->rd_stream, &h->rd_mask, &h->rd_sums, &h->rd_tbase, &h->rd_trec, &h->rd_start, &h->rd_nl, &h->rd_open, &h->rd_len, &h->rd_wild,
                           &h->rd_idlen, &h->rd_perm, &h->rd_obytes, &h->rd_oidlen, &h->rd_boff, &h->rd_ioff };
        for ( DevBuf * b : rel ) dev_free(h, *b);
        *nreads_out = nreads;
        return build_from_device(h);
        RG_API_END(h)
}

// the read table of the current set: lengths and wildcard flags (either may be NULL), in read order
int real_gpu_get_read_table(real_gpu * h, uint32_t * lengths, uint8_t * wildcard_flags)
{
        RG_API_BEGIN(h)
        if ( ! h->have_reads ) return fail(h, REAL_GPU_E_STATE, "no reads set");
        if ( lengths && h->nreads )
        {
                if ( ! h->src_len32 ) return fail(h, REAL_GPU_E_STATE, "get_read_table: the lengths are kept only for reads set by real_gpu_set_reads_fasta");
                { RG_CUDA(cudaMemcpyAsync(lengths, h->src_len32, h->nreads * 4, cudaMemcpyDeviceToHost, h->st)); RG_CUDA(cudaStreamSynchronize(h->st)); }
        }
        if ( wildcard_flags && h->nreads )
        {
                std::vector<uint32_t> bad(h->nreads);
                { RG_CUDA(cudaMemcpyAsync(bad.data(), h->bad.p, h->nreads * 4, cudaMemcpyDeviceToHost, h->st)); RG_CUDA(cudaStreamSynchronize(h->st)); }
                for ( uint64_t i = 0; i < h->nreads; ++i ) wildcard_flags[i] = bad[i] ? 1 : 0;
        }
        return REAL_GPU_OK;
        RG_API_END(h)
}

// the ids of the reads as set by real_gpu_set_read_ids / real_gpu_set_reads_fasta: offsets[count+1] and, when bytes is given,
// the id bytes (offsets[count] of them; call once with bytes = NULL to learn the size)
int real_gpu_get_read_ids(real_gpu * h, char * bytes, uint64_t * offsets)
{
        RG_API_BEGIN(h)
        if ( ! offsets ) return fail(h, REAL_GPU_E_ARG, "get_read_ids: null pointer");
        real_gpu::Format & F = h->fmt;
        if ( ! F.id_off.p ) return fail(h, REAL_GPU_E_STATE, "no ids set");
        { RG_CUDA(cudaMemcpyAsync(offsets, F.id_off.p, (F.id_count + 1) * 8, cudaMemcpyDeviceToHost, h->st)); RG_CUDA(cudaStreamSynchronize(h->st)); }
        if ( bytes && offsets[F.id_count] ) { RG_CUDA(cudaMemcpyAsync(bytes, F.ids.p, offsets[F.id_count], cudaMemcpyDeviceToHost, h->st)); RG_CUDA(cudaStreamSynchronize(h->st)); }
        return REAL_GPU_OK;
        RG_API_END(h)
}

// the packed bytes of the reads [first, first+count) of a 2 bit/base read set and their byte offsets (count+1, relative to the first)
int real_gpu_get_reads_packed(real_gpu * h, uint8_t * packed, uint64_t * byte_offsets)
{
        RG_API_BEGIN(h)
        if ( ! h->have_reads ) return fail(h, REAL_GPU_E_STATE, "no reads set");
        if ( ! h->src_packed || ! h->src_byte_offsets || ! byte_offsets ) return fail(h, REAL_GPU_E_STATE, "get_reads_packed: no packed read set with byte offsets");
        { RG_CUDA(cudaMemcpyAsync(byte_offsets, h->src_byte_offsets, (h->nreads + 1) * 8, cudaMemcpyDeviceToHost, h->st)); RG_CUDA(cudaStreamSynchronize(h->st)); }
        if ( packed && byte_offsets[h->nreads] ) { RG_CUDA(cudaMemcpyAsync(packed, h->src_packed, byte_offsets[h->nreads], cudaMemcpyDeviceToHost, h->st)); RG_CUDA(cudaStreamSynchronize(h->st)); }
        return REAL_GPU_OK;
        RG_API_END(h)
}

int real_gpu_set_reads_packed_device(real_gpu * h, const uint8_t * d_packed, uint32_t uniform_length, const uint8_t * d_wildcard_flags,
                                     const uint8_t * d_quality, uint64_t nreads)
{
        RG_API_BEGIN(h)
        if ( nreads && ! d_packed ) return fail(h, REAL_GPU_E_ARG, "set_reads_packed_device: null pointer");
        if ( ! uniform_length || uniform_length > 65535 ) return fail(h, REAL_GPU_E_ARG, "set_reads_packed_device: uniform_length must be 1..65535");
        if ( nreads >= (1ULL << 28) ) return fail(h, REAL_GPU_E_LIMIT, "set_reads: more than 2^28 reads in one set");
        h->have_reads = false;
        h->nreads = nreads; h->total_bases = (uint64_t)uniform_length * nreads; h->maxlen = uniform_length;
        dev_reserve(h, h->offs, (nreads + 1) * 8);
        dev_reserve(h, h->bad, (size_t)nreads * 4 + 16);
        h->src_packed = d_packed; h->src_mapped = nullptr; h->src_packed_uniform = uniform_length; h->src_byte_offsets = nullptr; h->src_len32 = nullptr;
        k_uniform_offsets<<<blocks_for(nreads + 1, 256), 256, 0, h->st>>>(ptr<uint64_t>(h->offs), nreads, uniform_length);
        RG_KERNEL_CHECK(); launch_count(h);
        if ( d_wildcard_flags && nreads )
        {
                k_flags_to_bad<<<blocks_for(nreads, 256), 256, 0, h->st>>>(d_wildcard_flags, nreads, ptr<uint32_t>(h->bad));
                RG_KERNEL_CHECK(); launch_count(h);
        }
        else
                RG_CUDA(cudaMemsetAsync(h->bad.p, 0, (size_t)nreads * 4 + 16, h->st));
        h->qual_present = false;
        if ( d_quality && (h->prm.scores || h->ll.p) )
        {
                dev_reserve(h, h->qual, h->total_bases + 64);
                if ( h->total_bases ) RG_CUDA(cudaMemcpyAsync(h->qual.p, d_quality, h->total_bases, cudaMemcpyDeviceToDevice, h->st));
                h->qual_present = true;
        }
        h->stats.h2d_reads_ms = 0;
        int const brc = build_from_device(h);
        RG_CUDA(cudaEventSynchronize(h->ev[3]));        // the reads are packed: the caller's buffers are not referenced any more
        flush_mask(h, true);    // a wildcard mask real_gpu_set_text_async has left behind travels now, behind the reads
        return brc;
        RG_API_END(h)
}

// scan in hit-list mode (regrowing the buffer if it was too small), score the hits, group them by read:
// afterwards hits_seg holds the hits of read r at [starts[r], starts[r] + counts[r])
static uint64_t collect_hits_by_read(real_gpu * h, int mode = 0)
{
        if ( h->hit_cap == 0 )
        {
                uint64_t const cap = std::max<uint64_t>(1u << 16, 2 * h->nreads);
                dev_alloc(h, h->hits_raw, cap * sizeof(RawHit));
                h->hit_cap = cap;              // only once the buffer exists
        }
        uint64_t found = run_scan(h, mode);
        if ( found > h->hit_cap )
        {
                // the buffer was too small: the kernel counted everything, so size it exactly
                uint64_t const cap = found + found / 8 + 1024;
                h->hit_cap = 0;
                dev_alloc(h, h->hits_raw, cap * sizeof(RawHit));
                h->hit_cap = cap;
                if ( h->comm.nranks > 1 && h->comm.window.p )
                        // Sharded tables: a scan is a sequence of rounds all ranks take part in (the hand-over flags count them).
                        // A rank that rescanned on its own would run rounds no peer joins -- and would pair with the peers' NEXT
                        // call.  The decision has to be collective: this call fails on this rank, the buffer is already enlarged.
                        throw LimitError("sharded tables: the hit buffer of this rank was too small for " + std::to_string(found) +
                                         " hits; it has been enlarged -- repeat the call on EVERY rank");
                found = run_scan(h, mode);
                if ( found > h->hit_cap ) throw CudaError("hit count changed between scans");
        }
        if ( found >= (1ULL << 32) ) throw LimitError("more than 2^32 hits in one call");
        RG_CUDA(cudaEventRecord(h->ev[0], h->st));
        dev_reserve(h, h->counts, h->nreads * 4 + 16);
        dev_reserve(h, h->starts, h->nreads * 4 + 16);
        dev_reserve(h, h->cursor, h->nreads * 4 + 16);
        RG_CUDA(cudaMemsetAsync(h->counts.p, 0, h->nreads * 4 + 16, h->st));
        if ( found )
        {
                if ( h->prm.scores && mode == 0 )
                {
                        k_score_hits<<<blocks_for(found, 256), 256, 0, h->st>>>(ptr<RawHit>(h->hits_raw), found, ptr<double>(h->ll),
                                ptr<uint64_t>(h->text) + TEXT_PAD_WORDS, h->shard_begin, read_src(h), ptr<uint32_t>(h->rlen),
                                h->qual_present ? ptr<uint8_t>(h->qual) : nullptr, ptr<uint64_t>(h->offs));
                        RG_KERNEL_CHECK(); launch_count(h);
                }
                // counting sort by read
                dev_reserve(h, h->scantmp, scan_temp_elems(h->nreads) * 4 + 64);
                dev_reserve(h, h->hits_seg, found * sizeof(RawHit));
                RG_CUDA(cudaMemsetAsync(h->cursor.p, 0, h->nreads * 4, h->st));
                k_hit_count<<<blocks_for(found, 256), 256, 0, h->st>>>(ptr<RawHit>(h->hits_raw), found, ptr<uint32_t>(h->counts));
                RG_KERNEL_CHECK(); launch_count(h);
                uint32_t nl = 0;
                exclusive_scan_u32(ptr<uint32_t>(h->counts), ptr<uint32_t>(h->starts), h->nreads, ptr<uint32_t>(h->scantmp), h->st, &nl);
                launch_count(h, nl);
                k_hit_scatter<<<blocks_for(found, 256), 256, 0, h->st>>>(ptr<RawHit>(h->hits_raw), found, ptr<uint32_t>(h->starts), ptr<uint32_t>(h->cursor), ptr<RawHit>(h->hits_seg));
                RG_KERNEL_CHECK(); launch_count(h);
                // reads with more hits than one thread should sort (post.cuh, SEG_SMALL)
                dev_reserve(h, h->large_list, (found / SEG_SMALL + 16) * 4);
                RG_CUDA(cudaMemsetAsync(h->large_list.p, 0, 4, h->st));
                k_mark_large<<<blocks_for(h->nreads, 256), 256, 0, h->st>>>(ptr<uint32_t>(h->counts), h->nreads, ptr<uint32_t>(h->large_list) + 4, ptr<uint32_t>(h->large_list));
                RG_KERNEL_CHECK(); launch_count(h);
        }
        return found;
}

// sorts the segments of the reads k_mark_large has listed (one CTA each); the raw hit buffer serves as scratch space
static void sort_large_segments(real_gpu * h, int mode, const uint64_t * bounds, uint32_t nblocks)
{
        SortLargeParams SP;
        SP.seg = ptr<RawHit>(h->hits_seg); SP.tmp = ptr<RawHit>(h->hits_raw);
        SP.starts = ptr<uint32_t>(h->starts); SP.counts = ptr<uint32_t>(h->counts);
        SP.list = ptr<uint32_t>(h->large_list) + 4; SP.nlarge = ptr<uint32_t>(h->large_list);
        SP.rlen = ptr<uint32_t>(h->rlen); SP.seedl = h->prm.seedl; SP.bounds = bounds; SP.nblocks = nblocks;
        unsigned const grid = (unsigned)(h->sm_count * 4);
        if ( mode == 0 ) k_sort_large<0><<<grid, 256, 0, h->st>>>(SP);
        else if ( mode == 1 ) k_sort_large<1><<<grid, 256, 0, h->st>>>(SP);
        else k_sort_large<2><<<grid, 256, 0, h->st>>>(SP);
        RG_KERNEL_CHECK(); launch_count(h);
}

} // extern "C"

namespace
{
// the body of real_gpu_match_all / real_gpu_match_all_packed: rows of 40 bytes (ABI struct) or of 16 bytes to the host
int match_all_common(real_gpu * h, bool packed, const void ** rows, uint64_t * nhits)
{
        int const rc = check_ready(h);
        if ( rc ) return rc;
        *rows = nullptr; *nhits = 0;
        h->stats.scan_launches = 0;
        uint64_t const found = collect_hits_by_read(h);
        size_t const rowbytes = packed ? sizeof(real_gpu_hit16) : sizeof(real_gpu_hit);
        if ( found )
        {
                dev_reserve(h, h->hits_out, found * sizeof(real_gpu_hit));
                if ( packed ) dev_reserve(h, h->hits_out16, found * sizeof(real_gpu_hit16));
                sort_large_segments(h, 0, nullptr, 1);
                k_hit_order<real_gpu_hit><<<blocks_for(h->nreads, 128), 128, 0, h->st>>>(ptr<RawHit>(h->hits_seg), ptr<uint32_t>(h->starts), ptr<uint32_t>(h->counts),
                                                                                        h->nreads, h->fileid, ptr<real_gpu_hit>(h->hits_out),
                                                                                        packed ? ptr<real_gpu_hit16>(h->hits_out16) : nullptr);
                RG_KERNEL_CHECK(); launch_count(h);
        }
        RG_CUDA(cudaEventRecord(h->ev[1], h->st));
        if ( found * rowbytes > h->host_hits_cap * sizeof(real_gpu_hit) )
        {
                if ( h->host_hits ) cudaFreeHost(h->host_hits);
                h->host_hits = nullptr; h->host_hits_cap = 0;
                uint64_t const cap = found * rowbytes / sizeof(real_gpu_hit) + found / 4 + 1024;
                RG_CUDA(cudaMallocHost(&h->host_hits, cap * sizeof(real_gpu_hit)));
                h->host_hits_cap = cap;
        }
        if ( found )
                RG_CUDA(cudaMemcpyAsync(h->host_hits, packed ? h->hits_out16.p : h->hits_out.p, found * rowbytes, cudaMemcpyDeviceToHost, h->st));
        RG_CUDA(cudaEventRecord(h->ev[2], h->st));
        RG_CUDA(cudaStreamSynchronize(h->st));
        h->stats.post_ms = elapsed(h->ev[0], h->ev[1]);
        h->stats.d2h_ms = elapsed(h->ev[1], h->ev[2]);
        *rows = h->host_hits;
        *nhits = found;
        h->fmt.nrows_all = found;
        return REAL_GPU_OK;
}
} // namespace

extern "C" {

int real_gpu_match_all(real_gpu * h, const real_gpu_hit ** hits, uint64_t * nhits)
{
        RG_API_BEGIN(h)
        if ( ! hits || ! nhits ) return fail(h, REAL_GPU_E_ARG, "match_all: null pointer");
        return match_all_common(h, false, reinterpret_cast<const void **>(hits), nhits);
        RG_API_END(h)
}

int real_gpu_match_all_packed(real_gpu * h, const real_gpu_hit16 ** rows, uint64_t * nhits)
{
        RG_API_BEGIN(h)
        if ( ! rows || ! nhits ) return fail(h, REAL_GPU_E_ARG, "match_all_packed: null pointer");
        return match_all_common(h, true, reinterpret_cast<const void **>(rows), nhits);
        RG_API_END(h)
}

// first window of every reference text block (matchUniqueImplementation.cpp:1208-1244: n_list windows per block)
static uint32_t block_bounds(real_gpu * h)
{
        if ( ! h->n_list ) return 1;
        if ( h->text_pending )
        {
                // real_gpu_set_text_async: the window counts read the wildcard mask, which may still be on its way (or not even sent)
                flush_mask(h);
                RG_CUDA(cudaStreamWaitEvent(h->st, h->evc[1], 0));
        }
        uint32_t const seedl = h->prm.seedl;
        uint64_t const ngroups = (h->n_total + 63) / 64;
        dev_reserve(h, h->win_valid, ngroups * 8 + 64);
        dev_reserve(h, h->win_counts, ngroups * 4 + 64);
        dev_reserve(h, h->scantmp, scan_temp_elems(ngroups) * 4 + 64);
        k_window_counts<<<blocks_for(ngroups, 256), 256, 0, h->st>>>(ptr<uint64_t>(h->nmask) + TEXT_PAD_WORDS, h->n_total, seedl, ngroups,
                                                                     ptr<uint64_t>(h->win_valid), ptr<uint32_t>(h->win_counts));
        RG_KERNEL_CHECK(); launch_count(h);
        uint32_t lastc = 0, lastp = 0, nl = 0;
        RG_CUDA(cudaMemcpyAsync(&lastc, ptr<uint32_t>(h->win_counts) + (ngroups - 1), 4, cudaMemcpyDeviceToHost, h->st));
        exclusive_scan_u32(ptr<uint32_t>(h->win_counts), ptr<uint32_t>(h->win_counts), ngroups, ptr<uint32_t>(h->scantmp), h->st, &nl);
        launch_count(h, nl);
        RG_CUDA(cudaMemcpyAsync(&lastp, ptr<uint32_t>(h->win_counts) + (ngroups - 1), 4, cudaMemcpyDeviceToHost, h->st));
        RG_CUDA(cudaStreamSynchronize(h->st));
        if ( h->n_total >= (1ULL << 32) )
                throw LimitError("reference text blocks (n_list) on a text of 2^32 or more bases: the window prefix sums are 32 bit");
        uint64_t const nwin = (uint64_t)lastc + lastp;
        uint64_t const nb = nwin ? (nwin + h->n_list - 1) / h->n_list : 1;
        if ( nb <= 1 ) return 1;
        if ( nb > (1u << 24) ) throw CudaError("more than 2^24 reference text blocks");
        dev_reserve(h, h->bounds, nb * 8 + 64);
        k_block_bounds<<<blocks_for(nb, 64), 64, 0, h->st>>>(ptr<uint64_t>(h->win_valid), ptr<uint32_t>(h->win_counts), ngroups, h->n_list, (uint32_t)nb, ptr<uint64_t>(h->bounds));
        RG_KERNEL_CHECK(); launch_count(h);
        return (uint32_t)nb;
}

int real_gpu_match_unique(real_gpu * h)
{
        RG_API_BEGIN(h)
        int const rc = check_ready(h);
        if ( rc ) return rc;
        if ( h->nrec + 1 > 65536 )
                return REAL_GPU_OK;   // the reference skips such files (matchUniqueImplementation.cpp:1139-1143)
        h->stats.scan_launches = 0;
        h->stats.post_ms = 0; h->stats.d2h_ms = 0;
        if ( ! h->prm.scores )
        {
                run_scan(h, 1);         // order independent: folded in the scan itself
                return REAL_GPU_OK;
        }
        // with scores the fold depends on the reference's visiting order (matchUniqueImplementation.cpp:179-248):
        // collect the hits of this file, then replay them per read in that order
        if ( h->comm.nranks > 1 )
                return fail(h, REAL_GPU_E_ARG, "match_unique with scores is order dependent: not available with sharded tables");
        if ( h->shard_begin != 0 || h->shard_len != h->n_total || h->own_begin != 0 || h->own_end != h->n_total )
                return fail(h, REAL_GPU_E_ARG, "match_unique with scores needs the whole file in one shard (the fold is order dependent)");
        uint64_t const found = collect_hits_by_read(h);
        if ( found )
        {
                uint32_t const nb = block_bounds(h);
                ReplayParams R;
                R.seg = ptr<RawHit>(h->hits_seg); R.starts = ptr<uint32_t>(h->starts); R.counts = ptr<uint32_t>(h->counts); R.rlen = ptr<uint32_t>(h->rlen);
                R.nreads = h->nreads; R.seedl = h->prm.seedl; R.fileid = h->fileid; R.filter_mult = h->prm.filter_mult;
                R.bounds = nb > 1 ? ptr<uint64_t>(h->bounds) : nullptr; R.nblocks = nb;
                R.info = ptr<unsigned long long>(h->info); R.score = ptr<float>(h->scores);
                sort_large_segments(h, 1, R.bounds, nb);
                k_unique_replay<<<blocks_for(h->nreads, 128), 128, 0, h->st>>>(R);
                RG_KERNEL_CHECK(); launch_count(h);
        }
        RG_CUDA(cudaEventRecord(h->ev[1], h->st));
        RG_CUDA(cudaStreamSynchronize(h->st));
        h->stats.post_ms = elapsed(h->ev[0], h->ev[1]);
        return REAL_GPU_OK;
        RG_API_END(h)
}

int real_gpu_get_unique_range(real_gpu * h, uint64_t first, uint64_t count, uint64_t * info, float * scores)
{
        RG_API_BEGIN(h)
        if ( ! h->have_reads ) return fail(h, REAL_GPU_E_STATE, "no reads set");
        if ( ! info ) return fail(h, REAL_GPU_E_ARG, "get_unique: null pointer");
        if ( first > h->nreads || count > h->nreads - first ) return fail(h, REAL_GPU_E_ARG, "get_unique: range outside the read set");
        RG_CUDA(cudaEventRecord(h->ev[0], h->st));
        if ( count ) RG_CUDA(cudaMemcpyAsync(info, ptr<uint64_t>(h->info) + first, count * 8, cudaMemcpyDeviceToHost, h->st));
        RG_CUDA(cudaEventRecord(h->ev[1], h->st));
        RG_CUDA(cudaStreamSynchronize(h->st));
        h->stats.d2h_ms = elapsed(h->ev[0], h->ev[1]);
        if ( scores )
        {
                if ( h->prm.scores && count ) RG_CUDA(cudaMemcpy(scores, ptr<float>(h->scores) + first, count * 4, cudaMemcpyDeviceToHost));
                else for ( uint64_t i = 0; i < count; ++i ) scores[i] = 0.0f;
        }
        return REAL_GPU_OK;
        RG_API_END(h)
}

int real_gpu_get_unique(real_gpu * h, uint64_t * info, float * scores)
{
        if ( ! h ) return REAL_GPU_E_ARG;
        return real_gpu_get_unique_range(h, 0, h->nreads, info, scores);
}

int real_gpu_unique_checksum(real_gpu * h, uint64_t first, uint64_t count, uint64_t * checksum)
{
        RG_API_BEGIN(h)
        if ( ! h->have_reads ) return fail(h, REAL_GPU_E_STATE, "no reads set");
        if ( ! checksum ) return fail(h, REAL_GPU_E_ARG, "unique_checksum: null pointer");
        if ( first > h->nreads || count > h->nreads - first ) return fail(h, REAL_GPU_E_ARG, "unique_checksum: range outside the read set");
        dev_reserve(h, h->counters, 8 * 8);
        RG_CUDA(cudaMemsetAsync(h->counters.p, 0, 8, h->st));
        if ( count )
        {
                k_unique_checksum<<<(unsigned)std::min<uint64_t>(blocks_for(count, 256), (uint64_t)h->sm_count * 8), 256, 0, h->st>>>(
                        ptr<unsigned long long>(h->info), first, count, ptr<unsigned long long>(h->counters));
                RG_KERNEL_CHECK(); launch_count(h);
        }
        unsigned long long v = 0;
        RG_CUDA(cudaMemcpyAsync(&v, h->counters.p, 8, cudaMemcpyDeviceToHost, h->st));
        RG_CUDA(cudaStreamSynchronize(h->st));
        *checksum = v;
        return REAL_GPU_OK;
        RG_API_END(h)
}

int real_gpu_reset_unique(real_gpu * h)
{
        RG_API_BEGIN(h)
        if ( ! h->have_reads ) return fail(h, REAL_GPU_E_STATE, "no reads set");
        RG_CUDA(cudaMemsetAsync(h->info.p, 0, (size_t)h->nreads * 8 + 16, h->st));
        if ( h->gaps.p ) RG_CUDA(cudaMemsetAsync(h->gaps.p, 0, (size_t)h->nreads * sizeof(real_gpu_gapinfo) + 16, h->st));
        if ( h->prm.scores )
        {
                k_fill_f32<<<blocks_for(h->nreads + 1, 256), 256, 0, h->st>>>(ptr<float>(h->scores), h->nreads, -FLT_MAX);
                RG_KERNEL_CHECK(); launch_count(h);
        }
        RG_CUDA(cudaStreamSynchronize(h->st));
        return REAL_GPU_OK;
        RG_API_END(h)
}

int real_gpu_set_block_windows(real_gpu * h, uint64_t n_list)
{
        if ( ! h ) return REAL_GPU_E_ARG;
        h->n_list = n_list;
        return REAL_GPU_OK;
}

int real_gpu_unique_export_keys(real_gpu * h, uint64_t * d_keys)
{
        RG_API_BEGIN(h)
        if ( ! h->have_reads ) return fail(h, REAL_GPU_E_STATE, "no reads set");
        if ( ! d_keys ) return fail(h, REAL_GPU_E_ARG, "null pointer");
        if ( h->nreads )
        {
                k_unique_export<<<blocks_for(h->nreads, 256), 256, 0, h->st>>>(ptr<unsigned long long>(h->info), h->nreads, d_keys);
                RG_KERNEL_CHECK(); launch_count(h);
        }
        RG_CUDA(cudaStreamSynchronize(h->st));
        return REAL_GPU_OK;
        RG_API_END(h)
}

int real_gpu_unique_export_ties(real_gpu * h, const uint64_t * d_min_keys, uint8_t * d_ties)
{
        RG_API_BEGIN(h)
        if ( ! h->have_reads ) return fail(h, REAL_GPU_E_STATE, "no reads set");
        if ( ! d_min_keys || ! d_ties ) return fail(h, REAL_GPU_E_ARG, "null pointer");
        if ( h->nreads )
        {
                k_unique_ties<<<blocks_for(h->nreads, 256), 256, 0, h->st>>>(ptr<unsigned long long>(h->info), h->nreads, d_min_keys, d_ties);
                RG_KERNEL_CHECK(); launch_count(h);
        }
        RG_CUDA(cudaStreamSynchronize(h->st));
        return REAL_GPU_OK;
        RG_API_END(h)
}

int real_gpu_unique_import(real_gpu * h, const uint64_t * d_min_keys, const uint8_t * d_tie_sums)
{
        RG_API_BEGIN(h)
        if ( ! h->have_reads ) return fail(h, REAL_GPU_E_STATE, "no reads set");
        if ( ! d_min_keys || ! d_tie_sums ) return fail(h, REAL_GPU_E_ARG, "null pointer");
        if ( h->nreads )
        {
                k_unique_import<<<blocks_for(h->nreads, 256), 256, 0, h->st>>>(ptr<unsigned long long>(h->info), h->nreads, d_min_keys, d_tie_sums);
                RG_KERNEL_CHECK(); launch_count(h);
        }
        RG_CUDA(cudaStreamSynchronize(h->st));
        return REAL_GPU_OK;
        RG_API_END(h)
}

int real_gpu_match_gaps(real_gpu * h, uint64_t n_list_windows)
{
        RG_API_BEGIN(h)
        int const rc = check_ready(h);
        if ( rc ) return rc;
        if ( ! h->ll.p )
                return fail(h, REAL_GPU_E_ARG, "match_gaps needs the scoring table (real_gpu_params::ll_table)");
        if ( h->comm.nranks > 1 )
                return fail(h, REAL_GPU_E_ARG, "match_gaps is order dependent: not available with sharded tables");
        if ( h->shard_begin != 0 || h->shard_len != h->n_total || h->own_begin != 0 || h->own_end != h->n_total )
                return fail(h, REAL_GPU_E_ARG, "match_gaps needs the whole file in one shard (the fold is order dependent)");
        if ( h->nrec + 1 > 65536 )
                return REAL_GPU_OK;
        if ( n_list_windows ) h->n_list = n_list_windows;
        h->stats.scan_launches = 0;
        uint64_t const found = collect_hits_by_read(h, 2);
        if ( found )
        {
                dev_reserve(h, h->gapres, found * sizeof(GapRes) + 64);
                sort_large_segments(h, 2, nullptr, 1);          // long segments in replay order before their results are computed
                GapParams G;
                G.seg = ptr<RawHit>(h->hits_seg); G.ncand = found; G.ll = ptr<double>(h->ll);
                G.text = ptr<uint64_t>(h->text) + TEXT_PAD_WORDS; G.nmask = ptr<uint64_t>(h->nmask) + TEXT_PAD_WORDS; G.shard_begin = h->shard_begin;
                G.rec = ptr<uint64_t>(h->rec); G.nrec = h->nrec;
                G.rs = read_src(h); G.rlen = ptr<uint32_t>(h->rlen);
                G.quality = h->qual_present ? ptr<uint8_t>(h->qual) : nullptr; G.offsets = ptr<uint64_t>(h->offs);
                G.seedl = h->prm.seedl; G.scores = h->prm.scores;
                G.res = ptr<GapRes>(h->gapres);
                k_gap_dp<<<blocks_for(found, 128), 128, 0, h->st>>>(G);
                RG_KERNEL_CHECK(); launch_count(h);
                uint32_t const nb = block_bounds(h);
                GapReplayParams R;
                R.seg = ptr<RawHit>(h->hits_seg); R.res = ptr<GapRes>(h->gapres); R.starts = ptr<uint32_t>(h->starts); R.counts = ptr<uint32_t>(h->counts);
                R.nreads = h->nreads; R.scores = h->prm.scores;
                R.bounds = nb > 1 ? ptr<uint64_t>(h->bounds) : nullptr; R.nblocks = nb;
                R.info = ptr<unsigned long long>(h->info); R.score = ptr<float>(h->scores); R.gaps = ptr<real_gpu_gapinfo>(h->gaps);
                k_gap_replay<<<blocks_for(h->nreads, 128), 128, 0, h->st>>>(R);
                RG_KERNEL_CHECK(); launch_count(h);
        }
        RG_CUDA(cudaEventRecord(h->ev[1], h->st));
        RG_CUDA(cudaStreamSynchronize(h->st));
        h->stats.post_ms = elapsed(h->ev[0], h->ev[1]);
        return REAL_GPU_OK;
        RG_API_END(h)
}

int real_gpu_get_gaps(real_gpu * h, real_gpu_gapinfo * gaps)
{
        RG_API_BEGIN(h)
        if ( ! h->have_reads ) return fail(h, REAL_GPU_E_STATE, "no reads set");
        if ( ! gaps ) return fail(h, REAL_GPU_E_ARG, "get_gaps: null pointer");
        if ( h->nreads ) RG_CUDA(cudaMemcpy(gaps, h->gaps.p, h->nreads * sizeof(real_gpu_gapinfo), cudaMemcpyDeviceToHost));
        return REAL_GPU_OK;
        RG_API_END(h)
}


// ---- sharded tables ----------------------------------------------------------------------------

static int comm_finish_connect(real_gpu * h)
{
        real_gpu::Comm & CM = h->comm;
        uint32_t * fl[SC_MAX_RANKS];
        for ( int r = 0; r < SC_MAX_RANKS; ++r ) fl[r] = reinterpret_cast<uint32_t *>(CM.base[(uint32_t)r < CM.nranks ? r : 0]);
        RG_CUDA(cudaMemcpy(CM.ptrs.p, fl, sizeof(fl), cudaMemcpyHostToDevice));
        CM.connected = true;
        return REAL_GPU_OK;
}

int real_gpu_comm_init(real_gpu * h, uint32_t rank, uint32_t nranks, uint64_t round_positions, void * handle_out)
{
        RG_API_BEGIN(h)
        if ( nranks < 1 || nranks > (uint32_t)SC_MAX_RANKS || rank >= nranks ) return fail(h, REAL_GPU_E_ARG, "comm_init: rank/nranks out of range (at most 8 ranks)");
        real_gpu::Comm & CM = h->comm;
        if ( CM.window.p ) return fail(h, REAL_GPU_E_STATE, "comm_init: already initialised");
        drop_prepared(h);
        if ( round_positions == 0 ) round_positions = SC_MAX_ROUND;
        round_positions = std::min<uint64_t>(SC_MAX_ROUND, ((round_positions + SC_TILE_POS - 1) / SC_TILE_POS) * SC_TILE_POS);
        CM.nranks = nranks; CM.rank = rank; CM.epoch = 0; CM.round_positions = round_positions; CM.connected = false;
        for ( uint32_t r = 0; r <= nranks; ++r ) CM.bucket_lo[r] = (uint32_t)(((uint64_t)r * SC_MAX_BUCKETS) / nranks);
        uint64_t const per = (round_positions + nranks - 1) / nranks;
        CM.seg_cap = (uint32_t)(((per + SC_UNIT - 1) / SC_UNIT) * SC_UNIT + (uint64_t)SC_MAX_BUCKETS * SC_UNIT);
        CM.meta_off = 256;
        CM.recs_off = 16384;
        size_t const bytes = CM.recs_off + (size_t)nranks * CM.seg_cap * sizeof(uint4);
        dev_alloc(h, CM.window, bytes);
        dev_alloc(h, CM.ptrs, SC_MAX_RANKS * sizeof(void *));
        dev_alloc(h, CM.pairs, 2048 * 4);
        dev_alloc(h, CM.error, 16);
        dev_reserve(h, h->part_meta, (1100 + 256 * SC_CURSOR_STRIDE) * 4);
        dev_reserve(h, h->counters, 8 * 8);
        RG_CUDA(cudaMemset(CM.window.p, 0, CM.recs_off));
        RG_CUDA(cudaMemset(CM.error.p, 0, 16));
        for ( int i = 0; i < 2; ++i ) RG_CUDA(cudaEventCreateWithFlags(&CM.ev[i], cudaEventDisableTiming));
        RG_CUDA(cudaDeviceSynchronize());
        CM.base[rank] = reinterpret_cast<char *>(CM.window.p);
        h->have_reads = false;            // the index has to be (re)built for this rank's buckets
        if ( handle_out )
        {
                cudaIpcMemHandle_t ih;
                RG_CUDA(cudaIpcGetMemHandle(&ih, CM.window.p));
                static_assert(sizeof(ih) == REAL_GPU_COMM_HANDLE_BYTES, "cudaIpcMemHandle_t size");
                memcpy(handle_out, &ih, sizeof(ih));
        }
        if ( nranks == 1 ) return comm_finish_connect(h);
        return REAL_GPU_OK;
        RG_API_END(h)
}

int real_gpu_set_bucket_shard(real_gpu * h, uint32_t rank, uint32_t nranks)
{
        RG_API_BEGIN(h)
        if ( nranks < 1 || nranks > (uint32_t)SC_MAX_RANKS || rank >= nranks ) return fail(h, REAL_GPU_E_ARG, "set_bucket_shard: rank/nranks out of range (at most 8 ranks)");
        real_gpu::Comm & CM = h->comm;
        if ( CM.window.p ) return fail(h, REAL_GPU_E_STATE, "set_bucket_shard: the handle is already a rank of a peer-memory group (real_gpu_comm_init)");
        drop_prepared(h);
        CM.nranks = nranks; CM.rank = rank; CM.connected = false;
        for ( uint32_t r = 0; r <= nranks; ++r ) CM.bucket_lo[r] = (uint32_t)(((uint64_t)r * SC_MAX_BUCKETS) / nranks);
        h->have_reads = false;            // the index has to be (re)built for this rank's buckets
        return REAL_GPU_OK;
        RG_API_END(h)
}

int real_gpu_comm_connect(real_gpu * h, const void * all_handles)
{
        RG_API_BEGIN(h)
        real_gpu::Comm & CM = h->comm;
        if ( ! CM.window.p ) return fail(h, REAL_GPU_E_STATE, "comm_connect: call real_gpu_comm_init first");
        if ( ! all_handles ) return fail(h, REAL_GPU_E_ARG, "comm_connect: null pointer");
        for ( uint32_t r = 0; r < CM.nranks; ++r )
        {
                if ( r == CM.rank || CM.ipc_opened[r] ) continue;
                cudaIpcMemHandle_t ih;
                memcpy(&ih, static_cast<const char *>(all_handles) + (size_t)r * REAL_GPU_COMM_HANDLE_BYTES, sizeof(ih));
                void * p = nullptr;
                RG_CUDA(cudaIpcOpenMemHandle(&p, ih, cudaIpcMemLazyEnablePeerAccess));
                CM.base[r] = reinterpret_cast<char *>(p);
                CM.ipc_opened[r] = true;
        }
        return comm_finish_connect(h);
        RG_API_END(h)
}

int real_gpu_comm_connect_local(real_gpu * h, real_gpu * const * peers)
{
        RG_API_BEGIN(h)
        real_gpu::Comm & CM = h->comm;
        if ( ! CM.window.p ) return fail(h, REAL_GPU_E_STATE, "comm_connect_local: call real_gpu_comm_init first");
        if ( ! peers ) return fail(h, REAL_GPU_E_ARG, "comm_connect_local: null pointer");
        for ( uint32_t r = 0; r < CM.nranks; ++r )
        {
                real_gpu * q = peers[r];
                if ( ! q || ! q->comm.window.p || q->comm.nranks != CM.nranks || q->comm.rank != r || q->comm.seg_cap != CM.seg_cap )
                        return fail(h, REAL_GPU_E_ARG, "comm_connect_local: peer handle is not an initialised rank of the same group");
                if ( q->prm.device != h->prm.device )
                {
                        cudaError_t const e = cudaDeviceEnablePeerAccess(q->prm.device, 0);
                        if ( e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled ) RG_CUDA(e);
                        (void)cudaGetLastError();
                }
                CM.base[r] = reinterpret_cast<char *>(q->comm.window.p);
                CM.local[r] = q;
        }
        return comm_finish_connect(h);
        RG_API_END(h)
}

// ---- peer-memory fold ---------------------------------------------------------------------------

static int fold_finish_connect(real_gpu * h)
{
        real_gpu::Fold & FD = h->fold;
        uint32_t * fl[SC_MAX_RANKS];
        for ( int r = 0; r < SC_MAX_RANKS; ++r ) fl[r] = reinterpret_cast<uint32_t *>(FD.base[(uint32_t)r < FD.nranks ? r : 0]);
        RG_CUDA(cudaMemcpy(FD.ptrs.p, fl, sizeof(fl), cudaMemcpyHostToDevice));
        FD.connected = true;
        return REAL_GPU_OK;
}

static FoldPeers fold_peers(real_gpu::Fold const & FD, uint32_t parity)
{
        FoldPeers FP;
        for ( uint32_t r = 0; r < (uint32_t)SC_MAX_RANKS; ++r )
                FP.stage[r] = reinterpret_cast<unsigned long long *>(FD.base[r < FD.nranks ? r : 0] + FD.stage_off) + (uint64_t)parity * FD.nranks * FD.seg;
        return FP;
}

static void fold_push(real_gpu * h, uint32_t parity)
{
        real_gpu::Fold & FD = h->fold;
        uint64_t const per = (h->nreads + FD.nranks - 1) / FD.nranks;
        dim3 const grid((unsigned)std::max<uint64_t>(1, std::min<uint64_t>((per + 255) / 256, 4096)), FD.nranks);
        k_fold_push<<<grid, 256, 0, h->st>>>(ptr<unsigned long long>(h->info), h->nreads, FD.nranks, FD.rank, FD.seg, fold_peers(FD, parity));
        RG_KERNEL_CHECK(); launch_count(h);
}

static void fold_merge(real_gpu * h, uint32_t parity)
{
        real_gpu::Fold & FD = h->fold;
        uint64_t const b = (h->nreads * FD.rank) / FD.nranks, e = (h->nreads * (FD.rank + 1)) / FD.nranks;
        if ( e > b )
        {
                k_fold_merge<<<blocks_for(e - b, 256), 256, 0, h->st>>>(fold_peers(FD, parity).stage[FD.rank], FD.nranks, FD.seg, e - b, ptr<unsigned long long>(h->info) + b);
                RG_KERNEL_CHECK(); launch_count(h);
        }
}

static int fold_check(real_gpu * h)
{
        real_gpu::Fold & FD = h->fold;
        if ( ! FD.window.p || ! FD.connected ) return fail(h, REAL_GPU_E_STATE, "fold_unique: call real_gpu_fold_init and real_gpu_fold_connect* first");
        if ( ! h->have_reads ) return fail(h, REAL_GPU_E_STATE, "no reads set");
        if ( h->prm.scores ) return fail(h, REAL_GPU_E_ARG, "fold_unique: the fold with scores is order dependent (needs one handle)");
        if ( h->nreads > FD.cap ) return fail(h, REAL_GPU_E_LIMIT, "fold_unique: more reads than real_gpu_fold_init was sized for");
        return REAL_GPU_OK;
}

int real_gpu_fold_init(real_gpu * h, uint32_t rank, uint32_t nranks, uint64_t max_reads, void * handle_out)
{
        RG_API_BEGIN(h)
        if ( nranks < 1 || nranks > (uint32_t)SC_MAX_RANKS || rank >= nranks ) return fail(h, REAL_GPU_E_ARG, "fold_init: rank/nranks out of range (at most 8 ranks)");
        real_gpu::Fold & FD = h->fold;
        if ( FD.window.p ) return fail(h, REAL_GPU_E_STATE, "fold_init: already initialised");
        FD.nranks = nranks; FD.rank = rank; FD.epoch = 0; FD.cap = max_reads; FD.connected = false;
        FD.seg = (((max_reads + nranks - 1) / nranks) + 1) & ~1ULL;
        size_t const bytes = FD.stage_off + (size_t)2 * nranks * FD.seg * 8 + 64;
        dev_alloc(h, FD.window, bytes);
        dev_alloc(h, FD.ptrs, SC_MAX_RANKS * sizeof(void *));
        dev_alloc(h, FD.error, 16);
        RG_CUDA(cudaMemset(FD.window.p, 0, FD.stage_off));
        RG_CUDA(cudaMemset(FD.error.p, 0, 16));
        RG_CUDA(cudaEventCreateWithFlags(&FD.ev, cudaEventDisableTiming));
        RG_CUDA(cudaDeviceSynchronize());
        FD.base[rank] = reinterpret_cast<char *>(FD.window.p);
        if ( handle_out )
        {
                cudaIpcMemHandle_t ih;
                RG_CUDA(cudaIpcGetMemHandle(&ih, FD.window.p));
                memcpy(handle_out, &ih, sizeof(ih));
        }
        if ( nranks == 1 ) return fold_finish_connect(h);
        return REAL_GPU_OK;
        RG_API_END(h)
}

int real_gpu_fold_connect(real_gpu * h, const void * all_handles)
{
        RG_API_BEGIN(h)
        real_gpu::Fold & FD = h->fold;
        if ( ! FD.window.p ) return fail(h, REAL_GPU_E_STATE, "fold_connect: call real_gpu_fold_init first");
        if ( ! all_handles ) return fail(h, REAL_GPU_E_ARG, "fold_connect: null pointer");
        for ( uint32_t r = 0; r < FD.nranks; ++r )
        {
                if ( r == FD.rank || FD.ipc_opened[r] ) continue;
                cudaIpcMemHandle_t ih;
                memcpy(&ih, static_cast<const char *>(all_handles) + (size_t)r * REAL_GPU_COMM_HANDLE_BYTES, sizeof(ih));
                void * p = nullptr;
                RG_CUDA(cudaIpcOpenMemHandle(&p, ih, cudaIpcMemLazyEnablePeerAccess));
                FD.base[r] = reinterpret_cast<char *>(p);
                FD.ipc_opened[r] = true;
        }
        return fold_finish_connect(h);
        RG_API_END(h)
}

int real_gpu_fold_connect_local(real_gpu * h, real_gpu * const * peers)
{
        RG_API_BEGIN(h)
        real_gpu::Fold & FD = h->fold;
        if ( ! FD.window.p ) return fail(h, REAL_GPU_E_STATE, "fold_connect_local: call real_gpu_fold_init first");
        if ( ! peers ) return fail(h, REAL_GPU_E_ARG, "fold_connect_local: null pointer");
        for ( uint32_t r = 0; r < FD.nranks; ++r )
        {
                real_gpu * q = peers[r];
                if ( ! q || ! q->fold.window.p || q->fold.nranks != FD.nranks || q->fold.rank != r || q->fold.seg != FD.seg )
                        return fail(h, REAL_GPU_E_ARG, "fold_connect_local: peer handle is not an initialised rank of the same group");
                if ( q->prm.device != h->prm.device )
                {
                        cudaError_t const e = cudaDeviceEnablePeerAccess(q->prm.device, 0);
                        if ( e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled ) RG_CUDA(e);
                        (void)cudaGetLastError();
                }
                FD.base[r] = reinterpret_cast<char *>(q->fold.window.p);
                FD.local[r] = q;
        }
        return fold_finish_connect(h);
        RG_API_END(h)
}

int real_gpu_fold_unique(real_gpu * h)
{
        RG_API_BEGIN(h)
        int const rc = fold_check(h);
        if ( rc ) return rc;
        real_gpu::Fold & FD = h->fold;
        if ( FD.local[FD.rank] ) return fail(h, REAL_GPU_E_STATE, "fold_unique: ranks of one process fold with real_gpu_fold_unique_group");
        long long wait_ms = 30000;
        if ( const char * e = getenv("REAL_GPU_COMM_TIMEOUT_MS") ) wait_ms = atoll(e);
        ++FD.epoch;
        uint32_t const parity = FD.epoch & 1;
        // Two staging areas, used alternately: a peer can be at most one exchange ahead of this rank (its next exchange waits
        // for this rank's signal, which is issued behind this rank's merge), so nobody writes into an area that is still read.
        RG_CUDA(cudaEventRecord(h->ev[0], h->st));
        fold_push(h, parity);
        k_comm_signal<<<1, 32, 0, h->st>>>(ptr<uint32_t *>(FD.ptrs), FD.nranks, FD.rank, 0, FD.epoch);
        RG_KERNEL_CHECK();
        k_comm_wait<<<1, 32, 0, h->st>>>(reinterpret_cast<uint32_t *>(FD.base[FD.rank]), FD.nranks, 0, FD.epoch, wait_ms * 2000000LL, ptr<uint32_t>(FD.error));
        RG_KERNEL_CHECK(); launch_count(h, 2);
        fold_merge(h, parity);
        RG_CUDA(cudaEventRecord(h->ev[1], h->st));
        uint32_t cerr = 0;
        RG_CUDA(cudaMemcpyAsync(&cerr, FD.error.p, 4, cudaMemcpyDeviceToHost, h->st));
        RG_CUDA(cudaStreamSynchronize(h->st));
        h->stats.fold_ms = elapsed(h->ev[0], h->ev[1]);
        if ( cerr ) return fail(h, REAL_GPU_E_CUDA, "fold_unique: timed out waiting for rank " + std::to_string(cerr - 1));
        return REAL_GPU_OK;
        RG_API_END(h)
}

int real_gpu_fold_unique_group(real_gpu * const * handles, uint32_t n)
{
        if ( ! handles || n == 0 || n > (uint32_t)SC_MAX_RANKS ) return REAL_GPU_E_ARG;
        for ( uint32_t r = 0; r < n; ++r )
                if ( ! handles[r] ) return REAL_GPU_E_ARG;
        real_gpu * h = handles[0];
        try
        {
                for ( uint32_t r = 0; r < n; ++r )
                {
                        h = handles[r];
                        RG_CUDA(cudaSetDevice(h->prm.device));
                        finish_build(h);
                        int const rc = fold_check(h);
                        if ( rc ) return rc;
                        if ( h->fold.nranks != n || h->fold.rank != r || ! h->fold.local[r] )
                                return fail(h, REAL_GPU_E_ARG, "fold_unique_group: handles[r] must be rank r of a group connected with real_gpu_fold_connect_local");
                        if ( h->nreads != handles[0]->nreads ) return fail(h, REAL_GPU_E_ARG, "fold_unique_group: the ranks hold different read sets");
                }
                // everybody pushes, then everybody merges what it was sent: the streams wait for each other through events
                for ( uint32_t r = 0; r < n; ++r )
                {
                        h = handles[r];
                        RG_CUDA(cudaSetDevice(h->prm.device));
                        RG_CUDA(cudaEventRecord(h->ev[0], h->st));
                        fold_push(h, 0);
                        RG_CUDA(cudaEventRecord(h->fold.ev, h->st));
                }
                for ( uint32_t r = 0; r < n; ++r )
                {
                        h = handles[r];
                        RG_CUDA(cudaSetDevice(h->prm.device));
                        for ( uint32_t q = 0; q < n; ++q )
                                if ( q != r ) RG_CUDA(cudaStreamWaitEvent(h->st, handles[q]->fold.ev, 0));
                        fold_merge(h, 0);
                        RG_CUDA(cudaEventRecord(h->ev[1], h->st));
                }
                for ( uint32_t r = 0; r < n; ++r )
                {
                        h = handles[r];
                        RG_CUDA(cudaSetDevice(h->prm.device));
                        RG_CUDA(cudaStreamSynchronize(h->st));
                        h->stats.fold_ms = elapsed(h->ev[0], h->ev[1]);
                }
        }
        catch ( std::exception const & e ) { return fail(h, REAL_GPU_E_CUDA, e.what()); }
        return REAL_GPU_OK;
}


// ---- output lines formatted on the device (csrc/format.cuh) -----------------------------------------

int real_gpu_set_read_ids(real_gpu * h, uint64_t first, uint64_t count, const char * bytes, const uint64_t * offsets)
{
        RG_API_BEGIN(h)
        if ( ! offsets || (count && ! bytes && offsets[count] != offsets[0]) ) return fail(h, REAL_GPU_E_ARG, "set_read_ids: null pointer");
        for ( uint64_t i = 0; i < count; ++i )
                if ( offsets[i+1] < offsets[i] ) return fail(h, REAL_GPU_E_ARG, "set_read_ids: offsets not ascending");
        uint64_t const nbytes = offsets[count] - offsets[0];
        dev_reserve(h, h->fmt.ids, nbytes + 16);
        dev_reserve(h, h->fmt.id_off, (count + 1) * 8);
        if ( nbytes ) RG_CUDA(cudaMemcpyAsync(h->fmt.ids.p, bytes + offsets[0], nbytes, cudaMemcpyHostToDevice, h->st));
        std::vector<uint64_t> rel;
        const uint64_t * src = offsets;
        if ( offsets[0] != 0 )
        {
                rel.resize(count + 1);
                for ( uint64_t i = 0; i <= count; ++i ) rel[i] = offsets[i] - offsets[0];
                src = rel.data();
        }
        RG_CUDA(cudaMemcpyAsync(h->fmt.id_off.p, src, (count + 1) * 8, cudaMemcpyHostToDevice, h->st));
        RG_CUDA(cudaStreamSynchronize(h->st));
        h->fmt.id_first = first; h->fmt.id_count = count; h->fmt.id_bytes = nbytes;
        return REAL_GPU_OK;
        RG_API_END(h)
}

int real_gpu_set_record_names(real_gpu * h, uint32_t fileid, uint32_t nrecords, const char * bytes, const uint64_t * offsets, const uint64_t * record_starts)
{
        RG_API_BEGIN(h)
        if ( fileid >= 64 ) return fail(h, REAL_GPU_E_LIMIT, "set_record_names: fileid >= 64");
        if ( ! offsets || ! record_starts || (nrecords && ! bytes && offsets[nrecords] != offsets[0]) ) return fail(h, REAL_GPU_E_ARG, "set_record_names: null pointer");
        for ( uint32_t i = 0; i < nrecords; ++i )
                if ( offsets[i+1] < offsets[i] ) return fail(h, REAL_GPU_E_ARG, "set_record_names: offsets not ascending");
        real_gpu::Format & F = h->fmt;
        F.file_names[fileid].assign(bytes + offsets[0], bytes + offsets[nrecords]);
        F.file_name_off[fileid].resize(nrecords + 1);
        for ( uint32_t i = 0; i <= nrecords; ++i ) F.file_name_off[fileid][i] = offsets[i] - offsets[0];
        F.file_starts[fileid].assign(record_starts, record_starts + nrecords);
        for ( uint32_t i = 0; i < nrecords; ++i ) F.max_name = std::max<uint64_t>(F.max_name, offsets[i+1] - offsets[i]);
        F.tables_dirty = true;
        return REAL_GPU_OK;
        RG_API_END(h)
}

} // extern "C"

namespace
{

// the record tables of all files on the device: names, name offsets and record starts by global record index
void format_upload_tables(real_gpu * h)
{
        real_gpu::Format & F = h->fmt;
        if ( ! F.tables_dirty ) return;
        std::vector<uint32_t> first(65, 0);
        std::vector<char> names; std::vector<uint64_t> noff, starts;
        for ( int f = 0; f < 64; ++f )
        {
                first[f] = (uint32_t)starts.size();
                for ( size_t r = 0; r < F.file_starts[f].size(); ++r )
                {
                        noff.push_back(names.size() + F.file_name_off[f][r]);
                        starts.push_back(F.file_starts[f][r]);
                }
                names.insert(names.end(), F.file_names[f].begin(), F.file_names[f].end());
        }
        first[64] = (uint32_t)starts.size();
        noff.push_back(names.size());
        starts.push_back(0);
        // (noff[r+1] is the end of record r's name: the names of a file are back to back and the files follow each other)
        dev_reserve(h, F.names, names.size() + 16);
        dev_reserve(h, F.name_off, noff.size() * 8);
        dev_reserve(h, F.rec_start, starts.size() * 8);
        dev_reserve(h, F.file_first, 65 * 4);
        if ( ! names.empty() ) RG_CUDA(cudaMemcpyAsync(F.names.p, names.data(), names.size(), cudaMemcpyHostToDevice, h->st));
        RG_CUDA(cudaMemcpyAsync(F.name_off.p, noff.data(), noff.size() * 8, cudaMemcpyHostToDevice, h->st));
        RG_CUDA(cudaMemcpyAsync(F.rec_start.p, starts.data(), starts.size() * 8, cudaMemcpyHostToDevice, h->st));
        RG_CUDA(cudaMemcpyAsync(F.file_first.p, first.data(), 65 * 4, cudaMemcpyHostToDevice, h->st));
        RG_CUDA(cudaStreamSynchronize(h->st));      // the staging vectors go out of scope
        F.tables_dirty = false;
}

template<bool ALL>
int format_items(real_gpu * h, uint64_t first, uint64_t count, const char ** bytes, uint64_t * nbytes, uint64_t * nlines)
{
        real_gpu::Format & F = h->fmt;
        *bytes = nullptr; *nbytes = 0;
        if ( nlines ) *nlines = 0;
        if ( ! count ) return REAL_GPU_OK;
        format_upload_tables(h);
        FormatParams P;
        memset(&P, 0, sizeof(P));
        P.rs = read_src(h); P.rlen = ptr<uint32_t>(h->rlen);
        P.ids = ptr<char>(F.ids); P.id_off = ptr<uint64_t>(F.id_off); P.id_first = F.id_first;
        P.file_first = ptr<uint32_t>(F.file_first); P.names = ptr<char>(F.names); P.name_off = ptr<uint64_t>(F.name_off); P.rec_start = ptr<uint64_t>(F.rec_start);
        P.scores = h->prm.scores;
        P.info = ptr<unsigned long long>(h->info); P.score = ptr<float>(h->scores); P.hits = ptr<real_gpu_hit>(h->hits_out);
        P.first = first; P.count = count;
        dev_reserve(h, F.len, (count + 2) * 4);
        dev_reserve(h, F.off, (count + 2) * 4);
        dev_reserve(h, h->scantmp, scan_temp_elems(count) * 4 + 64);
        P.len = ptr<uint32_t>(F.len); P.off = ptr<uint32_t>(F.off);
        dev_reserve(h, h->counters, 8 * 8);
        RG_CUDA(cudaMemsetAsync(h->counters.p, 0, 8, h->st));
        P.nlines = ptr<unsigned long long>(h->counters);
        // the byte offsets of a batch are 32 bit: a bound on its bytes (ids of the whole set + the longest possible rest per item)
        if ( F.id_bytes + count * ((uint64_t)h->maxlen + F.max_name + 96) >= (1ULL << 32) )
                throw LimitError("format: this many items may take more than 4 GiB of output; format fewer per call");
        RG_CUDA(cudaEventRecord(h->ev[0], h->st));
        k_fmt_len<ALL><<<blocks_for(count, 256), 256, 0, h->st>>>(P);
        RG_KERNEL_CHECK(); launch_count(h);
        uint32_t nl = 0;
        exclusive_scan_u32(P.len, ptr<uint32_t>(F.off), count, ptr<uint32_t>(h->scantmp), h->st, &nl);
        launch_count(h, nl);
        uint32_t last[2] = {0, 0};
        unsigned long long nl_host = 0;
        RG_CUDA(cudaMemcpyAsync(&nl_host, P.nlines, 8, cudaMemcpyDeviceToHost, h->st));
        RG_CUDA(cudaMemcpyAsync(&last[0], ptr<uint32_t>(F.off) + (count - 1), 4, cudaMemcpyDeviceToHost, h->st));
        RG_CUDA(cudaMemcpyAsync(&last[1], ptr<uint32_t>(F.len) + (count - 1), 4, cudaMemcpyDeviceToHost, h->st));
        RG_CUDA(cudaStreamSynchronize(h->st));
        uint64_t const total = (uint64_t)last[0] + last[1];
        if ( ! total ) { if ( nlines ) *nlines = 0; return REAL_GPU_OK; }
        dev_reserve(h, F.out, total + 16);
        P.out = ptr<char>(F.out);
        k_fmt_write<ALL><<<(unsigned)std::min<uint64_t>((count + FMT_WARPS - 1) / FMT_WARPS, (uint64_t)h->sm_count * 16), FMT_WARPS * 32, 0, h->st>>>(P);
        RG_KERNEL_CHECK(); launch_count(h);
        RG_CUDA(cudaEventRecord(h->ev[1], h->st));
        int const b = F.flip; F.flip ^= 1;
        if ( F.host_cap[b] < total )
        {
                if ( F.host[b] ) cudaFreeHost(F.host[b]);
                F.host[b] = nullptr; F.host_cap[b] = 0;
                size_t const cap = total + total / 8 + 4096;
                RG_CUDA(cudaMallocHost(&F.host[b], cap));
                F.host_cap[b] = cap;
        }
        RG_CUDA(cudaMemcpyAsync(F.host[b], F.out.p, total, cudaMemcpyDeviceToHost, h->st));
        RG_CUDA(cudaEventRecord(h->ev[2], h->st));
        RG_CUDA(cudaStreamSynchronize(h->st));
        h->stats.post_ms = elapsed(h->ev[0], h->ev[1]);
        h->stats.d2h_ms = elapsed(h->ev[1], h->ev[2]);
        *bytes = F.host[b]; *nbytes = total;
        if ( nlines ) *nlines = nl_host;
        return REAL_GPU_OK;
}

} // namespace

extern "C" {

int real_gpu_format_unique(real_gpu * h, uint64_t first, uint64_t count, const char ** bytes, uint64_t * nbytes, uint64_t * nlines)
{
        RG_API_BEGIN(h)
        if ( ! bytes || ! nbytes ) return fail(h, REAL_GPU_E_ARG, "format_unique: null pointer");
        if ( ! h->have_reads ) return fail(h, REAL_GPU_E_STATE, "no reads set");
        if ( first > h->nreads || count > h->nreads - first ) return fail(h, REAL_GPU_E_ARG, "format_unique: range outside the read set");
        if ( first < h->fmt.id_first || first + count > h->fmt.id_first + h->fmt.id_count )
                return fail(h, REAL_GPU_E_STATE, "format_unique: the ids of these reads have not been set (real_gpu_set_read_ids)");
        if ( count >= (1ULL << 26) ) return fail(h, REAL_GPU_E_LIMIT, "format_unique: more than 2^26 reads in one call");
        return format_items<false>(h, first, count, bytes, nbytes, nlines);
        RG_API_END(h)
}

int real_gpu_format_all(real_gpu * h, uint64_t first_row, uint64_t count, const char ** bytes, uint64_t * nbytes)
{
        RG_API_BEGIN(h)
        if ( ! bytes || ! nbytes ) return fail(h, REAL_GPU_E_ARG, "format_all: null pointer");
        if ( ! h->have_reads ) return fail(h, REAL_GPU_E_STATE, "no reads set");
        if ( first_row > h->fmt.nrows_all || count > h->fmt.nrows_all - first_row ) return fail(h, REAL_GPU_E_ARG, "format_all: range outside the rows of the last real_gpu_match_all");
        if ( h->fmt.id_first != 0 || h->fmt.id_count < h->nreads )
                return fail(h, REAL_GPU_E_STATE, "format_all: the ids of all reads must be set (real_gpu_set_read_ids)");
        if ( count >= (1ULL << 26) ) return fail(h, REAL_GPU_E_LIMIT, "format_all: more than 2^26 rows in one call");
        return format_items<true>(h, first_row, count, bytes, nbytes, nullptr);
        RG_API_END(h)
}

int real_gpu_selftest_format_scores(int device, const float * values, uint64_t n, char * out16)
{
        try
        {
                RG_CUDA(cudaSetDevice(device));
                float * dv = nullptr; char * dout = nullptr;
                RG_CUDA(cudaMalloc(&dv, n * 4 + 16));
                RG_CUDA(cudaMalloc(&dout, n * 16 + 16));
                RG_CUDA(cudaMemcpy(dv, values, n * 4, cudaMemcpyHostToDevice));
                if ( n ) k_fmt_selftest<<<blocks_for(n, 256), 256>>>(dv, n, dout);
                cudaError_t const e = cudaDeviceSynchronize();
                if ( e == cudaSuccess ) cudaMemcpy(out16, dout, n * 16, cudaMemcpyDeviceToHost);
                cudaFree(dv); cudaFree(dout);
                return e == cudaSuccess ? REAL_GPU_OK : REAL_GPU_E_CUDA;
        }
        catch ( ... ) { return REAL_GPU_E_CUDA; }
}

int real_gpu_get_stats(real_gpu * h, real_gpu_stats * out)
{
        if ( ! out ) return REAL_GPU_E_ARG;
        RG_API_BEGIN(h)
        *out = h->stats;
        return REAL_GPU_OK;
        RG_API_END(h)
}

void * real_gpu_stream(real_gpu * h) { return h ? (void *)h->st : nullptr; }
uint64_t real_gpu_device_bytes(const real_gpu * h) { return h ? h->held : 0; }

int real_gpu_synth_text(int device, uint64_t seed, uint64_t first_word, uint64_t nwords, uint32_t n_per_million,
                        uint64_t * d_words, uint64_t * d_nmask_or_null)
{
        try
        {
                RG_CUDA(cudaSetDevice(device));
                if ( nwords )
                {
                        k_synth_text<<<blocks_for(nwords, 256), 256>>>(seed, first_word, nwords, d_nmask_or_null ? n_per_million : 0, d_words);
                        RG_KERNEL_CHECK();
                        if ( d_nmask_or_null )
                        {
                                if ( first_word & 1 ) return REAL_GPU_E_ARG;
                                uint64_t const nm = (nwords + 1) / 2;
                                k_synth_nmask<<<blocks_for(nm, 256), 256>>>(seed, first_word >> 1, nm, n_per_million, d_nmask_or_null);
                                RG_KERNEL_CHECK();
                        }
                }
                RG_CUDA(cudaDeviceSynchronize());
        }
        catch ( std::exception const & e ) { fprintf(stderr, "real_gpu_synth_text: %s\n", e.what()); return REAL_GPU_E_CUDA; }
        return REAL_GPU_OK;
}

int real_gpu_synth_reads(int device, uint64_t seed, const uint64_t * d_words, const uint64_t * d_nmask_or_null, uint64_t text_n,
                         uint64_t total_reads, uint64_t first_read, uint64_t nreads, uint32_t length, uint32_t sub_per_16384,
                         uint8_t * d_mapped, uint8_t * d_quality_or_null)
{
        try
        {
                RG_CUDA(cudaSetDevice(device));
                if ( length == 0 || length > 256 || text_n < length || total_reads == 0 ) return REAL_GPU_E_ARG;
                if ( nreads )
                {
                        k_synth_reads<<<blocks_for(nreads, 128), 128>>>(seed, d_words, d_nmask_or_null, text_n, total_reads, first_read, nreads, length,
                                                                       sub_per_16384, d_mapped, d_quality_or_null);
                        RG_KERNEL_CHECK();
                }
                RG_CUDA(cudaDeviceSynchronize());
        }
        catch ( std::exception const & e ) { fprintf(stderr, "real_gpu_synth_reads: %s\n", e.what()); return REAL_GPU_E_CUDA; }
        return REAL_GPU_OK;
}

} // extern "C"
