// K3: the text scan -- partition + probe + verify + report, the dominant kernels of the path.
//
// Replaces, for every seed window of the text and every read at once, the reference's per-read
// ::match (match.hpp:335-416): directory lookup + equal_range on the signature, seed error count
// against the complementary signature (:386-388), position / record / wildcard predicates
// (:391-398, RangeVector.hpp:59-66, AutoTextArray.hpp:167-172), rest-of-read Hamming distance
// (RestMatch.hpp:39-81) and the updater call (:410).
//
// Measured on B200 (tools/gather_bench.cu): random 32-byte sector reads run at ~40 G/s out of HBM
// (every one drags a 128-byte line: ~5 TB/s of DRAM traffic for 1.3 TB/s of useful sectors) but at
// ~290 G/s out of L2.  Three random table probes per text position straight into multi-GB tables
// therefore top out near 13 G positions/s.  So the scan first PARTITIONS the window starts of a text
// chunk by the first bases of their window -- all three table keys of a position begin with
// fragment 0, so that prefix is the top bits of every key -- and then probes bucket after bucket:
// while a bucket is being probed only 1/2^bucket_bits of each table is touched, a slice that stays
// in L2.
//
//   k_part_hist     TMA-staged text tiles -> bucket histogram
//   k_part_offsets  bucket starts (padded to whole work units) + sentinel records in the padding
//   k_part_scatter  TMA-staged text tiles -> 16-byte records {window word, the 16 bases in front of it,
//                   position} grouped by bucket (staged in shared memory, written run by run)
//   k_own_list      bucket shards (multi-GPU): the positions whose bucket this rank owns, as a dense list + their
//                   bucket histogram in one pass; k_part_scatter_list then forms the records of the list
//   k_bucket_probe  warps pull 512-record grabs in bucket order and walk them 64 records at a time:
//                   6 independent 4-byte probes per lane; set slot bits are compacted
//                   into the warp's shared-memory queue (stage A: rank -> entry chain -> seed test ->
//                   canonical-list rule), the survivors into a second queue (stage B: record / wildcard
//                   predicates, whole-read XOR+popcount distance, report), so that each stage runs with
//                   full warps and no block-wide barrier sits between them.
#pragma once

#include "common.cuh"
#include "index.cuh"

namespace realgpu
{

static const int SC_THREADS = 256;
static const int SC_WPT = 2;                                 // text words per thread and tile
static const int SC_TILE_WORDS = SC_THREADS * SC_WPT;
static const int SC_TILE_POS = SC_TILE_WORDS * 32;           // 16384 window starts per tile
static const int SC_HALO = 2;                                // words of halo in front and behind
static const int SC_SMEM_WORDS = SC_TILE_WORDS + 2 * SC_HALO; // 516 words = 4128 bytes (multiple of 16)
static const int SC_MAX_BUCKETS = 256;
static const int SC_CURSOR_STRIDE = 32;                      // u32 per bucket cursor: one 128-byte line each, so the global atomics spread over the L2 slices
static const int SC_UNIT = 512;                              // records per grab of the probe kernel (one global atomic per warp and grab)
static const int SC_RPT = 2;                                 // records per lane and step
static const int SC_PROBE_MINB = 3;                          // CTAs per SM of k_bucket_probe (register bound and launch cap, plan_scan)
static const int SC_QA_CAP = 32 + 96 * SC_RPT;               // per-warp stage A queue (set slot bits): drained from 32 up, a step adds <= 96 per record and lane
static const int SC_QB_CAP = 64;                             // per-warp stage B queue (seed test passed)
static const uint32_t SC_POS_NONE = 0xFFFFFFFFu;             // position word of a padding record
static const uint64_t SC_MAX_CHUNK = 0xFFF00000ull;         // positions per chunk: a record holds its position relative to the chunk in 32 bits (all ones = padding)
static const uint64_t SC_MAX_ROUND = 1ull << 30;             // sharded tables: positions per round (sizes the record areas of the windows)

static const int SC_MAX_RANKS = 8;                           // GPUs of one NVSwitch box that can share a scan (sharded tables)
static const int SC_META_STRIDE = SC_MAX_BUCKETS + 8;        // u32 per source in a rank's bucket-count area

struct TableDev
{
        const SlotWord * slots;
        const Entry * E;
        uint32_t hb;
        uint32_t nlists;
};

struct ScanParams
{
        const uint64_t * text;        // local word 0; valid from -TEXT_PAD_WORDS
        const uint64_t * nmask;       // local mask word 0
        uint64_t shard_begin;         // global position of local base 0
        uint64_t x_begin, x_end;      // local text positions whose keys are probed (by this rank, this round)
        uint64_t pos_base;            // local text position the record positions are relative to (first position of the round)
        uint64_t win_begin, win_end;  // local seed-window starts this shard evaluates
        uint64_t own_begin, own_end;  // GLOBAL hit start positions this shard reports
        TableDev tab[3];
        uint32_t seedl, F, keybits, seedkmax, totalkmax;        // seedl = the indexed seed bases (<= 32)
        uint32_t vseedl;              // seed length of the options; > seedl: the rest of the seed is tested at verification
        ReadSrc rs;                   // the bases of the reads: packed strands, or the caller's 2 bit/base input
        const uint32_t * rlen;
        const uint64_t * rec;         // nrec+1 global record starts
        uint32_t nrec;
        uint32_t fileid;
        // partition of the chunk [x_begin, x_end): x0 = first position of the chunk
        uint32_t bucket_bits;
        uint32_t entries_evict_normal;  // 1: the probe loads entries with evict_normal (a single chunk), else evict_first
        uint4 * recs;                 // records grouped by bucket: {window lo, window hi, 16 bases in front of it, position - pos_base}
        uint32_t * bucket_count;      // [SC_MAX_BUCKETS]
        uint32_t * bucket_start;      // [SC_MAX_BUCKETS+1] record index
        uint32_t * bucket_cursor;     // [SC_MAX_BUCKETS]
        uint32_t * unit_counter;      // work distribution of k_bucket_probe
        int mode;                     // 0 = report all hits, 1 = fold into the unique state, 2 = seed candidates of the gapped pass
        RawHit * hits;
        unsigned long long hit_cap;
        unsigned long long * hit_count;
        unsigned long long * info;
        unsigned long long * stats;   // [0] candidates  [1] seed-pass  [2] hits
        // Sharded tables (nranks > 1, one rank per GPU): rank r holds the tables of the buckets [bucket_lo[r], bucket_lo[r+1])
        // only.  Every rank partitions its slice of the round's positions and writes the records of a bucket straight
        // into the record area of the bucket's owner (peer memory over NVLink); the owner probes what arrived.
        uint32_t nranks, rank;
        uint32_t bucket_lo[SC_MAX_RANKS + 1];
        uint4 * peer_recs[SC_MAX_RANKS];        // record area of every rank (own included); source s writes from record s * seg_cap
        uint32_t * peer_meta[SC_MAX_RANKS];     // bucket-count area of every rank: [source][SC_META_STRIDE] padded record counts
        uint32_t seg_cap;                       // records a source may deliver to one rank in a round
        uint32_t * pair_grab;                   // probe side: first grab of every (own bucket, source) pair, bucket-major, + total
        uint32_t * pair_rec;                    //             first record of the pair in the local record area
        uint32_t npairs;
        // Bucket shards (real_gpu_set_bucket_shard): this handle indexes and probes the buckets [own_b_lo, own_b_lo + own_b_cnt)
        // only; it reads every text position of the chunk but forms records only of the positions whose bucket it owns.
        // own_b_cnt = SC_MAX_BUCKETS: no filter.
        uint32_t own_b_lo, own_b_cnt;
        uint32_t * list;              // bucket shard: positions (relative to pos_base) of the chunk this handle keeps
        unsigned long long * list_count;
        unsigned long long * nprobed; // positions this handle has formed records of (statistics)
};

__device__ __forceinline__ uint32_t bucket_owner(ScanParams const & P, uint32_t b)
{
        uint32_t r = 0;
        #pragma unroll
        for ( int i = 1; i < SC_MAX_RANKS; ++i )
                if ( (uint32_t)i < P.nranks && b >= P.bucket_lo[i] ) r = i;
        return r;
}

__device__ __forceinline__ uint32_t smem_u32(const void * p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t * bar, uint32_t count)
{
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t * bar, uint32_t bytes)
{
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t * bar, uint32_t parity)
{
        uint32_t done = 0;
        while ( ! done )
        {
                asm volatile(
                        "{\n\t"
                        ".reg .pred p;\n\t"
                        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                        "selp.u32 %0, 1, 0, p;\n\t"
                        "}" : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
        }
}
// 1-D bulk asynchronous copy global -> shared, completion signalled on the mbarrier (TMA unit)
__device__ __forceinline__ void bulk_load(void * dst, const void * src, uint32_t bytes, uint64_t * bar)
{
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     :: "r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// ---- reporting -------------------------------------------------------------------------------

// UpdateUniqueInfo<false>::update (matchUniqueImplementation.cpp:97-159) as an order-independent
// compare-and-swap: lowest error count wins, a second distinct position at that count makes the
// read NonUnique, '+' wins when both strands hit the same position (the reference probes the
// straight lists first).  The position kept in a NonUnique word is the smallest one seen, which
// makes the word deterministic (the reference keeps whichever came first).
__device__ __forceinline__ void unique_update(unsigned long long * slot, uint32_t inverted, uint32_t file, uint64_t pos, uint32_t k, uint32_t frag)
{
        unsigned long long old = *slot;
        while ( true )
        {
                uint32_t const st = umi_state(old);
                unsigned long long const take = umi_make(inverted ? ST_REVERSE : ST_STRAIGHT, file, pos, k, frag);
                unsigned long long neu = old;
                if ( st == ST_NOMATCH || st == ST_GAPPED )
                        neu = take;
                else if ( k < umi_err(old) )
                        neu = take;
                else if ( k == umi_err(old) )
                {
                        bool const same = (pos == umi_pos(old)) && (file == umi_file(old)) && (frag == umi_frag(old));
                        if ( st == ST_NONUNIQUE )
                        {
                                if ( file < umi_file(old) || (file == umi_file(old) && pos < umi_pos(old)) )
                                        neu = umi_with_state(take, ST_NONUNIQUE);
                        }
                        else if ( ! same )
                        {
                                bool const smaller = file < umi_file(old) || (file == umi_file(old) && pos < umi_pos(old));
                                neu = umi_with_state(smaller ? take : old, ST_NONUNIQUE);
                        }
                        else if ( ! inverted && st == ST_REVERSE )
                                neu = take;
                }
                if ( neu == old )
                        return;
                unsigned long long const prev = atomicCAS(slot, old, neu);
                if ( prev == old )
                        return;
                old = prev;
        }
}

// RangeVector::positionToRange (RangeVector.hpp:59-62): last record start <= pos
__device__ __forceinline__ uint32_t record_of(const uint64_t * __restrict__ rec, uint32_t nrec, uint64_t pos)
{
        uint32_t lo = 0, hi = nrec + 1;
        while ( lo < hi )
        {
                uint32_t const mid = (lo + hi) >> 1;
                if ( __ldg(rec + mid) <= pos ) lo = mid + 1; else hi = mid;
        }
        return lo - 1;
}

// AutoTextArray::isDontCareFree (AutoTextArray.hpp:167-172) on the raw mask bits
__device__ __forceinline__ bool wildcard_free(const uint64_t * __restrict__ nmask, uint64_t lpos, uint32_t len)
{
        uint64_t const first = lpos >> 6, last = (lpos + len - 1) >> 6;
        for ( uint64_t w = first; w <= last; ++w )
        {
                uint64_t m = __ldg(nmask + w);
                if ( m )
                {
                        if ( w == first ) m &= (~0ULL) >> (lpos & 63);
                        if ( w == last ) m &= (~0ULL) << (63 - ((lpos + len - 1) & 63));
                        if ( m ) return false;
                }
        }
        return true;
}


// ---- partition ---------------------------------------------------------------------------------

struct HistSmem
{
        uint64_t tile[2][SC_SMEM_WORDS];
        uint64_t bar[2];
        uint32_t cnt[SC_MAX_BUCKETS];
};

// valid positions of the word that starts at local position lx0, as a 32-bit mask (bit j = base j)
__device__ __forceinline__ uint32_t clip_mask(uint64_t lx0, uint64_t x_begin, uint64_t x_end)
{
        if ( lx0 + 32 <= x_begin || lx0 >= x_end ) return 0;
        uint32_t m = 0xFFFFFFFFu;
        if ( lx0 < x_begin ) m &= 0xFFFFFFFFu << (uint32_t)(x_begin - lx0);
        if ( lx0 + 32 > x_end ) m &= 0xFFFFFFFFu >> (uint32_t)(lx0 + 32 - x_end);
        return m;
}

// The positions j0 .. j0+7 (j0 a multiple of 8) of the text word w0 (w1 = the word behind it): bit u of the result is
// set when the 8-bit bucket (first 4 bases) of position j0+u lies in [lo, lo+cnt); top = the 16 bases from j0 on,
// bucket of position j0+u = (top >> (24 - 2u)) & 0xFF
__device__ __forceinline__ uint32_t own_mask8(uint64_t w0, uint64_t w1, uint32_t j0, uint32_t lo, uint32_t cnt, uint32_t & top)
{
        uint64_t const v = j0 ? ((w0 << (2*j0)) | (w1 >> (64 - 2*j0))) : w0;
        top = (uint32_t)(v >> 32);
        uint32_t m = 0;
        #pragma unroll
        for ( uint32_t u = 0; u < 8; ++u )
                m |= ((((top >> (24 - 2*u)) & 0xFFu) - lo < cnt) ? 1u : 0u) << u;
        return m;
}

// The positions of the text word w0 (w1 = the word behind it) whose 8-bit bucket (their first 4 bases) lies in
// [lo, lo+cnt): bit 63-2j of the result is set for position j.  When the range is an aligned power of two -- the case
// for 2, 4 or 8 ranks -- only the top bits of the bucket decide, and they are compared for all 32 positions at once.
__device__ __forceinline__ uint64_t kept_positions(uint64_t w0, uint64_t w1, uint32_t lo, uint32_t cnt)
{
        if ( (cnt & (cnt - 1)) == 0 && (lo & (cnt - 1)) == 0 )
        {
                uint32_t const nb = 8 - (31 - __clz(cnt));            // deciding bits
                uint32_t const want = lo >> (8 - nb);
                uint64_t eq = 0xAAAAAAAAAAAAAAAAULL;
                for ( uint32_t k = 0; k < nb; ++k )
                {
                        uint64_t const y = k ? ((w0 << k) | (w1 >> (64 - k))) : w0;
                        eq &= ((want >> (nb - 1 - k)) & 1u) ? y : ~y;
                }
                return eq;
        }
        uint64_t eq = 0;
        #pragma unroll
        for ( uint32_t j0 = 0; j0 < 32; j0 += 8 )
        {
                uint32_t top;
                uint32_t const m = own_mask8(w0, w1, j0, lo, cnt, top);
                #pragma unroll
                for ( uint32_t u = 0; u < 8; ++u )
                        eq |= (uint64_t)((m >> u) & 1u) << (63 - 2 * (j0 + u));
        }
        return eq;
}
// the same restricted to the positions [x_begin, x_end); lx0 = position of base 0 of w0
__device__ __forceinline__ uint64_t kept_positions_clipped(uint64_t w0, uint64_t w1, uint32_t lo, uint32_t cnt, uint64_t lx0, uint64_t x_begin, uint64_t x_end)
{
        if ( lx0 + 32 <= x_begin || lx0 >= x_end ) return 0;
        uint64_t eq = kept_positions(w0, w1, lo, cnt);
        if ( lx0 < x_begin ) eq &= (~0ULL) >> (2 * (uint32_t)(x_begin - lx0));
        if ( lx0 + 32 > x_end ) eq &= (~0ULL) << (2 * (uint32_t)(lx0 + 32 - x_end));
        return eq;
}

// bucket histogram of the chunk (shared-memory reductions, then one global reduction per CTA and bucket)
__global__ void __launch_bounds__(SC_THREADS) k_part_hist(ScanParams P)
{
        extern __shared__ __align__(128) unsigned char sc_smem[];
        HistSmem & S = *reinterpret_cast<HistSmem *>(sc_smem);

        uint64_t const first_tile = P.x_begin / SC_TILE_POS;
        uint64_t const end_tile = (P.x_end + SC_TILE_POS - 1) / SC_TILE_POS;
        uint32_t const bbits = P.bucket_bits;
        uint32_t const bsh = 64 - (bbits ? bbits : 1);
        uint32_t const bmask = bbits ? 0xFFFFFFFFu : 0u;

        if ( threadIdx.x == 0 )
        {
                mbar_init(&S.bar[0], 1);
                mbar_init(&S.bar[1], 1);
                asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        S.cnt[threadIdx.x] = 0;
        __syncthreads();

        uint64_t tile_id = first_tile + blockIdx.x;
        if ( threadIdx.x == 0 && tile_id < end_tile )
        {
                mbar_expect_tx(&S.bar[0], SC_SMEM_WORDS * 8);
                bulk_load(&S.tile[0][0], P.text + (int64_t)tile_id * SC_TILE_WORDS - SC_HALO, SC_SMEM_WORDS * 8, &S.bar[0]);
        }

        for ( uint32_t it = 0; tile_id < end_tile; tile_id += gridDim.x, ++it )
        {
                uint32_t const buf = it & 1;
                uint64_t const next_tile = tile_id + gridDim.x;
                if ( threadIdx.x == 0 && next_tile < end_tile )
                {
                        mbar_expect_tx(&S.bar[buf ^ 1], SC_SMEM_WORDS * 8);
                        bulk_load(&S.tile[buf ^ 1][0], P.text + (int64_t)next_tile * SC_TILE_WORDS - SC_HALO, SC_SMEM_WORDS * 8, &S.bar[buf ^ 1]);
                }
                mbar_wait(&S.bar[buf], (it >> 1) & 1);
                const uint64_t * tw = &S.tile[buf][SC_HALO];
                uint64_t const tile_x0 = tile_id * SC_TILE_POS;
                #pragma unroll
                for ( int k = 0; k < SC_WPT; ++k )
                {
                        uint32_t const wi = threadIdx.x + k * SC_THREADS;
                        uint64_t const w0 = tw[wi], w1 = tw[wi + 1];
                        uint32_t m = clip_mask(tile_x0 + (uint64_t)wi * 32, P.x_begin, P.x_end);
                        if ( P.own_b_cnt < SC_MAX_BUCKETS && ! (m == 0xFFFFFFFFu && bbits == 8) )
                        {
                                // bucket shard: only the positions of the own buckets are counted (8-bit buckets).  Whole words take
                                // the path below and count every position -- 32 cheap reductions beat picking the kept positions out
                                // one by one at every rank count (measured, r02) -- and the counts of foreign buckets are dropped at the end
                                uint64_t eq = kept_positions_clipped(w0, w1, P.own_b_lo, P.own_b_cnt, tile_x0 + (uint64_t)wi * 32, P.x_begin, P.x_end);
                                while ( eq )
                                {
                                        uint32_t const j = (uint32_t)__clzll(eq) >> 1;
                                        eq &= ~(0x8000000000000000ULL >> (2 * j));
                                        uint64_t const v = j ? ((w0 << (2*j)) | (w1 >> (64 - 2*j))) : w0;
                                        atomicAdd(&S.cnt[(uint32_t)(v >> 56)], 1u);
                                }
                                continue;
                        }
                        if ( m == 0xFFFFFFFFu && bbits == 8 )
                        {
                                // a whole word of 8-bit buckets: 32-bit funnel shifts over the three halves that hold them
                                uint32_t const hi = (uint32_t)(w0 >> 32), lo = (uint32_t)w0, nx = (uint32_t)(w1 >> 32);
                                #pragma unroll
                                for ( int j = 0; j < 16; ++j )
                                {
                                        atomicAdd(&S.cnt[__funnelshift_l(lo, hi, 2*j) >> 24], 1u);
                                        atomicAdd(&S.cnt[__funnelshift_l(nx, lo, 2*j) >> 24], 1u);
                                }
                                continue;
                        }
                        while ( m )
                        {
                                uint32_t const j = __ffs(m) - 1;
                                m &= m - 1;
                                uint64_t const v = j ? ((w0 << (2*j)) | (w1 >> (64 - 2*j))) : w0;
                                atomicAdd(&S.cnt[(uint32_t)(v >> bsh) & bmask], 1u);
                        }
                }
                __syncthreads();   // tile[buf] is free again
        }
        uint32_t const c = S.cnt[threadIdx.x];
        if ( c && (P.own_b_cnt >= SC_MAX_BUCKETS || threadIdx.x - P.own_b_lo < P.own_b_cnt) ) atomicAdd(P.bucket_count + threadIdx.x, c);
}

// ---- partition, scatter pass ---------------------------------------------------------------------
// Records are first laid out bucket by bucket in shared memory and then copied out run by run, so every global store
// instruction writes whole consecutive records of one bucket: scattering records straight from the threads that produce
// them leaves ~200 KB of half-written lines open per CTA, more than L2 holds for a full grid (measured: 2 GB of DRAM reads
// and 5 GB of writes for 3 GB of records, 10 ms per 250 M positions).  Ranks come from a warp-level multisplit (ballots
// of the bucket bits: rank_word): shared-memory atomics that return a value serialise far too much for this.
//
// Dense form (every position of the chunk, or those of the own buckets of a two-rank bucket shard): tiles of 8192
// positions, one text word per thread.  What is staged is the 2-byte offset of a position in its tile, not its 16-byte
// record: the copy-out rebuilds the record from the text words of the tile, which are in shared memory anyway.  Staging
// costs 4 bytes of shared-memory traffic per record instead of 32, and the small staging array lets a tile be four times
// as large as with staged records, so the per-tile bucket work and barriers are paid four times less often per position
// and a bucket's run in a tile is ~32 records (whole lines) instead of ~8 (measured, DESIGN 4.3).
static const int PD_THREADS = 256;                            // threads per CTA; thread b also acts for bucket b
static const int PD_MINB = 4;                                 // CTAs per SM (64 registers)
static const int PD_TILE_WORDS = PD_THREADS;                  // one text word per thread
static const int PD_TILE_POS = PD_TILE_WORDS * 32;            // 8192
static const int PD_SMEM_WORDS = PD_TILE_WORDS + 2 * SC_HALO; // 260 words = 2080 bytes
static_assert(PD_THREADS == SC_MAX_BUCKETS, "the bucket work gives every thread one bucket");
static_assert(SC_TILE_POS % PD_TILE_POS == 0, "a tile must not reach past the last tile of k_part_hist (the text padding)");
static_assert(PD_TILE_POS <= 65536, "tile offsets are staged in 16 bits");

struct ScatterSmem
{
        uint64_t tile[2][PD_SMEM_WORDS];                   // bulk-copy destinations first: 16-byte aligned
        uint64_t bar[2];
        uint4 quad[2 * PD_TILE_WORDS];                     // quad h: the 64 bases [16h-16, 16h+48) of the tile, as 4 half-words
        uint4 * dst[SC_MAX_BUCKETS];                       // per tile: record area of the bucket's owner + first record of the tile's run - first staging slot
        uint4 * area[SC_MAX_BUCKETS];                      // record area of the bucket's owner
        uint32_t wcnt[PD_THREADS / 32][SC_MAX_BUCKETS];    // per-warp counts, then running slots
        uint32_t loc[SC_MAX_BUCKETS + 1];                  // first staging slot of a bucket
        uint32_t wsum[SC_MAX_BUCKETS / 32];                // bucket totals per warp of bucket threads (exclusive scan)
        uint16_t stage[PD_TILE_POS];                       // offset of the position in the tile, bucket-major
};

// the bucket of base j of the text word w0 (w1 = the word behind it): the top bits of the 16 bases from j on
__device__ __forceinline__ uint32_t bucket_at(uint64_t w0, uint64_t w1, uint32_t j, uint32_t bsh, uint32_t bmask)
{
        uint32_t const top = j < 16 ? __funnelshift_l((uint32_t)w0, (uint32_t)(w0 >> 32), 2 * j)
                                    : __funnelshift_l((uint32_t)(w1 >> 32), (uint32_t)w0, 2 * j - 32);
        return (top >> bsh) & bmask;
}

// "the lanes whose bit p of the stream w0:w1 (p = 0: the top bit of w0) equals mine", one ballot per bit plane
__device__ __forceinline__ uint32_t agree_plane(uint64_t w0, uint64_t w1, uint32_t p)
{
        uint32_t const half = p < 32 ? (uint32_t)(w0 >> 32) : p < 64 ? (uint32_t)w0 : (uint32_t)(w1 >> 32);
        uint32_t bal, flip;
        ballot_bit(half, 0x80000000u >> (p & 31), bal, flip);
        return bal ^ flip;
}

// Phase 3 of k_part_scatter: ranks the valid positions m of the thread's text word w0 (w1 = the word behind it) inside
// their buckets with a warp multisplit and stages their tile offsets.  The matches of four steps are issued together:
// their result latency is what this phase waits for.  PLANES (8-bit buckets): the bucket of position j is bits 2j ..
// 2j+7 of the stream w0:w1, so consecutive positions share six of their eight bit planes; each plane's ballot is taken
// once for the word (70 ballots for its 32 positions, against 256 for one multisplit per position).
template <bool PLANES>
__device__ __forceinline__ void rank_word(ScatterSmem & S, uint64_t w0, uint64_t w1, uint32_t m, uint32_t wi, int wid, uint32_t lt,
                                          uint32_t bsh, uint32_t bmask)
{
        uint32_t E[72];
        #pragma unroll
        for ( uint32_t jb = 0; jb < 32; jb += 4 )
        {
                if ( PLANES )
                {
                        #pragma unroll
                        for ( uint32_t p = jb ? 2 * jb + 6 : 0; p < 2 * jb + 14; ++p ) E[p] = agree_plane(w0, w1, p);
                }
                uint32_t b[4], peers[4];
                #pragma unroll
                for ( uint32_t u = 0; u < 4; ++u )
                {
                        uint32_t const j = jb + u;
                        b[u] = bucket_at(w0, w1, j, bsh, bmask);
                        if ( PLANES )
                                peers[u] = __ballot_sync(0xffffffffu, (m >> j) & 1) & E[2*j] & E[2*j+1] & E[2*j+2] & E[2*j+3]
                                           & E[2*j+4] & E[2*j+5] & E[2*j+6] & E[2*j+7];
                        else
                                peers[u] = peers_u8(b[u], (m >> j) & 1);
                }
                #pragma unroll
                for ( uint32_t u = 0; u < 4; ++u )
                {
                        bool const ok = (m >> (jb + u)) & 1;
                        uint32_t const below = __popc(peers[u] & lt);
                        uint32_t pre = 0;
                        if ( ok ) pre = S.wcnt[wid][b[u]];
                        __syncwarp();
                        if ( ok && below == 0 ) S.wcnt[wid][b[u]] = pre + __popc(peers[u]);
                        __syncwarp();
                        if ( ok ) S.stage[pre + below] = (uint16_t)(wi * 32 + jb + u);
                }
        }
}

__global__ void __launch_bounds__(PD_THREADS, PD_MINB) k_part_scatter(ScanParams P)
{
        extern __shared__ __align__(128) unsigned char sc_smem[];
        ScatterSmem & S = *reinterpret_cast<ScatterSmem *>(sc_smem);

        uint64_t const first_tile = P.x_begin / PD_TILE_POS;
        uint64_t const end_tile = (P.x_end + PD_TILE_POS - 1) / PD_TILE_POS;
        uint32_t const bbits = P.bucket_bits;
        uint32_t const bsh = 32 - (bbits ? bbits : 1);
        uint32_t const bmask = bbits ? 0xFFFFFFFFu : 0u;
        uint32_t const fsh = 64 - 2 * P.seedl;
        bool const filter = P.own_b_cnt < SC_MAX_BUCKETS;          // bucket shard: only the positions of the own buckets
        int const lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
        uint32_t const lt = (1u << lane) - 1;

        if ( threadIdx.x == 0 )
        {
                mbar_init(&S.bar[0], 1);
                mbar_init(&S.bar[1], 1);
                asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        #pragma unroll
        for ( int w = 0; w < PD_THREADS / 32; ++w ) S.wcnt[w][threadIdx.x] = 0;
        S.area[threadIdx.x] = P.peer_recs[bucket_owner(P, threadIdx.x)];
        __syncthreads();

        uint64_t tile_id = first_tile + blockIdx.x;
        if ( threadIdx.x == 0 && tile_id < end_tile )
        {
                mbar_expect_tx(&S.bar[0], PD_SMEM_WORDS * 8);
                bulk_load(&S.tile[0][0], P.text + (int64_t)tile_id * PD_TILE_WORDS - SC_HALO, PD_SMEM_WORDS * 8, &S.bar[0]);
        }

        for ( uint32_t it = 0; tile_id < end_tile; tile_id += gridDim.x, ++it )
        {
                uint32_t const buf = it & 1;
                uint64_t const next_tile = tile_id + gridDim.x;
                if ( threadIdx.x == 0 && next_tile < end_tile )
                {
                        mbar_expect_tx(&S.bar[buf ^ 1], PD_SMEM_WORDS * 8);
                        bulk_load(&S.tile[buf ^ 1][0], P.text + (int64_t)next_tile * PD_TILE_WORDS - SC_HALO, PD_SMEM_WORDS * 8, &S.bar[buf ^ 1]);
                }
                mbar_wait(&S.bar[buf], (it >> 1) & 1);
                const uint64_t * tw = &S.tile[buf][SC_HALO];
                uint64_t const tile_x0 = tile_id * PD_TILE_POS;

                // (1) this thread's word: the two quads of its half-words for the copy-out (the halo covers tw[-1] and
                // tw[PD_TILE_WORDS]), the valid positions m, their per-warp bucket counts (reductions without return value)
                uint32_t const wi = threadIdx.x;
                uint64_t const w0 = tw[wi], w1 = tw[wi + 1];
                {
                        uint32_t const wm_lo = (uint32_t)tw[(int)wi - 1];
                        uint32_t const w0_hi = (uint32_t)(w0 >> 32), w0_lo = (uint32_t)w0, w1_hi = (uint32_t)(w1 >> 32);
                        S.quad[2 * wi] = make_uint4(wm_lo, w0_hi, w0_lo, w1_hi);
                        S.quad[2 * wi + 1] = make_uint4(w0_hi, w0_lo, w1_hi, (uint32_t)w1);
                }
                uint32_t m = clip_mask(tile_x0 + (uint64_t)wi * 32, P.x_begin, P.x_end);
                if ( filter )
                {
                        #pragma unroll
                        for ( uint32_t j = 0; j < 32; ++j )
                                if ( bucket_at(w0, w1, j, bsh, bmask) - P.own_b_lo >= P.own_b_cnt ) m &= ~(1u << j);
                }
                #pragma unroll
                for ( uint32_t j = 0; j < 32; ++j )
                        if ( (m >> j) & 1 )
                                atomicAdd(&S.wcnt[wid][bucket_at(w0, w1, j, bsh, bmask)], 1u);
                __syncthreads();
                // (2) bucket b (thread b): totals -> staging layout, global run reservation, per-warp running slots.  The exclusive
                // scan over the 256 bucket totals is a warp scan + one barrier
                uint32_t bstart = 0, reserved = 0;
                {
                        uint32_t tot = 0;
                        #pragma unroll
                        for ( int w = 0; w < PD_THREADS / 32; ++w ) tot += S.wcnt[w][threadIdx.x];
                        uint32_t const incl = warp_incl_scan(tot, lane);
                        if ( lane == 31 ) S.wsum[wid] = incl;
                        // the run's first record is needed at the copy-out only: the global atomic that reserves it stays in
                        // flight while the tile is ranked -- its result must not be touched before
                        if ( tot )
                        {
                                bstart = P.bucket_start[threadIdx.x];
                                reserved = atomicAdd(P.bucket_cursor + threadIdx.x * SC_CURSOR_STRIDE, tot);
                        }
                        __syncthreads();
                        uint32_t base = 0;
                        #pragma unroll
                        for ( int w = 0; w < SC_MAX_BUCKETS / 32 - 1; ++w )
                                if ( w < wid ) base += S.wsum[w];
                        uint32_t const ex = base + incl - tot;
                        S.loc[threadIdx.x] = ex;
                        if ( threadIdx.x == SC_MAX_BUCKETS - 1 ) S.loc[SC_MAX_BUCKETS] = ex + tot;
                        uint32_t run = ex;
                        #pragma unroll
                        for ( int w = 0; w < PD_THREADS / 32; ++w )
                        {
                                uint32_t const c = S.wcnt[w][threadIdx.x];
                                S.wcnt[w][threadIdx.x] = run;
                                run += c;
                        }
                }
                __syncthreads();
                // (3) warp multisplit: one position per lane and step; the group leader advances the warp's slot counter
                if ( bbits == 8 ) rank_word<true>(S, w0, w1, m, wi, wid, lt, bsh, bmask);
                else rank_word<false>(S, w0, w1, m, wi, wid, lt, bsh, bmask);
                // where staging slot 0 would go if it belonged to this bucket: the copy-out adds the slot number
                S.dst[threadIdx.x] = S.area[threadIdx.x] + ((int64_t)(bstart + reserved) - (int64_t)S.loc[threadIdx.x]);
                __syncthreads();
                // the per-warp counters are free from here on (the copy-out does not read them): cleared for the next tile now,
                // under the barrier that ends the copy-out
                #pragma unroll
                for ( int w = 0; w < PD_THREADS / 32; ++w ) S.wcnt[w][threadIdx.x] = 0;
                // (4) copy out: consecutive threads write consecutive records of a bucket run; four records in flight per thread.
                // A record at offset o = 16h + r needs the bases [o-16, o+32), which lie in quad h: one 16-byte load, then
                // funnel shifts by 2r cut the 16 bases in front and the two halves of the window.  Its bucket comes from its window
                {
                        uint32_t const n = S.loc[SC_MAX_BUCKETS];
                        uint32_t const pos0 = (uint32_t)(tile_x0 - P.pos_base);     // may wrap for the clipped first tile; the sums below do not
                        uint32_t i = threadIdx.x;
                        for ( ; i < n; i += 4 * PD_THREADS )
                        {
                                uint32_t o[4];
                                uint4 q[4];
                                #pragma unroll
                                for ( int u = 0; u < 4; ++u ) o[u] = i + u * PD_THREADS < n ? S.stage[i + u * PD_THREADS] : 0u;
                                #pragma unroll
                                for ( int u = 0; u < 4; ++u ) q[u] = S.quad[o[u] >> 4];
                                #pragma unroll
                                for ( int u = 0; u < 4; ++u )
                                {
                                        if ( i + u * PD_THREADS >= n ) break;
                                        uint32_t const sh = 2 * (o[u] & 15);
                                        uint32_t const before = __funnelshift_l(q[u].y, q[u].x, sh);   // the 16 bases in front of the window
                                        uint32_t const vhi = __funnelshift_l(q[u].z, q[u].y, sh);
                                        uint32_t const vlo = __funnelshift_l(q[u].w, q[u].z, sh);
                                        uint64_t const win = (((uint64_t)vhi << 32) | vlo) >> fsh;
                                        uint4 * const d = S.dst[(vhi >> bsh) & bmask];
                                        d[i + u * PD_THREADS] = make_uint4((uint32_t)win, (uint32_t)(win >> 32), before, pos0 + o[u]);
                                }
                        }
                }
                __syncthreads();   // tile[buf], the quads, staging and the counters are free again
        }
}

// ---- partition of a bucket shard -------------------------------------------------------------------
// The multi-GPU form of the partition when the tables are sharded by bucket and every GPU holds the whole text
// (real_gpu_set_bucket_shard): the rank reads EVERY position of the chunk but keeps only those whose bucket belongs
// to it, 1/nranks of them.  Testing a position costs about one instruction (kept_positions: bit sliced over the 32
// positions of a text word); ranking and staging a record is what is expensive.  So one light pass (k_own_list) writes
// the kept positions as a dense list of 4-byte descriptors and counts them per bucket on the way -- no separate
// histogram pass -- and a staged scatter kernel then forms the records of the list (k_part_scatter_list) at its usual cost
// per record.  No record crosses NVLink: the only exchange of a bucket-sharded scan is the fold of the per-read results.
//
// The list kernel stages whole records: its positions are scattered over the text, so there is no tile of text words in
// shared memory a record could be rebuilt from.  Tiles of 2048 listed positions.
static const int PS_THREADS = 256;                            // threads per CTA; thread b also acts for bucket b
static const int PS_PPT = 8;                                  // listed positions per thread
static const int PS_TILE_POS = PS_THREADS * PS_PPT;           // 2048

struct ListScatterSmem
{
        uint4 stage[PS_TILE_POS];                          // record, bucket-major
        uint32_t wcnt[PS_THREADS / 32][SC_MAX_BUCKETS];    // per-warp counts, then running slots
        uint32_t loc[SC_MAX_BUCKETS + 1];                  // first staging slot of a bucket
        uint32_t wsum[SC_MAX_BUCKETS / 32];                // bucket totals per warp of bucket threads (exclusive scan)
        uint4 * dst[SC_MAX_BUCKETS];                       // per tile: record area + first record of the tile's run - first staging slot
};

__global__ void __launch_bounds__(PS_THREADS, 1024 / PS_THREADS) k_part_scatter_list(ScanParams P)
{
        extern __shared__ __align__(128) unsigned char sc_smem[];
        ListScatterSmem & S = *reinterpret_cast<ListScatterSmem *>(sc_smem);

        uint64_t const nlist = *P.list_count;
        uint64_t const end_tile = (nlist + PS_TILE_POS - 1) / PS_TILE_POS;
        uint32_t const bbits = P.bucket_bits;
        uint32_t const bsh = 64 - (bbits ? bbits : 1);
        uint32_t const bmask = bbits ? 0xFFFFFFFFu : 0u;
        uint32_t const fsh = 64 - 2 * P.seedl;
        int const lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
        uint32_t const lt = (1u << lane) - 1;

        #pragma unroll
        for ( int w = 0; w < PS_THREADS / 32; ++w ) S.wcnt[w][threadIdx.x] = 0;
        __syncthreads();

        for ( uint64_t tile_id = blockIdx.x; tile_id < end_tile; tile_id += gridDim.x )
        {
                // the PS_PPT positions of this thread: window word v, the 32 bases in front of it, position field, validity mask m
                uint64_t wv[PS_PPT];
                uint32_t wbefore[PS_PPT], wpos[PS_PPT];
                uint32_t m = 0;
                {
                        uint64_t const i0 = tile_id * PS_TILE_POS + (uint64_t)threadIdx.x * PS_PPT;
                        #pragma unroll
                        for ( uint32_t u = 0; u < PS_PPT; ++u )
                        {
                                bool const ok = i0 + u < nlist;
                                uint32_t const p = ok ? __ldcs(P.list + i0 + u) : 0u;
                                uint64_t const lx = P.pos_base + p;
                                const uint64_t * tw = P.text + (lx >> 5);
                                uint32_t const j = (uint32_t)(lx & 31);
                                uint64_t const wm = __ldg(tw - 1), w0 = __ldg(tw), w1 = __ldg(tw + 1);
                                wv[u] = j ? ((w0 << (2*j)) | (w1 >> (64 - 2*j))) : w0;
                                wbefore[u] = (uint32_t)(j ? ((wm << (2*j)) | (w0 >> (64 - 2*j))) : wm);
                                wpos[u] = p;
                                m |= (ok ? 1u : 0u) << u;
                        }
                }

                // (1) per-warp bucket counts (reductions without return value)
                #pragma unroll
                for ( uint32_t u = 0; u < PS_PPT; ++u )
                        if ( (m >> u) & 1 )
                                atomicAdd(&S.wcnt[wid][(uint32_t)(wv[u] >> bsh) & bmask], 1u);
                __syncthreads();
                // (2) bucket b (thread b): totals -> staging layout, global run reservation, per-warp running slots
                uint32_t bstart = 0, reserved = 0;
                {
                        uint32_t tot = 0;
                        #pragma unroll
                        for ( int w = 0; w < PS_THREADS / 32; ++w ) tot += S.wcnt[w][threadIdx.x];
                        uint32_t const incl = warp_incl_scan(tot, lane);
                        if ( lane == 31 ) S.wsum[wid] = incl;
                        if ( tot )
                        {
                                bstart = P.bucket_start[threadIdx.x];
                                reserved = atomicAdd(P.bucket_cursor + threadIdx.x * SC_CURSOR_STRIDE, tot);
                        }
                        __syncthreads();
                        uint32_t base = 0;
                        #pragma unroll
                        for ( int w = 0; w < SC_MAX_BUCKETS / 32 - 1; ++w )
                                if ( w < wid ) base += S.wsum[w];
                        uint32_t const ex = base + incl - tot;
                        S.loc[threadIdx.x] = ex;
                        if ( threadIdx.x == SC_MAX_BUCKETS - 1 ) S.loc[SC_MAX_BUCKETS] = ex + tot;
                        uint32_t run = ex;
                        #pragma unroll
                        for ( int w = 0; w < PS_THREADS / 32; ++w )
                        {
                                uint32_t const c = S.wcnt[w][threadIdx.x];
                                S.wcnt[w][threadIdx.x] = run;
                                run += c;
                        }
                }
                __syncthreads();
                // (3) warp multisplit: one position per lane and step; the group leader advances the warp's slot counter
                #pragma unroll
                for ( uint32_t jb = 0; jb < PS_PPT; jb += 4 )
                {
                        uint32_t b[4], peers[4];
                        #pragma unroll
                        for ( uint32_t u = 0; u < 4; ++u )
                        {
                                b[u] = (uint32_t)(wv[jb + u] >> bsh) & bmask;
                                peers[u] = peers_u8(b[u], (m >> (jb + u)) & 1);
                        }
                        #pragma unroll
                        for ( uint32_t u = 0; u < 4; ++u )
                        {
                                bool const ok = (m >> (jb + u)) & 1;
                                uint32_t const below = __popc(peers[u] & lt);
                                uint32_t pre = 0;
                                if ( ok ) pre = S.wcnt[wid][b[u]];
                                __syncwarp();
                                if ( ok && below == 0 ) S.wcnt[wid][b[u]] = pre + __popc(peers[u]);
                                __syncwarp();
                                if ( ok )
                                {
                                        uint64_t const win = wv[jb + u] >> fsh;
                                        S.stage[pre + below] = make_uint4((uint32_t)win, (uint32_t)(win >> 32), wbefore[jb + u], wpos[jb + u]);
                                }
                        }
                }
                S.dst[threadIdx.x] = P.recs + ((int64_t)(bstart + reserved) - (int64_t)S.loc[threadIdx.x]);
                __syncthreads();
                #pragma unroll
                for ( int w = 0; w < PS_THREADS / 32; ++w ) S.wcnt[w][threadIdx.x] = 0;
                // (4) copy out: consecutive threads write consecutive records of a bucket run; four records in flight per thread
                {
                        uint32_t const n = S.loc[SC_MAX_BUCKETS];
                        uint32_t i = threadIdx.x;
                        for ( ; i + 3 * PS_THREADS < n; i += 4 * PS_THREADS )
                        {
                                uint4 r[4]; uint4 * d[4];
                                #pragma unroll
                                for ( int u = 0; u < 4; ++u ) r[u] = S.stage[i + u * PS_THREADS];
                                #pragma unroll
                                for ( int u = 0; u < 4; ++u ) d[u] = S.dst[(uint32_t)(((((uint64_t)r[u].y << 32) | r[u].x) << fsh) >> bsh) & bmask];
                                #pragma unroll
                                for ( int u = 0; u < 4; ++u ) d[u][i + u * PS_THREADS] = r[u];
                        }
                        for ( ; i < n; i += PS_THREADS )
                        {
                                uint4 const r = S.stage[i];
                                S.dst[(uint32_t)(((((uint64_t)r.y << 32) | r.x) << fsh) >> bsh) & bmask][i] = r;
                        }
                }
                __syncthreads();   // staging and the counters are free again
        }
}

static const int OL_THREADS = 256;
static const int OL_WPT = 4;                                  // consecutive text words per thread and tile
static const int OL_TILE_WORDS = OL_THREADS * OL_WPT;
static const int OL_TILE_POS = OL_TILE_WORDS * 32;            // 32768 positions

__global__ void __launch_bounds__(OL_THREADS) k_own_list(ScanParams P)
{
        __shared__ uint32_t cnt[SC_MAX_BUCKETS];
        __shared__ unsigned long long tile_base;
        cnt[threadIdx.x] = 0;
        __syncthreads();
        uint64_t const first_tile = P.x_begin / OL_TILE_POS;
        uint64_t const end_tile = (P.x_end + OL_TILE_POS - 1) / OL_TILE_POS;
        for ( uint64_t tile_id = first_tile + blockIdx.x; tile_id < end_tile; tile_id += gridDim.x )
        {
                uint64_t const w0i = tile_id * OL_TILE_WORDS + (uint64_t)threadIdx.x * OL_WPT;
                uint64_t w[OL_WPT + 1];
                #pragma unroll
                for ( int k = 0; k <= OL_WPT; ++k ) w[k] = __ldg(P.text + w0i + k);
                uint64_t eq[OL_WPT];
                uint32_t c = 0;
                #pragma unroll
                for ( int k = 0; k < OL_WPT; ++k )
                {
                        eq[k] = kept_positions_clipped(w[k], w[k+1], P.own_b_lo, P.own_b_cnt, (w0i + k) * 32, P.x_begin, P.x_end);
                        c += (uint32_t)__popcll(eq[k]);
                }
                uint32_t total;
                uint32_t const ex = block_excl_scan(c, &total);
                if ( threadIdx.x == 0 && total ) tile_base = atomicAdd(P.list_count, (unsigned long long)total);
                __syncthreads();
                if ( ! total ) continue;
                uint32_t * out = P.list + tile_base + ex;
                // one loop over the kept positions of all OL_WPT words of the thread: a loop per word leaves the lanes of a warp
                // waiting for the one with most kept positions in THAT word, four times over (13 of 32 lanes active, r02 capture)
                {
                        static_assert(OL_WPT == 4, "the word selects below are written out for four words");
                        uint32_t k = 0;
                        uint64_t e = eq[0], wa = w[0], wb = w[1];
                        while ( true )
                        {
                                while ( ! e && k < OL_WPT - 1 )
                                {
                                        ++k;
                                        e = (k == 1) ? eq[1] : ((k == 2) ? eq[2] : eq[3]);
                                        wa = wb;
                                        wb = (k == 1) ? w[2] : ((k == 2) ? w[3] : w[4]);
                                }
                                if ( ! e ) break;
                                uint32_t const j = (uint32_t)__clzll(e) >> 1;
                                e &= ~(0x8000000000000000ULL >> (2 * j));
                                uint64_t const v = j ? ((wa << (2*j)) | (wb >> (64 - 2*j))) : wa;
                                *out++ = (uint32_t)((w0i + k) * 32 - P.pos_base) + j;
                                atomicAdd(&cnt[(uint32_t)(v >> 56)], 1u);
                        }
                }
                __syncthreads();           // tile_base is free again
        }
        __syncthreads();
        if ( cnt[threadIdx.x] ) atomicAdd(P.bucket_count + threadIdx.x, cnt[threadIdx.x]);
}

// one block: bucket starts (every bucket padded to whole grabs), cursors, sentinel records in the padding.
// The records of bucket b go to the record area of b's owner, into this rank's segment of it (from record
// rank * seg_cap), bucket after bucket; the owner is told the padded size of every bucket it is sent.
__global__ void __launch_bounds__(SC_MAX_BUCKETS) k_part_offsets(ScanParams P)
{
        __shared__ uint32_t sc[SC_MAX_BUCKETS], st[SC_MAX_BUCKETS + 1];
        uint32_t const c = P.bucket_count[threadIdx.x];
        uint32_t const padded = ((c + SC_UNIT - 1) / SC_UNIT) * SC_UNIT;
        sc[threadIdx.x] = padded;
        __syncthreads();
        if ( threadIdx.x == 0 )
        {
                uint32_t a = 0;
                for ( uint32_t d = 0; d < P.nranks; ++d )
                {
                        a = P.rank * P.seg_cap;
                        for ( uint32_t b = P.bucket_lo[d]; b < P.bucket_lo[d+1]; ++b ) { st[b] = a; a += sc[b]; }
                }
                st[SC_MAX_BUCKETS] = a;            // single rank: the total (all buckets are in one area)
                *P.unit_counter = 0;
                if ( P.own_b_cnt < SC_MAX_BUCKETS )
                {
                        unsigned long long kept = 0;
                        for ( uint32_t b = 0; b < (uint32_t)SC_MAX_BUCKETS; ++b ) kept += P.bucket_count[b];
                        atomicAdd(P.nprobed, kept);
                }
        }
        __syncthreads();
        uint32_t const owner = bucket_owner(P, threadIdx.x);
        P.bucket_start[threadIdx.x] = st[threadIdx.x];
        if ( threadIdx.x == 0 ) P.bucket_start[SC_MAX_BUCKETS] = st[SC_MAX_BUCKETS];
        P.bucket_cursor[threadIdx.x * SC_CURSOR_STRIDE] = 0;
        uint4 * area = P.peer_recs[owner];
        for ( uint32_t r = st[threadIdx.x] + c; r < st[threadIdx.x] + padded; ++r )
                area[r] = make_uint4(0, 0, 0, SC_POS_NONE);
        if ( P.nranks > 1 )
                P.peer_meta[owner][P.rank * SC_META_STRIDE + threadIdx.x] = padded;
}

// ---- cross-rank hand-over (sharded tables) ----------------------------------------------------------
// flags[slot * SC_MAX_RANKS + source] in every rank's window holds the last round `source` has completed for
// that slot (0: its records of the round are delivered, 1: it has consumed the records it was sent).  Kernel
// boundaries order the data stores before the signal; the signal is a system-scope release store into peer
// memory, the wait an acquire load of local memory.
__global__ void k_comm_signal(uint32_t * const * peer_flags, uint32_t nranks, uint32_t rank, uint32_t slot, uint32_t epoch)
{
        if ( threadIdx.x < nranks )
        {
                __threadfence_system();
                uint32_t * f = peer_flags[threadIdx.x] + slot * SC_MAX_RANKS + rank;
                asm volatile("st.release.sys.global.u32 [%0], %1;" :: "l"(f), "r"(epoch) : "memory");
        }
}

// spins until every rank has signalled `epoch` (or later) in `slot`; gives up after timeout_cycles and raises *error
__global__ void k_comm_wait(const uint32_t * flags, uint32_t nranks, uint32_t slot, uint32_t epoch, long long timeout_cycles, uint32_t * error)
{
        if ( threadIdx.x < nranks )
        {
                const uint32_t * f = flags + slot * SC_MAX_RANKS + threadIdx.x;
                long long const t0 = clock64();
                uint32_t v;
                while ( true )
                {
                        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
                        if ( (int32_t)(v - epoch) >= 0 ) break;
                        if ( clock64() - t0 > timeout_cycles ) { *error = 1 + threadIdx.x; break; }
                        __nanosleep(200);
                }
        }
}

// owner side: the (bucket, source) pairs of the round in bucket-major order -> first grab / first record of each
static const int SC_PAIR_THREADS = 512;                      // >= own buckets * ranks for any rank count up to SC_MAX_RANKS
__global__ void __launch_bounds__(SC_PAIR_THREADS) k_comm_pairs(ScanParams P, const uint32_t * meta)
{
        __shared__ uint32_t roff[SC_MAX_RANKS][SC_MAX_BUCKETS];
        uint32_t const lo = P.bucket_lo[P.rank], nb = P.bucket_lo[P.rank + 1] - lo;
        if ( threadIdx.x < P.nranks )
        {
                uint32_t a = threadIdx.x * P.seg_cap;
                for ( uint32_t b = 0; b < nb; ++b ) { roff[threadIdx.x][b] = a; a += meta[threadIdx.x * SC_META_STRIDE + lo + b]; }
        }
        __syncthreads();
        uint32_t const npairs = nb * P.nranks;                // < SC_PAIR_THREADS
        uint32_t const p = threadIdx.x;
        uint32_t const b = p / P.nranks, src = p - b * P.nranks;
        uint32_t const g = (p < npairs) ? meta[src * SC_META_STRIDE + lo + b] / SC_UNIT : 0;
        uint32_t total;
        uint32_t const ex = block_excl_scan(g, &total);
        if ( p < npairs ) { P.pair_grab[p] = ex; P.pair_rec[p] = roff[src][b]; }
        if ( p == 0 ) { P.pair_grab[npairs] = total; *P.unit_counter = 0; }
}

// ---- probe -------------------------------------------------------------------------------------

struct ItemA { uint64_t win; uint32_t before; uint32_t post; };      // a set slot bit: window, bases in front, position in the chunk (entry index: ProbeSmem::qe, table: ProbeSmem::qt)
struct ItemB { uint64_t lp; uint32_t id; uint32_t exact; };           // an entry that passed the seed test (exact: bit f = fragment f matches exactly)

struct ProbeSmem
{
        ItemA qa[SC_THREADS / 32][SC_QA_CAP];
        ItemB qb[SC_THREADS / 32][SC_QB_CAP];
        uint32_t qe[SC_THREADS / 32][SC_QA_CAP];        // entry index (rank of the slot) of the stage A items
        uint8_t qt[SC_THREADS / 32][SC_QA_CAP];         // table of the stage A items
        uint32_t qbn[SC_THREADS / 32];
        uint32_t stat[3][SC_THREADS];                   // per thread: candidates, seed passes, hits (far below 2^32 per launch)
};

// Seeds longer than the indexed 32 bases: the seed test of ::match (match.hpp:386-388) over the WHOLE seed of strand
// `id` laid over the text at local position lstart (read start); a0 = first seed base in strand coordinates.  Returns
// false when the seed has more than seedkmax mismatches; exact = which of its four fragments match exactly.
__device__ __forceinline__ bool wide_seed_test(ScanParams const & P, uint32_t id, uint32_t L, uint64_t lstart, uint32_t a0, uint32_t & exact)
{
        uint32_t const Ft = P.vseedl >> 2;
        uint32_t seedk = 0;
        exact = 0;
        #pragma unroll
        for ( uint32_t f = 0; f < 4; ++f )
        {
                uint64_t const rf = strand_bases(P.rs, id, L, a0 + f * Ft, Ft) >> (64 - 2 * Ft);
                uint64_t const tf = text_word(P.text, lstart + a0 + f * Ft, Ft);
                uint32_t const kf = diffcount64(rf, tf);
                seedk += kf;
                if ( kf == 0 ) exact |= 1u << f;
        }
        return seedk <= P.seedkmax;
}

// whole-read Hamming distance of strand id of a 2 bit/base input read against the text at word tp, bit offset sh; gives up
// (returns more than kmax) once the count exceeds kmax.  The words are cut out four at a time, all their loads issued
// before the first is used: a warp that verifies does not probe, so the round trips must overlap, not queue up
// (one word per iteration cost the C3 scan 11 ms).
__device__ __forceinline__ uint32_t distance_packed(ReadSrc const & rs, uint32_t id, uint32_t L, const uint64_t * __restrict__ tp, uint32_t sh, uint32_t kmax)
{
        uint32_t const nw = (L + 31) >> 5;
        const uint8_t * p = packed_read(rs, id >> 1);
        bool const minus = id & 1;
        uint64_t prev = __ldg(tp);
        uint32_t k = 0;
        for ( uint32_t w0 = 0; w0 < nw; w0 += 4 )
        {
                uint64_t rw[4], tw[4];
                #pragma unroll
                for ( uint32_t u = 0; u < 4; ++u )
                        if ( w0 + u < nw )
                        {
                                uint32_t const w = w0 + u;
                                uint32_t const len = (w + 1 == nw) ? (L - 32*w) : 32;
                                rw[u] = packed_bases(p, minus ? (L - 32*w - len) : 32*w, len);
                                tw[u] = __ldg(tp + w + 1);
                        }
                #pragma unroll
                for ( uint32_t u = 0; u < 4; ++u )
                        if ( w0 + u < nw )
                        {
                                uint32_t const w = w0 + u;
                                uint32_t const len = (w + 1 == nw) ? (L - 32*w) : 32;
                                uint64_t r = rw[u] >> (64 - 2*len);
                                if ( minus ) r = revcomp_word(r, len);
                                uint64_t const tv = sh ? ((prev << sh) | (tw[u] >> (64 - sh))) : prev;
                                prev = tw[u];
                                k += diffcount64(r, tv >> (64 - 2*len));
                        }
                if ( k > kmax ) break;
        }
        return k;
}

// stage B: one read strand laid over seed window lp -- position / record / wildcard predicates,
// whole-read distance, report
template<bool WIDE, bool PACKED>
__device__ __forceinline__ uint32_t verify_and_report(ScanParams const & P, uint64_t lp, uint32_t id, uint32_t exact)
{
        uint32_t const strand = id & 1;
        uint32_t const read = id >> 1;
        if ( P.mode == 2 )
        {
                // gapped pass (match.hpp:477-499): only the seed is required to match; '+' strand only; reads still
                // NoMatch/Gapped; the seed window must lie inside one record and be wildcard free
                if ( strand ) return 0;
                uint32_t const st = umi_state(P.info[read]);
                if ( st != ST_NOMATCH && st != ST_GAPPED ) return 0;
                uint64_t const grpos = P.shard_begin + lp;
                if ( grpos < P.own_begin || grpos >= P.own_end ) return 0;
                uint32_t const gfrag = record_of(P.rec, P.nrec, grpos);
                if ( gfrag >= P.nrec || grpos + P.vseedl > __ldg(P.rec + gfrag + 1) ) return 0;
                if ( ! wildcard_free(P.nmask, lp, P.vseedl) ) return 0;
                if ( WIDE && ! wide_seed_test(P, id, __ldg(P.rlen + read), lp, 0, exact) ) return 0;
                unsigned long long const slot = atomicAdd(P.hit_count, 1ULL);
                if ( slot < P.hit_cap )
                {
                        RawHit h;
                        h.pm = rawhit_pack(grpos, 0, 0, gfrag);
                        h.read = read | (exact << 28);
                        h.score = 0.0f;
                        P.hits[slot] = h;
                }
                return 1;
        }
        uint32_t const L = __ldg(P.rlen + read);
        uint32_t const matchoffset = strand ? (L - P.seedl) : 0;          // RestMatch.hpp:84-89
        uint64_t const gp = P.shard_begin + lp;
        if ( gp < matchoffset ) return 0;                                   // match.hpp:393
        uint64_t const gpos = gp - matchoffset;
        if ( gpos < P.own_begin || gpos >= P.own_end ) return 0;
        uint64_t const lpos = gpos - P.shard_begin;
        if ( WIDE && ! wide_seed_test(P, id, L, lpos, strand ? (L - P.vseedl) : 0u, exact) ) return 0;

        // whole-read Hamming distance = seedk + restk (match.hpp:400-405); the words of the read and of the text under
        // it are fetched four at a time so that their latencies overlap (and overlap the predicates' loads below)
        const uint64_t * tp = P.text + (lpos >> 5);
        uint32_t const sh = (uint32_t)(lpos & 31) << 1;
        uint32_t const nw = (L + 31) >> 5;
        uint64_t prev = __ldg(tp);
        uint32_t k = 0, frag;
        if ( ! PACKED )
        {
                const uint64_t * rp = P.rs.rpack + (uint64_t)id * P.rs.W;
                uint64_t rw[4], tw[4];
                #pragma unroll
                for ( uint32_t u = 0; u < 4; ++u )
                        if ( u < nw ) { rw[u] = __ldg(rp + u); tw[u] = __ldg(tp + u + 1); }

                // RangeVector::isPositionValid && AutoTextArray::isDontCareFree (match.hpp:398)
                frag = record_of(P.rec, P.nrec, gpos);
                if ( frag >= P.nrec || gpos + L > __ldg(P.rec + frag + 1) ) return 0;
                if ( ! wildcard_free(P.nmask, lpos, L) ) return 0;

                for ( uint32_t w0 = 0; w0 < nw; w0 += 4 )
                {
                        if ( w0 )
                        {
                                #pragma unroll
                                for ( uint32_t u = 0; u < 4; ++u )
                                        if ( w0 + u < nw ) { rw[u] = __ldg(rp + w0 + u); tw[u] = __ldg(tp + w0 + u + 1); }
                        }
                        #pragma unroll
                        for ( uint32_t u = 0; u < 4; ++u )
                                if ( w0 + u < nw )
                                {
                                        uint32_t const w = w0 + u;
                                        uint32_t const len = (w + 1 == nw) ? (L - 32*w) : 32;
                                        uint64_t const tv = sh ? ((prev << sh) | (tw[u] >> (64 - sh))) : prev;      // = text_word(P.text, lpos + 32*w, .) before the final shift
                                        prev = tw[u];
                                        k += diffcount64(rw[u] >> (64 - 2*len), tv >> (64 - 2*len));
                                }
                        if ( k > P.totalkmax ) return 0;
                }
        }
        else
        {
                // 2 bit/base input: the strand's words are cut out of the caller's packed bytes
                frag = record_of(P.rec, P.nrec, gpos);
                if ( frag >= P.nrec || gpos + L > __ldg(P.rec + frag + 1) ) return 0;
                if ( ! wildcard_free(P.nmask, lpos, L) ) return 0;
                k = distance_packed(P.rs, id, L, tp, sh, P.totalkmax);
                if ( k > P.totalkmax ) return 0;
        }
        if ( P.mode == 1 )
                unique_update(P.info + read, strand, P.fileid, gpos, k, frag);
        else
        {
                unsigned long long const slot = atomicAdd(P.hit_count, 1ULL);
                if ( slot < P.hit_cap )
                {
                        RawHit h;
                        h.pm = rawhit_pack(gpos, k, strand, frag);
                        h.read = read | (exact << 28);     // which fragments of the seed are exact: decides the lists that see the hit (order-faithful replay)
                        h.score = 1.0f;
                        P.hits[slot] = h;
                }
        }
        return 1;
}

// stage A: a set slot bit with the index e of its first entry -> entry chain; per entry the seed test
// (match.hpp:386-388) and the canonical-list rule: of the up to six lists that reach a position,
// only the pair made of the two LOWEST exact fragments reports it (replaces unifyMatches' dedup)
template<bool WIDE, bool PACKED>
__device__ __forceinline__ void follow_item(ScanParams const & P, ItemA const & it, uint32_t e, int const table, ItemB * qb, uint32_t * qbn, uint32_t * lstats, uint64_t pol_e)
{
        uint32_t const F = P.F;
        uint64_t const fm = (1ULL << (2*F)) - 1;
        uint64_t const lx = P.pos_base + it.post;
        while ( e != ENTRY_NONE )
        {
                uint4 const raw = ld_hot_v4(P.tab[table].E + e, pol_e);
                uint64_t const eseed = ((uint64_t)raw.y << 32) | raw.x;
                uint32_t const t = raw.z & 3, id = raw.z >> 2;
                e = raw.w;
                if ( lx < (uint64_t)t * F ) continue;
                uint64_t const lp = lx - (uint64_t)t * F;                      // seed window start (local)
                if ( lp < P.win_begin || lp >= P.win_end ) continue;
                lstats[0] += 1;
                // the seed window starts t fragments in front of the probed position: its first t*F bases come
                // from the record's "before" word, the rest from the window word
                uint32_t const tb = 2 * t * F;
                uint64_t const win = t ? ((((uint64_t)it.before & ((1ULL << tb) - 1)) << (2*P.seedl - tb)) | (it.win >> tb)) : it.win;
                uint64_t x = eseed ^ win;
                x = ((x >> 1) | x) & 0x5555555555555555ULL;
                uint32_t const seedk = (uint32_t)__popcll(x);
                if ( seedk > P.seedkmax ) continue;
                int first = -1, second = -1;
                uint32_t exact4 = 0;
                #pragma unroll
                for ( int f = 0; f < 4; ++f )
                {
                        bool const exact = ((x >> (2*F*(3-f))) & fm) == 0;
                        if ( exact ) { exact4 |= 1u << f; if ( first < 0 ) first = f; else if ( second < 0 ) second = f; }
                }
                if ( first != (int)t || second != pair_second(table, (int)t) ) continue;
                lstats[1] += 1;
                uint32_t const o = atomicAdd(qbn, 1u);
                if ( o < SC_QB_CAP )
                {
                        ItemB ib; ib.lp = lp; ib.id = id; ib.exact = exact4;
                        qb[o] = ib;
                }
                else
                        lstats[2] += verify_and_report<WIDE, PACKED>(P, lp, id, exact4);          // queue full: handle it here
        }
}

// the warp's stage B queue
template<bool WIDE, bool PACKED>
__device__ __forceinline__ void drain_b_warp(ScanParams const & P, ItemB * qb, uint32_t * qbn, int lane, uint32_t * lstats)
{
        uint32_t const n = min(*qbn, (uint32_t)SC_QB_CAP);
        __syncwarp();
        for ( uint32_t i = lane; i < n; i += 32 )
        {
                ItemB const ib = qb[i];
                lstats[2] += verify_and_report<WIDE, PACKED>(P, ib.lp, ib.id, ib.exact);
        }
        __syncwarp();
        if ( lane == 0 ) *qbn = 0;
        __syncwarp();
}

// the warp's stage A queue (n items, the same value in every lane): full rounds of 32 from the top of the queue;
// with `flush` also the rest.  Returns the number of items left.  The statistics go to per-thread shared-memory
// counters so that the probe loop carries no state for this path.
template<bool WIDE, bool PACKED>
__device__ __forceinline__ uint32_t drain_a_warp(ScanParams const & P, ProbeSmem & S, uint32_t n, bool flush)
{
        int const lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
        const ItemA * qa = S.qa[wid];
        const uint32_t * qe = S.qe[wid];
        const uint8_t * qt = S.qt[wid];
        ItemB * qb = S.qb[wid];
        uint32_t * qbn = &S.qbn[wid];
        uint32_t lstats[3] = {0, 0, 0};
        // entries are touched about once per bucket pass: when several chunks stream them past, they go through L2 with
        // evict_first priority so that they do not push the presence words (probed several times per line) out of the
        // protected set (plan_scan)
        uint64_t const pol_e = P.entries_evict_normal ? policy_evict_normal() : policy_evict_first();
        while ( n >= 32 || (flush && n) )
        {
                uint32_t const take = n >= 32 ? 32u : n;
                if ( (uint32_t)lane < take )
                        follow_item<WIDE, PACKED>(P, qa[n - take + lane], qe[n - take + lane], (int)qt[n - take + lane], qb, qbn, lstats, pol_e);
                __syncwarp();
                n -= take;
                if ( *qbn >= 32 )
                        drain_b_warp<WIDE, PACKED>(P, qb, qbn, lane, lstats);
        }
        if ( flush && *qbn )
                drain_b_warp<WIDE, PACKED>(P, qb, qbn, lane, lstats);
        #pragma unroll
        for ( int s = 0; s < 3; ++s )
                if ( lstats[s] ) S.stat[s][threadIdx.x] += lstats[s];
        return n;
}

// the 512 records of grab g
__device__ __forceinline__ const uint4 * grab_records(ScanParams const & P, uint32_t g)
{
        if ( ! P.npairs )
                return P.recs + (uint64_t)g * SC_UNIT;
        uint32_t lo = 0, hi = P.npairs;                 // last pair with pair_grab <= g
        while ( hi - lo > 1 )
        {
                uint32_t const mid = (lo + hi) >> 1;
                if ( __ldg(P.pair_grab + mid) <= g ) lo = mid; else hi = mid;
        }
        return P.recs + (uint64_t)__ldg(P.pair_rec + lo) + (uint64_t)(g - __ldg(P.pair_grab + lo)) * SC_UNIT;
}

// WIDE: seeds longer than the indexed 32 bases (the whole-seed test costs registers the common case must not pay for)
template<bool WIDE, bool PACKED>
__global__ void __launch_bounds__(SC_THREADS, SC_PROBE_MINB) k_bucket_probe(const __grid_constant__ ScanParams P)
{
        extern __shared__ __align__(128) unsigned char sc_smem[];
        ProbeSmem & S = *reinterpret_cast<ProbeSmem *>(sc_smem);
        int const lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
        uint32_t const lt = (1u << lane) - 1;
        ItemA * qa = S.qa[wid];
        uint32_t * qe = S.qe[wid];
        uint8_t * qt = S.qt[wid];
        uint32_t qn = 0;                 // items in the stage A queue; warp uniform, kept in a register

        if ( lane == 0 ) S.qbn[wid] = 0;
        #pragma unroll
        for ( int s = 0; s < 3; ++s ) S.stat[s][threadIdx.x] = 0;
        __syncwarp();
        // single rank: the record area holds the buckets back to back, padded to whole grabs; sharded: the grabs are
        // numbered pair by pair (own bucket, source), see k_comm_pairs
        uint32_t const ngrabs = P.npairs ? P.pair_grab[P.npairs] : P.bucket_start[SC_MAX_BUCKETS] / SC_UNIT;

        uint32_t const F = P.F;
        uint32_t const kb = P.keybits;
        uint64_t const fm = (1ULL << (2*F)) - 1;
        bool const nlA = P.tab[0].nlists != 0, nlB = P.tab[1].nlists != 0, nlC = P.tab[2].nlists != 0;

        // grabs of 512 records are handed out in bucket order by a global counter, one per warp at a time, so all
        // warps of the grid work on the same bucket (slice) at any time; a warp draws its next grab before it
        // starts on the current one, and there is no block-wide barrier anywhere in the loop
        uint32_t g = 0;
        if ( lane == 0 ) g = atomicAdd(P.unit_counter, 1u);
        g = __shfl_sync(0xffffffffu, g, 0);
        int const NSTEP = SC_UNIT / (32 * SC_RPT);
        int const STEP_LINES = 32 * SC_RPT * (int)sizeof(uint4) / 128;          // 128-byte lines of records per step
        while ( g < ngrabs )
        {
                uint32_t gn = 0;
                if ( lane == 0 ) gn = atomicAdd(P.unit_counter, 1u);

                // The records of a step are not held in registers ahead of time (the candidate path below needs the
                // registers): they are pulled into L2 two steps ahead with prefetches -- across the grab boundary too --
                // and loaded when the step starts (holding the next step's records in registers instead: 83 vs 76 ms scan on C3).
                const uint4 * rp = grab_records(P, g);
                #pragma unroll 1
                for ( int step = 0; step < NSTEP; ++step )
                {
                        if ( step == NSTEP - 2 )
                                gn = __shfl_sync(0xffffffffu, gn, 0);
                        uint4 cur[SC_RPT];
                        {
                                int const ps = step + 2;
                                bool const pv = ps < NSTEP || gn < ngrabs;
                                const uint4 * pb = (ps < NSTEP) ? (rp + ps * 32 * SC_RPT) : (pv ? grab_records(P, gn) + (ps - NSTEP) * 32 * SC_RPT : rp);
                                if ( lane < STEP_LINES && pv )
                                        asm volatile("prefetch.global.L2 [%0];" :: "l"(pb + lane * 8));
                        }
                        #pragma unroll
                        for ( int k = 0; k < SC_RPT; ++k ) cur[k] = __ldcs(rp + step * 32 * SC_RPT + k * 32 + lane);
                        // one 8-byte probe per record and table: presence bits of the slot's word + rank of its first slot
                        SlotWord sw[SC_RPT][3];
                        uint32_t bits5[SC_RPT];          // bit index inside the word, 5 bits per table
                        #pragma unroll
                        for ( int k = 0; k < SC_RPT; ++k )
                        {
                                // padding records probe slot 0 of every table like anybody else (no divergent branch around the
                                // loads); their candidates are masked out below
                                uint64_t const win = ((uint64_t)cur[k].y << 32) | cur[k].x;
                                uint64_t const m0 = (win >> (6*F)) & fm;
                                bits5[k] = 0;
                                #pragma unroll
                                for ( int t = 0; t < 3; ++t )
                                {
                                        sw[k][t].bits = 0; sw[k][t].rank = 0;
                                        if ( t == 0 ? nlA : (t == 1 ? nlB : nlC) )           // warp uniform
                                        {
                                                uint64_t const mo = (win >> (2*F*(2 - t))) & fm;
                                                uint32_t const h = slot_of((m0 << (2*F)) | mo, kb, P.tab[t].hb);
                                                bits5[k] |= (h & 31) << (5 * t);
                                                sw[k][t] = ld_slotword(P.tab[t].slots + (h >> 5));
                                        }
                                }
                        }
                        // compact the set slot bits into the warp's stage A queue: one ballot per (record, table)
                        uint32_t cand = 0;
                        #pragma unroll
                        for ( int k = 0; k < SC_RPT; ++k )
                                #pragma unroll
                                for ( int t = 0; t < 3; ++t )
                                        cand |= ((cur[k].w != SC_POS_NONE) ? ((sw[k][t].bits >> ((bits5[k] >> (5 * t)) & 31)) & 1u) : 0u) << (k * 3 + t);
                        if ( __any_sync(0xffffffffu, cand != 0) )
                        {
                                #pragma unroll
                                for ( int k = 0; k < SC_RPT; ++k )
                                        #pragma unroll
                                        for ( int t = 0; t < 3; ++t )
                                        {
                                                bool const set = (cand >> (k * 3 + t)) & 1u;
                                                uint32_t const bal = __ballot_sync(0xffffffffu, set);
                                                if ( set )
                                                {
                                                        uint32_t const o = qn + __popc(bal & lt);
                                                        ItemA ia; ia.win = ((uint64_t)cur[k].y << 32) | cur[k].x; ia.before = cur[k].z; ia.post = cur[k].w;
                                                        qa[o] = ia;
                                                        qt[o] = (uint8_t)t;
                                                        qe[o] = sw[k][t].rank + __popc(sw[k][t].bits & ((1u << ((bits5[k] >> (5 * t)) & 31)) - 1));
                                                }
                                                qn += __popc(bal);
                                        }
                                __syncwarp();
                                if ( qn >= 32 )
                                        qn = drain_a_warp<WIDE, PACKED>(P, S, qn, false);
                        }
                }
                g = gn;
        }
        drain_a_warp<WIDE, PACKED>(P, S, qn, true);

        // statistics: one atomic per warp and counter
        #pragma unroll
        for ( int s = 0; s < 3; ++s )
        {
                unsigned long long v2 = S.stat[s][threadIdx.x];      // widened for the sum over the warp
                #pragma unroll
                for ( int o = 16; o > 0; o >>= 1 )
                        v2 += __shfl_xor_sync(0xffffffffu, v2, o);
                if ( (threadIdx.x & 31) == 0 && v2 )
                        atomicAdd(P.stats + s, v2);
        }
}

} // namespace realgpu
