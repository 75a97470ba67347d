// K1 (read packing, seed extraction) and K2 (read-side signature index) kernels.
//
// K1 replaces, per read, Pattern::computeMapped (Pattern.hpp:105-128),
// SignatureConstruction::signatureMapped / reverseMappedSignature
// (SignatureConstruction.hpp:218-280, 347-410) and RestWordBuffer::setupStraight/setupReverse
// (RestWordBuffer.hpp:56-78): both strands of every read are packed 2 bit/base, MSB first, into
// W words, and the 4-fragment seed of each strand is kept as one word.
//
// K2 replaces ListSet::sort + getLookupTable (ListSet.hpp:41-63, getLookupTable.hpp:25-51), on the
// READ side (BASELINE.json north_star).  The six pair lists collapse into three tables because a
// text position x sees the same 2-fragment key for several lists:
//   table A (adjacent fragments)  key(x) = bases [x,x+2F)               lists 0,3,5 at window x, x-F, x-2F
//   table B (one fragment apart)  key(x) = [x,x+F) ++ [x+2F,x+3F)       lists 1,4   at window x, x-F
//   table C (two apart)           key(x) = [x,x+F) ++ [x+3F,x+4F)       list  2     at window x
// Each table is a presence array over signature slots -- one 8-byte SlotWord {32 presence bits, rank of the
// word's first slot} per 32 slots, so that one 8-byte probe yields the bit and the entry index -- plus an
// entry array addressed by rank.
#pragma once

#include "common.cuh"
#include "prims.cuh"

namespace realgpu
{

// list id of (table, fragment offset t) and the fragment pair it keys on
__host__ __device__ __forceinline__ int list_of(int table, int t)
{
        // A: (0,1)->0 (1,2)->3 (2,3)->5 ; B: (0,2)->1 (1,3)->4 ; C: (0,3)->2
        return table == 0 ? (t == 0 ? 0 : (t == 1 ? 3 : 5)) : (table == 1 ? (t == 0 ? 1 : 4) : 2);
}
__host__ __device__ __forceinline__ int pair_second(int table, int t) { return t + 1 + table; }

// which (table,t) entries exist for a given seed error budget: a seed with at most s mismatching
// bases has at least 4-s exact fragments, and a match is reported through the pair made of its two
// LOWEST exact fragments only, so pairs that can never be that pair are not indexed.
__host__ __device__ __forceinline__ int table_lists(int table, uint32_t seedkmax)
{
        if ( seedkmax >= 2 ) return table == 0 ? 3 : (table == 1 ? 2 : 1);
        if ( seedkmax == 1 ) return table == 0 ? 2 : (table == 1 ? 1 : 0);
        return table == 0 ? 1 : 0;
}

// ---- K1 --------------------------------------------------------------------------------------

// `len` (1..32) mapped bytes starting at p, packed 2 bit/base MSB first and left aligned; *bad is set when a
// byte is not 0..3.  The bytes are fetched as aligned 32-bit words and realigned with funnel shifts; four
// bases are packed at a time with one multiply: for x = b0 | b1<<8 | b2<<16 | b3<<24 (each 0..3) the top byte
// of x * 0x40100401 is b0<<6 | b1<<4 | b2<<2 | b3 (the partial products land on disjoint bits).
__device__ __forceinline__ uint64_t pack_bytes(const uint8_t * __restrict__ p, uint32_t len, uint32_t & bad)
{
        uintptr_t const addr = reinterpret_cast<uintptr_t>(p);
        const uint32_t * q = reinterpret_cast<const uint32_t *>(addr & ~(uintptr_t)3);
        uint32_t const sh = (uint32_t)(addr & 3) * 8;
        uint32_t const nq = (uint32_t)((addr & 3) + len + 3) >> 2;        // aligned words that hold the bytes
        uint32_t w[9];
        #pragma unroll
        for ( uint32_t i = 0; i < 9; ++i )
                w[i] = (i < nq) ? __ldg(q + i) : 0u;
        uint64_t word = 0;
        #pragma unroll
        for ( uint32_t i = 0; i < 8; ++i )
        {
                uint32_t x = __funnelshift_r(w[i], w[i+1], sh);
                int const rem = (int)len - 4 * (int)i;                      // bytes of this group that belong to the read
                if ( rem < 4 ) x &= (rem <= 0) ? 0u : (0xFFFFFFFFu >> (8 * (4 - rem)));
                bad |= x & 0xFCFCFCFCu;
                uint32_t const packed = ((x & 0x03030303u) * 0x40100401u) >> 24;
                word |= (uint64_t)packed << (56 - 8 * i);
        }
        return word;
}

// one thread per (read, strand, word): word w of the '+' strand is read[32w, 32w+32); word w of the '-' strand
// is the reverse complement of read[L-32w-len, L-32w)
__global__ void __launch_bounds__(256) k_pack_reads(const uint8_t * __restrict__ mapped, const uint64_t * __restrict__ offsets,
                                                  uint64_t nreads, uint32_t W, uint64_t * __restrict__ rpack, uint32_t * __restrict__ bad)
{
        uint64_t const gid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if ( gid >= nreads * 2 * W ) return;
        uint32_t const w = (uint32_t)(gid % W);
        uint64_t const rs = gid / W;
        uint32_t const s = (uint32_t)(rs & 1);
        uint64_t const r = rs >> 1;
        uint64_t const o = offsets[r];
        uint32_t const L = (uint32_t)(offsets[r+1] - o);
        uint64_t word = 0;
        if ( 32 * w < L )
        {
                uint32_t const len = min(32u, L - 32 * w);
                uint32_t anybad = 0;
                if ( s == 0 )
                {
                        word = pack_bytes(mapped + o + 32 * w, len, anybad);
                        if ( anybad ) bad[r] = 1;
                }
                else
                {
                        uint64_t const fwd = pack_bytes(mapped + o + (L - 32 * w - len), len, anybad);
                        word = revcomp_word(fwd >> (64 - 2 * len), len) << (64 - 2 * len);
                }
        }
        rpack[gid] = word;
}

// The same for reads of at most PB_MAX_W words, both strands and the seeds in one pass: one thread per (read, word)
// packs the forward word once; the words of a read are exchanged through shared memory, and word w of the '-' strand
// is cut out of the (at most two) forward words that hold its bases.  Halves the byte loads and the packing work of
// k_pack_reads and replaces k_read_seeds (and the wildcard-flag array in between).
static const uint32_t PB_MAX_W = 64;
__global__ void __launch_bounds__(256) k_pack_both(const uint8_t * __restrict__ mapped, const uint64_t * __restrict__ offsets, uint64_t nreads, uint32_t W,
                                                 uint32_t seedl, uint32_t minlen, uint64_t * __restrict__ rpack, uint32_t * __restrict__ rlen, uint64_t * __restrict__ seeds,
                                                 uint32_t * __restrict__ usable)
{
        __shared__ uint64_t fw[256];
        __shared__ uint32_t sbad[256];
        uint32_t const rpb = 256 / W;                                 // reads per block
        uint32_t const rl = threadIdx.x / W, w = threadIdx.x - rl * W;
        uint64_t const r = (uint64_t)blockIdx.x * rpb + rl;
        bool const active = rl < rpb && r < nreads;
        sbad[threadIdx.x] = 0;
        __syncthreads();
        uint32_t L = 0;
        uint64_t word = 0;
        if ( active )
        {
                uint64_t const o = offsets[r];
                L = (uint32_t)(offsets[r+1] - o);
                if ( 32 * w < L )
                {
                        uint32_t anybad = 0;
                        word = pack_bytes(mapped + o + 32 * w, min(32u, L - 32 * w), anybad);
                        if ( anybad ) sbad[rl] = 1;
                }
                __stcs(rpack + (2 * r) * W + w, word);
        }
        fw[threadIdx.x] = word;
        __syncthreads();
        if ( ! active ) return;
        uint64_t rc = 0;
        if ( 32 * w < L )
        {
                uint32_t const len = min(32u, L - 32 * w);
                uint32_t const b0 = L - 32 * w - len;                  // first base of the stretch whose reverse complement this word is
                uint32_t const a = b0 >> 5, o2 = 2 * (b0 & 31);
                uint64_t const x0 = fw[rl * W + a], x1 = (a + 1 < W) ? fw[rl * W + a + 1] : 0ULL;
                uint64_t const fwd = (o2 ? ((x0 << o2) | (x1 >> (64 - o2))) : x0) >> (64 - 2 * len);
                rc = revcomp_word(fwd, len) << (64 - 2 * len);
        }
        __stcs(rpack + (2 * r + 1) * W + w, rc);
        if ( w == 0 )
        {
                bool const ok = (L >= minlen) && ! sbad[rl];          // minlen = the seed length of the options (>= the indexed seed length)
                rlen[r] = ok ? L : 0;
                usable[r] = ok ? 1 : 0;
                uint64_t const sf = fw[rl * W] >> (64 - 2 * seedl);
                seeds[2*r] = ok ? sf : 0;
                seeds[2*r+1] = ok ? revcomp_word(sf, seedl) : 0;
        }
}

__global__ void __launch_bounds__(256) k_uniform_offsets(uint64_t * __restrict__ offsets, uint64_t nreads, uint32_t L)
{
        uint64_t const i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if ( i <= nreads ) offsets[i] = i * L;
}

__global__ void __launch_bounds__(256) k_flags_to_bad(const uint8_t * __restrict__ flags, uint64_t nreads, uint32_t * __restrict__ bad)
{
        uint64_t const i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if ( i < nreads ) bad[i] = flags[i] ? 1u : 0u;
}

// one thread per read: usable length and the two strand seeds.
// seed word = seedl bases right aligned, fragment 0 in the top bits (what getTextWord(p,seedl) yields for the
// text window the strand is laid over); the '-' seed is the LAST seedl bases of the reverse complement strand
// (RestMatch.hpp:84-89) = the reverse complement of the first seedl bases of the read.
__global__ void __launch_bounds__(256) k_read_seeds(const uint64_t * __restrict__ offsets, uint64_t nreads, uint32_t W, uint32_t seedl, uint32_t minlen,
                                                  const uint64_t * __restrict__ rpack, const uint32_t * __restrict__ bad,
                                                  uint32_t * __restrict__ rlen, uint64_t * __restrict__ seeds, uint32_t * __restrict__ usable)
{
        uint64_t const r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if ( r >= nreads ) return;
        uint32_t const L = (uint32_t)(offsets[r+1] - offsets[r]);
        bool const ok = (L >= minlen) && ! bad[r];
        rlen[r] = ok ? L : 0;
        usable[r] = ok ? 1 : 0;
        uint64_t const sf = rpack[(2*r) * W] >> (64 - 2*seedl);
        seeds[2*r] = ok ? sf : 0;
        seeds[2*r+1] = ok ? revcomp_word(sf, seedl) : 0;
}

// 2 bit/base input (real_gpu_set_reads_packed*): nothing is repacked -- the scan verifies its candidates against the
// caller's bytes (ReadSrc, common.cuh) -- so K1 shrinks to the usable length and the two strand seeds of every read.
// One thread per read; lengths null = all reads have `uniform` bases.
__global__ void __launch_bounds__(256) k_seeds_packed(const uint8_t * __restrict__ packed, const uint64_t * __restrict__ byte_offsets,
                                                    const uint64_t * __restrict__ offsets, const uint32_t * __restrict__ len32, uint32_t uniform, uint64_t nreads, uint32_t seedl, uint32_t minlen,
                                                    const uint32_t * __restrict__ bad, uint32_t * __restrict__ rlen, uint64_t * __restrict__ seeds,
                                                    uint32_t * __restrict__ usable)
{
        uint64_t const r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if ( r >= nreads ) return;
        uint32_t const L = offsets ? (uint32_t)(offsets[r+1] - offsets[r]) : (len32 ? len32[r] : uniform);     // base offsets, lengths, or one length for all
        bool const ok = (L >= minlen) && ! bad[r];
        uint64_t sf = 0;
        if ( ok )
        {
                const uint8_t * p = packed + (byte_offsets ? byte_offsets[r] : r * (uint64_t)((uniform + 3) >> 2));
                sf = packed_bases(p, 0, seedl) >> (64 - 2*seedl);
        }
        rlen[r] = ok ? L : 0;
        usable[r] = ok ? 1 : 0;
        __stcs(seeds + 2*r, sf);
        __stcs(seeds + 2*r + 1, ok ? revcomp_word(sf, seedl) : 0);
}

// ---- K2 --------------------------------------------------------------------------------------

struct TableGeom
{
        uint32_t F;          // bases per fragment
        uint32_t keybits;    // 4F
        uint32_t hb;         // log2 slots
        uint32_t nlists;     // fragment offsets indexed in this table
        int table;           // 0,1,2
};

__device__ __forceinline__ uint64_t pair_key(uint64_t seed, uint32_t F, int a, int b)
{
        if ( F == 8 )
        {
                // -l 32: the four fragments are the four 16-bit fields of the seed; one byte permute puts fragment a over
                // fragment b (bytes 0-3 = low half f2:f3, bytes 4-7 = high half f0:f1; fragment f sits in bytes 7-2f, 6-2f)
                uint32_t const sel = ((7u - 2u * (uint32_t)a) << 12) | ((6u - 2u * (uint32_t)a) << 8) | ((7u - 2u * (uint32_t)b) << 4) | (6u - 2u * (uint32_t)b);
                return __byte_perm((uint32_t)seed, (uint32_t)(seed >> 32), sel);
        }
        uint64_t const fm = (F == 32) ? ~0ULL : ((1ULL << (2*F)) - 1);
        uint64_t const ma = (seed >> (2*F*(3-a))) & fm;
        uint64_t const mb = (seed >> (2*F*(3-b))) & fm;
        return (ma << (2*F)) | mb;
}

// The table build does not sort and uses no global atomics on the table itself.
//  (1) The entries of a table -- (strand seed, strand id, fragment offset), nlists per usable read strand -- are
//      grouped by the top e1 <= 8 bits of their slot with one staged partition pass (histogram, then a scatter
//      that lays the records out bucket by bucket in shared memory and writes whole runs),
//  (2) and each of those buckets again by the next e2 <= 8 bits, which leaves sub-buckets of a few thousand
//      entries whose slots span at most 2^16 slots = 2048 slot words.
//  (3) One CTA per sub-bucket then builds that piece of the table in shared memory: presence bits, ranks
//      (popcount scan), and the claim of E[rank] by the first entry of a slot; same-slot entries go behind the
//      distinct ones of the same sub-bucket and are chained through `next`.  E is addressed by "first grouped
//      entry of the sub-bucket + rank inside it", so no device-wide rank scan is needed, E holds exactly one
//      element per entry, and every global store of the build is part of a dense range.
// Measured before this layout (entries claimed with global CAS into bucket-sized slices of a 2x over-allocated,
// memset E): 45 of the 55 ms of the C3 index build were the bit / claim kernels waiting on random DRAM sectors.
static const int EP_IDS_PER_THREAD = 4;
static const int EP_TILE_IDS = 256 * EP_IDS_PER_THREAD;       // strand ids per tile
static const int EP_TILE_ENTRIES = EP_TILE_IDS * 3;
static const int EP_MAX_BUCKETS = 256;
static const int EP_CURSOR_STRIDE = 32;
static const uint32_t SUB_MAX_WORDS = 2048;                   // slot words of one sub-bucket (shared-memory arrays of k_build_sub)
static const uint32_t SUB_TARGET_ENTRIES = 4096;

struct EntryPartParams
{
        const uint64_t * seeds;       // 2*nreads strand seeds
        const uint32_t * usable;      // nreads
        uint64_t nids;                // 2*nreads
        TableGeom G;
        uint32_t ebits;               // level 1: bucket = slot >> (hb - ebits)
        uint32_t e2bits;              // level 2: sub-bucket = (slot >> (hb - ebits - e2bits)) & (2^e2bits - 1)
        uint64_t * ent_seed;          // level 1 output
        uint32_t * ent_val;
        uint64_t * ent2_seed;         // level 2 output
        uint32_t * ent2_val;
        uint32_t * bucket_count;      // [256]
        uint32_t * bucket_start;      // [257]
        uint32_t * bucket_cursor;     // [256 * EP_CURSOR_STRIDE]
        uint32_t * tile_start;        // [257] level 2: first tile of a level-1 bucket
        uint32_t * sub_count;         // [2^(ebits+e2bits)]
        uint32_t * sub_start;         // [2^(ebits+e2bits) + 1]
        uint32_t * sub_cursor;        // [2^(ebits+e2bits)]
        // sharded tables: this rank indexes only the entries with own_lo <= slot >> own_shift <= own_last
        uint32_t own_shift, own_lo, own_last;
};

__device__ __forceinline__ bool entry_owned(EntryPartParams const & P, uint32_t slot)
{
        uint32_t const p = slot >> P.own_shift;
        return p >= P.own_lo && p <= P.own_last;
}

// G.table == TABLE_ITEMS: the geometry of the fused build (build_tables_fused, real_gpu.cu).  When the slots are the keys
// themselves (hb == keybits), the slot of entry (table, t) starts with fragment t of the seed whatever the table is, so
// the entries (A,t), (B,t), (C,t) of a strand fall into the same bucket at every partition level of at most 2F bits: the
// build partitions ITEMS (strand, t) -- half as many as there are entries -- and only the sub-bucket kernel tells the
// tables apart.  The "slot" of an item is fragment t followed by zeros.
static const int TABLE_ITEMS = 3;
__device__ __forceinline__ uint32_t entry_slot(uint64_t seed, TableGeom const & G, uint32_t t)
{
        if ( G.table == TABLE_ITEMS )
        {
                uint32_t const fb = 2 * G.F;
                return (uint32_t)((seed >> (fb * (3 - t))) & ((1ULL << fb) - 1)) << (G.hb - fb);
        }
        return slot_of(pair_key(seed, G.F, (int)t, pair_second(G.table, (int)t)), G.keybits, G.hb);
}

// level-1 histograms of all three tables in one pass over the seeds (P[t].G.nlists == 0: table not built)
struct EntryPartParams3 { EntryPartParams P[3]; };
__global__ void __launch_bounds__(256) k_ent_hist3(const __grid_constant__ EntryPartParams3 Q)
{
        __shared__ uint32_t cnt[3][EP_MAX_BUCKETS];
        #pragma unroll
        for ( int t = 0; t < 3; ++t ) cnt[t][threadIdx.x] = 0;
        __syncthreads();
        EntryPartParams const & P0 = Q.P[0];
        uint64_t const stride = (uint64_t)gridDim.x * blockDim.x;
        for ( uint64_t id0 = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; id0 < P0.nids; id0 += 4 * stride )
        {
                uint64_t seed[4];
                bool ok[4];
                #pragma unroll
                for ( int k = 0; k < 4; ++k )
                {
                        uint64_t const id = id0 + (uint64_t)k * stride;
                        ok[k] = id < P0.nids;
                        seed[k] = ok[k] ? __ldcs(P0.seeds + id) : 0;
                        ok[k] = ok[k] && __ldg(P0.usable + (id >> 1));
                }
                #pragma unroll
                for ( int k = 0; k < 4; ++k )
                        if ( ok[k] )
                        {
                                #pragma unroll
                                for ( int tb = 0; tb < 3; ++tb )
                                {
                                        EntryPartParams const & P = Q.P[tb];
                                        uint32_t const sh = P.G.hb - P.ebits;
                                        for ( uint32_t t = 0; t < P.G.nlists; ++t )
                                        {
                                                uint32_t const slot = entry_slot(seed[k], P.G, t);
                                                if ( entry_owned(P, slot) ) atomicAdd(&cnt[tb][P.ebits ? (slot >> sh) : 0u], 1u);
                                        }
                                }
                        }
        }
        __syncthreads();
        #pragma unroll
        for ( int tb = 0; tb < 3; ++tb )
                if ( Q.P[tb].G.nlists && cnt[tb][threadIdx.x] ) atomicAdd(Q.P[tb].bucket_count + threadIdx.x, cnt[tb][threadIdx.x]);
}

// bucket starts, cursors, and the level-2 tiling (tiles never straddle a level-1 bucket)
__global__ void __launch_bounds__(EP_MAX_BUCKETS) k_ent_offsets(EntryPartParams P, uint32_t * total)
{
        __shared__ uint32_t sc[EP_MAX_BUCKETS];
        sc[threadIdx.x] = P.bucket_count[threadIdx.x];
        __syncthreads();
        if ( threadIdx.x == 0 )
        {
                uint32_t a = 0, tl = 0;
                for ( int b = 0; b < EP_MAX_BUCKETS; ++b )
                {
                        P.bucket_start[b] = a; a += sc[b];
                        P.tile_start[b] = tl; tl += (sc[b] + EP_TILE_ENTRIES - 1) / EP_TILE_ENTRIES;
                }
                P.bucket_start[EP_MAX_BUCKETS] = a;
                P.tile_start[EP_MAX_BUCKETS] = tl;
                *total = a;
        }
        P.bucket_cursor[threadIdx.x * EP_CURSOR_STRIDE] = 0;
}

struct EntryPartSmem
{
        uint64_t stage_seed[EP_TILE_ENTRIES];
        uint32_t stage_val[EP_TILE_ENTRIES];
        uint32_t wcnt[8][EP_MAX_BUCKETS];
        uint32_t loc[EP_MAX_BUCKETS + 1];
        uint32_t base[EP_MAX_BUCKETS];
        uint32_t wsum[8];
        uint8_t stage_b[EP_TILE_ENTRIES];
};

// steps (2) and (4) of a staged 256-way scatter tile, shared by both levels: turn the per-warp counts into the
// staging layout, reserve the tile's run in every bucket (cursor stride cs), and after the multisplit copy the
// staged entries out run by run
// returns the first output index of the tile's run in bucket threadIdx.x: the caller stores it to S.base after the
// multisplit, so that the global atomic behind it is in flight while the tile is ranked
// (as two addends: adding them here would make the thread wait for the atomic's round trip on the spot)
__device__ __forceinline__ uint2 ep_layout(EntryPartSmem & S, const uint32_t * __restrict__ start, uint32_t * __restrict__ cursor, uint32_t cs)
{
        uint32_t tot = 0;
        #pragma unroll
        for ( int w = 0; w < 8; ++w ) tot += S.wcnt[w][threadIdx.x];
        uint32_t blocktot;
        uint32_t const ex = block_excl_scan256(tot, &blocktot, S.wsum);        // (one barrier; every tile has more behind it)
        S.loc[threadIdx.x] = ex;
        if ( threadIdx.x == EP_MAX_BUCKETS - 1 ) S.loc[EP_MAX_BUCKETS] = blocktot;
        uint2 basev = make_uint2(0u, 0u);
        if ( tot )
        {
                basev.x = start[threadIdx.x];
                basev.y = atomicAdd(cursor + threadIdx.x * cs, tot);
        }
        uint32_t run = ex;
        #pragma unroll
        for ( int w = 0; w < 8; ++w )
        {
                uint32_t const c = S.wcnt[w][threadIdx.x];
                S.wcnt[w][threadIdx.x] = run;
                run += c;
        }
        return basev;
}
__device__ __forceinline__ void ep_place(EntryPartSmem & S, int wid, uint32_t lt, bool ok, uint32_t b, uint64_t seed, uint32_t val)
{
        uint32_t const peers = peers_u8(b, ok);
        uint32_t const below = __popc(peers & lt);
        uint32_t pre = 0;
        if ( ok ) pre = S.wcnt[wid][b];
        __syncwarp();
        if ( ok && below == 0 ) S.wcnt[wid][b] = pre + __popc(peers);
        __syncwarp();
        if ( ok )
        {
                uint32_t const slot = pre + below;
                S.stage_seed[slot] = seed;
                S.stage_val[slot] = val;
                S.stage_b[slot] = (uint8_t)b;
        }
}
__device__ __forceinline__ void ep_copy_out(EntryPartSmem & S, uint64_t * __restrict__ out_seed, uint32_t * __restrict__ out_val)
{
        // S.base[b] holds "first output index of the run - first staging slot of the bucket" (mod 2^32), so an entry costs one
        // dependent shared-memory load; four entries are in flight per thread
        uint32_t const n = S.loc[EP_MAX_BUCKETS];
        uint32_t i = threadIdx.x;
        for ( ; i + 3 * 256 < n; i += 4 * 256 )
        {
                uint32_t o[4]; uint64_t sd[4]; uint32_t vl[4];
                #pragma unroll
                for ( int u = 0; u < 4; ++u ) { o[u] = S.stage_b[i + u * 256]; sd[u] = S.stage_seed[i + u * 256]; vl[u] = S.stage_val[i + u * 256]; }
                #pragma unroll
                for ( int u = 0; u < 4; ++u ) o[u] = S.base[o[u]] + (i + u * 256);
                #pragma unroll
                for ( int u = 0; u < 4; ++u ) { out_seed[o[u]] = sd[u]; out_val[o[u]] = vl[u]; }
        }
        for ( ; i < n; i += 256 )
        {
                uint32_t const o = S.base[S.stage_b[i]] + i;
                out_seed[o] = S.stage_seed[i];
                out_val[o] = S.stage_val[i];
        }
}

// level 1: strand seeds -> entries grouped by the top ebits of their slot
__global__ void __launch_bounds__(256) k_ent_scatter(EntryPartParams P)
{
        extern __shared__ __align__(16) unsigned char ep_smem[];
        EntryPartSmem & S = *reinterpret_cast<EntryPartSmem *>(ep_smem);
        int const lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
        uint32_t const lt = (1u << lane) - 1;
        uint32_t const sh = P.G.hb - P.ebits;
        uint32_t const nl = P.G.nlists;
        #pragma unroll
        for ( int w = 0; w < 8; ++w ) S.wcnt[w][threadIdx.x] = 0;
        __syncthreads();

        uint64_t const ntiles = (P.nids + EP_TILE_IDS - 1) / EP_TILE_IDS;
        // the seeds of the next tile are fetched while the current one is ranked
        uint64_t seedn[EP_IDS_PER_THREAD];
        uint32_t usen[EP_IDS_PER_THREAD];
        #pragma unroll
        for ( int k = 0; k < EP_IDS_PER_THREAD; ++k )
        {
                uint64_t const id = (uint64_t)blockIdx.x * EP_TILE_IDS + (uint64_t)k * 256 + threadIdx.x;
                seedn[k] = (id < P.nids) ? __ldcs(P.seeds + id) : 0;
                usen[k] = (id < P.nids) ? __ldg(P.usable + (id >> 1)) : 0u;
        }
        for ( uint64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x )
        {
                uint64_t seed[EP_IDS_PER_THREAD];
                bool ok[EP_IDS_PER_THREAD];
                #pragma unroll
                for ( int k = 0; k < EP_IDS_PER_THREAD; ++k )
                {
                        seed[k] = seedn[k];
                        ok[k] = usen[k] != 0;
                        uint64_t const idn = (tile + gridDim.x) * EP_TILE_IDS + (uint64_t)k * 256 + threadIdx.x;
                        seedn[k] = (idn < P.nids) ? __ldcs(P.seeds + idn) : 0;
                        usen[k] = (idn < P.nids) ? __ldg(P.usable + (idn >> 1)) : 0u;
                }
                // (1) per-warp bucket counts
                #pragma unroll
                for ( int k = 0; k < EP_IDS_PER_THREAD; ++k )
                        if ( ok[k] )
                                for ( uint32_t t = 0; t < nl; ++t )
                                {
                                        uint32_t const slot = entry_slot(seed[k], P.G, t);
                                        if ( entry_owned(P, slot) ) atomicAdd(&S.wcnt[wid][P.ebits ? (slot >> sh) : 0u], 1u);
                                }
                __syncthreads();
                // (2) staging layout, global run reservation, per-warp running slots
                uint2 const basev = ep_layout(S, P.bucket_start, P.bucket_cursor, EP_CURSOR_STRIDE);
                __syncthreads();
                // (3) warp multisplit into the staging area
                #pragma unroll
                for ( int k = 0; k < EP_IDS_PER_THREAD; ++k )
                {
                        uint64_t const id = tile * EP_TILE_IDS + (uint64_t)k * 256 + threadIdx.x;
                        for ( uint32_t t = 0; t < nl; ++t )
                        {
                                uint32_t const slot = ok[k] ? entry_slot(seed[k], P.G, t) : 0u;
                                uint32_t const b = (ok[k] && P.ebits) ? (slot >> sh) : 0u;
                                ep_place(S, wid, lt, ok[k] && entry_owned(P, slot), b, seed[k], (uint32_t)(id << 2) | t);
                        }
                }
                S.base[threadIdx.x] = basev.x + basev.y - S.loc[threadIdx.x];
                __syncthreads();
                // (4) copy out run by run
                ep_copy_out(S, P.ent_seed, P.ent_val);
                __syncthreads();
                #pragma unroll
                for ( int w = 0; w < 8; ++w ) S.wcnt[w][threadIdx.x] = 0;
                __syncthreads();
        }
}

// level 1 of a bucket shard (real_gpu_set_bucket_shard / sharded tables): only the entries whose slot belongs to this
// rank are kept, 1/nranks of them.  Computing and testing a slot is cheap, ranking and staging an entry is not, so the
// kept entries are first compacted into a shared-memory list, which is ranked and written out EP_TILE_ENTRIES at a
// time with full warps (the same scheme as k_part_scatter_own in scan.cuh).
static const int EO_IDS_PER_THREAD = 2;
static const int EO_TILE_IDS = 256 * EO_IDS_PER_THREAD;
static const int EO_FLUSH = EP_TILE_ENTRIES - 256;
static const int EO_LIST_CAP = EO_FLUSH + EO_TILE_IDS * 3;

struct EntryOwnSmem
{
        EntryPartSmem P;
        uint64_t list_seed[EO_LIST_CAP];
        uint32_t list_val[EO_LIST_CAP];
        uint32_t add[4];
        uint8_t list_b[EO_LIST_CAP];
};

__device__ __forceinline__ void eo_flush(EntryPartParams const & P, EntryOwnSmem & SO, uint32_t first, uint32_t n)
{
        EntryPartSmem & S = SO.P;
        int const lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
        uint32_t const lt = (1u << lane) - 1;
        uint64_t seed[EP_TILE_ENTRIES / 256];
        uint32_t val[EP_TILE_ENTRIES / 256], b[EP_TILE_ENTRIES / 256];
        #pragma unroll
        for ( int k = 0; k < EP_TILE_ENTRIES / 256; ++k )
        {
                uint32_t const i = (uint32_t)k * 256 + threadIdx.x;
                bool const ok = i < n;
                seed[k] = ok ? SO.list_seed[first + i] : 0;
                val[k] = ok ? SO.list_val[first + i] : 0;
                b[k] = ok ? SO.list_b[first + i] : 0;
                if ( ok ) atomicAdd(&S.wcnt[wid][b[k]], 1u);
        }
        __syncthreads();
        uint2 const basev = ep_layout(S, P.bucket_start, P.bucket_cursor, EP_CURSOR_STRIDE);
        __syncthreads();
        #pragma unroll
        for ( int k = 0; k < EP_TILE_ENTRIES / 256; ++k )
                ep_place(S, wid, lt, (uint32_t)k * 256 + threadIdx.x < n, b[k], seed[k], val[k]);
        S.base[threadIdx.x] = basev.x + basev.y - S.loc[threadIdx.x];
        __syncthreads();
        ep_copy_out(S, P.ent_seed, P.ent_val);
        __syncthreads();
        #pragma unroll
        for ( int w = 0; w < 8; ++w ) S.wcnt[w][threadIdx.x] = 0;
        __syncthreads();
}

__global__ void __launch_bounds__(256, 2) k_ent_scatter_own(EntryPartParams P)
{
        extern __shared__ __align__(16) unsigned char ep_smem[];
        EntryOwnSmem & SO = *reinterpret_cast<EntryOwnSmem *>(ep_smem);
        int const lane = threadIdx.x & 31;
        uint32_t const sh = P.G.hb - P.ebits;
        uint32_t const nl = P.G.nlists;
        #pragma unroll
        for ( int w = 0; w < 8; ++w ) SO.P.wcnt[w][threadIdx.x] = 0;
        if ( threadIdx.x < 4 ) SO.add[threadIdx.x] = 0;
        __syncthreads();
        uint32_t n = 0, step = 0;

        uint64_t const ntiles = (P.nids + EO_TILE_IDS - 1) / EO_TILE_IDS;
        // the seeds of the next tile are fetched while the current one is worked on (two CTAs per SM do not hide the latency)
        uint64_t seedn[EO_IDS_PER_THREAD];
        uint32_t usen[EO_IDS_PER_THREAD];
        #pragma unroll
        for ( int k = 0; k < EO_IDS_PER_THREAD; ++k )
        {
                uint64_t const id = (uint64_t)blockIdx.x * EO_TILE_IDS + (uint64_t)k * 256 + threadIdx.x;
                seedn[k] = (id < P.nids) ? __ldcs(P.seeds + id) : 0;
                usen[k] = (id < P.nids) ? __ldg(P.usable + (id >> 1)) : 0u;
        }
        for ( uint64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++step )
        {
                uint64_t seed[EO_IDS_PER_THREAD];
                uint32_t slot[EO_IDS_PER_THREAD][3];
                bool okk[EO_IDS_PER_THREAD];
                uint32_t own = 0;                      // bit k*3+t: entry t of id k is kept
                #pragma unroll
                for ( int k = 0; k < EO_IDS_PER_THREAD; ++k )
                {
                        seed[k] = seedn[k];
                        okk[k] = usen[k] != 0;
                        uint64_t const idn = (tile + gridDim.x) * EO_TILE_IDS + (uint64_t)k * 256 + threadIdx.x;
                        seedn[k] = (idn < P.nids) ? __ldcs(P.seeds + idn) : 0;
                        usen[k] = (idn < P.nids) ? __ldg(P.usable + (idn >> 1)) : 0u;
                }
                #pragma unroll
                for ( int k = 0; k < EO_IDS_PER_THREAD; ++k )
                {
                        bool const ok = okk[k];
                        #pragma unroll
                        for ( uint32_t t = 0; t < 3; ++t )
                        {
                                slot[k][t] = (ok && t < nl) ? entry_slot(seed[k], P.G, t) : 0u;
                                if ( ok && t < nl && entry_owned(P, slot[k][t]) ) own |= 1u << (k * 3 + t);
                        }
                }
                uint32_t const c = __popc(own);
                uint32_t const incl = warp_incl_scan(c, lane);
                uint32_t wbase = 0;
                if ( lane == 31 && incl ) wbase = atomicAdd(&SO.add[step % 3], incl);
                wbase = __shfl_sync(0xffffffffu, wbase, 31);
                uint32_t o = n + wbase + incl - c;
                #pragma unroll
                for ( int k = 0; k < EO_IDS_PER_THREAD; ++k )
                {
                        uint64_t const id = tile * EO_TILE_IDS + (uint64_t)k * 256 + threadIdx.x;
                        #pragma unroll
                        for ( uint32_t t = 0; t < 3; ++t )
                                if ( (own >> (k * 3 + t)) & 1u )
                                {
                                        SO.list_seed[o] = seed[k];
                                        SO.list_val[o] = (uint32_t)(id << 2) | t;
                                        SO.list_b[o] = (uint8_t)(P.ebits ? (slot[k][t] >> sh) : 0u);
                                        ++o;
                                }
                }
                if ( threadIdx.x == 0 ) SO.add[(step + 1) % 3] = 0;
                __syncthreads();
                n += SO.add[step % 3];
                bool const last = tile + gridDim.x >= ntiles;
                while ( n >= (uint32_t)EO_FLUSH || (last && n) )
                {
                        uint32_t const take = min(n, (uint32_t)EP_TILE_ENTRIES);
                        eo_flush(P, SO, n - take, take);
                        n -= take;
                }
        }
}

// level 2 tiling: tile -> (level-1 bucket, first entry, entries)
__device__ __forceinline__ void ep2_tile(EntryPartParams const & P, uint32_t tile, uint32_t & b, uint32_t & first, uint32_t & n)
{
        uint32_t lo = 0, hi = 1u << P.ebits;                 // last bucket with tile_start <= tile
        while ( hi - lo > 1 )
        {
                uint32_t const mid = (lo + hi) >> 1;
                if ( P.tile_start[mid] <= tile ) lo = mid; else hi = mid;
        }
        b = lo;
        first = P.bucket_start[b] + (tile - P.tile_start[b]) * EP_TILE_ENTRIES;
        n = min((uint32_t)EP_TILE_ENTRIES, P.bucket_start[b+1] - first);
}

__global__ void __launch_bounds__(256) k_ent2_hist(EntryPartParams P)
{
        __shared__ uint32_t cnt[EP_MAX_BUCKETS];
        uint32_t const ntiles = P.tile_start[1u << P.ebits];
        uint32_t const sh = P.G.hb - P.ebits - P.e2bits, smask = (1u << P.e2bits) - 1;
        for ( uint32_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x )
        {
                uint32_t b, first, n;
                ep2_tile(P, tile, b, first, n);
                cnt[threadIdx.x] = 0;
                __syncthreads();
                for ( uint32_t i = threadIdx.x; i < n; i += 256 )
                        atomicAdd(&cnt[(entry_slot(__ldcs(P.ent_seed + first + i), P.G, __ldcs(P.ent_val + first + i) & 3) >> sh) & smask], 1u);
                __syncthreads();
                if ( threadIdx.x <= smask && cnt[threadIdx.x] ) atomicAdd(P.sub_count + ((b << P.e2bits) | threadIdx.x), cnt[threadIdx.x]);
                __syncthreads();
        }
}

// level 2: the entries of every level-1 bucket grouped again by the next e2bits of their slot
__global__ void __launch_bounds__(256, 4) k_ent2_scatter(EntryPartParams P)
{
        extern __shared__ __align__(16) unsigned char ep_smem[];
        EntryPartSmem & S = *reinterpret_cast<EntryPartSmem *>(ep_smem);
        int const lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
        uint32_t const lt = (1u << lane) - 1;
        uint32_t const ntiles = P.tile_start[1u << P.ebits];
        uint32_t const sh = P.G.hb - P.ebits - P.e2bits, smask = (1u << P.e2bits) - 1;
        #pragma unroll
        for ( int w = 0; w < 8; ++w ) S.wcnt[w][threadIdx.x] = 0;
        __syncthreads();
        for ( uint32_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x )
        {
                uint32_t b, first, n;
                ep2_tile(P, tile, b, first, n);
                uint64_t seed[EP_TILE_ENTRIES / 256];
                uint32_t val[EP_TILE_ENTRIES / 256];
                #pragma unroll
                for ( int k = 0; k < EP_TILE_ENTRIES / 256; ++k )
                {
                        uint32_t const i = (uint32_t)k * 256 + threadIdx.x;
                        seed[k] = (i < n) ? __ldcs(P.ent_seed + first + i) : 0;
                        val[k] = (i < n) ? __ldcs(P.ent_val + first + i) : 0;
                }
                #pragma unroll
                for ( int k = 0; k < EP_TILE_ENTRIES / 256; ++k )
                        if ( (uint32_t)k * 256 + threadIdx.x < n )
                                atomicAdd(&S.wcnt[wid][(entry_slot(seed[k], P.G, val[k] & 3) >> sh) & smask], 1u);
                __syncthreads();
                uint2 const basev = ep_layout(S, P.sub_start + (b << P.e2bits), P.sub_cursor + (b << P.e2bits), 1);
                __syncthreads();
                #pragma unroll
                for ( int k = 0; k < EP_TILE_ENTRIES / 256; ++k )
                {
                        bool const ok = (uint32_t)k * 256 + threadIdx.x < n;
                        ep_place(S, wid, lt, ok, (entry_slot(seed[k], P.G, val[k] & 3) >> sh) & smask, seed[k], val[k]);
                }
                S.base[threadIdx.x] = basev.x + basev.y - S.loc[threadIdx.x];
                __syncthreads();
                ep_copy_out(S, P.ent2_seed, P.ent2_val);
                __syncthreads();
                #pragma unroll
                for ( int w = 0; w < 8; ++w ) S.wcnt[w][threadIdx.x] = 0;
                __syncthreads();
        }
}

// One CTA per sub-bucket: the grouped entries [sub_start[sb], sub_start[sb+1]) all have slots in
// [sb << sub_shift, (sb+1) << sub_shift), i.e. `words` = max(1, 2^sub_shift / 32) slot words.  Dynamic shared
// memory: 3 * words u32 (presence bits, rank of the word's first slot, claimed bits).
static const uint32_t SUB_DUP_CAP = 512;       // same-slot entries of a sub-bucket that are chained in one go (more are chained one by one)
struct SubDup { uint64_t seed; uint32_t val; uint32_t r; };

__global__ void __launch_bounds__(256, 7) k_build_sub(const uint64_t * __restrict__ ent_seed, const uint32_t * __restrict__ ent_val, const uint32_t * __restrict__ sub_start,
                                                 TableGeom G, uint32_t sub_shift, uint32_t words, SlotWord * __restrict__ slots, Entry * __restrict__ E,
                                                 uint32_t * __restrict__ ndistinct, uint32_t first_sub)
{
        extern __shared__ __align__(16) uint32_t sub_smem[];
        uint32_t * bits = sub_smem, * rank = sub_smem + words, * claimed = sub_smem + 2 * words;
        __shared__ SubDup dup[SUB_DUP_CAP];
        __shared__ uint32_t ovf, ndup;
        uint32_t const sb = first_sub + blockIdx.x;
        uint32_t const s0 = sub_start[sb], s1 = sub_start[sb+1];
        uint32_t const slot0 = sb << sub_shift;                    // sub_shift == hb when there is a single sub-bucket (sb == 0)
        for ( uint32_t w = threadIdx.x; w < words; w += 256 ) { bits[w] = 0; claimed[w] = 0; }
        if ( threadIdx.x == 0 ) { ovf = 0; ndup = 0; }
        __syncthreads();
        // presence bits; four entries per thread and step, their loads issued together
        for ( uint32_t i0 = s0 + threadIdx.x; i0 < s1; i0 += 1024 )
        {
                uint64_t seed[4]; uint32_t val[4];
                #pragma unroll
                for ( int k = 0; k < 4; ++k )
                {
                        uint32_t const i = i0 + (uint32_t)k * 256;
                        seed[k] = (i < s1) ? __ldg(ent_seed + i) : 0;
                        val[k] = (i < s1) ? __ldg(ent_val + i) : 0;
                }
                #pragma unroll
                for ( int k = 0; k < 4; ++k )
                        if ( i0 + (uint32_t)k * 256 < s1 )
                        {
                                uint32_t const l = entry_slot(seed[k], G, val[k] & 3) - slot0;
                                atomicOr(&bits[l >> 5], 1u << (l & 31));
                        }
        }
        __syncthreads();
        // ranks: every thread owns a run of consecutive words
        uint32_t const wpt = (words + 255) / 256;
        uint32_t const w0 = threadIdx.x * wpt;
        uint32_t c = 0;
        for ( uint32_t w = w0; w < min(words, w0 + wpt); ++w ) c += __popc(bits[w]);
        uint32_t d;
        uint32_t run = s0 + block_excl_scan(c, &d);
        for ( uint32_t w = w0; w < min(words, w0 + wpt); ++w ) { rank[w] = run; run += __popc(bits[w]); }
        __syncthreads();
        for ( uint32_t w = threadIdx.x; w < words; w += 256 )
        {
                SlotWord sw; sw.bits = bits[w]; sw.rank = rank[w];
                slots[(uint64_t)sb * words + w] = sw;
        }
        for ( uint32_t r = threadIdx.x; r < d; r += 256 ) E[s0 + r].next = ENTRY_NONE;
        if ( threadIdx.x == 0 && d ) atomicAdd(ndistinct, d);
        __syncthreads();
        // entries: the first one of a slot claims E[rank]; the others (few: the tables are sparse) are set aside and chained
        // below by full warps -- chaining them where they are found leaves two or three lanes of a warp waiting for a
        // global atomic each time
        for ( uint32_t i0 = s0 + threadIdx.x; i0 < s1; i0 += 1024 )
        {
                uint64_t seed[4]; uint32_t val[4];
                #pragma unroll
                for ( int k = 0; k < 4; ++k )
                {
                        uint32_t const i = i0 + (uint32_t)k * 256;
                        seed[k] = (i < s1) ? __ldg(ent_seed + i) : 0;
                        val[k] = (i < s1) ? __ldg(ent_val + i) : 0;
                }
                #pragma unroll
                for ( int k = 0; k < 4; ++k )
                        if ( i0 + (uint32_t)k * 256 < s1 )
                        {
                                uint32_t const l = entry_slot(seed[k], G, val[k] & 3) - slot0;
                                uint32_t const bit = 1u << (l & 31);
                                uint32_t const r = rank[l >> 5] + __popc(bits[l >> 5] & (bit - 1));
                                if ( ! (atomicOr(&claimed[l >> 5], bit) & bit) )
                                {
                                        E[r].seed = seed[k];
                                        E[r].val = val[k];
                                }
                                else
                                {
                                        uint32_t const j = atomicAdd(&ndup, 1u);
                                        if ( j < SUB_DUP_CAP )
                                        {
                                                SubDup dd; dd.seed = seed[k]; dd.val = val[k]; dd.r = r;
                                                dup[j] = dd;
                                        }
                                        else
                                        {
                                                uint32_t const o = s0 + d + SUB_DUP_CAP + atomicAdd(&ovf, 1u);
                                                Entry en; en.seed = seed[k]; en.val = val[k];
                                                en.next = atomicExch(&E[r].next, o);
                                                E[o] = en;
                                        }
                                }
                        }
        }
        __syncthreads();
        // the set-aside entries go behind the distinct ones of this sub-bucket, in list order
        uint32_t const nd = min(ndup, SUB_DUP_CAP);
        for ( uint32_t j = threadIdx.x; j < nd; j += 256 )
        {
                SubDup const dd = dup[j];
                uint32_t const o = s0 + d + j;
                Entry en; en.seed = dd.seed; en.val = dd.val;
                en.next = atomicExch(&E[dd.r].next, o);
                E[o] = en;
        }
}

// The sub-bucket kernel of the fused build: the grouped ITEMS [sub_start[sb], sub_start[sb+1]) all carry a fragment t that
// starts with the prefix sb, so for every table the slots of their entries lie in [sb << sub_shift, (sb+1) << sub_shift).
// Three CTAs build that piece of the three tables, one each: item (strand, t) is an entry of table tb when t < nl[tb] (A: pairs
// (t,t+1), B: (t,t+2), C: (t,t+3)).  The entry arrays of the three tables use the ITEM numbering: the entries of a sub-bucket sit at
// the front of E[tb][sub_start[sb] ...) -- no per-table offsets are needed; B and C leave the tail of each range unused.
// Dynamic shared memory: presence bits and claimed bits (words u32 each) and the ranks of the words' first slots
// (words u16, relative to the sub-bucket: a sub-bucket spans at most 2^16 slots).
static const uint32_t SUB3_DUP_CAP = 256;
struct Build3Params
{
        const uint64_t * item_seed; const uint32_t * item_val; const uint32_t * sub_start;
        TableGeom G[3];                 // G[tb].nlists == 0: table not built
        uint32_t sub_shift, words, first_sub;
        SlotWord * slots[3]; Entry * E[3];
        uint32_t * ndistinct[3];
};

// One CTA per (sub-bucket, table) -- a third of the shared memory and fewer registers per CTA than one CTA for all three
// tables, so that enough CTAs are resident to hide the latencies of a kernel that is a chain of short phases (items -> presence
// bits -> ranks -> heads)
// FAST: -l 32 (fragments of 8 bases, 2^32 slots, sub-buckets of 2^16 slots): the slot of an entry relative to its sub-bucket is
// simply the second fragment of its pair, one 16-bit field of the seed -- the general path (entry_slot) spends some twenty
// instructions per entry and pass on runtime geometry
template<bool FAST>
__device__ __forceinline__ uint32_t sub_local_slot(uint64_t seed, TableGeom const & G, uint32_t t, int tb, uint32_t slot0)
{
        if ( FAST )
                return (uint32_t)(seed >> (16u * (2u - t - (uint32_t)tb))) & 0xFFFFu;
        return entry_slot(seed, G, t) - slot0;
}

static const int BUILD3_MINB = 6;                               // CTAs per SM of k_build_sub3 (register bound)
template<bool FAST>
__global__ void __launch_bounds__(256, BUILD3_MINB) k_build_sub3(const __grid_constant__ Build3Params P)
{
        extern __shared__ __align__(16) uint32_t sub_smem[];
        uint32_t const words = P.words;
        __shared__ SubDup dup[SUB3_DUP_CAP];
        __shared__ uint32_t ndup, dist;
        uint32_t const sb = P.first_sub + blockIdx.x / 3;
        int const tb = (int)(blockIdx.x % 3);
        TableGeom const & G = P.G[tb];
        if ( ! G.nlists ) return;
        uint32_t const s0 = P.sub_start[sb], s1 = P.sub_start[sb+1];
        uint32_t const slot0 = sb << P.sub_shift;
        // presence bits, claimed bits (u32 each), ranks (u16, relative to s0)
        uint32_t * bits = sub_smem, * claimed = bits + words;
        uint16_t * rank = reinterpret_cast<uint16_t *>(bits + 2 * words);
        // the items of the sub-bucket (some 55 KB) are pulled into L2 while the shared memory is cleared: the two passes below
        // wait for their item loads more than for anything else (a third of the stall samples), four loads per thread at a time
        for ( uint32_t i = s0 + threadIdx.x * 16; i < s1; i += 256 * 16 )
        {
                asm volatile("prefetch.global.L2 [%0];" :: "l"(P.item_seed + i));
                if ( ((i - s0) & 31) == 0 ) asm volatile("prefetch.global.L2 [%0];" :: "l"(P.item_val + i));
        }
        for ( uint32_t w = threadIdx.x; w < 2 * words + (words + 1) / 2; w += 256 ) sub_smem[w] = 0;
        if ( threadIdx.x == 0 ) ndup = 0;
        __syncthreads();
        // presence bits; four items per thread and step, their loads issued together
        for ( uint32_t i0 = s0 + threadIdx.x; i0 < s1; i0 += 1024 )
        {
                uint64_t seed[4]; uint32_t val[4];
                #pragma unroll
                for ( int k = 0; k < 4; ++k )
                {
                        uint32_t const i = i0 + (uint32_t)k * 256;
                        seed[k] = (i < s1) ? __ldg(P.item_seed + i) : 0;
                        val[k] = (i < s1) ? __ldg(P.item_val + i) : 0;
                }
                #pragma unroll
                for ( int k = 0; k < 4; ++k )
                        if ( i0 + (uint32_t)k * 256 < s1 )
                        {
                                uint32_t const t = val[k] & 3;
                                if ( t < G.nlists )
                                {
                                        uint32_t const l = sub_local_slot<FAST>(seed[k], G, t, tb, slot0);
                                        atomicOr(&bits[l >> 5], 1u << (l & 31));
                                }
                        }
        }
        __syncthreads();
        // ranks: every thread owns a run of consecutive words
        {
                uint32_t const wpt = (words + 255) / 256;
                uint32_t const w0 = threadIdx.x * wpt;
                uint32_t c = 0;
                for ( uint32_t w = w0; w < min(words, w0 + wpt); ++w ) c += __popc(bits[w]);
                uint32_t d;
                uint32_t run = block_excl_scan(c, &d);                    // < 2^16: a sub-bucket spans at most 2^16 slots
                for ( uint32_t w = w0; w < min(words, w0 + wpt); ++w ) { rank[w] = (uint16_t)run; run += __popc(bits[w]); }
                if ( threadIdx.x == 0 ) dist = d;
        }
        __syncthreads();
        for ( uint32_t w = threadIdx.x; w < words; w += 256 )
        {
                SlotWord sw; sw.bits = bits[w]; sw.rank = s0 + rank[w];
                P.slots[tb][(uint64_t)sb * words + w] = sw;
        }
        if ( threadIdx.x == 0 && dist ) atomicAdd(P.ndistinct[tb], dist);
        __syncthreads();
        // entries: the first one of a slot claims E[rank] and writes the whole 16-byte head (next = none) with one store; the
        // others (few: the tables are sparse) are set aside -- or, beyond the capacity of the list, parked in their final place
        // with the head's index in `next` -- and chained after the barrier, when every head stands
        Entry * E = P.E[tb];
        for ( uint32_t i0 = s0 + threadIdx.x; i0 < s1; i0 += 1024 )
        {
                uint64_t seed[4]; uint32_t val[4];
                #pragma unroll
                for ( int k = 0; k < 4; ++k )
                {
                        uint32_t const i = i0 + (uint32_t)k * 256;
                        seed[k] = (i < s1) ? __ldg(P.item_seed + i) : 0;
                        val[k] = (i < s1) ? __ldg(P.item_val + i) : 0;
                }
                #pragma unroll
                for ( int k = 0; k < 4; ++k )
                        if ( i0 + (uint32_t)k * 256 < s1 )
                        {
                                uint32_t const t = val[k] & 3;
                                if ( t < G.nlists )
                                {
                                        uint32_t const l = sub_local_slot<FAST>(seed[k], G, t, tb, slot0);
                                        uint32_t const bit = 1u << (l & 31);
                                        uint32_t const r = s0 + rank[l >> 5] + __popc(bits[l >> 5] & (bit - 1));
                                        if ( ! (atomicOr(&claimed[l >> 5], bit) & bit) )
                                        {
                                                Entry en; en.seed = seed[k]; en.val = val[k]; en.next = ENTRY_NONE;
                                                *reinterpret_cast<uint4 *>(E + r) = *reinterpret_cast<const uint4 *>(&en);
                                        }
                                        else
                                        {
                                                uint32_t const j = atomicAdd(&ndup, 1u);
                                                if ( j < SUB3_DUP_CAP )
                                                {
                                                        SubDup dd; dd.seed = seed[k]; dd.val = val[k]; dd.r = r;
                                                        dup[j] = dd;
                                                }
                                                else
                                                {
                                                        Entry en; en.seed = seed[k]; en.val = val[k]; en.next = r;
                                                        *reinterpret_cast<uint4 *>(E + s0 + dist + j) = *reinterpret_cast<const uint4 *>(&en);
                                                }
                                        }
                                }
                        }
        }
        __syncthreads();
        // the set-aside entries go behind the distinct ones of this sub-bucket
        uint32_t const nd = min(ndup, SUB3_DUP_CAP);          // (ndup counts every same-slot entry, parked ones included)
        for ( uint32_t j = threadIdx.x; j < nd; j += 256 )
        {
                SubDup const dd = dup[j];
                uint32_t const o = s0 + dist + j;
                Entry en; en.seed = dd.seed; en.val = dd.val;
                en.next = atomicExch(&E[dd.r].next, o);
                *reinterpret_cast<uint4 *>(E + o) = *reinterpret_cast<const uint4 *>(&en);
        }
        for ( uint32_t j = SUB3_DUP_CAP + threadIdx.x; j < ndup; j += 256 )
        {
                uint32_t const o = s0 + dist + j;
                uint32_t const r = E[o].next;                        // the head's index was parked here
                E[o].next = atomicExch(&E[r].next, o);
        }
}

} // namespace realgpu
