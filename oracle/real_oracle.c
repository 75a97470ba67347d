/* TEST INFRASTRUCTURE ONLY -- never linked, imported or called by the product path.
 *
 * CPU restatement of the reference's matching hot path (see real_oracle.h).  Each function
 * cites the reference file:line it follows (paths relative to /root/reference/src).
 * Parity status: PINNED -- checked against the reference's own objects via
 * oracle/_ref/ref_harness and against tests/golden/ fixtures produced by that harness.
 *
 * Known, deliberate definitions where the reference has undefined behaviour:
 *   - matchGaps reads MAXscore/MINgap/where/start uninitialised when no DP end cell
 *     qualifies (match.hpp:515-518); here they start as 0, so such a candidate records nothing.
 *   - quality values are used as `(ref<<8)|(read<<6)|q` without clamping (Scoring.hpp:72);
 *     here the index is additionally masked to the table size for memory safety.
 */
#include "real_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <float.h>

/* ------------------------------------------------------------------------------------------
 * bit helpers
 * ---------------------------------------------------------------------------------------- */

/* PopCountTable.hpp:113-131 : number of differing 2-bit symbols */
uint32_t oracle_diffcount64(uint64_t a, uint64_t b)
{
        uint64_t x = a ^ b;
        x = ((x >> 1) | x) & 0x5555555555555555ULL;
        return (uint32_t)__builtin_popcountll(x);
}

/* ERank222B.hpp:55-85 via AutoTextArray.hpp:122-125 : l bases starting at base i, right aligned */
uint64_t oracle_text_word(const uint64_t * words, uint64_t i, uint32_t l)
{
        if ( l == 0 )
                return 0;
        uint64_t const bit = i << 1;
        uint32_t nbits = l << 1;
        uint64_t w = bit >> 6;
        uint32_t const skip = (uint32_t)(bit & 63);
        uint32_t const avail = 64 - skip;
        uint64_t b = words[w];
        if ( skip )
                b &= (~0ULL) >> skip;
        if ( avail == nbits )
                return b;
        if ( nbits < avail )
                return b >> (avail - nbits);
        nbits -= avail;
        return (b << nbits) | (words[w+1] >> (64 - nbits));
}

static inline uint32_t text_symbol(const uint64_t * words, uint64_t i)
{
        return (uint32_t)((words[i >> 5] >> (62 - 2*(i & 31))) & 3);
}

static inline int nmask_bit(const uint64_t * nmask, uint64_t i)
{
        return (int)((nmask[i >> 6] >> (63 - (i & 63))) & 1);
}

/* AutoTextArray.hpp:167-172 : no wildcard among bases [i, i+l) (rank difference restated as a scan) */
int oracle_dontcare_free(const uint64_t * nmask, uint64_t i, uint64_t l)
{
        for ( uint64_t p = i; p < i + l; ++p )
                if ( nmask_bit(nmask, p) )
                        return 0;
        return 1;
}

/* RangeVector.hpp:59-62 : rank1(pos)-1 over the record-start bit vector */
uint32_t oracle_position_to_range(const uint64_t * record_starts, uint32_t nrecords, uint64_t pos)
{
        /* number of starts (including the sentinel) <= pos, minus one */
        uint32_t lo = 0, hi = nrecords + 1;
        while ( lo < hi )
        {
                uint32_t const mid = (lo + hi) >> 1;
                if ( record_starts[mid] <= pos )
                        lo = mid + 1;
                else
                        hi = mid;
        }
        return lo - 1;
}

/* RangeVector.hpp:63-66 */
int oracle_position_valid(const uint64_t * record_starts, uint32_t nrecords, uint64_t pos, uint32_t patl)
{
        uint32_t const range = oracle_position_to_range(record_starts, nrecords, pos);
        if ( range >= nrecords )
                return 0; /* pos at or beyond the sentinel: the reference would index past its table */
        return (pos + patl) <= record_starts[range+1];
}

/* ------------------------------------------------------------------------------------------
 * signatures
 * ---------------------------------------------------------------------------------------- */

typedef struct
{
        uint32_t syms[4];
        uint32_t bits[4];
} frag_layout;

/* SignatureConstruction.hpp:47-54 */
static frag_layout layout_for(uint32_t seedl)
{
        frag_layout F;
        F.syms[0] = F.syms[1] = F.syms[2] = seedl / 4;
        F.syms[3] = seedl - 3 * (seedl / 4);
        for ( int i = 0; i < 4; ++i )
                F.bits[i] = F.syms[i] << 1;
        return F;
}

/* SignatureConstruction.hpp:218-280 : forward fragments of read[0..seedl) */
void oracle_fragments(const uint8_t * mapped, uint32_t seedl, uint32_t m[4])
{
        frag_layout const F = layout_for(seedl);
        uint32_t o = 0;
        for ( int f = 0; f < 4; ++f )
        {
                uint32_t v = 0;
                for ( uint32_t i = 0; i < F.syms[f]; ++i )
                        v = (v << 2) | (mapped[o++] & 3);
                m[f] = v;
        }
}

/* SignatureConstruction.hpp:347-410 : fragments of the reverse complement of read[0..seedl) */
void oracle_reverse_fragments(const uint8_t * mapped, uint32_t seedl, uint32_t m[4])
{
        frag_layout const F = layout_for(seedl);
        /* fragment 3 is built from read[0..syms3) backwards, fragment 2 from the next syms2, ... */
        uint32_t o = 0;
        for ( int f = 3; f >= 0; --f )
        {
                uint32_t v = 0;
                for ( uint32_t i = 0; i < F.syms[f]; ++i )
                        v = (v << 2) | (3 - (mapped[o + F.syms[f] - 1 - i] & 3));
                m[f] = v;
                o += F.syms[f];
        }
}

static const int PAIR_A[6] = {0,0,0,1,1,2};
static const int PAIR_B[6] = {1,2,3,2,3,3};

/* SignatureConstruction.hpp:62-67 */
void oracle_pair_signatures(const uint32_t m[4], uint32_t seedl, uint64_t s[6])
{
        frag_layout const F = layout_for(seedl);
        for ( int k = 0; k < 6; ++k )
                s[k] = (((uint64_t)m[PAIR_A[k]]) << F.bits[PAIR_B[k]]) | (uint64_t)m[PAIR_B[k]];
        /* a 32 bit signature type truncates (real.cpp:217-220) -- nothing to cut for seedl <= 32 */
}

/* ------------------------------------------------------------------------------------------
 * rest of the read
 * ---------------------------------------------------------------------------------------- */

/* RestMatch.hpp:214-318 via RestWordBuffer.hpp:56-78 ; returns the number of words written */
uint32_t oracle_rest_words(const uint8_t * mapped, uint32_t patl, uint32_t seedl, int inverted, uint64_t * out)
{
        uint32_t const restlen = patl - seedl;
        uint32_t const full = restlen / 32;
        uint32_t const frac = restlen - full * 32;
        uint32_t nw = 0;
        if ( ! inverted )
        {
                uint32_t o = seedl;
                for ( uint32_t i = 0; i < full; ++i )
                {
                        uint64_t w = 0;
                        for ( uint32_t j = 0; j < 32; ++j )
                                w = (w << 2) | (mapped[o++] & 3);
                        out[nw++] = w;
                }
                if ( frac )
                {
                        uint64_t w = 0;
                        for ( uint32_t j = 0; j < frac; ++j )
                                w = (w << 2) | (mapped[o++] & 3);
                        out[nw++] = w;
                }
        }
        else
        {
                uint32_t o = patl;
                for ( uint32_t i = 0; i < full; ++i )
                {
                        uint64_t w = 0;
                        for ( uint32_t j = 0; j < 32; ++j )
                                w = (w << 2) | (3 - (mapped[--o] & 3));
                        out[nw++] = w;
                }
                if ( frac )
                {
                        uint64_t w = 0;
                        for ( uint32_t j = 0; j < frac; ++j )
                                w = (w << 2) | (3 - (mapped[--o] & 3));
                        out[nw++] = w;
                }
        }
        return nw;
}

/* RestMatch.hpp:39-81 */
uint32_t oracle_rest_distance(const uint64_t * restwords, uint32_t patl, uint32_t seedl, const uint64_t * words, uint64_t o)
{
        uint32_t const restlen = patl - seedl;
        uint32_t const full = restlen / 32;
        uint32_t const frac = restlen - full * 32;
        uint32_t dist = 0;
        for ( uint32_t i = 0; i < full; ++i, o += 32 )
                dist += oracle_diffcount64(restwords[i], oracle_text_word(words, o, 32));
        if ( frac )
                dist += oracle_diffcount64(restwords[full], oracle_text_word(words, o, frac));
        return dist;
}

/* ------------------------------------------------------------------------------------------
 * scoring
 * ---------------------------------------------------------------------------------------- */

/* Scoring.cpp:27-35 */
static const double Q_PRB[65] = {
   1.0000000, 0.7943282, 0.6309573, 0.5011872, 0.3981072, 0.3162278, 0.2511886, 0.1995262, 0.1584893, 0.1258925,
   0.1000000, 0.0794328, 0.0630957, 0.0501187, 0.0398107, 0.0316228, 0.0251189, 0.0199526, 0.0158489, 0.0125893,
   0.0100000, 0.0079433, 0.0063096, 0.0050119, 0.0039811, 0.0031623, 0.0025119, 0.0019953, 0.0015849, 0.0012589,
   0.0010000, 0.0007943, 0.0006310, 0.0005012, 0.0003981, 0.0003162, 0.0002512, 0.0001995, 0.0001585, 0.0001259,
   0.0001000, 0.0000794, 0.0000631, 0.0000501, 0.0000398, 0.0000316, 0.0000251, 0.0000200, 0.0000158, 0.0000126,
   0.0000100, 0.0000079, 0.0000063, 0.0000050, 0.0000040, 0.0000032, 0.0000025, 0.0000020, 0.0000016, 0.0000013,
   0.0000010, 0.0000008, 0.0000006, 0.0000005, 0.0000004
};

/* Scoring.cpp:61-133 (odds ratios) and :155-171 (per-quality log score) */
void oracle_build_ll(double similarity, double gc, double trans, double err, double gcmut_bias, double * ll)
{
        double odds[4][4];
        double bg[4];
        double const transit = trans * (1 - similarity);
        double const transver = (1 - trans) * (1 - similarity);

        bg[0] = (1 - gc) / 2; bg[3] = (1 - gc) / 2;
        bg[1] = gc / 2;       bg[2] = gc / 2;

        double const bias = gcmut_bias * (1 - gc) / gc;

        /* transitions */
        odds[0][2] = transit / (bias + 1) / (1 - gc);
        odds[3][1] = transit / (bias + 1) / (1 - gc);
        odds[2][0] = transit / (bias + 1) / gc * bias;
        odds[1][3] = transit / (bias + 1) / gc * bias;
        /* transversions */
        odds[0][1] = transver / 2 / (bias + 1) / (1 - gc);
        odds[3][2] = transver / 2 / (bias + 1) / (1 - gc);
        odds[0][3] = transver / 2 / (bias + 1) / (1 - gc);
        odds[3][0] = transver / 2 / (bias + 1) / (1 - gc);
        odds[1][0] = transver / 2 / (bias + 1) / gc * bias;
        odds[2][3] = transver / 2 / (bias + 1) / gc * bias;
        odds[1][2] = transver / 2 / (bias + 1) / gc * bias;
        odds[2][1] = transver / 2 / (bias + 1) / gc * bias;
        /* conservation */
        odds[0][0] = 1 - odds[0][1] - odds[0][2] - odds[0][3];
        odds[3][3] = 1 - odds[3][0] - odds[3][1] - odds[3][2];
        odds[2][2] = 1 - odds[2][0] - odds[2][1] - odds[2][3];
        odds[1][1] = 1 - odds[1][0] - odds[1][2] - odds[1][3];

        for ( int x = 0; x < 4; ++x )
                for ( int y = 0; y < 4; ++y )
                {
                        odds[x][y] *= 1 - err;
                        odds[x][y] /= bg[y];
                }

        for ( unsigned c0 = 0; c0 < 4; ++c0 )
                for ( unsigned c1 = 0; c1 < 4; ++c1 )
                        for ( unsigned q = 0; q < 64; ++q )
                                ll[(c0 << 8) | (c1 << 6) | q] = log(odds[c0][c1]) / log(2.0) * (1 - Q_PRB[q]);
}

/* ComputeScore.hpp:50-190 : 1.0 + sum of LL over the read, double accumulation in index order,
 * '-' strand reads the reverse complement and the qualities back to front; returned as float */
float oracle_compute_score(const double * ll, const uint64_t * words, const uint8_t * mapped, const uint8_t * quality,
                           uint64_t pos, uint32_t patl, int inverted)
{
        double raw = 1.0f;
        for ( uint32_t i = 0; i < patl; ++i )
        {
                uint32_t const ref = text_symbol(words, pos + i);
                uint32_t readbase, q;
                if ( inverted )
                {
                        uint8_t const b = mapped[patl - 1 - i];
                        readbase = (b < 4) ? (3u - b) : b;
                        q = quality ? quality[patl - 1 - i] : 30;
                }
                else
                {
                        readbase = mapped[i];
                        q = quality ? quality[i] : 30;
                }
                raw += ll[((ref << 8) | (readbase << 6) | q) & 1023];
        }
        return (float)raw;
}

/* ------------------------------------------------------------------------------------------
 * text block index: six stably sorted signature lists (MapTextFile.hpp:181-230, ListSet.hpp:41-63)
 * ---------------------------------------------------------------------------------------- */

/* MapTextFile.hpp:115-179 : a window is emitted iff its seedl bases hold no wildcard */
uint64_t oracle_count_windows(const uint64_t * nmask, uint64_t n, uint32_t seedl)
{
        uint64_t run = 0, cnt = 0;
        for ( uint64_t i = 0; i < n; ++i )
        {
                run = nmask_bit(nmask, i) ? 0 : run + 1;
                if ( run >= seedl )
                        ++cnt;
        }
        return cnt;
}

typedef struct
{
        uint64_t nwin;          /* windows in this block */
        uint32_t * wpos;        /* window start positions, text order */
        uint64_t * sig[6];      /* signature of window w in list k (text order) */
        uint64_t * skey[6];     /* list k sorted by signature */
        uint32_t * sidx[6];     /* window index of sorted entry */
} block_index;

static void block_free(block_index * B)
{
        free(B->wpos);
        for ( int k = 0; k < 6; ++k ) { free(B->sig[k]); free(B->skey[k]); free(B->sidx[k]); }
        memset(B, 0, sizeof(*B));
}

/* stable LSD sort of (key, idx) by key: restates the observable effect of
 * ParallelRadixSort.hpp:50-214 / u_sort.hpp:105-131 (equal signatures keep text order) */
static void stable_sort_pairs(uint64_t * key, uint32_t * idx, uint64_t n)
{
        if ( n < 2 )
                return;
        uint64_t * k2 = (uint64_t *)malloc(n * sizeof(uint64_t) + 8);
        uint32_t * i2 = (uint32_t *)malloc(n * sizeof(uint32_t) + 8);
        size_t * cnt = (size_t *)malloc(65537 * sizeof(size_t));
        for ( int pass = 0; pass < 4; ++pass )
        {
                int const sh = 16 * pass;
                memset(cnt, 0, 65537 * sizeof(size_t));
                for ( uint64_t i = 0; i < n; ++i )
                        cnt[((key[i] >> sh) & 0xFFFF) + 1]++;
                if ( cnt[((key[0] >> sh) & 0xFFFF) + 1] == n )
                        continue; /* every key has the same digit */
                for ( int d = 0; d < 65536; ++d )
                        cnt[d+1] += cnt[d];
                for ( uint64_t i = 0; i < n; ++i )
                {
                        size_t const o = cnt[(key[i] >> sh) & 0xFFFF]++;
                        k2[o] = key[i];
                        i2[o] = idx[i];
                }
                memcpy(key, k2, n * sizeof(uint64_t));
                memcpy(idx, i2, n * sizeof(uint32_t));
        }
        free(k2); free(i2); free(cnt);
}

/* builds the index of windows [first, first+count) of the file's window sequence */
static int block_build(block_index * B, const oracle_text * T, uint32_t seedl, const uint32_t * allwpos, uint64_t first, uint64_t count)
{
        frag_layout const F = layout_for(seedl);
        memset(B, 0, sizeof(*B));
        B->nwin = count;
        B->wpos = (uint32_t *)malloc(count * sizeof(uint32_t) + 8);
        memcpy(B->wpos, allwpos + first, count * sizeof(uint32_t));
        for ( int k = 0; k < 6; ++k )
        {
                B->sig[k] = (uint64_t *)malloc(count * sizeof(uint64_t) + 8);
                B->skey[k] = (uint64_t *)malloc(count * sizeof(uint64_t) + 8);
                B->sidx[k] = (uint32_t *)malloc(count * sizeof(uint32_t) + 8);
        }
        #pragma omp parallel for schedule(static)
        for ( int64_t w = 0; w < (int64_t)count; ++w )
        {
                uint64_t const p = B->wpos[w];
                uint32_t m[4];
                uint64_t o = p;
                for ( int f = 0; f < 4; ++f )
                {
                        m[f] = (uint32_t)oracle_text_word(T->words, o, F.syms[f]);
                        o += F.syms[f];
                }
                uint64_t s[6];
                oracle_pair_signatures(m, seedl, s);
                for ( int k = 0; k < 6; ++k )
                {
                        B->sig[k][w] = s[k];
                        B->skey[k][w] = s[k];
                        B->sidx[k][w] = (uint32_t)w;
                }
        }
        #pragma omp parallel for schedule(dynamic,1)
        for ( int k = 0; k < 6; ++k )
                stable_sort_pairs(B->skey[k], B->sidx[k], count);
        return 0;
}

/* getLookupTable.hpp:25-51 + std::equal_range (match.hpp:376-381): the bucket directory only
 * narrows the binary search, so the range is the plain equal range of the sorted list */
static void equal_range_u64(const uint64_t * a, uint64_t n, uint64_t key, uint64_t * lo_out, uint64_t * hi_out)
{
        uint64_t lo = 0, hi = n;
        while ( lo < hi ) { uint64_t const mid = (lo + hi) >> 1; if ( a[mid] < key ) lo = mid + 1; else hi = mid; }
        uint64_t const first = lo;
        hi = n;
        while ( lo < hi ) { uint64_t const mid = (lo + hi) >> 1; if ( a[mid] <= key ) lo = mid + 1; else hi = mid; }
        *lo_out = first;
        *hi_out = lo;
}

static uint32_t * enumerate_windows(const oracle_text * T, uint32_t seedl, uint64_t * nwin_out)
{
        uint64_t const nwin = oracle_count_windows(T->nmask, T->n, seedl);
        uint32_t * wpos = (uint32_t *)malloc(nwin * sizeof(uint32_t) + 8);
        uint64_t run = 0, c = 0;
        for ( uint64_t i = 0; i < T->n; ++i )
        {
                run = nmask_bit(T->nmask, i) ? 0 : run + 1;
                if ( run >= seedl )
                        wpos[c++] = (uint32_t)(i + 1 - seedl);
        }
        *nwin_out = nwin;
        return wpos;
}

/* ------------------------------------------------------------------------------------------
 * per read context (RestWordBuffer.hpp:33-78, RestMatch.hpp:84-111)
 * ---------------------------------------------------------------------------------------- */

/* reads of up to 65535 bases (the product's limit): the rest of the read is at most 65535 - 4 bases, 2048 words.
 * Two such buffers make read_ctx 32 KB, well inside a thread's stack. */
#define ORACLE_MAX_REST_WORDS 2048

typedef struct
{
        const uint8_t * mapped;
        const uint8_t * quality;
        uint32_t patl;
        uint64_t patid;
        int usable;
        uint64_t fw[6], rv[6];
        uint64_t rest_fw[ORACLE_MAX_REST_WORDS], rest_rv[ORACLE_MAX_REST_WORDS];
        float epsilon;
} read_ctx;

/* skip rules of matchAllImplementation.cpp:273-289 / matchUniqueImplementation.cpp:379-394 */
static void read_setup(read_ctx * C, const oracle_params * P, const oracle_reads * R, uint64_t r)
{
        C->mapped = R->mapped + R->offsets[r];
        C->quality = R->quality ? (R->quality + R->offsets[r]) : 0;
        C->patl = (uint32_t)(R->offsets[r+1] - R->offsets[r]);
        C->patid = r;
        C->usable = (C->patl >= P->seedl) && (C->patl - P->seedl <= 32u * ORACLE_MAX_REST_WORDS);
        for ( uint32_t i = 0; i < C->patl; ++i )
                if ( C->mapped[i] > 3 )
                        C->usable = 0;
        if ( ! C->usable )
                return;
        uint32_t m[4];
        oracle_fragments(C->mapped, P->seedl, m);
        oracle_pair_signatures(m, P->seedl, C->fw);
        oracle_reverse_fragments(C->mapped, P->seedl, m);
        oracle_pair_signatures(m, P->seedl, C->rv);
        oracle_rest_words(C->mapped, C->patl, P->seedl, 0, C->rest_fw);
        oracle_rest_words(C->mapped, C->patl, P->seedl, 1, C->rest_rv);
        C->epsilon = (float)(P->filter_mult * C->patl);
}

/* ------------------------------------------------------------------------------------------
 * updaters
 * ---------------------------------------------------------------------------------------- */

/* UniqueMatchInfo.hpp:26-39 */
#define UMI_POSBITS 35
#define UMI_FILESHIFT 35
#define UMI_ERRSHIFT 41
#define UMI_FRAGSHIFT 45
#define UMI_STATESHIFT 61
#define UMI_POSMASK ((1ULL << UMI_POSBITS) - 1)
enum { ST_NOMATCH = 0, ST_STRAIGHT = 1, ST_REVERSE = 2, ST_GAPPED = 3, ST_NONUNIQUE = 4 };

static inline uint32_t umi_state(uint64_t d) { uint64_t s = d >> UMI_STATESHIFT; return s > 4 ? 4 : (uint32_t)s; }
static inline uint64_t umi_pos(uint64_t d) { return d & UMI_POSMASK; }
static inline uint32_t umi_file(uint64_t d) { return (uint32_t)((d >> UMI_FILESHIFT) & 63); }
static inline uint32_t umi_err(uint64_t d) { return (uint32_t)((d >> UMI_ERRSHIFT) & 15); }
static inline uint32_t umi_frag(uint64_t d) { return (uint32_t)((d >> UMI_FRAGSHIFT) & 0xFFFF); }
static inline uint64_t umi_set_state(uint64_t d, uint32_t s) { return (d & ~(7ULL << UMI_STATESHIFT)) | ((uint64_t)s << UMI_STATESHIFT); }
static inline uint64_t umi_set_pos(uint64_t d, uint64_t p) { return (d & ~UMI_POSMASK) | p; }
static inline uint64_t umi_take(uint64_t d, int inverted, uint32_t file, uint32_t pos, uint32_t k, uint32_t frag)
{
        d = umi_set_state(d, inverted ? ST_REVERSE : ST_STRAIGHT);
        d = umi_set_pos(d, pos);
        d = (d & ~(63ULL << UMI_FILESHIFT)) | ((uint64_t)file << UMI_FILESHIFT);
        d = (d & ~(15ULL << UMI_ERRSHIFT)) | ((uint64_t)k << UMI_ERRSHIFT);
        d = (d & ~(0xFFFFULL << UMI_FRAGSHIFT)) | ((uint64_t)frag << UMI_FRAGSHIFT);
        return d;
}

typedef struct
{
        int mode;               /* 0 = all, 1 = unique */
        int scores;
        /* all */
        oracle_hit * hits; uint64_t nhits, cap;
        uint64_t patid; uint32_t block;
        /* unique */
        uint64_t * info; float * score;
} sink;

/* matchAllImplementation.cpp:172-181 */
static void sink_all(sink * S, int inverted, uint32_t file, uint32_t pos, uint32_t k, float score, uint32_t frag)
{
        if ( S->nhits == S->cap )
        {
                S->cap = S->cap ? 2 * S->cap : 16;
                S->hits = (oracle_hit *)realloc(S->hits, S->cap * sizeof(oracle_hit));
        }
        oracle_hit * H = &S->hits[S->nhits++];
        H->patid = S->patid; H->pos = pos; H->file = file; H->frag = frag; H->k = k;
        H->inverted = inverted ? 1 : 0; H->score = score; H->block = S->block;
}

/* matchUniqueImplementation.cpp:97-159 */
static void sink_unique_plain(uint64_t * info, int inverted, uint32_t file, uint32_t pos, uint32_t k, uint32_t frag)
{
        uint64_t d = *info;
        switch ( umi_state(d) )
        {
                case ST_NOMATCH: case ST_GAPPED:
                        d = umi_take(d, inverted, file, pos, k, frag);
                        break;
                case ST_STRAIGHT: case ST_REVERSE:
                        if ( k < umi_err(d) )
                                d = umi_take(d, inverted, file, pos, k, frag);
                        else if ( k == umi_err(d) && (pos != umi_pos(d) || file != umi_file(d) || frag != umi_frag(d)) )
                                d = umi_set_state(d, ST_NONUNIQUE);
                        break;
                case ST_NONUNIQUE:
                        if ( k < umi_err(d) )
                                d = umi_take(d, inverted, file, pos, k, frag);
                        break;
        }
        *info = d;
}

/* matchUniqueImplementation.cpp:179-248 */
static void sink_unique_scored(uint64_t * info, float * sc, int inverted, uint32_t file, uint32_t pos, uint32_t k, float score, float epsilon, uint32_t frag)
{
        uint64_t d = *info;
        switch ( umi_state(d) )
        {
                case ST_NOMATCH: case ST_GAPPED:
                        d = umi_take(d, inverted, file, pos, k, frag);
                        *sc = score;
                        break;
                case ST_STRAIGHT: case ST_REVERSE:
                        if ( score > *sc + epsilon )
                        {
                                d = umi_take(d, inverted, file, pos, k, frag);
                                *sc = score;
                        }
                        else if ( (score > *sc - epsilon) && (pos != umi_pos(d) || file != umi_file(d) || frag != umi_frag(d)) )
                                d = umi_set_state(d, ST_NONUNIQUE);
                        break;
                case ST_NONUNIQUE:
                        if ( score > *sc + epsilon )
                        {
                                d = umi_take(d, inverted, file, pos, k, frag);
                                *sc = score;
                        }
                        break;
        }
        *info = d;
}

/* ------------------------------------------------------------------------------------------
 * the probe: match.hpp:335-416
 * ---------------------------------------------------------------------------------------- */

static void probe_list(const oracle_params * P, const oracle_text * T, const block_index * B, const read_ctx * C,
                       int k, int inverted, sink * S)
{
        uint64_t const s_a = inverted ? C->rv[k] : C->fw[k];
        uint64_t const s_b = inverted ? C->rv[5-k] : C->fw[5-k];
        uint32_t const restlen = C->patl - P->seedl;
        uint32_t const matchoffset = inverted ? restlen : 0;                           /* RestMatch.hpp:84-89 */
        int32_t const textrestoffset = inverted ? -(int32_t)restlen : (int32_t)P->seedl; /* RestMatch.hpp:104-111 */
        const uint64_t * restwords = inverted ? C->rest_rv : C->rest_fw;

        uint64_t lo, hi;
        equal_range_u64(B->skey[k], B->nwin, s_a, &lo, &hi);
        for ( uint64_t e = lo; e < hi; ++e )
        {
                uint32_t const w = B->sidx[k][e];
                uint32_t const seedk = oracle_diffcount64(s_b, B->sig[5-k][w]);
                if ( seedk > P->seedkmax )
                        continue;
                uint32_t const rpos = B->wpos[w];
                if ( rpos < matchoffset )
                        continue;
                uint32_t const pos = rpos - matchoffset;
                if ( ! (oracle_position_valid(T->record_starts, T->nrecords, pos, C->patl) && oracle_dontcare_free(T->nmask, pos, C->patl)) )
                        continue;
                uint32_t const restpos = rpos + (uint32_t)textrestoffset;
                uint32_t const restk = oracle_rest_distance(restwords, C->patl, P->seedl, T->words, restpos);
                uint32_t const totalk = seedk + restk;
                if ( totalk > P->totalkmax )
                        continue;
                uint32_t const frag = oracle_position_to_range(T->record_starts, T->nrecords, pos);
                float const score = P->scores ? oracle_compute_score(P->ll, T->words, C->mapped, C->quality, pos, C->patl, inverted) : 1.0f;
                if ( S->mode == 0 )
                        sink_all(S, inverted, T->fileid, pos, totalk, score, frag);
                else if ( S->scores )
                        sink_unique_scored(S->info, S->score, inverted, T->fileid, pos, totalk, score, C->epsilon, frag);
                else
                        sink_unique_plain(S->info, inverted, T->fileid, pos, totalk, frag);
        }
}

/* matchAllImplementation.cpp:122-136 : (k,pos,file,frag,score,inverted) */
static int hit_less(const oracle_hit * A, const oracle_hit * B)
{
        if ( A->k != B->k ) return A->k < B->k;
        if ( A->pos != B->pos ) return A->pos < B->pos;
        if ( A->file != B->file ) return A->file < B->file;
        if ( A->frag != B->frag ) return A->frag < B->frag;
        if ( (double)A->score != (double)B->score ) return (double)A->score < (double)B->score;
        return A->inverted < B->inverted;
}
static int hit_cmp(const void * a, const void * b)
{
        const oracle_hit * A = (const oracle_hit *)a; const oracle_hit * B = (const oracle_hit *)b;
        if ( hit_less(A,B) ) return -1;
        if ( hit_less(B,A) ) return 1;
        return 0;
}

/* matchAllImplementation.cpp:150-161 : sort + drop adjacent equals; returns the new count */
static uint64_t unify_hits(oracle_hit * H, uint64_t n)
{
        if ( ! n ) return 0;
        qsort(H, n, sizeof(oracle_hit), hit_cmp);
        uint64_t o = 1;
        for ( uint64_t i = 1; i < n; ++i )
                if ( hit_cmp(&H[i], &H[i-1]) != 0 )
                        H[o++] = H[i];
        return o;
}

/* AllMatcher::match, matchAllImplementation.cpp:261-355 */
static void read_match_all(const oracle_params * P, const oracle_text * T, const block_index * B, const read_ctx * C, sink * S)
{
        if ( ! C->usable ) return;
        for ( int k = 0; k < 6; ++k ) probe_list(P, T, B, C, k, 0, S);
        for ( int k = 0; k < 6; ++k ) probe_list(P, T, B, C, k, 1, S);
}

/* UniqueMatcher::match, matchUniqueImplementation.cpp:369-500 (incl. the 0-error shortcut :434,470) */
static void read_match_unique(const oracle_params * P, const oracle_text * T, const block_index * B, const read_ctx * C, sink * S)
{
        if ( ! C->usable ) return;
        probe_list(P, T, B, C, 0, 0, S);
        int const uni0s = (umi_state(*S->info) == ST_STRAIGHT) && (umi_err(*S->info) == 0);
        if ( ! uni0s || P->scores )
                for ( int k = 1; k < 6; ++k ) probe_list(P, T, B, C, k, 0, S);
        probe_list(P, T, B, C, 0, 1, S);
        int const uni0r = (umi_state(*S->info) == ST_REVERSE) && (umi_err(*S->info) == 0);
        if ( ! uni0r || P->scores )
                for ( int k = 1; k < 6; ++k ) probe_list(P, T, B, C, k, 1, S);
}

static int hit_order_cmp(const void * a, const void * b)
{
        const oracle_hit * A = (const oracle_hit *)a; const oracle_hit * B = (const oracle_hit *)b;
        if ( A->block != B->block ) return A->block < B->block ? -1 : 1;
        if ( A->patid != B->patid ) return A->patid < B->patid ? -1 : 1;
        return hit_cmp(a, b);
}

int64_t oracle_match_all(const oracle_params * P, const oracle_text * T, const oracle_reads * R, oracle_hit * out, uint64_t cap)
{
        if ( T->n < P->seedl ) return 0;                         /* matchAllImplementation.cpp:415-419 */
        uint64_t nwin = 0;
        uint32_t * wpos = enumerate_windows(T, P->seedl, &nwin);
        uint64_t const nlist = P->n_list ? P->n_list : (nwin ? nwin : 1);
        uint64_t total = 0;
        uint32_t block = 0;

        for ( uint64_t first = 0; first < nwin; first += nlist, ++block )
        {
                uint64_t const count = (nwin - first < nlist) ? (nwin - first) : nlist;
                block_index B;
                block_build(&B, T, P->seedl, wpos, first, count);

                oracle_hit * merged = 0; uint64_t nmerged = 0, cmerged = 0;
                #pragma omp parallel
                {
                        sink S; memset(&S, 0, sizeof(S));
                        S.mode = 0; S.scores = P->scores; S.block = block;
                        oracle_hit * mine = 0; uint64_t nmine = 0, cmine = 0;
                        #pragma omp for schedule(dynamic,256)
                        for ( int64_t r = 0; r < (int64_t)R->nreads; ++r )
                        {
                                read_ctx C;
                                read_setup(&C, P, R, (uint64_t)r);
                                S.nhits = 0; S.patid = (uint64_t)r;
                                read_match_all(P, T, &B, &C, &S);
                                uint64_t const u = unify_hits(S.hits, S.nhits);
                                if ( nmine + u > cmine )
                                {
                                        cmine = 2 * (nmine + u) + 16;
                                        mine = (oracle_hit *)realloc(mine, cmine * sizeof(oracle_hit));
                                }
                                if ( u ) memcpy(mine + nmine, S.hits, u * sizeof(oracle_hit));
                                nmine += u;
                        }
                        #pragma omp critical
                        {
                                if ( nmerged + nmine > cmerged )
                                {
                                        cmerged = 2 * (nmerged + nmine) + 16;
                                        merged = (oracle_hit *)realloc(merged, cmerged * sizeof(oracle_hit));
                                }
                                if ( nmine ) memcpy(merged + nmerged, mine, nmine * sizeof(oracle_hit));
                                nmerged += nmine;
                        }
                        free(mine);
                        free(S.hits);
                }
                qsort(merged, nmerged, sizeof(oracle_hit), hit_order_cmp);
                for ( uint64_t i = 0; i < nmerged; ++i, ++total )
                        if ( total < cap )
                                out[total] = merged[i];
                free(merged);
                block_free(&B);
        }
        free(wpos);
        return (int64_t)total;
}

void oracle_unique_init(uint64_t nreads, uint64_t * info, float * score)
{
        for ( uint64_t i = 0; i < nreads; ++i )
        {
                info[i] = 0;                                       /* UniqueMatchInfo.hpp:172 */
                if ( score ) score[i] = -FLT_MAX;                  /* UniqueMatchInfo.hpp:190 */
        }
}

int oracle_match_unique(const oracle_params * P, const oracle_text * T, const oracle_reads * R, uint64_t * info, float * score)
{
        if ( T->n < P->seedl ) return 0;                          /* matchUniqueImplementation.cpp:1133-1137 */
        if ( T->nrecords + 1 > 65536 ) return 0;                  /* :1139-1143 (ranges.size() incl. sentinel) */
        if ( P->scores && ! score ) return -1;
        uint64_t nwin = 0;
        uint32_t * wpos = enumerate_windows(T, P->seedl, &nwin);
        uint64_t const nlist = P->n_list ? P->n_list : (nwin ? nwin : 1);

        for ( uint64_t first = 0; first < nwin; first += nlist )
        {
                uint64_t const count = (nwin - first < nlist) ? (nwin - first) : nlist;
                block_index B;
                block_build(&B, T, P->seedl, wpos, first, count);
                #pragma omp parallel for schedule(dynamic,256)
                for ( int64_t r = 0; r < (int64_t)R->nreads; ++r )
                {
                        read_ctx C;
                        read_setup(&C, P, R, (uint64_t)r);
                        sink S; memset(&S, 0, sizeof(S));
                        S.mode = 1; S.scores = P->scores;
                        S.info = &info[r]; S.score = score ? &score[r] : 0;
                        read_match_unique(P, T, &B, &C, &S);
                }
                block_free(&B);
        }
        free(wpos);
        return 0;
}

/* ------------------------------------------------------------------------------------------
 * gapped extension: match.hpp:16-332, 428-602
 * ---------------------------------------------------------------------------------------- */

/* match.hpp:16-29 */
static double total_scoring(uint32_t gap, double cur, double open, double extend, double offset)
{
        if ( gap % 3 == 0 )
                return cur + (gap * extend) + open + offset;
        return cur + (gap * extend) + open;
}

typedef struct { double maxscore; uint32_t mingap, where, start, gap_pos; int assigned; } gap_result;

/* agm (match.hpp:267-332) + opt_solution (:159-260) + backtracing (:115-152) on full, zeroed
 * (n+1)x(m+1) matrices exactly as AgmMatrix (:66-81) lays them out */
static gap_result gapped_dp(const oracle_params * P, const oracle_text * T, const read_ctx * C, uint64_t rpos, uint32_t n, uint32_t m)
{
        uint32_t const MAXgap = 3;
        double const MINscore = -100.0, open = -1.0, extend = -1.0, offset = -1.0;
        size_t const W = (size_t)m + 1;
        double * G = (double *)calloc((size_t)(n+1) * W, sizeof(double));
        uint32_t * H = (uint32_t *)calloc((size_t)(n+1) * W, sizeof(uint32_t));
        uint64_t const ri = rpos + P->seedl - 1;
        uint32_t const rj = P->seedl - 1;

        for ( uint32_t i = 1; i < n + 1; ++i )
        {
                if ( i < MAXgap + 1 ) H[(size_t)i*W + 0] = i;
                uint32_t const left = ((int)i - (int)MAXgap > 0) ? (i - MAXgap) : 1;       /* j_limits, match.hpp:50-64 */
                uint32_t const right = (i + MAXgap > m) ? m : (i + MAXgap);
                for ( uint32_t j = left; j <= right; ++j )
                {
                        if ( j < MAXgap + 1 ) H[0*W + j] = j;
                        uint32_t const q = C->quality ? C->quality[j + rj] : 30;
                        double const sub = P->ll[((text_symbol(T->words, i + ri) << 8) | ((uint32_t)C->mapped[j + rj] << 6) | q) & 1023];
                        if ( i == j )
                        {
                                G[(size_t)i*W + j] = G[(size_t)(i-1)*W + (j-1)] + sub;
                                H[(size_t)i*W + j] = 0;
                        }
                        else
                        {
                                uint32_t const d = (i < j) ? i : j;
                                double const mis = G[(size_t)(i-1)*W + (j-1)] + sub;
                                double const gap = G[(size_t)d*W + d];
                                G[(size_t)i*W + j] = (mis < gap) ? gap : mis;              /* std::max(mis,gap) */
                                if ( gap > mis ) H[(size_t)i*W + j] = (i < j) ? (j - i) : (i - j);
                                else H[(size_t)i*W + j] = 0;
                        }
                }
        }

        /* The reference's MAXscore / MINgap / where / start are UNINITIALISED locals of ::matchGaps (match.hpp:518-522) that
         * opt_solution assigns only when some end cell of the band reaches MINscore.  When none does (a seed hit whose rest
         * of the read does not align at all) the reference goes on with whatever its stack held -- in practice the values
         * of the candidate evaluated before, possibly of another read: undefined behaviour that no restatement can follow.
         * Here such a candidate counts as "no gap found" (MINgap = 0), and `assigned` = 0 tells the caller that the
         * reference's own result for this read is not defined. */
        gap_result R; R.maxscore = 0; R.mingap = 0; R.where = 0; R.start = 0; R.gap_pos = 0; R.assigned = 0;
        double score = MINscore;
        uint32_t const up = ((int)m - (int)MAXgap < 0) ? 0 : (m - MAXgap);                    /* i_limits, match.hpp:33-47 */
        uint32_t const down = (m + MAXgap > n) ? n : (m + MAXgap);
        for ( uint32_t i = up; i <= down; ++i )
        {
                double const g = G[(size_t)i*W + m];
                if ( i < m )
                {
                        if ( g >= MINscore && m - i <= MAXgap )
                        {
                                double const t = total_scoring(m - i, g, open, extend, offset);
                                if ( t > score ) { score = t; R.maxscore = t; R.mingap = m - i; R.where = 1; R.start = i; R.assigned = 1; }
                        }
                }
                else if ( i > m )
                {
                        if ( g >= MINscore && i - m <= MAXgap )
                        {
                                double const t = total_scoring(i - m, g, open, extend, offset);
                                if ( t > score ) { score = t; R.maxscore = t; R.mingap = i - m; R.where = 2; R.start = i; R.assigned = 1; }
                        }
                }
                else
                {
                        if ( g >= MINscore )
                        {
                                double const t = total_scoring(0, g, open, extend, offset);
                                if ( t > score ) { score = t; R.maxscore = t; R.mingap = 0; R.where = 0; R.start = m; R.assigned = 1; }
                        }
                }
        }
        if ( m + MAXgap > n )
        {
                uint32_t const left = ((int)n - (int)MAXgap > 0) ? (n - MAXgap) : 1;       /* j_limits(n, m, ...) */
                uint32_t const right = (n + MAXgap > m) ? m : (n + MAXgap);
                for ( uint32_t j = left; j < right; ++j )
                {
                        double const g = G[(size_t)n*W + j];
                        if ( g >= MINscore && n - j <= MAXgap )
                        {
                                double const t = total_scoring(n - j, g, open, extend, offset);
                                if ( t > score ) { score = t; R.maxscore = t; R.mingap = n - j; R.where = 3; R.start = j; R.assigned = 1; }
                        }
                }
        }

        /* backtracing, match.hpp:115-152 */
        {
                int i, j;
                if ( R.where == 1 || R.where == 2 ) { i = (int)R.start; j = (int)m; }
                else { i = (int)n; j = (int)R.start; }
                R.gap_pos = 0;
                while ( i >= 0 && j >= 0 )
                {
                        if ( H[(size_t)i*W + j] == 0 ) { --i; --j; }
                        else { R.gap_pos = (i > j) ? (uint32_t)j : (uint32_t)i; break; }
                }
        }
        free(G); free(H);
        return R;
}

/* ::matchGaps, match.hpp:428-602 */
static void probe_list_gaps(const oracle_params * P, const oracle_text * T, const block_index * B, const read_ctx * C,
                            int k, int inverted, uint64_t * info, float * sc, oracle_gap * gap, uint8_t * undefined)
{
        uint64_t const s_a = inverted ? C->rv[k] : C->fw[k];
        uint64_t const s_b = inverted ? C->rv[5-k] : C->fw[5-k];
        uint32_t const st0 = umi_state(*info);
        if ( !(st0 == ST_NOMATCH || st0 == ST_GAPPED) )
                return;
        uint64_t lo, hi;
        equal_range_u64(B->skey[k], B->nwin, s_a, &lo, &hi);
        for ( uint64_t e = lo; e < hi; ++e )
        {
                uint32_t const w = B->sidx[k][e];
                uint32_t const seedk = oracle_diffcount64(s_b, B->sig[5-k][w]);
                if ( seedk > P->seedkmax )
                        continue;
                uint32_t const rpos = B->wpos[w];
                if ( ! (oracle_position_valid(T->record_starts, T->nrecords, rpos, P->seedl) && oracle_dontcare_free(T->nmask, rpos, P->seedl)) )
                        continue;
                uint32_t const range = oracle_position_to_range(T->record_starts, T->nrecords, rpos);
                uint64_t const phigh = T->record_starts[range+1];
                if ( inverted )
                        continue;                                                      /* match.hpp:499, no else */
                double const seedscore = P->scores ? (double)oracle_compute_score(P->ll, T->words, C->mapped, C->quality, rpos, P->seedl, 0) : (double)1.0f;
                uint64_t n = phigh - P->seedl - rpos;
                if ( n > 2ULL * C->patl ) n = 2ULL * C->patl;
                uint64_t const m = C->patl - P->seedl;
                if ( !( n && m && oracle_dontcare_free(T->nmask, (uint64_t)rpos + P->seedl, n) ) )
                        continue;
                gap_result const G = gapped_dp(P, T, C, rpos, (uint32_t)n, (uint32_t)m);
                if ( ! G.assigned && undefined )
                        *undefined = 1;
                if ( ! G.mingap )
                        continue;
                double const complete = seedscore + G.maxscore;
                float const stored = (P->scores && sc) ? *sc : 0.0f;                   /* UniqueMatchInfo.hpp:178-185 */
                if ( umi_state(*info) == ST_NOMATCH )
                {
                        *info = umi_set_state(*info, ST_GAPPED);
                        if ( P->scores && sc ) *sc = (float)complete;
                        *info = umi_set_pos(*info, rpos);
                        gap->patid = (uint32_t)C->patid; gap->mingap = G.mingap; gap->where = G.where; gap->start = G.start; gap->gap_pos = G.gap_pos; gap->present = 1;
                }
                else if ( umi_state(*info) == ST_GAPPED )
                {
                        if ( complete > stored + 1e-6 )
                        {
                                if ( P->scores && sc ) *sc = (float)complete;
                                *info = umi_set_pos(*info, rpos);
                                gap->patid = (uint32_t)C->patid; gap->mingap = G.mingap; gap->where = G.where; gap->start = G.start; gap->gap_pos = G.gap_pos; gap->present = 1;
                        }
                        else if ( complete < stored - 1e-6 )
                        {
                        }
                        else
                                gap->present = 0;
                }
        }
}

int oracle_match_gaps(const oracle_params * P, const oracle_text * T, const oracle_reads * R, uint64_t * info, float * score, oracle_gap * gaps)
{
        return oracle_match_gaps_flagged(P, T, R, info, score, gaps, 0);
}

/* undefined (may be null): one byte per read, set when a candidate of the read left opt_solution's outputs unassigned */
int oracle_match_gaps_flagged(const oracle_params * P, const oracle_text * T, const oracle_reads * R, uint64_t * info, float * score, oracle_gap * gaps,
                              uint8_t * undefined)
{
        if ( T->n < P->seedl ) return 0;
        if ( T->nrecords + 1 > 65536 ) return 0;
        if ( ! P->ll ) return -1;
        uint64_t nwin = 0;
        uint32_t * wpos = enumerate_windows(T, P->seedl, &nwin);
        uint64_t const nlist = P->n_list ? P->n_list : (nwin ? nwin : 1);
        for ( uint64_t first = 0; first < nwin; first += nlist )
        {
                uint64_t const count = (nwin - first < nlist) ? (nwin - first) : nlist;
                block_index B;
                block_build(&B, T, P->seedl, wpos, first, count);
                #pragma omp parallel for schedule(dynamic,256)
                for ( int64_t r = 0; r < (int64_t)R->nreads; ++r )
                {
                        uint32_t const st = umi_state(info[r]);
                        if ( !(st == ST_NOMATCH || st == ST_GAPPED) )                  /* matchUniqueImplementation.cpp:508 */
                                continue;
                        read_ctx C;
                        read_setup(&C, P, R, (uint64_t)r);
                        if ( ! C.usable )
                                continue;
                        for ( int k = 0; k < 6; ++k ) probe_list_gaps(P, T, &B, &C, k, 0, &info[r], score ? &score[r] : 0, &gaps[r], undefined ? &undefined[r] : 0);
                        for ( int k = 0; k < 6; ++k ) probe_list_gaps(P, T, &B, &C, k, 1, &info[r], score ? &score[r] : 0, &gaps[r], undefined ? &undefined[r] : 0);
                }
                block_free(&B);
        }
        free(wpos);
        return 0;
}
