// Shared device/host helpers of libreal_gpu.so (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdexcept>
#include <string>
#include <cstdio>

namespace realgpu
{

struct CudaError : public std::runtime_error
{
        explicit CudaError(std::string const & s) : std::runtime_error(s) {}
};

#define RG_CUDA(expr)                                                                          \
        do {                                                                                   \
                cudaError_t rg_e_ = (expr);                                                    \
                if ( rg_e_ != cudaSuccess )                                                    \
                {                                                                              \
                        char rg_buf_[512];                                                     \
                        snprintf(rg_buf_, sizeof(rg_buf_), "%s failed: %s (%s:%d)", #expr,     \
                                 cudaGetErrorString(rg_e_), __FILE__, __LINE__);               \
                        throw realgpu::CudaError(rg_buf_);                                     \
                }                                                                              \
        } while (0)

#define RG_KERNEL_CHECK() RG_CUDA(cudaGetLastError())

// ---- layouts shared by kernels -------------------------------------------------------------

// zero words kept in front of and behind the device copy of the text / N mask so that unaligned
// extracts and tile halos never leave the allocation
static const uint32_t TEXT_PAD_WORDS = 64;

// presence table: one 8-byte word per 32 slots = {presence bits, rank of the word's first slot}; a probe is ONE
// 8-byte load that yields both the bit and, if it is set, the index of the slot's entry
struct __align__(8) SlotWord
{
        uint32_t bits;
        uint32_t rank;
};
static const uint32_t RANK_BLOCK_WORDS = 2048;      // slot words per block of the ranking kernels (tables are padded to it)

static const uint32_t ENTRY_NONE = 0xFFFFFFFFu;

// one index entry: the read strand's whole seed, (strand id << 2 | fragment offset), chain link
struct __align__(16) Entry
{
        uint64_t seed;
        uint32_t val;
        uint32_t next;
};

// raw hit as emitted by the scan kernel (16 bytes)
struct __align__(16) RawHit
{
        uint64_t pm;     // pos:35 | k:4 | strand:1 | frag:24
        uint32_t read;
        float score;
};

__host__ __device__ inline uint64_t rawhit_pack(uint64_t pos, uint32_t k, uint32_t strand, uint32_t frag)
{
        return pos | ((uint64_t)k << 35) | ((uint64_t)strand << 39) | ((uint64_t)frag << 40);
}
__host__ __device__ inline uint32_t rawhit_read(uint32_t r) { return r & 0x0FFFFFFFu; }      // RawHit::read = read | exact-fragment mask << 28
__host__ __device__ inline uint32_t rawhit_exact(uint32_t r) { return r >> 28; }
__host__ __device__ inline uint64_t rawhit_pos(uint64_t pm) { return pm & ((1ULL << 35) - 1); }
__host__ __device__ inline uint32_t rawhit_k(uint64_t pm) { return (uint32_t)((pm >> 35) & 15); }
__host__ __device__ inline uint32_t rawhit_strand(uint64_t pm) { return (uint32_t)((pm >> 39) & 1); }
__host__ __device__ inline uint32_t rawhit_frag(uint64_t pm) { return (uint32_t)((pm >> 40) & 0xFFFFFF); }

// UniqueMatchInfo word (UniqueMatchInfo.hpp:26-39)
#define UMI_FILESHIFT 35
#define UMI_ERRSHIFT 41
#define UMI_FRAGSHIFT 45
#define UMI_STATESHIFT 61
#define UMI_POSMASK ((1ULL << 35) - 1)
enum { ST_NOMATCH = 0, ST_STRAIGHT = 1, ST_REVERSE = 2, ST_GAPPED = 3, ST_NONUNIQUE = 4 };

__host__ __device__ inline uint32_t umi_state(uint64_t d) { uint64_t s = d >> UMI_STATESHIFT; return s > 4 ? 4u : (uint32_t)s; }
__host__ __device__ inline uint64_t umi_pos(uint64_t d) { return d & UMI_POSMASK; }
__host__ __device__ inline uint32_t umi_file(uint64_t d) { return (uint32_t)((d >> UMI_FILESHIFT) & 63); }
__host__ __device__ inline uint32_t umi_err(uint64_t d) { return (uint32_t)((d >> UMI_ERRSHIFT) & 15); }
__host__ __device__ inline uint32_t umi_frag(uint64_t d) { return (uint32_t)((d >> UMI_FRAGSHIFT) & 0xFFFF); }
__host__ __device__ inline uint64_t umi_make(uint32_t state, uint32_t file, uint64_t pos, uint32_t k, uint32_t frag)
{
        return pos | ((uint64_t)file << UMI_FILESHIFT) | ((uint64_t)k << UMI_ERRSHIFT) | ((uint64_t)frag << UMI_FRAGSHIFT) | ((uint64_t)state << UMI_STATESHIFT);
}
__host__ __device__ inline uint64_t umi_with_state(uint64_t d, uint32_t s) { return (d & ~(7ULL << UMI_STATESHIFT)) | ((uint64_t)s << UMI_STATESHIFT); }

// ---- bit helpers ----------------------------------------------------------------------------

// number of differing 2-bit symbols (PopCountTable.hpp:113-131)
__device__ __forceinline__ uint32_t diffcount64(uint64_t a, uint64_t b)
{
        uint64_t x = a ^ b;
        x = ((x >> 1) | x) & 0x5555555555555555ULL;
        return (uint32_t)__popcll(x);
}

// l (1..32) bases starting at base i, right aligned (AutoTextArray.hpp:122-125); `words` may be
// indexed one word past the last base (padding)
__device__ __forceinline__ uint64_t text_word(const uint64_t * __restrict__ words, uint64_t i, uint32_t l)
{
        uint64_t const w = i >> 5;
        uint32_t const sh = (uint32_t)(i & 31) << 1;
        uint64_t const a = __ldg(words + w);
        uint64_t const b = __ldg(words + w + 1);
        uint64_t v = sh ? ((a << sh) | (b >> (64 - sh))) : a;
        return v >> (64 - 2*l);
}

// reverse complement of the `len` bases held right aligned in x
__device__ __forceinline__ uint64_t revcomp_word(uint64_t x, uint32_t len)
{
        uint64_t y = __brevll(~x);                                                     // complement, reverse all bits
        y = ((y >> 1) & 0x5555555555555555ULL) | ((y & 0x5555555555555555ULL) << 1);   // put the two bits of every base back in order
        return y >> (64 - 2*len);
}

// ---- where the bases of the reads live ---------------------------------------------------------
// Byte-per-base input (real_gpu_set_reads*) is packed once into `rpack`: both strands of every read, W words each,
// 32 bases per word MSB first, left aligned (RestWordBuffer.hpp:33-78 for all reads at once).  Input that already is
// 2 bit/base (real_gpu_set_reads_packed*: 4 bases per byte, first base in bits 7..6, every read on a byte boundary --
// the reference's rewritten pattern file, TemporaryFile.hpp:231-268) is NOT repacked: the few candidates that reach
// the verification cut their words straight out of the packed bytes, the '-' strand by reverse complement.
struct ReadSrc
{
        const uint64_t * rpack;       // strand id s = 2*read + strand at rpack + s * W, or null
        uint32_t W;
        uint32_t ubytes;              // packed input of uniform length: bytes per read (0: boffs)
        const uint8_t * packed;
        const uint64_t * boffs;       // nreads+1 byte offsets into packed
};

// `len` (1..32) bases from base `first` on of the packed read that starts at byte p, LEFT aligned.  Reads aligned 32-bit
// words only, and none that does not hold a wanted byte.
__device__ __forceinline__ uint64_t packed_bases(const uint8_t * __restrict__ p, uint32_t first, uint32_t len)
{
        uintptr_t const addr = reinterpret_cast<uintptr_t>(p) + (first >> 2);
        const uint32_t * q = reinterpret_cast<const uint32_t *>(addr & ~(uintptr_t)3);
        uint32_t const sh = (uint32_t)(addr & 3) * 8;
        uint32_t const bo = 2 * (first & 3);
        uint32_t const nbytes = (bo + 2 * len + 7) >> 3;                        // <= 9
        uint32_t const nq = (uint32_t)((addr & 3) + nbytes + 3) >> 2;          // <= 3
        uint32_t const w0 = __ldg(q), w1 = nq > 1 ? __ldg(q + 1) : 0u, w2 = nq > 2 ? __ldg(q + 2) : 0u;
        // bytes in memory order -> most significant byte first
        uint32_t const hi = __byte_perm(__funnelshift_r(w0, w1, sh), 0, 0x0123);
        uint32_t const lo = __byte_perm(__funnelshift_r(w1, w2, sh), 0, 0x0123);
        uint64_t v = ((uint64_t)hi << 32) | lo;
        if ( bo )
        {
                uint32_t const b8 = (w2 >> sh) & 0xFFu;                           // the ninth byte
                v = (v << bo) | (uint64_t)(b8 >> (8 - bo));
        }
        return len == 32 ? v : (v & (~0ULL << (64 - 2 * len)));
}

__device__ __forceinline__ const uint8_t * packed_read(ReadSrc const & S, uint32_t read)
{
        return S.packed + (S.ubytes ? (uint64_t)read * S.ubytes : __ldg(S.boffs + read));
}

// `len` (1..32) bases from base `first` on of strand id (= 2*read + strand) of a read of L bases, LEFT aligned.
// '-' strand = reverse complement of the read: its bases [first, first+len) are read[L-first-len, L-first) mirrored.
__device__ __forceinline__ uint64_t strand_bases(ReadSrc const & S, uint32_t id, uint32_t L, uint32_t first, uint32_t len)
{
        if ( S.rpack )
        {
                const uint64_t * rp = S.rpack + (uint64_t)id * S.W;
                uint32_t const w = first >> 5, o = 2 * (first & 31);
                uint64_t v = __ldg(rp + w);
                if ( o )
                {
                        v <<= o;
                        if ( o + 2 * len > 64 ) v |= __ldg(rp + w + 1) >> (64 - o);
                }
                return len == 32 ? v : (v & (~0ULL << (64 - 2 * len)));
        }
        const uint8_t * p = packed_read(S, id >> 1);
        if ( ! (id & 1) )
                return packed_bases(p, first, len);
        uint64_t const fwd = packed_bases(p, L - first - len, len) >> (64 - 2 * len);
        return revcomp_word(fwd, len) << (64 - 2 * len);
}

__device__ __forceinline__ uint64_t splitmix64(uint64_t x)
{
        uint64_t z = x + 0x9E3779B97F4A7C15ULL;
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
        return z ^ (z >> 31);
}

// slot of a pair signature in a presence table with 2^hb slots.  Signatures that already fit are
// used as they are (no collisions between different signatures); wider ones are folded, keeping
// their top SLOT_PREFIX_BITS bits in place so that a key prefix still selects a contiguous slice of the
// table (the multi-pass scan relies on that).
static const uint32_t SLOT_PREFIX_BITS = 8;
__host__ __device__ __forceinline__ uint32_t slot_of(uint64_t key, uint32_t keybits, uint32_t hb)
{
        if ( keybits <= hb )
                return (uint32_t)key;
        uint32_t const low = hb - SLOT_PREFIX_BITS;
        uint32_t const top = (uint32_t)(key >> (keybits - SLOT_PREFIX_BITS));
        return (top << low) | (uint32_t)((key * 0x9E3779B97F4A7C15ULL) >> (64 - low));
}

// Loads from the hot table slices (presence bits, entries).  Measured on B200
// (tools/l2_resident_bench.cu): loads issued as ld.global.nc.L1::no_allocate are kept in L2 with low
// priority -- a randomly probed 32 MB table already drops from ~278 to ~180 G probes/s, 64 MB to
// ~105 -- while plain loads or loads carrying an evict_last policy hold ~275 G/s up to 64 MB, also with
// a stream of touch-once data flowing through L2 at the same time.
__device__ __forceinline__ uint64_t policy_evict_normal()
{
        uint64_t pol;
        asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(pol));
        return pol;
}
__device__ __forceinline__ uint64_t policy_evict_first()
{
        uint64_t pol;
        asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
        return pol;
}
__device__ __forceinline__ uint32_t ld_hot_u32(const uint32_t * p, uint64_t pol)
{
        uint32_t v;
        asm volatile("ld.global.L2::cache_hint.u32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
        return v;
}
// probe of the presence table: a plain load (normal L2 priority).  The touch-once streams that pass through L2 at
// the same time (text records, entries) are loaded evict_first, which is what keeps the probed slice resident.
__device__ __forceinline__ SlotWord ld_slotword(const SlotWord * p)
{
        SlotWord v;
        asm volatile("ld.global.v2.u32 {%0,%1}, [%2];" : "=r"(v.bits), "=r"(v.rank) : "l"(p));
        return v;
}
__device__ __forceinline__ SlotWord ld_hot_slotword(const SlotWord * p, uint64_t pol)
{
        SlotWord v;
        asm volatile("ld.global.L2::cache_hint.v2.u32 {%0,%1}, [%2], %3;" : "=r"(v.bits), "=r"(v.rank) : "l"(p), "l"(pol));
        return v;
}
__device__ __forceinline__ uint4 ld_hot_v4(const void * p, uint64_t pol)
{
        uint4 v;
        asm volatile("ld.global.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p), "l"(pol));
        return v;
}

} // namespace realgpu
