// deflate.cu - L1 per-chunk DEFLATE with a preset dictionary (spec: README.md:288, 1159-1198;
// the skeleton's mz_deflateInit2(..., 15, ...) / mz_deflate(FINISH) at README.md:2374, 2378;
// resolved to one RFC 1950 stream per chunk with FDICT in SURVEY.md §0.2 C5).
//
// zlib walks hash chains serially; here the best match of EVERY position is found in parallel
// and the zlib level-6 lazy rule becomes a pure function next(p), so the parse is chain
// following.  Three kernels per batch of chunks, so that no phase leaves a CTA idle:
//
//  parse_kernel    one CTA per chunk (persistent, three size classes; the next chunk's descriptor and bytes are fetched
//                  while the current one is parsed).
//     P0 stage chunk in shared memory + Adler-32      P4 match search as RUNS, one lane per SORTED index: a
//     P1 histogram of 4-byte hashes (13 bits)            screen (own candidates = preceding lanes, dictionary
//     P2 scan -> bucket starts                            candidates = one 16-byte bucket record), pairs
//     P3 tile-ordered scatter; positions of one           compacted by ballots into two per-warp lists and
//        bucket that fell into one tile are put in        extended 32 at a time
//        order by the thread of their first slot      P4c prefix max of run ends -> match words
//        (positions ascending: nearest-first search,  P5 per-32-byte-range backward DP of chain exits
//        deterministic output)                         P6 hop the true chain across ranges
//                                                      P7 symbol histograms + compact u16 token stream
//  huffman_kernel  one WARP per chunk: length-limited Huffman lengths (two-queue merge by lane 0,
//                  everything else lane-parallel), canonical codes, dynamic header, block type
//                  choice (stored / fixed / dynamic by exact cost, like zlib).
//  encode_kernel   one CTA per chunk: token -> bit strings, block scan of bit counts, parallel
//                  emission (atomicOr only on words shared by two threads), zlib header/trailer.
//  pack_kernel     compacts the per-chunk stage slots into the caller's blob.
// Every stream inflates under stock zlib and the total size stays within 2 % of zlib level 6; beyond that every stream
// equals, byte for byte, the one of the test suite's sequential CPU model of these kernels (candidate sets, run heads
// with the sentinels below, lazy parse, Huffman codes, block types, multi-block and stored streams).
#include <stdlib.h>

#include <vector>

#include "ctx.cuh"
#include "deflate_core.h"

using namespace dfl;

namespace {

constexpr int OWN_CAP = 4;        // nearest own-chunk candidates examined per position, at most (large class)
// Own-chunk candidates per size class.  On the 8 KiB-average corpus most matches of a short chunk come from the preset
// dictionary: with two own candidates instead of four the small class loses 0.06 % (4 KiB chunks) to 0.2 % (8 KiB CDC
// chunks) of size and stays at zlib-6 parity (1.0001x), while a 32 KiB chunk would lose 1.8 % - so the depth follows
// the class (CPU size model of the test suite: own/dict 4/4, 3/4, 2/4 -> 0.9978 / 0.9985 / 1.0001 x zlib-6 on CDC chunks;
// 0.9982 / 0.9994 / 1.0020 on 16 KiB; 1.0051 / 1.0115 / 1.0231 on 32 KiB).
constexpr int OWN_SMALL = 2, OWN_MEDIUM = 3, OWN_LARGE = 4;
constexpr int DICT_CAP = 4;       // nearest dictionary candidates examined per position (one 16-byte bucket record)
constexpr int DICT_HASH_BITS = 15; // the dictionary index lives in global memory: finer buckets, fewer false candidates
constexpr uint32_t DICT_BUCKETS = 1u << DICT_HASH_BITS;
constexpr uint32_t DICT_MAX = 32768;
// Size classes of parse_kernel (bytes per chunk): the small class keeps its match words in shared memory, the medium
// and large ones in global scratch; small and medium fit two CTAs per SM, large one.  On the 8 KiB-average corpus
// 87 % of the bytes are small (<= 13 KiB: the most that lets two CTAs share an SM), 12.5 % medium (13-20 KiB), < 0.5 % large.
constexpr uint32_t NMAX_SMALL = 13312, NMAX_MEDIUM = 20480, NMAX_LARGE = 32768;
constexpr int N_CLASS = 3, LONG_CLASS = 3;   // class 3: longer than NMAX_LARGE (multi-block streams)
static_assert(NMAX_LARGE / 512 <= 64, "P3b keeps one moved-bit per element of a thread");
constexpr int T_PARSE = 512;
constexpr int TILE_SHIFT = 9;       // log2(T_PARSE): a scatter tile is T_PARSE consecutive positions
static_assert((1 << TILE_SHIFT) == T_PARSE, "TILE_SHIFT");
constexpr int T_ENCODE = 256;
constexpr int HUFF_WARPS = 8;
constexpr uint32_t BATCH_SMALL = 32768, BATCH_MEDIUM = 16384, BATCH_LARGE = 8192;  // chunks per batch (bounds the token scratch)
// Chunks longer than NMAX_LARGE become one zlib stream of several DEFLATE blocks of LONG_BLOCK input bytes.
// Block b >= 1 is parsed like any chunk, with the PREVIOUS block of the same chunk in the role of the preset
// dictionary (indexed on the device), which gives every position zlib's full 32 KiB window.
constexpr uint32_t LONG_BLOCK = 32768;
constexpr uint32_t BATCH_LONG = 96;   // blocks per batch: each carries a 0.5 MB dictionary index
// log2 of the range length of the chain passes in the small class.  16-byte ranges keep all 512 threads busy on an
// 8 KiB chunk but double the range-to-range hops of P6; measured slower (kt20 vs kt21), so both classes use 32.
constexpr int RS_SMALL = 5;
constexpr uint32_t REC_WORDS = 320;                          // 288 lit/len + 32 dist counters / codes

// Device image of the dictionary index (SLOT_DEFLATE_DICT), built on the host once per dictionary.
// One 16-byte record per bucket of 4-byte hashes: the four nearest (largest position first) dictionary
// positions of that bucket, each in the "K" layout that parse_kernel also gives every chunk position:
//     pos << 17 | 1 << 16 (valid) | tag << 8 | prev
// tag = byte 1 of the hash product (a filter only: phase B compares the real bytes), prev = the byte before pos
// (DICT_PREV0 before position 0).  One LDG.128 per chunk position screens all four candidates; a candidate c
// starts a run at a position with signature s iff ((c ^ s) & 0x1ffff) - 1 < 0xff (both valid, same tag, different
// previous byte), and it lies inside the window iff c >= threshold << 17 - two compares per candidate.
// The two sentinels differ, so chunk position 0 against dictionary position 0 is always a run head.  Being fixed bytes,
// they also decide three other pairs: no run starts at own source 0 against a position preceded by 0xFE, at chunk
// position 0 against a dictionary position preceded by 0xFE, or at dictionary position 0 against a chunk position
// preceded by 0xFF (the match is lost unless another candidate finds it).  Blocks of a long chunk see the same
// sentinels, not the real bytes before them.  Testing position 0 in the screen instead would add instructions to its
// hottest loop for at most about 1e-6 of the size (CPU model, CDC chunks: 0 bytes on int32 data, 1 byte in 1.38 MB on
// random bytes that are 60 % 0xFE / 0xFF; text never contains those bytes); the CPU model restates this rule (prev0 = 1).
constexpr uint32_t DICT_PREV0 = 0xFFu, CHUNK_PREV0 = 0xFEu;
struct DictDev {
    uint8_t bytes[DICT_MAX + 32];
    uint4 bk4[DICT_BUCKETS];
};

// Per-chunk record handed from kernel to kernel (indexed by job within the batch).
struct ChunkRec {
    uint32_t n;         // chunk length
    uint32_t n_words;   // u16 token words
    uint32_t adler;
    uint32_t mode;      // 0 stored, 1 fixed, 2 dynamic
    uint32_t hdr_bits;
    uint32_t flags;     // REC_MULTI: one block of a multi-block stream (never stored on its own); REC_LAST: BFINAL
    uint32_t bits;      // bits of the whole block (header + tokens + end-of-block) in the chosen mode
    uint32_t pad;
};
constexpr uint32_t REC_MULTI = 1, REC_LAST = 2;

struct DeflArgs {
    const uint8_t* data;
    uint64_t start0;
    const uint64_t* cuts;
    const uint64_t* select;  // may be null
    const DictDev* dict;
    uint32_t dict_len, dict_adler;
    int level;
    const uint32_t* list;    // selection slots of this size class (long class: one entry per BLOCK)
    const uint32_t* blk;     // long class: block number inside the chunk (null otherwise)
    const DictDev* long_dicts;  // long class: per batch job, the index of the previous block
    const uint8_t* stored_flag; // stored_kernel: only the list entries flagged here (null = all)
    uint32_t job0, job1;     // batch = list[job0 .. job1)
    uint32_t nmax;
    uint8_t* stage;
    const uint64_t* slot_off;
    uint64_t* sizes;
    uint32_t* match;         // per-CTA scratch, nmax words each (large class)
    uint16_t* tokens;        // [batch job][nmax] u16 words (<= one word per input byte)
    uint32_t* hist;          // [batch job][REC_WORDS]: symbol counts, then canonical codes
    uint8_t* hdrs;           // [batch job][640] dynamic header bytes
    ChunkRec* recs;          // [batch job]
    unsigned int* counter;
    unsigned long long* stat;  // per-call counters in ctx scratch: [0] token words, [1] input bytes, [2] chunks parsed
};

// Per-phase cycle counters of parse_kernel (thread 0 of every CTA, summed over chunks); read by
// hmse_debug_deflate_prof.  A dozen clock reads per chunk: negligible.
__device__ unsigned long long g_prof[16];
#define PROF(i)                                                     \
    if (t == 0) {                                                   \
        const long long now__ = clock64();                          \
        atomicAdd(&g_prof[i], (unsigned long long)(now__ - tprev)); \
        tprev = now__;                                              \
    }

constexpr uint32_t CNT_WORDS = NBUCKET / 2 + 36;  // bucket table; later the pair lists, then the 32 x 64 block-exit table
// Per-warp lists of (position, source) pairs awaiting extension, one for own-chunk sources and one for dictionary
// sources (each is extended by code that knows its address space).  A list holds < 32 left-overs plus what one window
// of 32 - OWN positions can add.
__host__ __device__ constexpr uint32_t own_cap(int own) { return (31u + (32u - own) * own + 7u) & ~7u; }
__host__ __device__ constexpr uint32_t dict_cap(int own) { return (31u + (32u - own) * DICT_CAP + 7u) & ~7u; }
__host__ __device__ constexpr uint32_t cnt_words(int own) {   // words of the bucket-table region (the pair lists may need more than the table)
    return (own_cap(own) + dict_cap(own)) * (T_PARSE / 32) > CNT_WORDS ? (own_cap(own) + dict_cap(own)) * (T_PARSE / 32) : CNT_WORDS;
}
constexpr uint32_t PAD_FRONT = 16;   // bytes before the chunk in shared memory: the last one is the "byte before position 0"
constexpr uint32_t BIG_GROUP = 16;   // P3b: same-tile groups up to this size are sorted by the thread of their first slot
constexpr uint32_t PAD_SORTED = 16;  // bytes between the chunk's slack and s_sorted (keeps the 16-byte alignment of what follows)

struct ParseSm {  // fixed-size shared state of parse_kernel
    uint32_t hist[REC_WORDS];
    uint16_t bentry[32];
    uint32_t warp_tmp[40];
    uint32_t job, blkno;        // the chunk (or block of a long chunk) being parsed: fetched by thread 0 while the
    uint64_t cs, len;           //   previous one was parsed (job >= job1: none left)
    uint64_t pf_cs;             // next chunk, announced early so that all threads can prefetch it into L2
    uint32_t pf_len, big_n;     // big_n: same-tile groups too long for one thread (P3b), sorted by the whole CTA
    uint32_t nx_job, nx_k, nx_blk, big_g;   // the descriptor being fetched (thread 0's state: kept here, not in registers
    uint64_t nx_j, nx_cs, nx_len;          //   that every thread would carry through all phases)
    uint32_t adler_a, adler_b;
    uint8_t lsym[256];          // length symbol - 257 of match length 3 + i (P7 looks it up instead of computing it)
};

// Dictionary bucket of a 4-byte value; the own-chunk bucket hash4(v) is its top HASH_BITS bits.
__host__ __device__ __forceinline__ uint32_t hash_dict(uint32_t v) { return (v * 0x9E3779B1u) >> (32 - DICT_HASH_BITS); }
// K-layout record of position `pos` whose four bytes are v and whose preceding byte is prev
constexpr uint32_t K_VALID = 0x10000u, K_LOW = 0x1ffffu, K_POS = 0xfffe0000u;
__host__ __device__ __forceinline__ uint32_t k_record(uint32_t v, uint32_t prev, uint32_t pos) {
    return (pos << 17) | K_VALID | ((v * 0x9E3779B1u) & 0xff00u) | prev;
}
__device__ __forceinline__ bool k_head(uint32_t cand, uint32_t sig) { return ((cand ^ sig) & K_LOW) - 1u < 0xffu; }

__device__ __forceinline__ uint32_t ld32u(const uint32_t* w, uint32_t off) {
    const uint32_t i = off >> 2;
    return __funnelshift_r(w[i], w[i + 1], (off & 3) * 8);
}
__device__ __forceinline__ uint32_t ldg32u(const uint8_t* base, uint32_t off) {
    const uint32_t* w = reinterpret_cast<const uint32_t*>(base) + (off >> 2);
    return __funnelshift_r(__ldg(w), __ldg(w + 1), (off & 3) * 8);
}

// Exclusive scan of one u32 per thread; *total = block sum (same value in every thread).  tmp = 32 words of shared
// memory.  ONE barrier: every warp folds the totals of the warps before it by itself (a REDUX) instead of waiting for a
// scan by warp 0 and two more barriers.  The caller keeps a barrier between two uses of the same tmp.
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t* tmp, uint32_t* total) {
    const unsigned lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (unsigned)o) inc += t;
    }
    if (lane == 31) tmp[w] = inc;
    __syncthreads();
    const uint32_t tv = lane < nw ? tmp[lane] : 0u;
    *total = __reduce_add_sync(0xffffffffu, tv);
    return inc - v + __reduce_add_sync(0xffffffffu, lane < w ? tv : 0u);
}

// Exclusive prefix MAX of one u32 per thread (identity 0), same scheme.
__device__ __forceinline__ uint32_t block_excl_scan_max(uint32_t v, uint32_t* tmp) {
    const unsigned lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (unsigned)o) inc = max(inc, t);
    }
    uint32_t exc = __shfl_up_sync(0xffffffffu, inc, 1);
    if (lane == 0) exc = 0;
    if (lane == 31) tmp[w] = inc;
    __syncthreads();
    const uint32_t tv = lane < nw && lane < w ? tmp[lane] : 0u;
    return max(exc, __reduce_max_sync(0xffffffffu, tv));
}

// Length of the common prefix of chunk[p ..] (shared memory words d32) and src[q ..] (generic pointer: the
// chunk itself or the dictionary text), continuing from l, at most lim; 8 bytes per step.
__device__ __forceinline__ uint32_t extend_run(const uint32_t* d32, const uint32_t* src, uint32_t p, uint32_t q,
                                               uint32_t l, uint32_t lim) {
    while (l < lim) {
        const uint32_t x0 = ld32u(d32, p + l) ^ ld32u(src, q + l);
        const uint32_t x1 = ld32u(d32, p + l + 4) ^ ld32u(src, q + l + 4);
        if (x0) {
            l += (uint32_t)(__ffs((int)x0) - 1) >> 3;
            break;
        }
        if (x1) {
            l += 4 + ((uint32_t)(__ffs((int)x1) - 1) >> 3);
            break;
        }
        l += 8;
    }
    return l > lim ? lim : l;
}

// Per-range passes touch element 32*r + j from lane r: a skew of one element per 32 makes those
// accesses conflict free in shared memory.
__device__ __forceinline__ uint32_t SK(uint32_t p) { return p + (p >> 5); }

// Shared-memory words addressed by their 32-bit shared-window address: the pair lists of P4 are written by predicated
// stores (no branch around a one-instruction body, whatever the compiler's mood) and read back the same way.
__device__ __forceinline__ void sts_if(uint32_t saddr, uint32_t v, bool p) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t@q st.shared.b32 [%0], %1;\n\t}" ::"r"(saddr), "r"(v), "r"((uint32_t)p));
}
__device__ __forceinline__ uint32_t lds_w(uint32_t saddr) {
    uint32_t v;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(saddr));
    return v;
}

// Global loads with an L1 policy.  Two CTAs of the small class leave the SM about 28 KB of L1: the dictionary TEXT (<= 32 KB,
// read by every extension step) should live there, so the loads that would wash it out do not allocate - the 512 KB of
// bucket records (one random 16-byte record per position) and the chunk bytes (read once).
__device__ __forceinline__ uint4 ldg_stream4(const uint4* p) {
    uint4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ uint32_t ldg_keep(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.global.nc.L1::evict_last.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}

// Match word: bits 16..24 length (0 = literal), bit 15 "lazy: emit as literal", bits 0..14 distance-1.
__device__ __forceinline__ bool mw_is_match(uint32_t mw) { return (mw >> 16) != 0 && !(mw & 0x8000u); }

// =================================================================================================
// parse_kernel
// =================================================================================================
// RS: log2 of the range length of the chain passes P4c-P7; OWN: own-chunk candidates per position; MSM: the match
// words live in shared memory (small class: every access to them is an LDS/STS/ATOMS with a 32-bit address) or in
// global scratch (a.match).
template <int RS, int OWN, bool MSM>
__global__ void __launch_bounds__(T_PARSE, 2) parse_kernel(DeflArgs a) {
    static_assert(OWN >= 1 && OWN <= OWN_CAP, "own candidates");
    constexpr int WIN = 32 - OWN;   // new sorted indices per window: the first OWN lanes only carry context
    constexpr uint32_t RL = 1u << RS;
    constexpr uint32_t CW = cnt_words(OWN);
    extern __shared__ __align__(16) uint8_t smem[];
    constexpr uint32_t T = T_PARSE;   // the launch uses exactly T_PARSE threads: strides and per-thread shares are constants
    const uint32_t t = threadIdx.x;
    const unsigned lane = t & 31, warp = t >> 5;
    constexpr unsigned nwarps = T >> 5;
    const uint32_t nmax = a.nmax;
    // layout: [PAD_FRONT | chunk, nmax + 16 | PAD_SORTED | sorted | bucket table | range entries | ParseSm | match words]
    uint32_t* s_data32 = reinterpret_cast<uint32_t*>(smem + PAD_FRONT);            // nmax + 16 bytes
    const uint8_t* s_data = smem + PAD_FRONT;
    const size_t o_sorted = (size_t)PAD_FRONT + nmax + 16 + PAD_SORTED;
    uint16_t* s_sorted = reinterpret_cast<uint16_t*>(smem + o_sorted);            // nmax u16 (later: exits, skewed)
    uint32_t* s_cnt32 = reinterpret_cast<uint32_t*>(smem + o_sorted + 2 * (size_t)(nmax + nmax / 32));  // CW words
    uint16_t* s_E = reinterpret_cast<uint16_t*>(s_cnt32);  // bucket h = sorted[E[h] .. E[h+1])
    uint8_t* s_entry = reinterpret_cast<uint8_t*>(s_cnt32 + CW);                  // nmax/16 bytes: entry offset of every range
    ParseSm* sm = reinterpret_cast<ParseSm*>(s_entry + nmax / 16);
    uint8_t* s_tail = reinterpret_cast<uint8_t*>(sm) + ((sizeof(ParseSm) + 15) & ~15u);
    // small class: match words in shared memory (skewed); the list of buckets to sort borrows that
    // space before P4.  large class: match words in global scratch, the list has its own space.
    uint32_t* mptr;
    if constexpr (MSM) mptr = reinterpret_cast<uint32_t*>(s_tail);
    else mptr = a.match + (size_t)blockIdx.x * (nmax + nmax / 32);
    uint16_t* s_exit = s_sorted;
    // the byte "before position 0" of every chunk (never equal to DICT_PREV0: (0, 0) is always a run head), so that the
    // signature of a position needs no special case for p == 0; never overwritten
    if (t == 0) {
        reinterpret_cast<uint32_t*>(smem)[PAD_FRONT / 4 - 1] = CHUNK_PREV0 << 24;
        sm->big_n = 0;
    }
    for (uint32_t i = t; i < 256; i += T) {
        uint32_t sy, eb, ev;
        len_sym(i + 3, sy, eb, ev);
        sm->lsym[i] = (uint8_t)(sy - 257);
    }

    // Thread 0 fetches the descriptor of the NEXT chunk while the current one is parsed, one dependent global load per
    // phase (work counter -> list -> selection -> cut points), so that a chunk starts without that chain of round trips;
    // as soon as the next chunk's bytes are known every thread prefetches a share of them into L2.
    auto next_job = [&](int step) {   // thread 0 only
        if (step == 0) sm->nx_job = a.job0 + atomicAdd(a.counter, 1u);
        const uint32_t nj = sm->nx_job;
        if (nj >= a.job1) return;
        if (step == 1) {
            sm->nx_k = a.list[nj];
            sm->nx_blk = a.blk ? a.blk[nj] : 0u;
        } else if (step == 2) {
            sm->nx_j = a.select ? a.select[sm->nx_k] : (uint64_t)sm->nx_k;
        } else if (step == 3) {
            const uint64_t j = sm->nx_j;
            const uint64_t c0 = j ? a.cuts[j - 1] : a.start0;
            sm->nx_cs = c0;
            sm->nx_len = a.cuts[j] - c0;
        }
    };
    auto publish_job = [&]() {        // thread 0 only, after the last reader of the current descriptor
        sm->job = sm->nx_job;
        sm->blkno = sm->nx_blk;
        sm->cs = sm->nx_cs;
        sm->len = sm->nx_len;
    };
    if (t == 0) {
        for (int st = 0; st < 4; st++) next_job(st);
        publish_job();
        sm->pf_len = 0;
    }
    for (;;) {
        __syncthreads();
        const uint32_t job = sm->job;
        if (job >= a.job1) break;
        long long tprev = clock64();
        const uint32_t bj = job - a.job0;  // index inside the batch
        uint64_t cs = sm->cs, len = sm->len;
        const uint32_t blkno = sm->blkno;
        uint32_t rec_flags = 0;
        if (a.blk) {   // one block of a long chunk
            rec_flags = REC_MULTI | ((uint64_t)(blkno + 1) * LONG_BLOCK >= len ? REC_LAST : 0u);
            cs += (uint64_t)blkno * LONG_BLOCK;
            len = len - (uint64_t)blkno * LONG_BLOCK < LONG_BLOCK ? len - (uint64_t)blkno * LONG_BLOCK : LONG_BLOCK;
        }
        const uint32_t n = (uint32_t)len;
        const uint8_t* src = a.data + cs;
        // the dictionary of this job: the preset one, or (blocks after the first) the previous block
        const DictDev* dict = blkno ? a.long_dicts + bj : a.dict;
        const uint32_t dlen = blkno ? LONG_BLOCK : a.dict_len;

        // ---- P0: stage the chunk (byte-unaligned source -> aligned words) with its Adler-32 partial sums
        //      taken from the words in flight (byte sum and position-weighted byte sum of a word are one
        //      instruction each), clear tables ---------------------------------------------------------
        {
            const uint32_t nw = (n + 3) >> 2;
            uint32_t sa = 0, sb = 0;   // sb <= 16 words x 32768 x 1020 per thread: no overflow
            auto sums = [&](uint32_t v, uint32_t wi) {   // Adler-32 partial sums of chunk word wi (already masked to the chunk)
                const uint32_t bs = __vsadu4(v, 0u);
                sa += bs;
                sb += (n - 4 * wi) * bs - __dp4a(v, 0x03020100u, 0u);   // sum over bytes of (n - position) * byte
            };
            const uint32_t mis = (uint32_t)((uintptr_t)src & 15);
            if (src - mis >= a.data) {
                // 16-byte vectors: every thread has all its loads in flight at once (two vectors of the chunk, each
                // assembled from the aligned vector it starts in and the next one), so the stage costs one memory round
                // trip instead of one per 4-byte word.  Source vector j holds bytes of the chunk iff j < nsrc: the last
                // one ends within the 16 bytes of slack the interface asks for.
                const uint4* vsrc = reinterpret_cast<const uint4*>(src - mis);
                const uint32_t nsrc = (n + mis + 15) >> 4;
                const uint32_t nvec = min((nw + 4 + 3) >> 2, (nmax + 16) / 16);   // output vectors, zero slack included
                const uint32_t q = mis >> 2, sh = (mis & 3) * 8;
                uint4* dst = reinterpret_cast<uint4*>(s_data32);
                auto emit = [&](uint32_t iv, const uint4& A, const uint4& B) {
                    const uint32_t s8[8] = {A.x, A.y, A.z, A.w, B.x, B.y, B.z, B.w};
                    uint32_t u[7], w[5], o[4];
#pragma unroll
                    for (int k = 0; k < 7; k++) u[k] = (q & 1) ? s8[k + 1] : s8[k];
#pragma unroll
                    for (int k = 0; k < 5; k++) w[k] = (q & 2) ? u[k + 2] : u[k];
#pragma unroll
                    for (int k = 0; k < 4; k++) {
                        const uint32_t wi = 4 * iv + k;
                        uint32_t v = __funnelshift_r(w[k], w[k + 1], sh);
                        if (wi >= nw) v = 0;
                        else if (n - 4 * wi < 4) v &= (1u << (8 * (n - 4 * wi))) - 1;
                        sums(v, wi);
                        o[k] = v;
                    }
                    dst[iv] = make_uint4(o[0], o[1], o[2], o[3]);
                };
                const uint4 z4 = make_uint4(0, 0, 0, 0);
                for (uint32_t iv = t; iv < nvec; iv += 2 * T) {
                    const uint32_t iv1 = iv + T;
                    uint4 A0 = z4, B0 = z4, A1 = z4, B1 = z4;
                    if (iv < nsrc) A0 = ldg_stream4(vsrc + iv);
                    if (mis && iv + 1 < nsrc) B0 = ldg_stream4(vsrc + iv + 1);
                    if (iv1 < nvec) {
                        if (iv1 < nsrc) A1 = ldg_stream4(vsrc + iv1);
                        if (mis && iv1 + 1 < nsrc) B1 = ldg_stream4(vsrc + iv1 + 1);
                    }
                    emit(iv, A0, B0);
                    if (iv1 < nvec) emit(iv1, A1, B1);
                }
            } else {   // a first chunk less than 16 bytes into a buffer that is only 4-byte aligned: word loads
                const uint32_t kmis = mis & 3;
                const uint32_t* wsrc = reinterpret_cast<const uint32_t*>(src - kmis);
                for (uint32_t i = t; i < nw + 4 && i < (nmax + 16) / 4; i += T) {
                    uint32_t v = 0;
                    if (i < nw) {
                        uint32_t lo = __ldg(wsrc + i);
                        uint32_t hi = kmis ? __ldg(wsrc + i + 1) : 0u;
                        v = __funnelshift_r(lo, hi, kmis * 8);
                        const uint32_t rem = n - 4 * i;  // bytes of this word inside the chunk
                        if (rem < 4) v &= (1u << (8 * rem)) - 1;
                        sums(v, i);
                    }
                    s_data32[i] = v;
                }
            }
            for (uint32_t i = t; i < CNT_WORDS; i += T) s_cnt32[i] = 0;   // (the bucket table proper: the rest of the region only holds pair lists)
            for (uint32_t i = t; i < REC_WORDS; i += T) sm->hist[i] = 0;
            sb %= 65521u;
            // only the two block totals are needed: one REDUX per warp, sixteen partial sums in shared memory
            const uint32_t wa = __reduce_add_sync(0xffffffffu, sa), wb = __reduce_add_sync(0xffffffffu, sb);
            if (lane == 0) {
                sm->warp_tmp[warp] = wa;        // <= 16 x 512 x 1020
                sm->warp_tmp[16 + warp] = wb;   // < 32 x 65521
            }
            __syncthreads();                    // (also orders the staging before its readers)
            if (warp == 0) {   // thread 0 is the only reader of the two sums (at the end of the chunk): no barrier after this
                const uint32_t tot_a = __reduce_add_sync(0xffffffffu, lane < nwarps ? sm->warp_tmp[lane] : 0u);
                const uint32_t tot_b = __reduce_add_sync(0xffffffffu, lane < nwarps ? sm->warp_tmp[16 + lane] : 0u);
                if (lane == 0) {
                    sm->adler_a = (1u + tot_a) % 65521u;
                    sm->adler_b = (n % 65521u + tot_b) % 65521u;
                }
            }
        }
        PROF(0)
        if (t == 0 && a.level != 0) next_job(0);
        const uint32_t nh = n >= 4 ? n - 3 : 0;  // hashed positions
        PROF(1)
        uint32_t n_words = 0;
        // 13-bit hash of every position, kept for the scatter and the bucket fix-up (upper half of the match words,
        // which are not written before P4)
        uint16_t* s_h16 = reinterpret_cast<uint16_t*>(mptr) + nmax;
        if (a.level != 0) {
            // ---- P1: hash histogram (count of bucket h lives at E[h+1]); four positions per step from two words ----
            for (uint32_t i = t; 4 * i < nh; i += T) {
                const uint32_t w0 = s_data32[i], w1 = s_data32[i + 1];
                uint32_t hh[4];
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    hh[q] = hash4(q ? __funnelshift_r(w0, w1, 8 * q) : w0);
                    if (4 * i + q < nh) {
                        const uint32_t h1 = hh[q] + 1;
                        atomicAdd(&s_cnt32[h1 >> 1], 1u << (16 * (h1 & 1)));
                    }
                }
                reinterpret_cast<uint2*>(s_h16)[i] = make_uint2(hh[0] | (hh[1] << 16), hh[2] | (hh[3] << 16));
            }
            __syncthreads();
            // ---- P2: exclusive scan: E[h+1] = start of bucket h (cursor), E[0] = 0.  E[0] holds no count, so this is
            //      the exclusive scan of the u16 array E[0 .. NBUCKET] itself.  A thread owns two 16-byte vectors, one in
            //      each half of the table (consecutive lanes read consecutive vectors: conflict-free LDS.128), scans its
            //      16 entries in registers, and ONE block scan carries both halves at once (half A in the low 16 bits of
            //      the packed sum, half B in the high 16: neither exceeds 32765).
            {
                static_assert(NBUCKET / 2 == 8 * T_PARSE, "two 16-byte vectors per thread");
                uint4* v4 = reinterpret_cast<uint4*>(s_cnt32);
                const uint4 va = v4[t], vb = v4[T_PARSE + t];
                uint32_t wa[4] = {va.x, va.y, va.z, va.w}, wb[4] = {vb.x, vb.y, vb.z, vb.w};
                uint32_t sa = 0, sb = 0;
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    sa += (wa[q] & 0xffffu) + (wa[q] >> 16);
                    sb += (wb[q] & 0xffffu) + (wb[q] >> 16);
                }
                const uint32_t packed = sa | (sb << 16);
                uint32_t inc = packed;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t tt = __shfl_up_sync(0xffffffffu, inc, o);
                    if (lane >= (unsigned)o) inc += tt;
                }
                if (lane == 31) sm->warp_tmp[warp] = inc;
                __syncthreads();
                // every warp folds the totals of the warps before it by itself (packed sums: no carry between the halves)
                const uint32_t tv = lane < nwarps ? sm->warp_tmp[lane] : 0u;
                const uint32_t tot = __reduce_add_sync(0xffffffffu, tv);
                const uint32_t ex = inc - packed + __reduce_add_sync(0xffffffffu, lane < warp ? tv : 0u);
                if (t == 0) s_E[NBUCKET] = (uint16_t)((tot & 0xffffu) + (tot >> 16));   // the entry past the last full word: everything before it
                uint32_t ra = ex & 0xffffu, rb = (ex >> 16) + (tot & 0xffffu);
#pragma unroll
                for (int q = 0; q < 4; q++) {   // word = E[2k] | E[2k+1] << 16 -> run | (run + E[2k]) << 16
                    const uint32_t ca = wa[q], cb = wb[q];
                    wa[q] = ra * 0x10001u + (ca << 16);
                    wb[q] = rb * 0x10001u + (cb << 16);
                    ra += (ca & 0xffffu) + (ca >> 16);
                    rb += (cb & 0xffffu) + (cb >> 16);
                }
                v4[t] = make_uint4(wa[0], wa[1], wa[2], wa[3]);
                v4[T_PARSE + t] = make_uint4(wb[0], wb[1], wb[2], wb[3]);
            }
            __syncthreads();
            PROF(2)
            if (t == 0) next_job(1);
            // ---- P3: scatter tile by tile (cursors count up to the bucket ends): buckets end up ordered by position
            //      except for same-hash positions that were scattered in the same tile (common in text: a word repeated
            //      within 512 bytes).  Such a group is contiguous in the bucket, and it is complete at the barrier that
            //      ends its tile: in the next trip every thread looks at the slot to the right of the one it filled - a
            //      position of the same tile there (same tile <=> the two differ only below the tile bits) makes the slot
            //      a candidate for the fix-up below.  The test runs in the shadow of the next tile's atomic; a slot the
            //      chunk has not filled yet holds a stale position, which at worst adds a candidate.
            //      The loop is a three-stage pipeline, one barrier a trip: a trip ISSUES the atomic of its tile and goes to
            //      the barrier without touching the result (the barrier orders the atomics of consecutive tiles whether or
            //      not their values have come back); the next trip stores the position into the slot the atomic returned;
            //      the trip after that looks at the right-hand neighbour.
            uint16_t* wlist = reinterpret_cast<uint16_t*>(mptr) + warp * (nmax / 16);   // <= 32 candidates per tile and warp
            uint32_t wcnt = 0;   // warp-uniform
            {
                if (t == 0) s_sorted[nh] = 0xFFFFu;   // no tile holds position 0xFFFF
                const uint32_t lt = (1u << lane) - 1u;
                constexpr uint32_t NONE = 0xffffffffu;
                uint32_t chk_slot = NONE, chk_p = 0;   // stored in the trip before: neighbour not looked at yet
                uint32_t hn = t < nh ? (uint32_t)s_h16[t] : 0u;   // the hash of the position this trip scatters
                // cur_*: this trip's atomic (issued here, consumed in the next trip); prv_*: the one issued a trip ago
                auto trip = [&](uint32_t p0, uint32_t& cur_old, uint32_t& cur_sh, uint32_t& cur_p, uint32_t prv_old, uint32_t prv_sh,
                                uint32_t prv_p) {
                    const uint32_t p = p0 + t;
                    cur_p = NONE;
                    if (p < nh) {
                        const uint32_t h1 = hn + 1;
                        cur_sh = 16 * (h1 & 1);
                        cur_old = atomicAdd(&s_cnt32[h1 >> 1], 1u << cur_sh);
                        cur_p = p;
                    }
                    const bool cand = chk_slot != NONE && ((uint32_t)s_sorted[chk_slot + 1] ^ chk_p) < (uint32_t)T_PARSE;
                    const uint32_t b = __ballot_sync(0xffffffffu, cand);
                    if (cand) wlist[wcnt + __popc(b & lt)] = (uint16_t)chk_slot;
                    wcnt += __popc(b);
                    chk_slot = NONE;
                    if (prv_p != NONE) {
                        chk_slot = (prv_old >> prv_sh) & 0xffffu;
                        chk_p = prv_p;
                        s_sorted[chk_slot] = (uint16_t)prv_p;
                    }
                    if (p + T < nh) hn = s_h16[p + T];
                    __syncthreads();
                };
                uint32_t oa = 0, sa = 0, pa = NONE, ob = 0, sb = 0, pb = NONE;
                for (uint32_t p0 = 0; p0 < nh + 2 * T; p0 += 2 * T) {   // the last two trips only drain the pipeline
                    trip(p0, oa, sa, pa, ob, sb, pb);
                    trip(p0 + T, ob, sb, pb, oa, sa, pa);
                }
            }
            PROF(3)
            if (t == 0) next_job(2);
            // ---- P3b: the element in the FIRST slot of a group (a neighbour belongs to the same bucket iff its stored hash
            //      agrees) sorts the whole group in place - groups are tiny, and one thread per group means no temporary
            //      copy: whatever a concurrent reader finds in a slot of a group that is being sorted is some member of that
            //      group, which has the tile and the bucket the reader tests for.
            {
                auto sort_group = [&](uint32_t i) {   // i: a candidate slot
                    const uint32_t p = s_sorted[i], r = s_sorted[i + 1];
                    const uint32_t h = s_h16[p];
                    if ((r ^ p) >= (uint32_t)T_PARSE || s_h16[r] != h) return;          // another tile, or the next bucket
                    if (i) {
                        const uint32_t l = s_sorted[i - 1];
                        if ((l ^ p) < (uint32_t)T_PARSE && s_h16[l] == h) return;       // not the first slot of its group
                    }
                    uint32_t g = 2;
                    for (; g <= BIG_GROUP; g++) {                                         // (the sentinel at nh ends the last group)
                        const uint32_t q = s_sorted[i + g];
                        if ((q ^ p) >= (uint32_t)T_PARSE || s_h16[q] != h) break;
                    }
                    if (g > BIG_GROUP) {   // repetitive data (a run of one byte fills a tile with ONE group): left to the whole CTA
                        s_cnt32[atomicAdd(&sm->big_n, 1u)] = i;
                        return;
                    }
                    for (uint32_t x = 1; x < g; x++) {                                    // insertion sort of g (mostly 2) positions
                        const uint32_t v = s_sorted[i + x];
                        uint32_t y = x;
                        for (; y > 0; y--) {
                            const uint32_t u = s_sorted[i + y - 1];
                            if (u < v) break;
                            s_sorted[i + y] = (uint16_t)u;
                        }
                        s_sorted[i + y] = (uint16_t)v;
                    }
                };
                __syncwarp();
                for (uint32_t j = lane; j < wcnt; j += 32) sort_group(wlist[j]);
            }
            __syncthreads();
            if (const uint32_t nbig = sm->big_n) {   // CTA-uniform; never taken on text
                // A long group (up to a whole tile) by all threads: its extent by one test per slot and a minimum, then a
                // rank sort - thread x counts the members smaller than its own (all positions differ) and moves it there.
                // One thread would need a quadratic number of dependent steps: milliseconds per chunk on constant data.
                for (uint32_t bg = 0; bg < nbig; bg++) {
                    const uint32_t i0 = s_cnt32[bg];
                    const uint32_t p = s_sorted[i0], h = s_h16[p];
                    if (t == 0) sm->big_g = T;
                    __syncthreads();
                    {
                        const uint32_t q = i0 + t <= nh ? (uint32_t)s_sorted[i0 + t] : 0xFFFFu;
                        if ((q ^ p) >= (uint32_t)T_PARSE || s_h16[q & 0x7fffu] != h) atomicMin(&sm->big_g, t);
                    }
                    __syncthreads();
                    const uint32_t g = sm->big_g;
                    uint32_t v = 0, rank = 0;
                    if (t < g) {
                        v = s_sorted[i0 + t];
                        for (uint32_t j = 0; j < g; j++) rank += (uint32_t)s_sorted[i0 + j] < v;
                    }
                    __syncthreads();
                    if (t < g) s_sorted[i0 + rank] = (uint16_t)v;
                }
                __syncthreads();
                if (t == 0) sm->big_n = 0;
            }
            PROF(4)
            if (t == 0) {   // the next chunk's bytes are known: announce them for the L2 prefetch below
                next_job(3);
                uint64_t pc = sm->nx_cs, pl = sm->nx_len;
                if (a.blk) {
                    pc += (uint64_t)sm->nx_blk * LONG_BLOCK;
                    pl = pl - (uint64_t)sm->nx_blk * LONG_BLOCK < LONG_BLOCK ? pl - (uint64_t)sm->nx_blk * LONG_BLOCK : LONG_BLOCK;
                }
                sm->pf_cs = pc;
                sm->pf_len = sm->nx_job < a.job1 ? (uint32_t)pl : 0u;
            }
            // ---- P4: matches as RUNS.  A pair (position p, source q) whose four bytes agree and whose
            //      preceding bytes differ starts a run: every position p+k inside it has a match of
            //      length end-(p+k) at the same distance, so only run heads are extended and
            //      best[p] = (prefix max over start positions of the run ends) - p  (P4c below).
            //      Phase A, one lane per SORTED index (windows of 32 - OWN lanes + OWN lanes of context), is a
            //      pure screen: the nearest own candidates are the preceding lanes (their signatures come
            //      by shuffle), the four nearest dictionary candidates come in one 16-byte bucket record.
            //      The surviving (position, source) pairs are compacted slot by slot (one ballot each) into two
            //      per-warp lists - own-chunk sources and dictionary sources - and extended 32 at a time
            //      (phase B), so the byte comparison runs with full warps, from shared memory for the one
            //      list and through the read-only path for the other.
            for (uint32_t i = t; i < n + (n >> 5); i += T) mptr[i] = 0;   // run keys: end << 15 | (32768 - dist)
            __syncthreads();
            {   // the next chunk, one 128-byte line per thread: in L2 by the time its P0 runs
                const uint32_t pl = sm->pf_len;
                const uint8_t* pb = a.data + sm->pf_cs;
                for (uint32_t o = t * 128u; o < pl; o += T * 128u) asm volatile("prefetch.global.L2 [%0];" ::"l"(pb + o));
            }
            {
                const uint32_t* dictw = reinterpret_cast<const uint32_t*>(dict->bytes);
                const uint4* bk4 = dict->bk4;
                const bool use_dict = dlen != 0;
                // the bucket table is dead (E is not needed to walk s_sorted): its region holds the pair lists
                // (lists are addressed by shared-window addresses: 32-bit arithmetic, one multiply-add per store)
                const uint32_t olist = (uint32_t)__cvta_generic_to_shared(s_cnt32) + warp * 4u * (own_cap(OWN) + dict_cap(OWN));
                const uint32_t dlist = olist + 4u * own_cap(OWN);
                uint32_t otop = olist, dtop = dlist;           // list ends (warp-uniform)
                const uint32_t lt = (1u << lane) - 1u;
                const uint32_t nwin = (nh + WIN - 1) / WIN;
                const int win_gap = (int)WSIZE - (int)dlen;    // a dictionary position q is inside the window of p iff q + win_gap >= p
                const uint32_t* smem32 = reinterpret_cast<const uint32_t*>(smem);
                struct StA { uint32_t sig; uint4 bk; };
                // sig: the K-layout record of the lane's position (pos << 17 | valid | tag << 8 | previous byte); lanes
                // outside the index range carry 0
                // (the bucket record of a lane without a position keeps its old value: nothing reads it while sig == 0)
                auto stageA = [&](uint32_t w, StA& r) {
                    r.sig = 0;
                    const int i = (int)(WIN * w) - OWN + (int)lane;
                    // (a window past the last one only reads in-range context elements that nobody consumes)
                    if ((uint32_t)i < nh) {
                        const uint32_t p = s_sorted[i];
                        // bytes p-1 .. p+3 lie in two consecutive words: one pair of loads serves both the value and
                        // the byte before it (position 0 finds CHUNK_PREV0 in the pad before the chunk)
                        const uint32_t off = p + (PAD_FRONT - 1);
                        const uint32_t w0 = smem32[off >> 2], w1 = smem32[(off >> 2) + 1];
                        const uint32_t o3 = off & 3u;
                        const uint32_t v = __funnelshift_rc(w0, w1, o3 * 8u + 8u);   // bytes p .. p+3 (clamped shift: 32 -> w1)
                        const uint32_t prod = v * 0x9E3779B1u;
                        // byte 0 <- byte o3 of w0 (the previous byte), byte 1 <- byte 1 of the product (the tag)
                        const uint32_t lowh = __byte_perm(w0, prod, o3 | 0x50u);
                        r.sig = (lowh & 0xffffu) | (p * 0x20000u + K_VALID);
                        if (use_dict && lane >= OWN) r.bk = ldg_stream4(&bk4[prod >> (32 - DICT_HASH_BITS)]);
                    }
                };
                // phase B: common prefix of chunk[p ..] and src[q ..], 8 bytes per step from three words a side
                auto extend_own = [&](uint32_t first, uint32_t count) {
                    if (lane < count) {
                        const uint32_t rec = lds_w(first + 4u * lane);
                        const uint32_t p = rec & 0x7fffu, q = rec >> 17;
                        const uint32_t lim = n - p;
                        const uint32_t sa = p * 8u, sb = q * 8u;   // funnel shifts take the amount modulo 32
                        const uint32_t* A = s_data32 + (p >> 2);
                        const uint32_t* B = s_data32 + (q >> 2);
                        uint32_t a0 = A[0], b0 = B[0], l = 0;
                        for (;;) {
                            const uint32_t a1 = A[1], a2 = A[2], b1 = B[1], b2 = B[2];
                            const uint32_t x0 = __funnelshift_r(a0, a1, sa) ^ __funnelshift_r(b0, b1, sb);
                            if (x0) {
                                l += (uint32_t)(__ffs((int)x0) - 1) >> 3;
                                break;
                            }
                            const uint32_t x1 = __funnelshift_r(a1, a2, sa) ^ __funnelshift_r(b1, b2, sb);
                            if (x1) {
                                l += 4 + ((uint32_t)(__ffs((int)x1) - 1) >> 3);
                                break;
                            }
                            l += 8;
                            if (l >= lim) break;
                            a0 = a2; b0 = b2;
                            A += 2; B += 2;
                        }
                        l = min(l, lim);
                        if (l >= 4) atomicMax(&mptr[SK(p)], ((p + l) << 15) | (32768u - (p - q)));
                    }
                };
                auto extend_dict = [&](uint32_t first, uint32_t count) {
                    if (lane < count) {
                        const uint32_t rec = lds_w(first + 4u * lane);
                        const uint32_t p = rec & 0x7fffu, q = rec >> 17;
                        const uint32_t lim = min(n - p, dlen - q);   // matches do not run from the dictionary into the chunk
                        const uint32_t sa = p * 8u, sb = q * 8u;
                        const uint32_t* A = s_data32 + (p >> 2);
                        const uint32_t* B = dictw + (q >> 2);
                        uint32_t a0 = A[0], b0 = ldg_keep(B), l = 0;
                        for (;;) {
                            const uint32_t a1 = A[1], a2 = A[2], b1 = ldg_keep(B + 1), b2 = ldg_keep(B + 2);
                            const uint32_t x0 = __funnelshift_r(a0, a1, sa) ^ __funnelshift_r(b0, b1, sb);
                            if (x0) {
                                l += (uint32_t)(__ffs((int)x0) - 1) >> 3;
                                break;
                            }
                            const uint32_t x1 = __funnelshift_r(a1, a2, sa) ^ __funnelshift_r(b1, b2, sb);
                            if (x1) {
                                l += 4 + ((uint32_t)(__ffs((int)x1) - 1) >> 3);
                                break;
                            }
                            l += 8;
                            if (l >= lim) break;
                            a0 = a2; b0 = b2;
                            A += 2; B += 2;
                        }
                        l = min(l, lim);
                        if (l >= 4) atomicMax(&mptr[SK(p)], ((p + l) << 15) | (32768u - (p + dlen - q)));
                    }
                };
                // phase A on one staged window.  A candidate (own: the signature of a preceding lane; dictionary: a
                // bucket record) starts a run here when k_head() holds - both valid, the same tag, a different previous
                // byte; the tag is only a filter (same bucket and same tag, different bytes: 1 in 256): phase B compares
                // the real bytes from the first one.
                auto screen = [&](const StA& cur) {
                    const uint32_t sig = cur.sig;
                    const bool act = lane >= OWN && sig != 0;
                    const uint32_t p = sig >> 17;
                    // inside the window  <=>  pos + (WSIZE - dlen) >= p  <=>  record >= max(p - (WSIZE - dlen), 0) << 17
                    const uint32_t thrK = (uint32_t)max((int)p - win_gap, 0) << 17;
                    const uint32_t c[DICT_CAP] = {cur.bk.x, cur.bk.y, cur.bk.z, cur.bk.w};
                    uint32_t sq[OWN];
                    bool ho[OWN], hd[DICT_CAP];
                    uint32_t bo[OWN], bd[DICT_CAP];
                    // all tests first, then all ballots, then the stores: six independent chains
#pragma unroll
                    for (int d = 0; d < OWN; d++) {
                        sq[d] = __shfl_up_sync(0xffffffffu, sig, d + 1);   // (a lane below d + 1 reads itself: never a head)
                        ho[d] = act && k_head(sq[d], sig);
                    }
#pragma unroll
                    for (int u = 0; u < DICT_CAP; u++) hd[u] = act && c[u] >= thrK && k_head(c[u], sig);
#pragma unroll
                    for (int d = 0; d < OWN; d++) bo[d] = __ballot_sync(0xffffffffu, ho[d]);
#pragma unroll
                    for (int u = 0; u < DICT_CAP; u++) bd[u] = __ballot_sync(0xffffffffu, hd[u]);
#pragma unroll
                    for (int d = 0; d < OWN; d++) {
                        sts_if(otop + 4u * __popc(bo[d] & lt), (sq[d] & K_POS) | p, ho[d]);
                        otop += 4u * __popc(bo[d]);
                    }
#pragma unroll
                    for (int u = 0; u < DICT_CAP; u++) {
                        sts_if(dtop + 4u * __popc(bd[u] & lt), (c[u] & K_POS) | p, hd[u]);
                        dtop += 4u * __popc(bd[u]);
                    }
                    __syncwarp();
                    while (otop - olist >= 128u) {
                        otop -= 128u;
                        extend_own(otop, 32);
                    }
                    while (dtop - dlist >= 128u) {
                        dtop -= 128u;
                        extend_dict(dtop, 32);
                    }
                    __syncwarp();
                };
                // two windows in flight per warp; each staged window is refilled right after it is consumed, so the
                // staging registers never move
                StA s0, s1;
                s0.bk = s1.bk = make_uint4(0, 0, 0, 0);
                stageA(warp, s0);
                stageA(warp + nwarps, s1);
                for (uint32_t w = warp; w < nwin;) {   // warp-uniform trip count
                    screen(s0);
                    stageA(w + 2 * nwarps, s0);
                    w += nwarps;
                    if (w >= nwin) break;
                    screen(s1);
                    stageA(w + 2 * nwarps, s1);
                    w += nwarps;
                }
                if (otop != olist) extend_own(olist, (otop - olist) >> 2);
                if (dtop != dlist) extend_dict(dlist, (dtop - dlist) >> 2);
            }
            __syncthreads();
            PROF(5)

            // ranges of RL positions (16 in the small class, so that all threads have one; 32 in the large),
            // blocked over threads; within a range the skewed index is SK(first) + offset
            const uint32_t R = (n + RL - 1) >> RS;
            const uint32_t rpt = (R + T - 1) / T;
            const uint32_t r0 = t * rpt, r1 = (r0 + rpt < R) ? r0 + rpt : R;
            // ---- P4c: run keys -> match words: a forward prefix max over positions (thread-local over its
            //      own ranges, one block scan of the per-thread maxima in between) ---------------------------
            {
                uint32_t loc = 0;
                for (uint32_t r = r0; r < r1; r++) {
                    const uint32_t ps = r << RS, cnt = (ps + RL < n) ? RL : n - ps;
                    const uint32_t* mp = mptr + SK(ps);
                    for (uint32_t q = 0; q < cnt; q++) loc = max(loc, mp[q]);
                }
                uint32_t run = block_excl_scan_max(loc, sm->warp_tmp);
                for (uint32_t r = r0; r < r1; r++) {
                    const uint32_t ps = r << RS, cnt = (ps + RL < n) ? RL : n - ps;
                    uint32_t* mp = mptr + SK(ps);
                    for (uint32_t q = 0; q < cnt; q++) {
                        run = max(run, mp[q]);
                        const uint32_t end = run >> 15, p = ps + q;
                        uint32_t mw = 0;
                        if (end >= p + 4) {
                            const uint32_t L = min(end - p, (uint32_t)MAX_MATCH);
                            mw = (L << 16) | (32767u - (run & 0x7fffu));
                        }
                        mp[q] = mw;
                    }
                }
            }
            __syncthreads();
            PROF(9)
            // ---- P5: backward DP: exit[p] = first chain position past p's range -------------
            for (uint32_t r = r0; r < r1; r++) {
                const uint32_t ps = r << RS, pe = (ps + RL < n) ? ps + RL : n;
                uint32_t nxt_len = pe < n ? (mptr[SK(pe)] >> 16) : 0;
                uint32_t* mp = mptr + SK(ps);
                uint16_t* xp = s_exit + SK(ps);
                for (uint32_t q = pe - ps; q-- > 0;) {
                    const uint32_t mw = mp[q];
                    const uint32_t L = mw >> 16;
                    const bool lazy_lit = L != 0 && L < (uint32_t)MAX_LAZY && nxt_len > L;
                    if (lazy_lit) mp[q] = mw | 0x8000u;
                    const uint32_t next = ps + q + ((L == 0 || lazy_lit) ? 1u : L);
                    xp[q] = (uint16_t)(next >= pe ? next : xp[next - ps]);
                    nxt_len = L;
                }
            }
            for (uint32_t r = t; r < R; r += T) s_entry[r] = 0xFF;
            __syncthreads();
            PROF(6)
            // ---- P6: hop the true chain across ranges, two levels.  A warp owns a block of 32 ranges
            //      (1024 bytes).  (a) lane e follows the chain that enters the block's first ranges at
            //      the e-th possible position and records where it leaves the block; (b) one thread
            //      hops block to block through those tables; (c) lane 0 of every warp re-walks its block
            //      from the true entry and marks the per-range entries. -----------------------------------
            {
                uint16_t* s_bexit = s_E;          // [block][258]: exit of a chain entering the block at offset o (E is dead)
                uint16_t* s_bentry = sm->bentry;  // [block]: true entry position (0xFFFF = not visited)
                const uint32_t NB = (n + 1023) >> 10;
                // (a) a chain almost always enters a block within its first 64 positions (only a match
                //     longer than that jumps further); those 64 entry points are tabulated in parallel
                for (uint32_t item = warp; item < 2 * NB; item += nwarps) {
                    const uint32_t blk = item >> 1, o = ((item & 1) << 5) + lane;
                    const uint32_t bs = blk << 10, be = (bs + 1024 < n) ? bs + 1024 : n;
                    if (bs + o < be) {
                        uint32_t p = bs + o;
                        while (p < be) p = s_exit[SK(p)];
                        s_bexit[blk * 64 + o] = (uint16_t)p;
                    }
                    if ((item & 1) == 0 && lane == 0) s_bentry[blk] = 0xFFFF;
                }
                __syncthreads();
                if (t == 0) {  // (b)
                    uint32_t p = 0;
                    while (p < n) {
                        const uint32_t blk = p >> 10, o = p & 1023;
                        s_bentry[blk] = (uint16_t)p;
                        if (o < 64) {
                            p = s_bexit[blk * 64 + o];
                        } else {  // rare: walk this block directly
                            const uint32_t be = ((blk << 10) + 1024 < n) ? (blk << 10) + 1024 : n;
                            while (p < be) p = s_exit[SK(p)];
                        }
                    }
                }
                __syncthreads();
                for (uint32_t blk = warp; blk < NB; blk += nwarps) {  // (c)
                    if (lane == 0 && s_bentry[blk] != 0xFFFF) {
                        const uint32_t be = ((blk << 10) + 1024 < n) ? (blk << 10) + 1024 : n;
                        uint32_t p = s_bentry[blk];
                        while (p < be) {
                            s_entry[p >> RS] = (uint8_t)(p & (RL - 1));
                            p = s_exit[SK(p)];
                        }
                    }
                }
            }
            __syncthreads();
            PROF(7)
            // ---- P7: symbol histograms + token words (literal: byte; match: 0x8000|len, dist-1).  A thread walks the
            //      tokens of its ranges twice (count, then write); lanes hold literals and matches at the same time, so a
            //      step is written without a branch on the token kind: the first symbol is the byte or a looked-up length
            //      symbol, the distance symbol comes from a logarithm and is counted under a predicate. ----
            uint32_t words = 0;
            for (uint32_t r = r0; r < r1; r++) {
                const uint32_t e = s_entry[r];
                if (e == 0xFF) continue;
                const uint32_t pe = ((r << RS) + RL < n) ? (r << RS) + RL : n;
                for (uint32_t p = (r << RS) + e; p < pe;) {
                    const uint32_t mw = mptr[SK(p)];
                    const bool m = mw_is_match(mw);
                    const uint32_t L = mw >> 16, d = mw & 0x7fffu;   // d = distance - 1
                    const uint32_t s1 = m ? 257u + sm->lsym[m ? L - 3 : 0u] : (uint32_t)s_data[p];
                    atomicAdd(&sm->hist[s1], 1u);
                    const uint32_t eb = (uint32_t)(31 - __clz((int)(d | 2u))) - 1u;   // 0 for d < 4
                    const uint32_t sy = d < 4 ? d : 2 * eb + 2 + ((d >> eb) & 1u);
                    if (m) atomicAdd(&sm->hist[288 + sy], 1u);
                    words += m ? 2u : 1u;
                    p += m ? L : 1u;
                }
            }
            uint32_t w_off = block_excl_scan(words, sm->warp_tmp, &n_words);
            // the token words are gathered in shared memory (the exit table is dead after P6) and leave as 16-byte
            // vectors: written where they are produced, every 2-byte store of a warp would touch its own 32-byte sector
            uint16_t* s_tok = s_exit;   // n_words <= n
            for (uint32_t r = r0; r < r1; r++) {
                const uint32_t e = s_entry[r];
                if (e == 0xFF) continue;
                const uint32_t pe = ((r << RS) + RL < n) ? (r << RS) + RL : n;
                for (uint32_t p = (r << RS) + e; p < pe;) {
                    const uint32_t mw = mptr[SK(p)];
                    const bool m = mw_is_match(mw);
                    const uint32_t L = mw >> 16;
                    s_tok[w_off] = m ? (uint16_t)(0x8000u | L) : (uint16_t)s_data[p];
                    if (m) s_tok[w_off + 1] = (uint16_t)(mw & 0x7fffu);
                    w_off += m ? 2u : 1u;
                    p += m ? L : 1u;
                }
            }
            __syncthreads();
            {
                uint4* tk4 = reinterpret_cast<uint4*>(a.tokens + (size_t)bj * nmax);   // nmax is a multiple of 8 words
                const uint4* st4 = reinterpret_cast<const uint4*>(s_tok);
                for (uint32_t i = t; i < (n_words + 7) / 8; i += T) tk4[i] = st4[i];   // (the last vector may carry stale words)
            }
            for (uint32_t i = t; i < REC_WORDS; i += T)
                a.hist[(size_t)bj * REC_WORDS + i] = sm->hist[i] + (i == (uint32_t)EOB ? 1u : 0u);
        }
        if (t == 0) {
            ChunkRec rec;
            rec.n = n;
            rec.n_words = n_words;
            rec.adler = (sm->adler_b << 16) | sm->adler_a;
            rec.mode = a.level == 0 ? 0u : 2u;
            rec.hdr_bits = 0;
            rec.flags = rec_flags;
            rec.bits = 0;
            rec.pad = 0;
            a.recs[bj] = rec;
            if (a.level == 0)
                for (int st = 0; st < 4; st++) next_job(st);
            publish_job();
            atomicAdd(&a.stat[0], (unsigned long long)n_words);
            atomicAdd(&a.stat[1], (unsigned long long)n);
            atomicAdd(&a.stat[2], 1ull);
        }
        PROF(8)
        if (t == 0) atomicAdd(&g_prof[15], 1ull);
    }
}

// =================================================================================================
// huffman_kernel: one warp per chunk
// =================================================================================================
struct HuffSm {
    uint32_t freq[REC_WORDS];
    uint32_t codes[REC_WORDS];
    HuffWork hw;
    DynHeader dh;
    uint32_t hdr[160];     // dynamic header bits
    uint32_t bl32[16];
    uint32_t small[32];    // per-length running counts / code-length-code frequencies
    uint32_t n_used, cost_dyn, cost_fix, mode, hdr_bits, bits;
    unsigned long long kraft;
};

// ---- warp-collective pieces of the Huffman construction -------------------------------------------------

// Code lengths of one tree whose k >= 2 leaves lie sorted ascending by (freq, symbol) in hw.w[0..k) / hw.order[0..k).
// The caller has zeroed lens[] for the unused symbols.  Two-queue merge on lane 0, everything else lane-parallel;
// depth overflow is repaired on the per-length histogram like zlib's gen_bitlen.
__device__ void warp_tree_lengths(HuffWork& hw, uint32_t k, int maxbits, uint8_t* lens, uint32_t* bl32,
                                  unsigned long long* kraft, unsigned lane) {
    if (lane < 16) bl32[lane] = 0;
    if (lane == 0) {
        *kraft = 0;
        huff_merge(hw, (int)k);
    }
    __syncwarp();
    const uint32_t root = 2 * k - 2;
    unsigned long long kr = 0;   // the Kraft sum: per-lane partial sums, one reduction (a 64-bit shared atomic is a CAS loop)
    for (uint32_t i = lane; i < k; i += 32) {
        uint32_t node = i, dpt = 0;
        while (node != root) {
            node = hw.parent[node];
            dpt++;
        }
        if (dpt > (uint32_t)maxbits) dpt = (uint32_t)maxbits;
        atomicAdd(&bl32[dpt], 1u);
        kr += 1ull << (maxbits - dpt);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) kr += __shfl_xor_sync(0xffffffffu, kr, o);
    if (lane == 0) *kraft = kr;
    __syncwarp();
    if (lane == 0) {
        for (int b = 0; b < 16; b++) hw.bl_count[b] = (uint16_t)bl32[b];
        huff_fix_overflow(hw.bl_count, maxbits, *kraft);
    }
    __syncwarp();
    for (uint32_t i = lane; i < k; i += 32) {  // rarest leaves take the longest codes
        uint32_t cum = 0, L = 1;
        for (int bits = maxbits; bits >= 1; bits--) {
            cum += hw.bl_count[bits];
            if (i < cum) {
                L = (uint32_t)bits;
                break;
            }
        }
        lens[hw.order[i]] = (uint8_t)L;
    }
    __syncwarp();
}

// Leaves of an alphabet of at most 32 symbols (lane = symbol, f = its count, 0 beyond the alphabet) sorted into
// hw.w / hw.order by (freq, symbol); at least two codes are forced like zlib's build_tree.  Returns the leaf count.
__device__ uint32_t warp_sort_small(uint32_t f, HuffWork& hw, unsigned lane) {
    uint32_t used = __ballot_sync(0xffffffffu, f != 0);
    if (__popc(used) < 2) {
        if (used == 0) {
            if (lane < 2) f = 1;
        } else if (used & 1u) {
            if (lane == 1) f = 1;
        } else if (lane == 0) {
            f = 1;
        }
        used = __ballot_sync(0xffffffffu, f != 0);
    }
    uint32_t rank = 0;
#pragma unroll
    for (int j = 0; j < 32; j++) {
        const uint32_t fj = __shfl_sync(0xffffffffu, f, j);
        rank += (fj != 0) && (fj < f || (fj == f && (unsigned)j < lane));
    }
    if (f) {
        hw.w[rank] = f;
        hw.order[rank] = (uint16_t)lane;
    }
    __syncwarp();
    return (uint32_t)__popc(used);
}

// zlib's run-length coding of one tree's code lengths (scan_tree / send_tree, rle_lengths in deflate_core.h), position
// parallel: every position learns the start and the end of its run (two passes over the 32-wide slices, forwards and
// backwards) and decides by itself whether an entry begins there.  out[base..) receives sym | extra << 8 in order;
// returns the entry count.  ts / te: n u16 of scratch each.
__device__ uint32_t warp_rle(const uint8_t* lens, uint32_t n, uint16_t* out, uint32_t out_base, uint16_t* ts, uint16_t* te,
                             unsigned lane) {
    const uint32_t upto = lane == 31 ? 0xffffffffu : (2u << lane) - 1;   // lanes 0 .. lane
    const uint32_t nslices = (n + 31) >> 5;
    uint32_t carry = 0;
    for (uint32_t sl = 0; sl < nslices; sl++) {
        const uint32_t base = sl << 5, i = base + lane;
        const uint32_t v = i < n ? lens[i] : 0x1FFu;
        uint32_t vp = __shfl_up_sync(0xffffffffu, v, 1);
        if (lane == 0) vp = base ? lens[base - 1] : 0x2FFu;
        const uint32_t hm = __ballot_sync(0xffffffffu, i < n && v != vp);
        const uint32_t m = hm & upto;
        const uint32_t st = m ? base + 31 - (uint32_t)__clz((int)m) : carry;
        if (i < n) ts[i] = (uint16_t)st;
        carry = __shfl_sync(0xffffffffu, st, 31);
    }
    uint32_t carry_e = n;
    for (uint32_t sl = nslices; sl-- > 0;) {
        const uint32_t base = sl << 5, i = base + lane;
        const uint32_t v = i < n ? lens[i] : 0x1FFu;
        uint32_t vp = __shfl_up_sync(0xffffffffu, v, 1);
        if (lane == 0) vp = base ? lens[base - 1] : 0x2FFu;
        const uint32_t hm = __ballot_sync(0xffffffffu, i < n && v != vp);
        const uint32_t m = hm & ~upto;
        if (i < n) te[i] = (uint16_t)(m ? base + (uint32_t)__ffs((int)m) - 1 : carry_e);
        if (hm) carry_e = base + (uint32_t)__ffs((int)hm) - 1;
    }
    __syncwarp();
    const uint32_t lt = (1u << lane) - 1;
    uint32_t count = 0;
    for (uint32_t sl = 0; sl < nslices; sl++) {
        const uint32_t i = (sl << 5) + lane;
        bool emit = false;
        uint32_t entry = 0;
        if (i < n) {
            const uint32_t v = lens[i], st = ts[i], r = te[i] - st, o = i - st;
            if (v == 0) {   // full 138-runs, then 18 / 17 / up to two literal zeros
                const uint32_t full = r / 138, rem = r - 138 * full;
                if (o < 138 * full) {
                    emit = o % 138 == 0;
                    entry = 18u | ((138u - 11u) << 8);
                } else if (rem >= 11) {
                    emit = o == 138 * full;
                    entry = 18u | ((rem - 11u) << 8);
                } else if (rem >= 3) {
                    emit = o == 138 * full;
                    entry = 17u | ((rem - 3u) << 8);
                } else {
                    emit = true;
                    entry = 0;
                }
            } else if (o == 0) {   // the length itself, then repeats of 6, then 16 / up to two literals
                emit = true;
                entry = v;
            } else {
                const uint32_t R = r - 1, o1 = o - 1, full = R / 6, rem = R - 6 * full;
                if (o1 < 6 * full) {
                    emit = o1 % 6 == 0;
                    entry = 16u | (3u << 8);
                } else if (rem >= 3) {
                    emit = o1 == 6 * full;
                    entry = 16u | ((rem - 3u) << 8);
                } else {
                    emit = true;
                    entry = v;
                }
            }
        }
        const uint32_t bm = __ballot_sync(0xffffffffu, emit);
        if (emit) out[out_base + count + __popc(bm & lt)] = (uint16_t)entry;
        count += __popc(bm);
    }
    __syncwarp();
    return count;
}

// Appends (val, nb <= 17) entries to a zeroed bit string of 32-bit words, 32 entries per call in lane order;
// `bitpos` is the running length (warp-uniform).
__device__ __forceinline__ void warp_put_bits(uint32_t* words, uint32_t& bitpos, uint32_t val, uint32_t nb, unsigned lane) {
    uint32_t inc = nb;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (unsigned)o) inc += t;
    }
    const uint32_t off = bitpos + inc - nb;
    if (nb) {
        atomicOr(&words[off >> 5], val << (off & 31));
        if ((off & 31) + nb > 32) atomicOr(&words[(off >> 5) + 1], val >> (32 - (off & 31)));
    }
    bitpos += __shfl_sync(0xffffffffu, inc, 31);
}

__global__ void __launch_bounds__(HUFF_WARPS * 32) huffman_kernel(DeflArgs a) {
    extern __shared__ __align__(16) uint8_t smem[];
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    HuffSm& s = reinterpret_cast<HuffSm*>(smem)[warp];
    const uint32_t n_jobs = a.job1 - a.job0;
    for (uint32_t bj = blockIdx.x * HUFF_WARPS + warp; bj < n_jobs; bj += gridDim.x * HUFF_WARPS) {
        ChunkRec rec = a.recs[bj];
        if (rec.mode == 0) continue;  // level 0: stored, nothing to build
        uint32_t* g = a.hist + (size_t)bj * REC_WORDS;
        uint32_t used = 0;
        for (uint32_t i = lane; i < REC_WORDS; i += 32) {
            const uint32_t f = g[i];
            s.freq[i] = f;
            s.codes[i] = 0;
            used += (i < (uint32_t)NLIT) && f != 0;
        }
        if (lane < 16) s.bl32[lane] = 0;
        if (lane == 0) {
            s.cost_dyn = 0;
            s.cost_fix = 0;
            s.kraft = 0;
        }
#pragma unroll
        for (int o = 16; o; o >>= 1) used += __shfl_xor_sync(0xffffffffu, used, o);
        __syncwarp();
        if (used < 2) {  // EOB is always used; force a second code like zlib (trees.c build_tree)
            if (lane == 0) s.freq[s.freq[0] ? 1 : 0] = 1;
            used = 2;
            __syncwarp();
        }
        const uint32_t k_used = used;
        // leaves of the literal/length tree sorted by (freq, symbol): a stable LSD radix sort of the used symbols,
        // two passes of 8 bits (freq <= 32768); in-pass ranks from match_any groups taken in symbol order
        for (uint32_t sy = lane; sy < (uint32_t)NLIT; sy += 32) s.dh.lit_lens[sy] = 0;
        {
            uint32_t* hist = s.hw.w + 288;   // 256 counters; the leaves (< 288) and the merge do not reach them yet
            uint32_t* tf = s.codes;          // pass-1 output: frequencies ...
            uint16_t* ts = s.hw.parent;      // ... and symbols (both are written for real only later)
            const uint32_t lt = (1u << lane) - 1;
#pragma unroll 1
            for (int pass = 0; pass < 2; pass++) {
                const uint32_t count = pass ? k_used : (uint32_t)NLIT;
                for (uint32_t i = lane; i < 256; i += 32) hist[i] = 0;
                __syncwarp();
                for (uint32_t i = lane; i < count; i += 32) {
                    const uint32_t f = pass ? tf[i] : s.freq[i];
                    if (f) atomicAdd(&hist[(f >> (8 * pass)) & 255u], 1u);
                }
                __syncwarp();
                {   // exclusive scan: lane owns bins 8*lane .. 8*lane+7
                    uint32_t c[8], sum = 0;
#pragma unroll
                    for (int q = 0; q < 8; q++) {
                        c[q] = hist[8 * lane + q];
                        sum += c[q];
                    }
                    uint32_t inc = sum;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const uint32_t tt = __shfl_up_sync(0xffffffffu, inc, o);
                        if (lane >= (unsigned)o) inc += tt;
                    }
                    uint32_t run = inc - sum;
#pragma unroll
                    for (int q = 0; q < 8; q++) {
                        hist[8 * lane + q] = run;
                        run += c[q];
                    }
                }
                __syncwarp();
                for (uint32_t base = 0; base < count; base += 32) {
                    const uint32_t i = base + lane;
                    const uint32_t f = i < count ? (pass ? tf[i] : s.freq[i]) : 0u;
                    const uint32_t sy = pass ? (uint32_t)ts[i < count ? i : 0] : i;
                    const uint32_t d = (f >> (8 * pass)) & 255u;
                    const uint32_t peers = __match_any_sync(0xffffffffu, f ? d : 256u + lane);
                    const uint32_t rank = __popc(peers & lt);
                    const uint32_t off = f ? hist[d] : 0u;
                    __syncwarp();
                    if (f) {
                        if (pass) {
                            s.hw.w[off + rank] = f;
                            s.hw.order[off + rank] = (uint16_t)sy;
                        } else {
                            tf[off + rank] = f;
                            ts[off + rank] = (uint16_t)sy;
                        }
                        if (rank == 0) hist[d] = off + __popc(peers);
                    }
                    __syncwarp();
                }
            }
            for (uint32_t i = lane; i < REC_WORDS; i += 32) s.codes[i] = 0;   // the sort borrowed them
        }
        __syncwarp();
        // literal/length tree, then the distance tree (30 symbols: one per lane)
        warp_tree_lengths(s.hw, k_used, 15, s.dh.lit_lens, s.bl32, &s.kraft, lane);
        {
            if (lane < 32) s.dh.dist_lens[lane] = 0;
            __syncwarp();
            const uint32_t kd = warp_sort_small(lane < (unsigned)NDIST ? s.freq[288 + lane] : 0u, s.hw, lane);
            warp_tree_lengths(s.hw, kd, 15, s.dh.dist_lens, s.bl32, &s.kraft, lane);
        }
        // canonical codes + block cost, both trees: per-length counts -> first code of every length (lane 0),
        // then the symbols in order, 32 at a time: code = first[len] + symbols of that length seen so far
        {
            uint32_t* cnt = s.bl32;          // [16] per-length counts, then first codes
            uint32_t* seen = s.small;        // [16] running counts
            const uint32_t lt = (1u << lane) - 1;
            uint32_t cd = 0, cf = 0;
#pragma unroll 1
            for (int tree = 0; tree < 2; tree++) {
                const uint8_t* lens = tree ? s.dh.dist_lens : s.dh.lit_lens;
                const uint32_t nsy = tree ? NDIST : NLIT, cbase = tree ? 288u : 0u;
                if (lane < 16) {
                    cnt[lane] = 0;
                    seen[lane] = 0;
                }
                __syncwarp();
                for (uint32_t sy = lane; sy < nsy; sy += 32)
                    if (lens[sy]) atomicAdd(&cnt[lens[sy]], 1u);
                __syncwarp();
                if (lane == 0) {
                    uint32_t code = 0, prev = 0;
                    for (int b = 1; b < 16; b++) {
                        code = (code + prev) << 1;
                        prev = cnt[b];
                        cnt[b] = code;
                    }
                }
                __syncwarp();
                for (uint32_t base = 0; base < nsy; base += 32) {
                    const uint32_t sy = base + lane;
                    const uint32_t l = sy < nsy ? lens[sy] : 0u;
                    const uint32_t peers = __match_any_sync(0xffffffffu, l ? l : 100u + lane);
                    const uint32_t rank = __popc(peers & lt);
                    const uint32_t before = l ? seen[l] : 0u;
                    __syncwarp();
                    if (l && rank == 0) seen[l] = before + __popc(peers);
                    __syncwarp();
                    if (sy < nsy) {
                        s.codes[cbase + sy] = l ? (l << 16) | bitrev(cnt[l] + before + rank, (int)l) : 0u;
                        const uint32_t f = g[cbase + sy];  // true counts (without the forced code)
                        const uint32_t xb = tree ? (uint32_t)dsym_extra((int)sy) : (sy > 256 ? (uint32_t)lsym_extra((int)sy) : 0u);
                        cd += f * (l + xb);
                        cf += f * ((tree ? 5u : (uint32_t)fixed_lit_len((int)sy)) + xb);
                    }
                }
                __syncwarp();
            }
            if (cd) atomicAdd(&s.cost_dyn, cd);
            if (cf) atomicAdd(&s.cost_fix, cf);
        }
        __syncwarp();
        // ---- dynamic header plan: trimmed alphabets, run-length coded lengths, the code-length code -------------
        uint32_t nlit, ndist, n_rle, ncl, dyn_hdr_bits;
        {
            uint32_t last = 0;
            for (uint32_t sy = lane; sy < (uint32_t)NLIT; sy += 32)
                if (s.dh.lit_lens[sy]) last = sy + 1;
#pragma unroll
            for (int o = 16; o; o >>= 1) last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
            nlit = last > 257 ? last : 257;
            const uint32_t dm = __ballot_sync(0xffffffffu, lane < (unsigned)NDIST && s.dh.dist_lens[lane] != 0);
            ndist = dm ? 32 - (uint32_t)__clz((int)dm) : 1;
            uint16_t* ts = s.hw.parent;
            uint16_t* te = s.hw.parent + 288;
            n_rle = warp_rle(s.dh.lit_lens, nlit, s.dh.rle, 0, ts, te, lane);
            n_rle += warp_rle(s.dh.dist_lens, ndist, s.dh.rle, n_rle, ts, te, lane);
            // code-length code: frequencies, lengths (limit 7), canonical codes - 19 symbols, one per lane
            s.small[lane] = 0;
            __syncwarp();
            for (uint32_t i = lane; i < n_rle; i += 32) atomicAdd(&s.small[s.dh.rle[i] & 0xff], 1u);
            __syncwarp();
            if (lane < (unsigned)NCL) s.dh.cl_lens[lane] = 0;
            const uint32_t kc = warp_sort_small(lane < (unsigned)NCL ? s.small[lane] : 0u, s.hw, lane);
            warp_tree_lengths(s.hw, kc, 7, s.dh.cl_lens, s.bl32, &s.kraft, lane);
            const uint32_t L = lane < (unsigned)NCL ? s.dh.cl_lens[lane] : 0u;
            uint32_t code = 0, prev = 0, first = 0;
#pragma unroll
            for (int b = 1; b <= 7; b++) {
                code = (code + prev) << 1;
                prev = __popc(__ballot_sync(0xffffffffu, L == (uint32_t)b));
                if (L == (uint32_t)b) first = code;
            }
            const uint32_t peers = __match_any_sync(0xffffffffu, L ? L : 100u + lane);
            const uint32_t clcode = L ? (L << 16) | bitrev(first + __popc(peers & ((1u << lane) - 1)), (int)L) : 0u;
            if (lane < (unsigned)NCL) s.dh.cl_codes[lane] = clcode;
            const uint32_t nz = __ballot_sync(0xffffffffu, lane < (unsigned)NCL && s.dh.cl_lens[cl_order((int)lane)] != 0);
            ncl = nz ? 32 - (uint32_t)__clz((int)nz) : 0;
            if (ncl < 4) ncl = 4;
            __syncwarp();
            uint32_t hb = 0;
            for (uint32_t i = lane; i < n_rle; i += 32) {
                const uint32_t sy = s.dh.rle[i] & 0xff;
                hb += s.dh.cl_lens[sy] + (sy == 16 ? 2u : sy == 17 ? 3u : sy == 18 ? 7u : 0u);
            }
#pragma unroll
            for (int o = 16; o; o >>= 1) hb += __shfl_xor_sync(0xffffffffu, hb, o);
            dyn_hdr_bits = 3 + 5 + 5 + 4 + 3 * ncl + hb;
        }
        // ---- block type by exact cost (like zlib), header bits -----------------------------------------------------
        const uint64_t dyn_bits = (uint64_t)dyn_hdr_bits + s.cost_dyn, fix_bits = 3ull + s.cost_fix;
        uint32_t mode_sel = dyn_bits < fix_bits ? 2u : 1u;
        const uint64_t best_bits = dyn_bits < fix_bits ? dyn_bits : fix_bits;
        const bool multi = (rec.flags & REC_MULTI) != 0;   // stored is decided for the whole stream (encode_long_kernel)
        if (!multi && (uint64_t)rec.n + 5 <= (best_bits + 7) / 8) mode_sel = 0;
        const uint32_t bfinal = (!multi || (rec.flags & REC_LAST)) ? 1u : 0u;
        uint32_t hbits = 0;
        for (uint32_t i = lane; i < 160; i += 32) s.hdr[i] = 0;
        __syncwarp();
        if (mode_sel == 2) {
            // entry 0: BFINAL, BTYPE = 2, HLIT, HDIST, HCLEN; entries 1..ncl: the code-length code lengths in their
            // transmission order; then the run-length coded lengths with their extra bits
            const uint32_t total = 1 + ncl + n_rle;
            for (uint32_t base = 0; base < total; base += 32) {
                const uint32_t e = base + lane;
                uint32_t val = 0, nb = 0;
                if (e == 0) {
                    val = bfinal | (2u << 1) | ((nlit - 257) << 3) | ((ndist - 1) << 8) | ((ncl - 4) << 13);
                    nb = 17;
                } else if (e <= ncl) {
                    val = s.dh.cl_lens[cl_order((int)(e - 1))];
                    nb = 3;
                } else if (e < total) {
                    const uint32_t r = s.dh.rle[e - 1 - ncl], sy = r & 0xff, c = s.dh.cl_codes[sy];
                    const uint32_t cl = c >> 16;
                    val = (c & 0xffffu) | ((r >> 8) << cl);
                    nb = cl + (sy == 16 ? 2u : sy == 17 ? 3u : sy == 18 ? 7u : 0u);
                }
                warp_put_bits(s.hdr, hbits, val, nb, lane);
            }
        } else if (mode_sel == 1) {
            if (lane == 0) s.hdr[0] = bfinal | (1u << 1);
            hbits = 3;
        }
        __syncwarp();
        if (lane == 0) {
            s.bits = (uint32_t)best_bits;
            s.mode = mode_sel;
            s.hdr_bits = hbits;
        }
        __syncwarp();
        const uint32_t mode = s.mode;
        if (mode == 1) {
            for (uint32_t i = lane; i < 288; i += 32) s.codes[i] = fixed_lit_code((int)i);
            s.codes[288 + lane] = fixed_dist_code((int)lane);
            __syncwarp();
        }
        for (uint32_t i = lane; i < REC_WORDS; i += 32) g[i] = s.codes[i];
        if (mode != 0) {
            const uint32_t hw32 = (s.hdr_bits + 31) >> 5;
            uint32_t* gh = reinterpret_cast<uint32_t*>(a.hdrs + (size_t)bj * 640);
            for (uint32_t i = lane; i < hw32; i += 32) gh[i] = s.hdr[i];
        }
        if (lane == 0) {
            a.recs[bj].mode = mode;
            a.recs[bj].hdr_bits = s.hdr_bits;
            a.recs[bj].bits = s.bits;
        }
        __syncwarp();
    }
}

// =================================================================================================
// encode_kernel: one CTA per chunk
// =================================================================================================
struct Emitter {
    uint32_t* out;      // 4-byte aligned start of the deflate bit stream
    uint64_t acc;
    uint32_t accbits, wi;
    bool first;
    __device__ __forceinline__ void begin(uint32_t* o, uint32_t bitoff) {
        out = o;
        wi = bitoff >> 5;
        accbits = bitoff & 31;
        acc = 0;
        first = true;
    }
    __device__ __forceinline__ void put(uint32_t v, uint32_t nb) {
        acc |= (uint64_t)v << accbits;
        accbits += nb;
        if (accbits >= 32) {
            if (first) atomicOr(out + wi, (uint32_t)acc);  // shared with the previous writer
            else out[wi] = (uint32_t)acc;
            first = false;
            acc >>= 32;
            accbits -= 32;
            wi++;
        }
    }
    __device__ __forceinline__ void end() {
        if (accbits) atomicOr(out + wi, (uint32_t)acc);
    }
};

// Bit strings of the token words.  Literals and match lengths come from a per-block table s_tab[512] of packed entries
// (value | bits << 27: a literal's code, or a length's code with its extra bits already appended - 20 bits at most), built
// once per block; distance words are computed (30 symbols from a logarithm) without a branch.  Every lane runs the same
// instructions whatever kind of word it holds: the loop used to serialise three divergent paths per step.
__device__ __forceinline__ uint32_t tab_index(uint32_t w) {   // literal 0..255 -> itself; length word 0x8000 | len -> 253 + len
    return (w & 0x8000u) ? 253u + (w & 0x1ffu) : w;
}
__device__ __forceinline__ void dist_bits(const uint32_t* codes, uint32_t d, uint32_t& val, uint32_t& nb) {   // d = distance - 1
    const uint32_t eb = (uint32_t)(31 - __clz((int)(d | 2u))) - 1u;       // 0 for d < 4
    const uint32_t sy = d < 4 ? d : 2 * eb + 2 + ((d >> eb) & 1u);
    const uint32_t c = codes[288 + sy], cl = c >> 16;
    val = (c & 0xffffu) | ((d & ((1u << eb) - 1u)) << cl);
    nb = cl + eb;
}
__device__ __forceinline__ void word_bits(const uint32_t* codes, const uint32_t* tab, uint32_t w, bool is_dist, uint32_t& val,
                                          uint32_t& nb) {
    const uint32_t e = tab[is_dist ? 0u : tab_index(w)];
    uint32_t dv, dn;
    dist_bits(codes, is_dist ? w : 0u, dv, dn);
    val = is_dist ? dv : (e & 0x7ffffffu);
    nb = is_dist ? dn : (e >> 27);
}

// Emits one coded block (mode 1 or 2) of batch job bj at bit offset bit0 of the stream words out32, which the
// caller has zeroed (words shared by two writers are OR-ed).  Collective over the CTA; returns the bit offset
// after the end-of-block code.
__device__ uint32_t emit_block(const DeflArgs& a, uint32_t bj, const ChunkRec& rec, uint32_t* out32, uint32_t bit0,
                               uint32_t* s_codes, uint32_t* s_tmp, uint32_t* s_hdr, uint32_t* s_tab) {
    const uint32_t T = T_ENCODE, t = threadIdx.x;
    __syncthreads();
    for (uint32_t i = t; i < REC_WORDS; i += T) s_codes[i] = a.hist[(size_t)bj * REC_WORDS + i];
    const uint32_t hbytes = (rec.hdr_bits + 7) >> 3;
    for (uint32_t i = t; i < 160; i += T) s_hdr[i] = 0;
    __syncthreads();
    {
        const uint8_t* gh = a.hdrs + (size_t)bj * 640;
        uint8_t* sh = reinterpret_cast<uint8_t*>(s_hdr);
        for (uint32_t i = t; i < hbytes; i += T) sh[i] = gh[i];
    }
    for (uint32_t i = t; i < 512; i += T) {   // the table: literal i, or match length i - 253
        uint32_t c, eb = 0, ev = 0;
        if (i < 256) {
            c = s_codes[i];
        } else {
            uint32_t sy;
            len_sym(i - 253, sy, eb, ev);
            c = s_codes[sy];
        }
        const uint32_t cl = c >> 16;
        s_tab[i] = (c & 0xffffu) | (ev << cl) | ((cl + eb) << 27);
    }
    __syncthreads();
    const uint16_t* tk = a.tokens + (size_t)bj * a.nmax;
    const uint32_t W = rec.n_words;
    const uint32_t per = (W + T - 1) / T;
    const uint32_t w0 = t * per < W ? t * per : W, w1 = w0 + per < W ? w0 + per : W;
    // the word before a thread's first one is a length word (so that the first one is a distance) iff it carries the flag
    // and is not itself a distance: a distance (<= 32767) never carries it, so only a length word before IT can mislead
    bool dist0 = false;
    if (w0) {
        const uint32_t p1 = tk[w0 - 1];
        dist0 = (p1 & 0x8000u) != 0;
        if (dist0 && w0 >= 2 && (tk[w0 - 2] & 0x8000u)) dist0 = false;   // (cannot happen: kept as the old code had it)
    }
    uint32_t bits = 0;
    {
        bool is_dist = dist0;
        for (uint32_t i = w0; i < w1; i++) {
            const uint32_t w = tk[i];
            uint32_t val, nb;
            word_bits(s_codes, s_tab, w, is_dist, val, nb);
            bits += nb;
            is_dist = !is_dist && (w & 0x8000u);   // a distance word never introduces another one
        }
    }
    uint32_t tok_bits;
    const uint32_t my_off = bit0 + rec.hdr_bits + block_excl_scan(bits, s_tmp, &tok_bits);
    const uint32_t eob = s_codes[EOB];
    if (t == 0) {  // header bits, word by word
        Emitter eh;
        eh.begin(out32, bit0);
        const uint32_t hb = rec.hdr_bits;
        for (uint32_t i = 0; i < (hb >> 5); i++) eh.put(s_hdr[i], 32);
        if (hb & 31) eh.put(s_hdr[hb >> 5] & ((1u << (hb & 31)) - 1), hb & 31);
        eh.end();
    }
    Emitter em;
    em.begin(out32, my_off);
    {
        bool is_dist = dist0;
        for (uint32_t i = w0; i < w1; i++) {
            const uint32_t w = tk[i];
            uint32_t val, nb;
            word_bits(s_codes, s_tab, w, is_dist, val, nb);
            em.put(val, nb);
            is_dist = !is_dist && (w & 0x8000u);
        }
    }
    em.end();
    if (t == T - 1) {  // EOB follows all tokens
        Emitter ee;
        ee.begin(out32, bit0 + rec.hdr_bits + tok_bits);
        ee.put(eob & 0xffffu, eob >> 16);
        ee.end();
    }
    return bit0 + rec.hdr_bits + tok_bits + (eob >> 16);
}

__device__ __forceinline__ void put_be32(uint8_t* p, uint32_t v) {
    p[0] = (uint8_t)(v >> 24);
    p[1] = (uint8_t)(v >> 16);
    p[2] = (uint8_t)(v >> 8);
    p[3] = (uint8_t)v;
}
// zlib stream header (2 bytes, + DICTID when a preset dictionary is in use) at slot + 2
__device__ __forceinline__ void put_zlib_header(const DeflArgs& a, uint8_t* slot) {
    uint8_t cmf, flg;
    zlib_header(a.dict_len != 0, cmf, flg);
    slot[2] = cmf;
    slot[3] = flg;
    if (a.dict_len) put_be32(slot + 4, a.dict_adler);
}

__global__ void __launch_bounds__(T_ENCODE) encode_kernel(DeflArgs a) {
    __shared__ uint32_t s_codes[REC_WORDS];
    __shared__ uint32_t s_tmp[40];
    __shared__ uint32_t s_hdr[160];
    __shared__ uint32_t s_tab[512];
    const uint32_t T = T_ENCODE, t = threadIdx.x;
    const uint32_t n_jobs = a.job1 - a.job0;
    for (uint32_t bj = blockIdx.x; bj < n_jobs; bj += gridDim.x) {
        __syncthreads();
        const ChunkRec rec = a.recs[bj];
        const uint32_t k = a.list[a.job0 + bj];
        uint8_t* slot = a.stage + a.slot_off[k];
        const uint32_t hdr_len = a.dict_len ? 6 : 2;
        uint32_t* out32 = reinterpret_cast<uint32_t*>(slot + 2 + hdr_len);  // slot is 16-aligned: 4 or 8
        const uint32_t n = rec.n;
        uint32_t stream_len;
        if (rec.mode != 0) {
            const uint32_t body = (rec.bits + 7) >> 3;
            stream_len = hdr_len + body + 4;
            // zero the deflate words (+ trailer spill) so shared boundary words can be OR-ed
            const uint32_t zw = (body + 4 + 3) >> 2;
            for (uint32_t i = t; i < zw; i += T) out32[i] = 0;
            emit_block(a, bj, rec, out32, 0, s_codes, s_tmp, s_hdr, s_tab);
            __syncthreads();
            if (t == 0) put_be32(slot + 2 + hdr_len + body, rec.adler);
        } else {
            // ---- stored block: n <= 32768 -> a single block ---------------------------------------
            const uint64_t j = a.select ? a.select[k] : (uint64_t)k;
            const uint8_t* src = a.data + (j ? a.cuts[j - 1] : a.start0);
            uint8_t* o = slot + 2 + hdr_len;
            if (t == 0) {
                o[0] = 1;
                o[1] = (uint8_t)n;
                o[2] = (uint8_t)(n >> 8);
                o[3] = (uint8_t)~n;
                o[4] = (uint8_t)(~n >> 8);
                put_be32(o + 5 + n, rec.adler);
            }
            for (uint32_t p = t; p < n; p += T) o[5 + p] = src[p];
            stream_len = hdr_len + 5 + n + 4;
        }
        if (t == 0) {
            put_zlib_header(a, slot);
            a.sizes[k] = stream_len;
        }
    }
}

// Long chunks: one CTA per chunk strings the coded blocks of its jobs together bit by bit.  If that is
// not smaller than stored blocks the chunk is flagged for stored_kernel instead.
struct LongArgs {
    const uint32_t* chunk_k;      // selection slot of long chunk i
    const uint32_t* chunk_first;  // its first job (index into the long job list)
    const uint32_t* chunk_nblk;
    uint8_t* stored_flag;         // [n_long]
    uint32_t c0, c1;              // chunks of this batch
};
__global__ void __launch_bounds__(T_ENCODE) encode_long_kernel(DeflArgs a, LongArgs la) {
    __shared__ uint32_t s_codes[REC_WORDS];
    __shared__ uint32_t s_tmp[40];
    __shared__ uint32_t s_hdr[160];
    __shared__ uint32_t s_tab[512];
    const uint32_t T = T_ENCODE, t = threadIdx.x;
    for (uint32_t ci = la.c0 + blockIdx.x; ci < la.c1; ci += gridDim.x) {
        __syncthreads();
        const uint32_t k = la.chunk_k[ci], nblk = la.chunk_nblk[ci];
        const uint32_t bj0 = la.chunk_first[ci] - a.job0;
        const uint64_t j = a.select ? a.select[k] : (uint64_t)k;
        const uint64_t n = a.cuts[j] - (j ? a.cuts[j - 1] : a.start0);
        uint64_t bits = 0;
        for (uint32_t b = 0; b < nblk; b++) bits += a.recs[bj0 + b].bits;
        const uint64_t body = (bits + 7) >> 3;
        if (body >= n + 5 * (n / 65535 + 1)) {
            if (t == 0) la.stored_flag[ci] = 1;
            continue;
        }
        uint8_t* slot = a.stage + a.slot_off[k];
        const uint32_t hdr_len = a.dict_len ? 6 : 2;
        uint32_t* out32 = reinterpret_cast<uint32_t*>(slot + 2 + hdr_len);
        const uint64_t zw = (body + 4 + 3) >> 2;
        for (uint64_t i = t; i < zw; i += T) out32[i] = 0;
        uint32_t bit = 0, ad_a = 1, ad_b = 0;
        for (uint32_t b = 0; b < nblk; b++) {
            const ChunkRec rec = a.recs[bj0 + b];
            bit = emit_block(a, bj0 + b, rec, out32, bit, s_codes, s_tmp, s_hdr, s_tab);
            // Adler-32 of a concatenation (zlib's adler32_combine)
            const uint32_t a2 = rec.adler & 0xffffu, b2 = rec.adler >> 16;
            const uint32_t rem = rec.n % 65521u;
            ad_b = (uint32_t)((ad_b + b2 + (uint64_t)rem * ((ad_a + 65520u) % 65521u)) % 65521u);
            ad_a = (ad_a + a2 + 65520u) % 65521u;
        }
        __syncthreads();
        if (t == 0) {
            put_be32(slot + 2 + hdr_len + body, (ad_b << 16) | ad_a);
            put_zlib_header(a, slot);
            a.sizes[k] = hdr_len + body + 4;
            la.stored_flag[ci] = 0;
        }
    }
}

// ---- helpers around the main kernels -------------------------------------------------------------

// Per selected chunk: worst-case slot size and size class list.  class 0: <= NMAX_SMALL,
// class 1: <= NMAX_LARGE, class 2: longer (multi-block stored path).
__global__ void classify_kernel(uint64_t start0, const uint64_t* __restrict__ cuts, const uint64_t* __restrict__ select,
                                uint64_t m, uint64_t* __restrict__ slot_size, uint32_t* __restrict__ lists,
                                uint32_t* __restrict__ list_n) {
    uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= m) return;
    const uint64_t j = select ? select[k] : k;
    const uint64_t s = j ? cuts[j - 1] : start0;
    const uint64_t len = cuts[j] - s;
    const uint64_t bound = len + 5 * (len / 65535 + 1) + 6 + 4 + 2 + 16;
    slot_size[k] = (bound + 15) & ~15ull;
    const int c = len <= NMAX_SMALL ? 0 : (len <= NMAX_MEDIUM ? 1 : (len <= NMAX_LARGE ? 2 : LONG_CLASS));
    const uint32_t pos = atomicAdd(&list_n[c], 1u);
    lists[(uint64_t)c * m + pos] = (uint32_t)k;
}

// Chunks longer than 32 KiB: stored blocks of <= 65535 bytes (valid zlib stream, ratio 1).
__global__ void __launch_bounds__(256)
stored_kernel(DeflArgs a) {
    __shared__ uint32_t s_a[256], s_b[256];
    for (uint32_t job = a.job0 + blockIdx.x; job < a.job1; job += gridDim.x) {
        if (a.stored_flag && !a.stored_flag[job]) continue;   // block-uniform
        const uint32_t k = a.list[job];
        const uint64_t j = a.select ? a.select[k] : (uint64_t)k;
        const uint64_t cs = j ? a.cuts[j - 1] : a.start0;
        const uint64_t n = a.cuts[j] - cs;
        const uint8_t* src = a.data + cs;
        uint8_t* slot = a.stage + a.slot_off[k];
        const uint32_t hdr_len = a.dict_len ? 6 : 2;
        uint8_t* o = slot + 2 + hdr_len;
        const uint64_t nblk = n / 65535 + 1;  // the last block may have length 0 only when n % 65535 == 0
        uint64_t sa = 0, sb = 0;
        for (uint64_t p = threadIdx.x; p < n; p += 256) {
            const uint64_t b = src[p];
            sa += b;
            sb = (sb + ((n - p) % 65521u) * b) % 65521u;
            const uint64_t blk = p / 65535;
            o[5 * (blk + 1) + p] = (uint8_t)b;
        }
        s_a[threadIdx.x] = (uint32_t)(sa % 65521u);
        s_b[threadIdx.x] = (uint32_t)sb;
        __syncthreads();
        if (threadIdx.x == 0) {
            uint64_t ta = 1, tb = n % 65521u;
            for (int i = 0; i < 256; i++) {
                ta += s_a[i];
                tb += s_b[i];
            }
            const uint32_t ad = (uint32_t)((tb % 65521u) << 16) | (uint32_t)(ta % 65521u);
            for (uint64_t b = 0; b < nblk; b++) {
                const uint64_t off = b * 65535;
                const uint32_t bl = (uint32_t)(n - off < 65535 ? n - off : 65535);
                uint8_t* h = o + off + 5 * b;
                h[0] = b == nblk - 1 ? 1 : 0;
                h[1] = (uint8_t)bl;
                h[2] = (uint8_t)(bl >> 8);
                h[3] = (uint8_t)~bl;
                h[4] = (uint8_t)(~bl >> 8);
            }
            uint8_t* tr = o + n + 5 * nblk;
            tr[0] = (uint8_t)(ad >> 24);
            tr[1] = (uint8_t)(ad >> 16);
            tr[2] = (uint8_t)(ad >> 8);
            tr[3] = (uint8_t)ad;
            uint8_t cmf, flg;
            zlib_header(a.dict_len != 0, cmf, flg);
            slot[2] = cmf;
            slot[3] = flg;
            if (a.dict_len) {
                slot[4] = (uint8_t)(a.dict_adler >> 24);
                slot[5] = (uint8_t)(a.dict_adler >> 16);
                slot[6] = (uint8_t)(a.dict_adler >> 8);
                slot[7] = (uint8_t)a.dict_adler;
            }
            a.sizes[k] = hdr_len + n + 5 * nblk + 4;
        }
        __syncthreads();
    }
}

// job_k[i] holds an index into the class-2 list: replace it by the selection slot stored there
__global__ void long_job_slot_kernel(uint32_t* __restrict__ job_k, uint32_t n, const uint32_t* __restrict__ list) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) job_k[i] = list[job_k[i]];
}

// lengths of the long chunks (class 2 list) for the host-side block plan
__global__ void long_len_kernel(uint64_t start0, const uint64_t* __restrict__ cuts, const uint64_t* __restrict__ select,
                                const uint32_t* __restrict__ list, uint32_t n, uint64_t* __restrict__ lens) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t j = select ? select[list[i]] : (uint64_t)list[i];
    lens[i] = cuts[j] - (j ? cuts[j - 1] : start0);
}

// Index of the previous block for every batch job with block number >= 1: the same 16-byte bucket records the
// host builds for the preset dictionary.  The four largest positions of a bucket are found by four rounds
// of atomicMax (round r admits positions below the winner of round r-1), then each winner is dressed with
// its tag and preceding byte.  One CTA per job; the records are read back through L2 (__ldcg).
__global__ void __launch_bounds__(1024) long_dict_kernel(DeflArgs a) {
    const uint32_t t = threadIdx.x;
    const uint32_t n_jobs = a.job1 - a.job0;
    for (uint32_t bj = blockIdx.x; bj < n_jobs; bj += gridDim.x) {
        const uint32_t blkno = a.blk[a.job0 + bj];
        if (!blkno) continue;
        const uint32_t k = a.list[a.job0 + bj];
        const uint64_t j = a.select ? a.select[k] : (uint64_t)k;
        const uint8_t* src = a.data + (j ? a.cuts[j - 1] : a.start0) + (uint64_t)(blkno - 1) * LONG_BLOCK;
        DictDev* dd = const_cast<DictDev*>(a.long_dicts) + bj;
        uint32_t* w = reinterpret_cast<uint32_t*>(dd->bk4);
        for (uint32_t i = t; i < LONG_BLOCK + 32; i += 1024) dd->bytes[i] = i < LONG_BLOCK ? src[i] : (uint8_t)0;
        for (uint32_t i = t; i < DICT_BUCKETS * 4; i += 1024) w[i] = 0;
        __syncthreads();
        auto le32 = [&](uint32_t q) {
            return (uint32_t)src[q] | ((uint32_t)src[q + 1] << 8) | ((uint32_t)src[q + 2] << 16) | ((uint32_t)src[q + 3] << 24);
        };
        for (int r = 0; r < DICT_CAP; r++) {
            for (uint32_t q = t; q + 3 < LONG_BLOCK; q += 1024) {
                const uint32_t h = hash_dict(le32(q));
                if (r == 0 || q + 1 < __ldcg(&w[h * 4 + r - 1])) atomicMax(&w[h * 4 + r], q + 1);
            }
            __syncthreads();
        }
        for (uint32_t i = t; i < DICT_BUCKETS * 4; i += 1024) {
            const uint32_t q1 = __ldcg(&w[i]);
            if (q1) {
                const uint32_t q = q1 - 1;
                w[i] = k_record(le32(q), q ? (uint32_t)src[q - 1] : DICT_PREV0, q);
            }
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256)
pack_kernel(const uint8_t* __restrict__ stage, const uint64_t* __restrict__ slot_off, const uint64_t* __restrict__ offs,
            uint64_t m, uint8_t* __restrict__ out, uint64_t out_cap) {
    for (uint64_t k = blockIdx.x; k < m; k += gridDim.x) {
        const uint8_t* s = stage + slot_off[k] + 2;
        const uint64_t o = offs[k], len = offs[k + 1] - o;
        if (o + len > out_cap) continue;
        uint8_t* d = out + o;
        // head bytes until d is 4-aligned, then words assembled from the (2-aligned) source
        uint64_t head = (4 - ((uintptr_t)d & 3)) & 3;
        if (head > len) head = len;
        if (threadIdx.x < head) d[threadIdx.x] = s[threadIdx.x];
        const uint64_t body = (len - head) >> 2;
        const uint8_t* sb = s + head;
        const uint32_t kmis = (uint32_t)((uintptr_t)sb & 3);
        const uint32_t* ws = reinterpret_cast<const uint32_t*>(sb - kmis);
        uint32_t* wd = reinterpret_cast<uint32_t*>(d + head);
        for (uint64_t i = threadIdx.x; i < body; i += 256) {
            uint32_t lo = ws[i], hi = kmis ? ws[i + 1] : 0u;
            wd[i] = __funnelshift_r(lo, hi, kmis * 8);
        }
        const uint64_t done = head + (body << 2);
        if (threadIdx.x < len - done) d[done + threadIdx.x] = s[done + threadIdx.x];
    }
}

uint32_t host_adler32(const uint8_t* d, size_t n) {
    uint32_t a = 1, b = 0;
    for (size_t i = 0; i < n; i++) {
        a = (a + d[i]) % 65521u;
        b = (b + a) % 65521u;
    }
    return (b << 16) | a;
}

// 128-bit fingerprint of the dictionary bytes (position-dependent mixes, summed), written straight into
// the mapped mailbox words 0..1: lets hmse_compress recognise the dictionary it has already indexed
// without copying 32 KiB to the host on every call.
__device__ __forceinline__ uint64_t mix64(uint64_t x) {
    x ^= x >> 30;
    x *= 0xBF58476D1CE4E5B9ull;
    x ^= x >> 27;
    x *= 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}
// out[2] = the Adler-32 of the same bytes (sum of bytes and position-weighted sum, n <= 32768: no overflow in 64 bits), so
// that a cached dictionary is only reused when fingerprint, length AND checksum agree.
__global__ void __launch_bounds__(256) dict_fingerprint_kernel(const uint8_t* __restrict__ d, uint32_t n, uint64_t* __restrict__ out) {
    __shared__ uint64_t s0[256], s1[256], s2[256], s3[256];
    uint64_t a = 0, b = 0, sa = 0, sb = 0;
    for (uint32_t i = threadIdx.x; i < n; i += 256) {
        const uint64_t x = ((uint64_t)i << 8) | d[i];
        a += mix64(x + 0x9E3779B97F4A7C15ull);
        b += mix64(x ^ 0xD6E8FEB86659FD93ull);
        sa += d[i];
        sb += (uint64_t)(n - i) * d[i];
    }
    s0[threadIdx.x] = a;
    s1[threadIdx.x] = b;
    s2[threadIdx.x] = sa;
    s3[threadIdx.x] = sb;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 1; i < 256; i++) {
            a += s0[i];
            b += s1[i];
            sa += s2[i];
            sb += s3[i];
        }
        out[0] = a;
        out[1] = b;
        out[2] = (((uint64_t)n + sb) % 65521u) << 16 | ((1 + sa) % 65521u);
    }
}

// Dictionary setup (the analogue of zlib's deflateSetDictionary): a <= 32 KiB one-off, indexed on
// the host and cached until the dictionary bytes change.  Not on the per-chunk path.
struct DictHost {
    uint8_t bytes[DICT_MAX];
    uint32_t len;
    uint32_t adler;
    uint64_t fp[2];
    int valid;
};

int ensure_dict(hmse_ctx* ctx, const uint8_t* d_zdict, uint32_t dict_len, uint32_t* adler, cudaStream_t st) {
    HMSE_SCRATCH(ctx, dev, DictDev*, SLOT_DEFLATE_DICT, sizeof(DictDev));
    DictHost* hd = (DictHost*)ctx->dict_host;
    if (!hd) {
        hd = (DictHost*)calloc(1, sizeof(DictHost));
        if (!hd) HMSE_FAIL(ctx, HMSE_E_NOMEM, "dictionary host copy");
        ctx->dict_host = hd;
    }
    KL(ctx);
    dict_fingerprint_kernel<<<1, 256, 0, st>>>(d_zdict, dict_len, ctx->pinned_dev);
    HMSE_LAUNCH_CHECK(ctx);
    HMSE_CUDA(ctx, cudaStreamSynchronize(st));
    const uint64_t fp0 = ctx->pinned[0], fp1 = ctx->pinned[1];
    const uint32_t dev_adler = (uint32_t)ctx->pinned[2];
    if (hd->valid && hd->len == dict_len && hd->fp[0] == fp0 && hd->fp[1] == fp1 && hd->adler == dev_adler) {
        *adler = hd->adler;
        return HMSE_OK;
    }
    static thread_local uint8_t tmp[DICT_MAX];
    HMSE_CUDA(ctx, cudaMemcpyAsync(tmp, d_zdict, dict_len, cudaMemcpyDeviceToHost, st));
    HMSE_CUDA(ctx, cudaStreamSynchronize(st));
    hd->fp[0] = fp0;
    hd->fp[1] = fp1;
    hd->valid = 0;
    memcpy(hd->bytes, tmp, dict_len);
    hd->len = dict_len;
    hd->adler = host_adler32(tmp, dict_len);
    DictDev* img = (DictDev*)calloc(1, sizeof(DictDev));
    if (!img) HMSE_FAIL(ctx, HMSE_E_NOMEM, "dictionary index");
    memcpy(img->bytes, tmp, dict_len);
    const uint32_t nh = dict_len >= 4 ? dict_len - 3 : 0;
    auto le32 = [&](uint32_t j) {
        return (uint32_t)tmp[j] | ((uint32_t)tmp[j + 1] << 8) | ((uint32_t)tmp[j + 2] << 16) | ((uint32_t)tmp[j + 3] << 24);
    };
    // ascending positions shift each bucket record by one slot: the largest DICT_CAP positions stay, nearest first
    for (uint32_t j = 0; j < nh; j++) {
        const uint32_t v = le32(j);
        uint4& b = img->bk4[hash_dict(v)];
        b.w = b.z;
        b.z = b.y;
        b.y = b.x;
        b.x = k_record(v, j ? (uint32_t)tmp[j - 1] : DICT_PREV0, j);
    }
    cudaError_t e = cudaMemcpyAsync(dev, img, sizeof(DictDev), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    free(img);
    if (e != cudaSuccess) HMSE_FAIL(ctx, HMSE_E_CUDA, "dictionary upload: %s", cudaGetErrorString(e));
    hd->valid = 1;
    *adler = hd->adler;
    return HMSE_OK;
}

size_t parse_smem(uint32_t nmax, bool match_smem, int own) {
    return (size_t)PAD_FRONT + nmax + 16 + PAD_SORTED + 2 * (size_t)(nmax + nmax / 32) + cnt_words(own) * 4 + nmax / 16 +
           ((sizeof(ParseSm) + 15) & ~15u) + (match_smem ? 4 * (size_t)(nmax + nmax / 32) : 0) + 32;
}

}  // namespace

HMSE_API int hmse_debug_deflate_prof(uint64_t* out16, int reset) {
    if (out16 && cudaMemcpyFromSymbol(out16, g_prof, sizeof(g_prof)) != cudaSuccess) return HMSE_E_CUDA;
    if (reset) {
        unsigned long long z[16] = {0};
        if (cudaMemcpyToSymbol(g_prof, z, sizeof(z)) != cudaSuccess) return HMSE_E_CUDA;
    }
    return HMSE_OK;
}

HMSE_API uint64_t hmse_compress_bound(uint64_t len) { return len + 5 * (len / 65535 + 1) + 6 + 4; }

HMSE_API int hmse_compress(hmse_ctx* ctx, const uint8_t* d_data, uint64_t start0, const uint64_t* d_cuts,
                           const uint64_t* d_select, uint64_t m, const uint8_t* d_zdict, uint32_t dict_len, int level,
                           uint8_t* d_out, uint64_t out_cap, uint64_t* d_offsets, uint64_t* total, void* stream) {
    if (!ctx) return HMSE_E_INVAL;
    cudaStream_t st = (cudaStream_t)stream;
    if (!total || !d_offsets) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compress: total/d_offsets is null");
    *total = 0;
    ctx->pack_valid = 0;
    if (dict_len > DICT_MAX) HMSE_FAIL(ctx, HMSE_E_INVAL, "dict_len must be <= 32768");
    if (dict_len && !d_zdict) HMSE_FAIL(ctx, HMSE_E_INVAL, "d_zdict is null");
    if (level != 0 && level != 6)
        HMSE_FAIL(ctx, HMSE_E_INVAL, "level must be 0 (stored blocks) or 6 (the match search is tuned against zlib level 6; "
                                     "other levels are not implemented)");
    if (m >= 0xFFFFFFFFull) HMSE_FAIL(ctx, HMSE_E_INVAL, "too many chunks in one call");
    if (m == 0) {
        HMSE_CUDA(ctx, cudaMemsetAsync(d_offsets, 0, 8, st));
        ctx->pack_m = ctx->pack_total = 0;
        ctx->pack_valid = 1;
        return HMSE_OK;
    }
    if (!d_data || !d_cuts) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compress: null pointer");
    if ((uintptr_t)d_data & 3) HMSE_FAIL(ctx, HMSE_E_INVAL, "d_data must be 4-byte aligned");

    uint32_t dict_adler = 0;
    if (dict_len) {
        int rc = ensure_dict(ctx, d_zdict, dict_len, &dict_adler, st);
        if (rc) return rc;
    }
    // misc: [slot_size m][slot_off m][sizes m+1][lists 4m u32][list_n 4 u32][totals 2 u64][stat 4 u64][counters]
    const size_t n_counters = m + 8;   // one work counter per batch; a long chunk may be a batch of its own
    const size_t misc_bytes = (3 * m + 2) * 8 + 4 * m * 4 + 64 + 32 + n_counters * 4 + 64;
    HMSE_SCRATCH(ctx, misc, uint8_t*, SLOT_DEFLATE_MISC, misc_bytes);
    uint64_t* slot_size = (uint64_t*)misc;
    uint64_t* slot_off = slot_size + m;
    uint64_t* sizes = slot_off + m;  // m + 1
    uint32_t* lists = (uint32_t*)(sizes + m + 1);
    uint32_t* list_n = lists + 4 * m;
    uint64_t* d_tot = (uint64_t*)(((uintptr_t)(list_n + 4) + 7) & ~(uintptr_t)7);  // [stage total, out total]
    unsigned long long* d_stat = (unsigned long long*)(d_tot + 2);   // per call and per ctx: contexts never share counters
    unsigned int* counters = (unsigned int*)(d_stat + 4);
    HMSE_CUDA(ctx, cudaMemsetAsync(list_n, 0, (size_t)((uint8_t*)(counters + n_counters) - (uint8_t*)list_n), st));
    KL(ctx);
    classify_kernel<<<(unsigned)div_up64(m, 256), 256, 0, st>>>(start0, d_cuts, d_select, m, slot_size, lists, list_n);
    HMSE_LAUNCH_CHECK(ctx);
    int rc = hmse_exclusive_scan_u64(ctx, slot_size, slot_off, m, d_tot, st);
    if (rc) return rc;
    volatile uint64_t* mail = ctx->pinned;
    if (int mrc = hmse_mail(ctx, 0, d_tot, 2, st)) return mrc;
    if (int mrc = hmse_mail(ctx, 2, list_n, 4, st)) return mrc;
    HMSE_CUDA(ctx, cudaStreamSynchronize(st));
    const uint64_t stage_bytes = mail[0];
    const uint32_t* hn = (const uint32_t*)(mail + 1);
    const uint32_t n_class[4] = {hn[0], hn[1], hn[2], hn[3]};
    HMSE_SCRATCH(ctx, stage, uint8_t*, SLOT_DEFLATE_STAGE, stage_bytes + 64);

    DeflArgs a;
    memset(&a, 0, sizeof(a));
    a.data = d_data;
    a.start0 = start0;
    a.cuts = d_cuts;
    a.select = d_select;
    a.dict = (const DictDev*)ctx->slot[SLOT_DEFLATE_DICT];
    a.dict_len = dict_len;
    a.dict_adler = dict_adler;
    a.level = level;
    a.stage = stage;
    a.slot_off = slot_off;
    a.sizes = sizes;
    a.stat = d_stat;

    const size_t sm_parse[N_CLASS] = {parse_smem(NMAX_SMALL, true, OWN_SMALL), parse_smem(NMAX_MEDIUM, false, OWN_MEDIUM),
                                      parse_smem(NMAX_LARGE, false, OWN_LARGE)};
    const size_t sm_huff = sizeof(HuffSm) * HUFF_WARPS;
    HMSE_CUDA(ctx, cudaFuncSetAttribute(parse_kernel<RS_SMALL, OWN_SMALL, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_parse[0]));
    HMSE_CUDA(ctx, cudaFuncSetAttribute(parse_kernel<5, OWN_MEDIUM, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_parse[1]));
    HMSE_CUDA(ctx, cudaFuncSetAttribute(parse_kernel<5, OWN_LARGE, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_parse[2]));
    HMSE_CUDA(ctx, cudaFuncSetAttribute(huffman_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_huff));
    const uint32_t nmax_c[N_CLASS] = {NMAX_SMALL, NMAX_MEDIUM, NMAX_LARGE};
    const uint32_t batch_c[N_CLASS] = {BATCH_SMALL, BATCH_MEDIUM, BATCH_LARGE};
    const uint32_t ctas_c[N_CLASS] = {(uint32_t)ctx->sm_count * 2, (uint32_t)ctx->sm_count * 2, (uint32_t)ctx->sm_count};

    // ---- plan of the long chunks (> NMAX_LARGE bytes): blocks of LONG_BLOCK bytes, batches aligned to chunks ----
    const uint32_t n_long = n_class[LONG_CLASS];
    std::vector<uint32_t> job_k, job_blk, ch_first, ch_nblk, batch_c0, batch_j0;   // batches: chunk / job boundaries
    std::vector<uint8_t> ch_stored;
    uint32_t long_jobs_max = 0, n_long_coded = 0;
    uint8_t* ldev = nullptr;   // [lens u64 n][first u32 n][nblk u32 n][flag u8 n (padded)][job_k][job_blk]
    size_t off_first = 0, off_nblk = 0, off_flag = 0, off_jk = 0, off_jb = 0;
    if (n_long) {
        std::vector<uint64_t> lens(n_long);
        HMSE_SCRATCH(ctx, lens_dev, uint64_t*, SLOT_DEFLATE_LONG, (size_t)n_long * 8);
        KL(ctx);
        long_len_kernel<<<(n_long + 255) / 256, 256, 0, st>>>(start0, d_cuts, d_select, lists + (size_t)LONG_CLASS * m, n_long, lens_dev);
        HMSE_LAUNCH_CHECK(ctx);
        HMSE_CUDA(ctx, cudaMemcpyAsync(lens.data(), lens_dev, (size_t)n_long * 8, cudaMemcpyDeviceToHost, st));
        HMSE_CUDA(ctx, cudaStreamSynchronize(st));
        ch_first.resize(n_long);
        ch_nblk.resize(n_long);
        ch_stored.assign(n_long, 0);
        batch_c0.push_back(0);
        batch_j0.push_back(0);
        for (uint32_t i = 0; i < n_long; i++) {
            const uint64_t nb = (lens[i] + LONG_BLOCK - 1) / LONG_BLOCK;
            ch_first[i] = (uint32_t)job_k.size();
            if (level == 0 || nb > 2048) {   // level 0, or a chunk beyond 64 MiB: stored blocks
                ch_nblk[i] = 0;
                ch_stored[i] = 1;
                continue;
            }
            ch_nblk[i] = (uint32_t)nb;
            n_long_coded++;
            if (job_k.size() - batch_j0.back() + nb > BATCH_LONG && job_k.size() > batch_j0.back()) {
                batch_c0.push_back(i);
                batch_j0.push_back((uint32_t)job_k.size());
            }
            for (uint32_t b = 0; b < nb; b++) {
                job_k.push_back(0);   // filled on the device side from the list: the host does not know k
                job_blk.push_back(b);
            }
        }
        batch_c0.push_back(n_long);
        batch_j0.push_back((uint32_t)job_k.size());
        for (size_t b = 0; b + 1 < batch_j0.size(); b++)
            if (batch_j0[b + 1] - batch_j0[b] > long_jobs_max) long_jobs_max = batch_j0[b + 1] - batch_j0[b];
        const size_t nj = job_k.size();
        off_first = (size_t)n_long * 8;
        off_nblk = off_first + (size_t)n_long * 4;
        off_flag = off_nblk + (size_t)n_long * 4;
        off_jk = (off_flag + n_long + 15) & ~(size_t)15;
        off_jb = off_jk + nj * 4;
        HMSE_SCRATCH(ctx, ld2, uint8_t*, SLOT_DEFLATE_LONG, off_jb + nj * 4 + 16);
        ldev = ld2;
        HMSE_CUDA(ctx, cudaMemcpyAsync(ldev + off_first, ch_first.data(), (size_t)n_long * 4, cudaMemcpyHostToDevice, st));
        HMSE_CUDA(ctx, cudaMemcpyAsync(ldev + off_nblk, ch_nblk.data(), (size_t)n_long * 4, cudaMemcpyHostToDevice, st));
        HMSE_CUDA(ctx, cudaMemcpyAsync(ldev + off_flag, ch_stored.data(), n_long, cudaMemcpyHostToDevice, st));
        if (nj) {
            // job -> selection slot: expand the chunk list by the block counts
            for (uint32_t i = 0; i < n_long; i++)
                for (uint32_t b = 0; b < ch_nblk[i]; b++) job_k[ch_first[i] + b] = i;   // index into the class list for now
            HMSE_CUDA(ctx, cudaMemcpyAsync(ldev + off_jk, job_k.data(), nj * 4, cudaMemcpyHostToDevice, st));
            HMSE_CUDA(ctx, cudaMemcpyAsync(ldev + off_jb, job_blk.data(), nj * 4, cudaMemcpyHostToDevice, st));
            KL(ctx);
            long_job_slot_kernel<<<(unsigned)((nj + 255) / 256), 256, 0, st>>>((uint32_t*)(ldev + off_jk), (uint32_t)nj, lists + (size_t)LONG_CLASS * m);
            HMSE_LAUNCH_CHECK(ctx);
        }
        HMSE_CUDA(ctx, cudaStreamSynchronize(st));   // the host vectors are pageable
    }

    // work scratch: tokens (u16 per input byte, per batch job), hist/codes, headers, records, large-class match
    size_t tok_bytes = 0, rec_jobs = 1;
    for (int c = 0; c < N_CLASS; c++) {
        const uint32_t jobs = n_class[c] < batch_c[c] ? n_class[c] : batch_c[c];
        if ((size_t)jobs * nmax_c[c] * 2 > tok_bytes) tok_bytes = (size_t)jobs * nmax_c[c] * 2;
        if (jobs > rec_jobs) rec_jobs = jobs;
    }
    if ((size_t)long_jobs_max * NMAX_LARGE * 2 > tok_bytes) tok_bytes = (size_t)long_jobs_max * NMAX_LARGE * 2;
    if (long_jobs_max > rec_jobs) rec_jobs = long_jobs_max;
    tok_bytes = (tok_bytes + 255) & ~(size_t)255;
    // CTAs that keep their match words in global scratch (one slot of NMAX_LARGE words each, whatever the class)
    uint32_t g_large = 0;
    for (int c = 1; c < N_CLASS; c++) {
        const uint32_t g = n_class[c] < ctas_c[c] ? n_class[c] : ctas_c[c];
        if (g > g_large) g_large = g;
    }
    if (long_jobs_max) {
        const uint32_t g = long_jobs_max < ctas_c[2] ? long_jobs_max : ctas_c[2];
        if (g > g_large) g_large = g;
    }
    const size_t work_bytes = tok_bytes + rec_jobs * (REC_WORDS * 4 + 640 + sizeof(ChunkRec)) +
                              (size_t)g_large * (NMAX_LARGE + NMAX_LARGE / 32) * 4 + 1024;
    HMSE_SCRATCH(ctx, work, uint8_t*, SLOT_DEFLATE_WORK, work_bytes);
    a.tokens = (uint16_t*)work;
    a.hist = (uint32_t*)(work + tok_bytes);
    a.hdrs = (uint8_t*)(a.hist + rec_jobs * REC_WORDS);
    a.recs = (ChunkRec*)(a.hdrs + rec_jobs * 640);
    a.match = (uint32_t*)(a.recs + rec_jobs);
    DictDev* long_dicts = nullptr;
    if (long_jobs_max) {
        HMSE_SCRATCH(ctx, ldicts, DictDev*, SLOT_DEFLATE_LDICT, (size_t)long_jobs_max * sizeof(DictDev));
        long_dicts = ldicts;
    }

    // one event pair per parse launch (timing mode): the roofline of the dominant kernel is per launch
    ctx->pev_n = 0;
    uint32_t n_parse = 0;
#define PARSE_EV(end)                                                                          \
    if (ctx->timing && ctx->pev_n < (uint32_t)HMSE_PARSE_EVENTS) {                            \
        cudaEventRecord(ctx->pev[2 * ctx->pev_n + (end)], st);                                \
        if (end) ctx->pev_n++;                                                                \
    }                                                                                          \
    if (end) n_parse++
    HT_BEGIN(ctx, HT_DEFLATE, st);
    uint32_t ci = 0;
    const uint32_t hmax = (uint32_t)ctx->sm_count * 3, emax = (uint32_t)ctx->sm_count * 8;
    for (int c = 0; c < N_CLASS; c++) {
        a.list = lists + (size_t)c * m;
        a.nmax = nmax_c[c];
        for (uint32_t j0 = 0; j0 < n_class[c]; j0 += batch_c[c]) {
            a.job0 = j0;
            a.job1 = j0 + batch_c[c] < n_class[c] ? j0 + batch_c[c] : n_class[c];
            a.counter = counters + ci++;
            const uint32_t jobs = a.job1 - a.job0;
            KL(ctx);
            PARSE_EV(0);
            if (c == 0) parse_kernel<RS_SMALL, OWN_SMALL, true><<<jobs < ctas_c[c] ? jobs : ctas_c[c], T_PARSE, sm_parse[c], st>>>(a);
            else if (c == 1) parse_kernel<5, OWN_MEDIUM, false><<<jobs < ctas_c[c] ? jobs : ctas_c[c], T_PARSE, sm_parse[c], st>>>(a);
            else parse_kernel<5, OWN_LARGE, false><<<jobs < ctas_c[c] ? jobs : ctas_c[c], T_PARSE, sm_parse[c], st>>>(a);
            PARSE_EV(1);
            if (level != 0) {
                const uint32_t hb = (jobs + HUFF_WARPS - 1) / HUFF_WARPS;
                KL(ctx);
                huffman_kernel<<<hb < hmax ? hb : hmax, HUFF_WARPS * 32, sm_huff, st>>>(a);
            }
            KL(ctx);
            encode_kernel<<<jobs < emax ? jobs : emax, T_ENCODE, 0, st>>>(a);
            HMSE_LAUNCH_CHECK(ctx);
        }
    }
    if (n_long) {
        // coded long chunks, batch by batch: previous-block indexes, parse, Huffman, bit-level concatenation
        LongArgs la;
        la.chunk_k = lists + (size_t)LONG_CLASS * m;
        la.chunk_first = (const uint32_t*)(ldev + off_first);
        la.chunk_nblk = (const uint32_t*)(ldev + off_nblk);
        la.stored_flag = ldev + off_flag;
        a.nmax = NMAX_LARGE;
        a.list = (const uint32_t*)(ldev + off_jk);
        a.blk = (const uint32_t*)(ldev + off_jb);
        a.long_dicts = long_dicts;
        for (size_t b = 0; n_long_coded && b + 1 < batch_j0.size(); b++) {
            a.job0 = batch_j0[b];
            a.job1 = batch_j0[b + 1];
            const uint32_t jobs = a.job1 - a.job0;
            if (!jobs) continue;
            a.counter = counters + ci++;
            KL(ctx);
            long_dict_kernel<<<jobs < (uint32_t)ctx->sm_count ? jobs : (uint32_t)ctx->sm_count, 1024, 0, st>>>(a);
            KL(ctx);
            PARSE_EV(0);
            parse_kernel<5, OWN_LARGE, false><<<jobs < ctas_c[2] ? jobs : ctas_c[2], T_PARSE, sm_parse[2], st>>>(a);
            PARSE_EV(1);
            const uint32_t hb = (jobs + HUFF_WARPS - 1) / HUFF_WARPS;
            KL(ctx);
            huffman_kernel<<<hb < hmax ? hb : hmax, HUFF_WARPS * 32, sm_huff, st>>>(a);
            la.c0 = batch_c0[b];
            la.c1 = batch_c0[b + 1];
            const uint32_t nc = la.c1 - la.c0;
            KL(ctx);
            encode_long_kernel<<<nc < emax ? nc : emax, T_ENCODE, 0, st>>>(a, la);
            HMSE_LAUNCH_CHECK(ctx);
        }
        // whatever stays (level 0, oversize, or not compressible): stored blocks
        a.list = lists + (size_t)LONG_CLASS * m;
        a.blk = nullptr;
        a.long_dicts = nullptr;
        a.stored_flag = ldev + off_flag;
        a.job0 = 0;
        a.job1 = n_long;
        KL(ctx);
        stored_kernel<<<n_long < 1024 ? n_long : 1024, 256, 0, st>>>(a);
        HMSE_LAUNCH_CHECK(ctx);
        a.stored_flag = nullptr;
    }
    HT_END(ctx, HT_DEFLATE, st);
    HMSE_CUDA(ctx, cudaMemsetAsync(sizes + m, 0, 8, st));
    rc = hmse_exclusive_scan_u64(ctx, sizes, d_offsets, m + 1, d_tot + 1, st);
    if (rc) return rc;
    if (int mrc = hmse_mail(ctx, 0, d_tot + 1, 2, st)) return mrc;
    if (int mrc = hmse_mail(ctx, 8, d_stat, 6, st)) return mrc;
    HMSE_CUDA(ctx, cudaStreamSynchronize(st));
    *total = mail[0];
    ctx->stat[0] = n_parse;
    ctx->stat[1] = mail[4];
    ctx->stat[2] = mail[5];
    ctx->stat[3] = mail[6];
    // the streams now sit in the stage slots; they stay there until the next hmse_compress on this ctx, so a caller
    // that did not know the size (d_out == NULL) or guessed too small packs them with hmse_compress_pack - no recompression
    ctx->pack_m = m;
    ctx->pack_total = mail[0];
    ctx->pack_valid = 1;
    if (!d_out && out_cap == 0) return HMSE_OK;   // sizes only
    if (!d_out || mail[0] > out_cap)
        HMSE_FAIL(ctx, HMSE_E_CAPACITY, "d_out capacity %llu < %llu bytes", (unsigned long long)out_cap,
                  (unsigned long long)mail[0]);
    return hmse_compress_pack(ctx, d_offsets, m, d_out, out_cap, stream);
}

HMSE_API int hmse_compress_pack(hmse_ctx* ctx, const uint64_t* d_offsets, uint64_t m, uint8_t* d_out, uint64_t out_cap,
                                void* stream) {
    if (!ctx) return HMSE_E_INVAL;
    cudaStream_t st = (cudaStream_t)stream;
    if (!ctx->pack_valid || m != ctx->pack_m)
        HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compress_pack: no staged result of %llu streams (call hmse_compress first)",
                  (unsigned long long)m);
    if (m == 0) return HMSE_OK;
    if (!d_offsets || !d_out) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compress_pack: null pointer");
    if (ctx->pack_total > out_cap)
        HMSE_FAIL(ctx, HMSE_E_CAPACITY, "d_out capacity %llu < %llu bytes", (unsigned long long)out_cap,
                  (unsigned long long)ctx->pack_total);
    const uint8_t* stage = (const uint8_t*)ctx->slot[SLOT_DEFLATE_STAGE];
    const uint64_t* slot_off = (const uint64_t*)ctx->slot[SLOT_DEFLATE_MISC] + m;   // [slot_size m][slot_off m] ...
    const uint64_t pg = m < (uint64_t)ctx->sm_count * 16 ? m : (uint64_t)ctx->sm_count * 16;
    HT_BEGIN(ctx, HT_PACK, st);
    KL(ctx);
    pack_kernel<<<(unsigned)pg, 256, 0, st>>>(stage, slot_off, d_offsets, m, d_out, out_cap);
    HMSE_LAUNCH_CHECK(ctx);
    HT_END(ctx, HT_PACK, st);
    return HMSE_OK;
}
