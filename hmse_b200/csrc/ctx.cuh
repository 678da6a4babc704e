// ctx.cuh - context, scratch slots and error plumbing shared by every translation unit.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/hmse.h"

#define HMSE_API extern "C" __attribute__((visibility("default")))

enum HmseSlot {
    SLOT_CDC_CFG = 0,   // device copy of gear table + parameters (CdcDev)
    SLOT_CDC_BITS,      // MaskS / MaskL candidate bitmaps, one bit per byte each
    SLOT_CDC_SEG,       // per-segment speculative + fix-up cut lists
    SLOT_CDC_META,      // per-segment entry/exit/count records and segment table, flags
    SLOT_CDC_FILES,     // first segment of every file (hmse_chunk_files)
    SLOT_SCAN,          // block sums of the generic exclusive scan
    SLOT_SHA_MISC,      // work counter
    SLOT_DEDUP_TABLE,   // open-addressing table of chunk indices
    SLOT_DEDUP_MISC,    // owner histogram / offsets for the partition step
    SLOT_DEDUP_OWNER,   // owner-side table + minimum gids of the sharded exchange (never the streaming table)
    SLOT_DEFLATE_STAGE, // per-chunk worst-case output slots
    SLOT_DEFLATE_MISC,  // sizes, slot offsets, class lists, counters
    SLOT_DEFLATE_DICT,  // hash-sorted index of the preset dictionary
    SLOT_DEFLATE_WORK,  // per-CTA match scratch for the large class
    SLOT_DEFLATE_LONG,  // block plan of chunks longer than 32 KiB
    SLOT_DEFLATE_LDICT, // per-block indexes of the previous block (long chunks)
    SLOT_MINHASH_MISC,  // work counter
    SLOT_LSH_SORT,      // radix-sort ping-pong buffers
    SLOT_LSH_MISC,      // digit histograms
    SLOT_INFLATE_MISC,  // work counter, error count
    SLOT_ARCHIVE_MISC,  // slot map and reference counts of the index build
    SLOT_DELTA_HEADS,   // bucket heads per (chunk, band) + root flags
    SLOT_DELTA_MISC,    // slot offsets, delta sizes, candidate list
    SLOT_DELTA_STAGE,   // per-candidate worst-case (len / 5) output slots
    SLOT_DELTA_BAD,     // error count of the decoder
    SLOT_CORPUS,
    SLOT_COMM_SMALL,    // counts / exits travelling through the all-gathers
    SLOT_COMM_SEND,     // records (dedup) or key columns (LSH) grouped by destination rank
    SLOT_COMM_RECV,     // what arrives, the owner's answers, the replies
    SLOT_READ_OPEN,     // record-number flags over delta-store positions, error word (hmse_read_open)
    SLOT_READ_PLAN,     // per-range lengths / first chunks / piece counts, need marks and their scans (hmse_read)
    SLOT_READ_WORK,     // need lists, per-stream statuses, piece offsets, gathered delta bytes
    SLOT_READ_DATA,     // the inflated stored chunks and applied deltas of one hmse_read batch
    SLOT_COMPOSE,       // source table, first-reference keys, candidate lists, gathered digests, scans (hmse_compose)
    SLOT_KNOWN_TABLE,   // digest table of the known lookup (never the streaming dedup table)
    SLOT_KNOWN,         // gathered digests, canon, plan and source addresses of hmse_compress_known
    SLOT_COUNT
};

// Timed regions (hmse_timing_ms ids; also in include/hmse.h)
constexpr int HMSE_PARSE_EVENTS = 128;
constexpr int HMSE_MAX_WORLD = 32;          // ranks per communicator (the counts matrix must fit the mailbox)
constexpr size_t HMSE_MAILBOX_BYTES = 16384;
enum HmseTimer {
    HT_SCAN = 0, HT_RESOLVE, HT_SHA, HT_DEDUP, HT_DEFLATE, HT_PACK, HT_MINHASH, HT_LSH, HT_INFLATE, HT_DELTA, HT_EXCHANGE,
    HT_READ_PLAN, HT_READ_COPY, HT_COMPOSE, HT_KNOWN, HT_COUNT
};
// HMSE_T_KNOWN is two spans (the lookup before the compression of the novel chunks, the merge after it): this private
// event pair holds the second, and hmse_timing_ms(HMSE_T_KNOWN) returns their sum
constexpr int HT_KNOWN_MERGE = HT_COUNT;
constexpr int HT_EVENT_PAIRS = HT_COUNT + 1;

struct hmse_ctx {
    int device;
    cudaEvent_t ev[2 * HT_EVENT_PAIRS];
    uint8_t ev_set[HT_EVENT_PAIRS];
    int timing;
    uint64_t launches;  // kernels launched through this ctx
    char err[512];
    void* slot[SLOT_COUNT];
    size_t slot_bytes[SLOT_COUNT];
    void* slot_base[SLOT_COUNT];  // what cudaMalloc returned (= slot[] unless guard bands surround the slot, HMSE_GUARD)
    uint64_t* pinned;  // small pinned host mailbox (HMSE_MAILBOX_BYTES), mapped: kernels write results into it directly
    uint64_t* pinned_dev;  // its device-side address
    int sm_count;
    // CDC state carried from scan to resolve
    uint64_t cdc_n_avail;
    hmse_cdc_cfg cdc_cfg;
    int cdc_cfg_valid;
    int cdc_have_scan;
    int cdc_rounds;
    // resolve state (incremental re-resolve)
    uint64_t seg_len, n_seg;
    uint64_t res_n_own;
    int res_eof, res_valid;
    // per-launch spans of the dominant kernel (parse_kernel) of the last hmse_compress, and what it moved
    cudaEvent_t pev[2 * HMSE_PARSE_EVENTS];
    uint32_t pev_n;
    uint64_t stat[4];  // [0] parse launches, [1] token words written, [2] input bytes parsed, [3] chunks parsed
    uint64_t dedup_cap, dedup_n;  // streaming dedup table (hmse_dedup_begin / hmse_dedup_append)
    void* dict_host;  // host copy + checksum of the indexed preset dictionary (deflate.cu)
    uint64_t pack_m, pack_total;  // streams / bytes staged by the last hmse_compress, still waiting in SLOT_DEFLATE_STAGE
    int pack_valid;               // (hmse_compress_pack copies them out without compressing again)
    uint64_t known_m, known_total;  // streams / bytes planned by the last hmse_compress_known (source addresses in SLOT_KNOWN)
    int known_valid;                // (hmse_compress_known_pack gathers them; any hmse_compress clears it)
    // multi-GPU (comm.cu)
    void* comm;       // ncclComm_t made by hmse_comm_init (null: callers pass their own)
    int comm_owned;
    int comm_rounds;  // stitch rounds of the last hmse_chunk_sharded
    uint64_t comm_stat[4];  // last exchange: bytes sent to / received from other ranks, records owned, records sent
};

#define HMSE_FAIL(ctx, code, ...)                              \
    do {                                                       \
        snprintf((ctx)->err, sizeof((ctx)->err), __VA_ARGS__); \
        return (code);                                         \
    } while (0)

#define HMSE_CUDA(ctx, call)                                                                   \
    do {                                                                                       \
        cudaError_t e__ = (call);                                                              \
        if (e__ != cudaSuccess) {                                                              \
            snprintf((ctx)->err, sizeof((ctx)->err), "%s:%d %s: %s", __FILE__, __LINE__, #call, \
                     cudaGetErrorString(e__));                                                 \
            return HMSE_E_CUDA;                                                                \
        }                                                                                      \
    } while (0)

#define HMSE_LAUNCH_CHECK(ctx) HMSE_CUDA(ctx, cudaGetLastError())
// counts a kernel launch; written before every <<< >>> so gpu_launches in bench.py is exact
#define KL(ctx) ((ctx)->launches++)
#define HT_BEGIN(ctx, id, st) \
    if ((ctx)->timing) cudaEventRecord((ctx)->ev[2 * (id)], (st))
#define HT_END(ctx, id, st)                                 \
    if ((ctx)->timing) {                                    \
        cudaEventRecord((ctx)->ev[2 * (id) + 1], (st));     \
        (ctx)->ev_set[id] = 1;                              \
    }

#define HMSE_SCRATCH(ctx, var, type, slot, bytes)                  \
    type var = (type)hmse_scratch((ctx), (slot), (size_t)(bytes)); \
    if (!(var)) return HMSE_E_NOMEM

// Grow-only scratch.  Returns nullptr (and sets err) on failure.  A grow synchronises the device
// (cudaFree) - steady-state calls with stable sizes never reallocate.
void* hmse_scratch(hmse_ctx* ctx, int slot, size_t bytes);

// Exclusive prefix sum of n u64 values (in may equal out).  d_total (device, may be null)
// receives the grand total.  Uses SLOT_SCAN.  Asynchronous on `stream`.
int hmse_exclusive_scan_u64(hmse_ctx* ctx, const uint64_t* d_in, uint64_t* d_out, uint64_t n,
                            uint64_t* d_total, cudaStream_t stream);

// Small results travel to the host through the mapped mailbox, written by a one-warp kernel: a
// cudaMemcpyAsync would queue behind whatever bulk copy occupies the device-to-host engine
// (the compressed blobs of the previous piece, when the caller streams), a store from an SM does not.
// Copies n32 32-bit words from d_src to mailbox word `word32` (4-byte units).  Asynchronous on `stream`.
int hmse_mail(hmse_ctx* ctx, uint32_t word32, const void* d_src, uint32_t n32, cudaStream_t stream);

// hmse_inflate without the host round trips: streams j = d_blob[d_begin[j] : d_end[j]) (d_end null: d_begin[j+1]),
// the dictionary's Adler-32 given by the caller.  Asynchronous on `stream`.
int hmse_inflate_ranges(hmse_ctx* ctx, const uint8_t* d_blob, const uint64_t* d_begin, const uint64_t* d_end, uint64_t m,
                        const uint8_t* d_zdict, uint32_t dict_len, uint32_t dict_adler, uint8_t* d_out,
                        const uint64_t* d_out_offsets, uint32_t* d_status, cudaStream_t stream);
uint32_t hmse_adler32_host(const uint8_t* d, size_t n);

// hmse_dedup's table over n keys (stride bytes apart, the digest first): canon[i] = smallest j with key j == key i,
// is_first[i] = (canon == i).  d_n (device, may be null) lowers n to a count only the device knows; the table is sized
// for n.  The table lives in scratch slot `slot`: SLOT_DEDUP_TABLE ends a streaming dedup session, any other slot
// leaves it alone.  Asynchronous on `stream`.
int hmse_dedup_table(hmse_ctx* ctx, const uint8_t* keys, uint64_t stride, uint64_t n, const uint64_t* d_n, int64_t* canon,
                     uint8_t* is_first, uint64_t* canon_gid, int slot, cudaStream_t stream);

// Where the streams staged by the last hmse_compress (m of them) sit: stream k starts at *stage + (*slot_off)[k] (device
// addresses).  Valid until the next hmse_compress on ctx; HMSE_E_INVAL when nothing of m streams is staged.
int hmse_compress_staged(hmse_ctx* ctx, uint64_t m, const uint8_t** stage, const uint64_t** slot_off);

// hmse_segment_copy with a source address per segment: d_dst[d_dst_off[i] : d_dst_off[i+1]) = the bytes at d_src_addr[i]
// (4 readable bytes must follow every segment).  Asynchronous on `stream`.
int hmse_segment_gather(hmse_ctx* ctx, const uint64_t* d_src_addr, uint8_t* d_dst, const uint64_t* d_dst_off, uint64_t n,
                        cudaStream_t stream);

// hmse_dedup_partition without the host round trip: d_counts[world] (device) receives the records per owner.
int hmse_dedup_partition_dev(hmse_ctx* ctx, const uint8_t* d_digests, uint64_t n, uint64_t id_base, uint32_t world,
                             uint8_t* d_records, uint32_t* d_perm, uint64_t* d_counts, cudaStream_t stream);

static inline uint64_t div_up64(uint64_t a, uint64_t b) { return (a + b - 1) / b; }
