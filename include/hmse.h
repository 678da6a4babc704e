/* hmse.h - C ABI of libhmse_b200.so: the HMSE data-reduction hot path on B200 (sm_100a).
 *
 * The reference (1Jamie/HMSE) defines this path only as a spec plus ESP-IDF skeletons; it has
 * no FFI.  Each entry point below replaces the spec function cited beside it, so a firmware or
 * host-side maintainer binds these where the skeleton called miniz / mbedtls / murmur3 (see
 * INTEGRATION.md for the ctypes binding that hmse_b200/ uses and the C call sequence).
 *
 * Conventions
 *  - extern "C", plain pointers and sizes.  Pointers named d_* are DEVICE pointers owned by the
 *    caller; everything else is host memory.  `stream` is a cudaStream_t passed as void*.
 *  - Every call returns an int status (HMSE_OK == 0, negative on error) and never throws;
 *    hmse_last_error(ctx) returns the text of the last failure on that context.
 *  - The library owns only scratch inside hmse_ctx (grown on demand, freed by hmse_destroy).
 *  - Kernels are enqueued on `stream`.  Calls that return a count to the host
 *    (hmse_chunk*, hmse_compress, hmse_dedup_partition) synchronise `stream` before returning;
 *    all others are asynchronous and their outputs are valid after the caller syncs `stream`.
 *  - One ctx per device per thread; a ctx is not thread-safe.
 *  - There is no CPU fallback: without a CUDA device every call fails with HMSE_E_CUDA.
 *
 * Chunk lists: a chunk list is (start0, cuts[n]) - chunk j is [j ? cuts[j-1] : start0, cuts[j]),
 * offsets relative to d_data.  This is the layout hmse_chunk* writes.
 */
#ifndef HMSE_H
#define HMSE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HMSE_OK 0
#define HMSE_E_INVAL (-1)    /* bad argument                                   */
#define HMSE_E_CAPACITY (-2) /* an output buffer is too small; needed size is returned */
#define HMSE_E_CUDA (-3)     /* CUDA runtime error (text in hmse_last_error)   */
#define HMSE_E_NOMEM (-4)    /* scratch allocation failed                      */
#define HMSE_E_NCCL (-5)     /* NCCL is missing or a collective failed (text in hmse_last_error) */

#define HMSE_ABI_VERSION 6

typedef struct hmse_ctx hmse_ctx;

/* FastCDC parameters (spec: README.md:289, 2444-2446; masks and Gear table per the FastCDC
 * paper the spec cites at README.md:2753-2755).  64 <= min <= avg <= max <= 1 MiB. */
typedef struct hmse_cdc_cfg {
    uint32_t min_size;
    uint32_t avg_size;
    uint32_t max_size;
    uint32_t reserved;
    uint64_t mask_s; /* tested while chunk length <  avg_size */
    uint64_t mask_l; /* tested while chunk length >= avg_size */
    uint64_t gear[256];
} hmse_cdc_cfg;

int hmse_abi_version(void);
int hmse_create(int device, hmse_ctx** out);
void hmse_destroy(hmse_ctx* ctx);
const char* hmse_last_error(hmse_ctx* ctx);
/* Bytes of device scratch currently held by ctx. */
uint64_t hmse_scratch_bytes(hmse_ctx* ctx);

/* Checked mode (test suite): with HMSE_GUARD=1 in the environment when the library is loaded, every scratch slot of a ctx
 * is surrounded by two 4 KiB guard bands; hmse_guard_check synchronises the device and fails with HMSE_E_INVAL (text
 * names the slot) when a kernel wrote outside its slot.  Without HMSE_GUARD it returns HMSE_E_INVAL. */
int hmse_guard_check(hmse_ctx* ctx);

/* ---- Measurement hooks (bench.py).  With timing enabled every entry point brackets its kernels
 *      with CUDA events on `stream`; hmse_timing_ms returns the last recorded span of a region. -- */
#define HMSE_T_SCAN 0
#define HMSE_T_RESOLVE 1
#define HMSE_T_SHA 2
#define HMSE_T_DEDUP 3
#define HMSE_T_DEFLATE 4
#define HMSE_T_PACK 5
#define HMSE_T_MINHASH 6
#define HMSE_T_LSH 7
#define HMSE_T_INFLATE 8
#define HMSE_T_DELTA 9
#define HMSE_T_EXCHANGE 10 /* the NCCL part of the last hmse_chunk_sharded / hmse_dedup_global / hmse_lsh_exchange */
#define HMSE_T_READ_PLAN 11 /* hmse_read steps 1-4: range checks, locate, pieces, need lists and their scans */
#define HMSE_T_READ_COPY 12 /* hmse_read: the pieces copied into the output, statuses folded per range */
#define HMSE_T_COMPOSE 13   /* hmse_compose: from the run checks to the last record written */
#define HMSE_T_KNOWN 14     /* hmse_compress_known: the lookup (steps 1-3) plus the stream lengths and offsets (step 5); the
                               compression of the novel chunks is HMSE_T_DEFLATE, the gather into d_out HMSE_T_PACK */
int hmse_timing(hmse_ctx* ctx, int enable);
int hmse_timing_ms(hmse_ctx* ctx, int id, float* ms);
/* Kernels launched through this ctx since hmse_create. */
uint64_t hmse_launch_count(hmse_ctx* ctx);
/* Facts about the last hmse_compress for the roofline of its dominant kernel (parse_kernel):
 * out4 = {parse launches, 16-bit token words written, input bytes parsed, chunks (blocks) parsed};
 * with timing enabled, *parse_ms_sum / *parse_ms_n = summed CUDA-event spans of (at most the first 128)
 * parse launches and how many were timed. */
int hmse_compress_stats(hmse_ctx* ctx, uint64_t* out4, float* parse_ms_sum, uint32_t* parse_ms_n);

/* ---- L2 chunking: replaces rabin_slide + the boundary loop of benchmark_fastcdc
 *      (README.md:2456-2464, 2475-2490). ------------------------------------------------- */

/* Whole stream: cuts of d_data[0:n).  d_cuts receives *n_cuts exclusive end offsets, strictly
 * increasing, last == n.  d_data must be 16-byte aligned.  On HMSE_E_CAPACITY *n_cuts holds the
 * required capacity. */
int hmse_chunk(hmse_ctx* ctx, const uint8_t* d_data, uint64_t n, const hmse_cdc_cfg* cfg,
               uint64_t* d_cuts, uint64_t cap, uint64_t* n_cuts, void* stream);

/* Many independent streams in one call.  File f = d_data[d_file_off[f] : d_file_off[f+1]) is chunked on its own,
 * exactly as hmse_chunk would chunk it in a buffer of its own (cuts at every file end; an empty file has no chunk).
 * d_file_off[n_files+1] (device) starts at 0, never decreases and ends at n; d_data as for hmse_chunk (16-byte aligned).
 * d_cuts receives one chunk list over the whole buffer (absolute offsets, start0 = 0); d_file_chunk[n_files+1] (device)
 * = index of each file's first chunk, d_file_chunk[n_files] = *n_cuts.  n / min_size + n_files + 1 always suffices as
 * cap; on HMSE_E_CAPACITY *n_cuts holds the capacity needed.  Bad offsets fail with HMSE_E_INVAL (checked on the
 * device, nothing written outside the outputs).  Synchronises `stream`. */
int hmse_chunk_files(hmse_ctx* ctx, const uint8_t* d_data, uint64_t n, const uint64_t* d_file_off, uint64_t n_files,
                     const hmse_cdc_cfg* cfg, uint64_t* d_cuts, uint64_t cap, uint64_t* n_cuts,
                     uint64_t* d_file_chunk, void* stream);

/* Sharded stream, step 1: candidate scan of d_data[0:n_avail) into ctx scratch. */
int hmse_chunk_scan(hmse_ctx* ctx, const uint8_t* d_data, uint64_t n_avail, const hmse_cdc_cfg* cfg,
                    void* stream);
/* Sharded stream, step 2 (repeatable): the chain of chunk starts s, entry <= s < n_own, over the
 * last scanned buffer.  eof != 0: the buffer ends the stream (n_own is ignored, = n_avail).
 * eof == 0: the stream continues; n_avail >= n_own + max_size is required.  *exit_off receives
 * the last cut (first chunk start >= n_own): the next shard's entry is exit_off - n_own.
 * Calling it again with another `entry` re-resolves incrementally. */
int hmse_chunk_resolve(hmse_ctx* ctx, const uint8_t* d_data, uint64_t n_own, uint64_t n_avail, int eof,
                       uint64_t entry, uint64_t* d_cuts, uint64_t cap, uint64_t* n_cuts,
                       uint64_t* exit_off, void* stream);
/* Copies the first n_words 64-bit words of the MaskS / MaskL candidate bitmaps of the last scan
 * (bit i of word w = byte position 64*w+i clears the mask on the full 64-byte window). */
int hmse_chunk_candidates(hmse_ctx* ctx, uint64_t* d_bits_s, uint64_t* d_bits_l, uint64_t n_words, void* stream);
/* Number of speculative fix-up rounds the last resolve needed (diagnostic). */
int hmse_chunk_last_rounds(hmse_ctx* ctx);

/* ---- L3 digest + exact dedup: replaces mbedtls_sha256 (README.md:2543) and the ChunkIndex
 *      lookup/insert rule (README.md:1264-1269, 1288-1292). -------------------------------- */

/* d_digests[j][32] = SHA-256 of chunk j. */
int hmse_digest(hmse_ctx* ctx, const uint8_t* d_data, uint64_t start0, const uint64_t* d_cuts,
                uint64_t n_chunks, uint8_t* d_digests, void* stream);

/* d_canon[i] = smallest j with digest j == digest i; d_is_first[i] = (canon == i). */
int hmse_dedup(hmse_ctx* ctx, const uint8_t* d_digests, uint64_t n, int64_t* d_canon,
               uint8_t* d_is_first, void* stream);

/* Streaming form of hmse_dedup over one growing digest array (the ChunkIndex insert rule applied
 * piece by piece, README.md:1542-1551).  hmse_dedup_begin sizes and clears the table for up to
 * max_chunks chunks; hmse_dedup_append inserts chunks [n_prev, n_prev + n_new) of d_digests_all
 * (whose first n_prev rows must be the ones appended so far, at the same address) and writes
 * d_canon[i - n_prev] = smallest j <= i with digest j == digest i (absolute indices),
 * d_is_first[i - n_prev] = (canon == i).  Results equal hmse_dedup over the whole array.
 * hmse_dedup uses the same table (it ends a streaming session); hmse_dedup_records has its own. */
int hmse_dedup_begin(hmse_ctx* ctx, uint64_t max_chunks, void* stream);
int hmse_dedup_append(hmse_ctx* ctx, const uint8_t* d_digests_all, uint64_t n_prev, uint64_t n_new,
                      int64_t* d_canon, uint8_t* d_is_first, void* stream);

/* d_select[0..*m) = ascending indices i with d_is_first[i] != 0 (the chunks to store/compress).
 * On HMSE_E_CAPACITY *m holds the required capacity. */
int hmse_dedup_select(hmse_ctx* ctx, const uint8_t* d_is_first, uint64_t n, uint64_t* d_select, uint64_t cap,
                      uint64_t* m, void* stream);

/* Multi-GPU dedup, sender side: groups records {digest[32], gid u64} by owner = le32(digest) %
 * world into d_records (40 B each, owner-major), d_perm[k] = local index of record k,
 * counts[world] (host) = records per owner.  gid = id_base + local index. */
int hmse_dedup_partition(hmse_ctx* ctx, const uint8_t* d_digests, uint64_t n, uint64_t id_base,
                         uint32_t world, uint8_t* d_records, uint32_t* d_perm, uint64_t* counts,
                         void* stream);
/* Owner side: d_canon_gid[k] = smallest gid among records with the same digest as record k. */
int hmse_dedup_records(hmse_ctx* ctx, const uint8_t* d_records, uint64_t m, uint64_t* d_canon_gid,
                       void* stream);
/* Sender side, after the return exchange: d_canon[d_perm[k]] = d_reply[k];
 * d_is_first[i] = (canon[i] == id_base + i). */
int hmse_dedup_scatter(hmse_ctx* ctx, const uint64_t* d_reply, const uint32_t* d_perm, uint64_t n,
                       uint64_t id_base, int64_t* d_canon, uint8_t* d_is_first, void* stream);

/* ---- Multi-GPU: one process per GPU, NCCL over NVLink (SURVEY.md section 8b "multi-GPU variant takes ncclComm_t and a
 *      global id base", 8e).  The reference is a single MCU (README.md:141-153) and has no counterpart; these entry
 *      points are what a host binding calls where the single-GPU flow calls hmse_chunk / hmse_dedup.
 *      `comm` is an ncclComm_t passed as void* (NCCL types stay out of this header) - the caller's own communicator, or
 *      NULL for the one hmse_comm_init created on this ctx.  NCCL is bound at run time (libnccl.so.2); without it these
 *      calls fail with HMSE_E_NCCL and everything else works.  Every rank of the communicator must make the same call. -- */
#define HMSE_UNIQUE_ID_BYTES 128
/* Rank 0: a fresh ncclUniqueId (128 bytes) to hand to every rank by any side channel. */
int hmse_comm_unique_id(uint8_t* out128);
/* ncclCommInitRank on ctx's device; the communicator belongs to ctx (freed by hmse_comm_destroy / hmse_destroy). */
int hmse_comm_init(hmse_ctx* ctx, const uint8_t* id128, int world, int rank);
int hmse_comm_destroy(hmse_ctx* ctx);
/* Size, rank and NCCL version (e.g. 22809) of `comm` (NULL: ctx's own); any out pointer may be null. */
int hmse_comm_info(hmse_ctx* ctx, void* comm, int* world, int* rank, int* nccl_version);
/* out[4 * r + q] (host) = vals4[q] of rank r: one ncclAllGather, one mailbox read (synchronises `stream`). */
int hmse_allgather_u64(hmse_ctx* ctx, void* comm, const uint64_t* vals4, uint64_t* out, void* stream);

/* L2 chunking of ONE stream held as contiguous byte-range shards: this rank holds d_data[0:n_avail) = its n_own owned
 * bytes + max_size bytes of look-ahead (eof != 0: the last shard, n_own is ignored).  Scan, speculative resolve from
 * offset 0, then rounds of { all-gather exits, re-resolve incrementally from the true entry } until no entry changes.
 * d_cuts / *n_cuts: the chunks that START in this shard (cuts relative to d_data); *entry = offset of the first one;
 * *id_base = chunks in the shards before this one; *n_total = chunks of the whole stream.  Concatenated over ranks the
 * cut lists equal hmse_chunk over the whole stream.  Synchronises `stream`. */
int hmse_chunk_sharded(hmse_ctx* ctx, void* comm, const uint8_t* d_data, uint64_t n_own, uint64_t n_avail, int eof,
                       const hmse_cdc_cfg* cfg, uint64_t* d_cuts, uint64_t cap, uint64_t* n_cuts, uint64_t* entry,
                       uint64_t* id_base, uint64_t* n_total, void* stream);
/* Global exact dedup (the ChunkIndex rule over the whole stream, README.md:1288-1292): d_canon[i] = smallest GLOBAL id
 * (id_base + local index on its rank) with the same digest anywhere, d_is_first[i] = (canon == id_base + i).  Records
 * travel to owner = le32(digest) % world and the answers back with ncclSend / ncclRecv groups on `stream`.
 * One host round trip (the counts); results are valid after the caller syncs `stream`. */
int hmse_dedup_global(hmse_ctx* ctx, void* comm, const uint8_t* d_digests, uint64_t n, uint64_t id_base, int64_t* d_canon,
                      uint8_t* d_is_first, void* stream);
/* Global LSH bucketing, exchange step: band b is owned by rank b % world.  d_keys[n][bands] (this rank's chunks, stream
 * order) -> d_owned[*n_total][*bands_owned] = the owned bands' keys of EVERY chunk of the stream, rows in global id
 * order (feed it to hmse_lsh_buckets with id_base 0; local column c is band rank + c * world).  *id_base = global id
 * of this rank's first chunk.  d_owned == NULL with owned_cap_rows == 0 only reports the sizes; on HMSE_E_CAPACITY
 * *n_total holds the rows needed. */
int hmse_lsh_exchange(hmse_ctx* ctx, void* comm, const uint64_t* d_keys, uint64_t n, uint32_t bands, uint64_t* d_owned,
                      uint64_t owned_cap_rows, uint64_t* n_total, uint64_t* id_base, uint32_t* bands_owned, void* stream);
/* Generic variable all-to-all on `stream`: the elements (elem_bytes each) of d_send are grouped by destination rank,
 * send_counts[world] (host) of them per rank; recv_counts[world] (host, out) = elements arriving from each rank, stored in
 * d_recv in rank order.  The counts travel first (one all-gather, one host round trip).  d_recv == NULL with
 * recv_cap == 0 is the size query: it only fills recv_counts and moves no data - a collective of its own that every
 * rank must make; the exchange proper follows with buffers of at least those sizes (d_recv non-null even when nothing
 * arrives).  Used by the cross-shard L4 steps
 * (heads back to the chunks' ranks, root flags to everybody, base chunk requests and their bytes). */
int hmse_alltoallv(hmse_ctx* ctx, void* comm, const void* d_send, const uint64_t* send_counts, void* d_recv,
                   uint64_t* recv_counts, uint32_t elem_bytes, uint64_t recv_cap, void* stream);
/* Facts about the last exchange on ctx: out4 = {bytes sent to other ranks, bytes received from other ranks, records
 * (or rows) owned after the exchange, records (rows) contributed}; *rounds = resync rounds of the last
 * hmse_chunk_sharded (may be null). */
int hmse_exchange_stats(hmse_ctx* ctx, uint64_t* out4, int* rounds);

/* ---- L1 DEFLATE: replaces mz_deflateInit2 / mz_deflate(FINISH) (README.md:2374, 2378). --- */

/* Worst-case bytes of one zlib stream for a chunk of `len` bytes. */
uint64_t hmse_compress_bound(uint64_t len);

/* One RFC 1950 stream (FDICT set when dict_len > 0) per selected chunk, packed back to back in
 * d_out in selection order; d_offsets[m+1] are the stream boundaries.  d_select[k] is a chunk
 * index (NULL = chunks 0..m-1).  dict_len <= 32768.  level: 6 (match search and lazy rule tuned against zlib
 * level 6) or 0 (stored blocks); anything else fails with HMSE_E_INVAL.  *total (host) = d_offsets[m].
 * d_out == NULL with out_cap == 0: everything but the final copy is done (sizes only, HMSE_OK).  On HMSE_E_CAPACITY
 * *total holds the required out_cap.  In both cases the streams stay staged inside ctx until the next hmse_compress and
 * hmse_compress_pack copies them out - the chunks are never compressed twice.
 * d_data: 4-byte aligned, and 16 readable bytes must follow the last chunk (chunks are staged with aligned 16-byte
 * vector loads: the vector that holds a chunk's last byte is read whole). */
int hmse_compress(hmse_ctx* ctx, const uint8_t* d_data, uint64_t start0, const uint64_t* d_cuts,
                  const uint64_t* d_select, uint64_t m, const uint8_t* d_zdict, uint32_t dict_len,
                  int level, uint8_t* d_out, uint64_t out_cap, uint64_t* d_offsets, uint64_t* total,
                  void* stream);

/* Packs the m streams staged by the last hmse_compress on ctx (same d_offsets) into d_out[0 : total). */
int hmse_compress_pack(hmse_ctx* ctx, const uint64_t* d_offsets, uint64_t m, uint8_t* d_out, uint64_t out_cap, void* stream);

/* Diagnostic: cycles spent per encoder phase (thread 0 of each CTA, summed over chunks) since
 * the last reset; out16[15] = chunks encoded.  Host pointer. */
int hmse_debug_deflate_prof(uint64_t* out16, int reset);

/* ---- Read path: replaces mz_inflateInit2 / mz_inflate (README.md:2397-2400, 1638-1640). -------------
 * Stream j = d_blob[d_offsets[j] : d_offsets[j+1]) is one RFC 1950 stream (any valid one with a window
 * <= 32 KiB: the output of hmse_compress or of stock zlib with the same preset dictionary) and is inflated
 * into d_out[d_out_offsets[j] : d_out_offsets[j+1]); the caller knows the raw sizes (the chunk index stores
 * them, README.md:1264-1269).  d_status[j] = 0 when the stream is well formed, yields exactly that many bytes
 * and its Adler-32 trailer (and DICTID, with a dictionary) agrees; otherwise an error code (1 header, 2 block
 * header, 3 code / distance, 4 overrun, 5 length, 6 checksum) - a bad stream never writes outside its range.
 * *n_bad (may be null) receives the number of non-zero statuses (synchronises `stream`). */
int hmse_inflate(hmse_ctx* ctx, const uint8_t* d_blob, const uint64_t* d_offsets, uint64_t m,
                 const uint8_t* d_zdict, uint32_t dict_len, uint8_t* d_out, const uint64_t* d_out_offsets,
                 uint32_t* d_status, uint64_t* n_bad, void* stream);

/* ---- Archive records (README.md:1264-1269 ChunkIndex, 1312 pointer records) and stream reassembly. ------
 * d_index[k] (40 B, packed) = { sha256 of unique chunk k = chunk d_select[k], u32 lba = d_offsets[k] >> 9,
 * u16 length = compressed bytes, u16 refcount (saturating) }; d_pointers[i] (8 B) = { u32 lba, u16 d_offsets[s] & 511,
 * u16 raw length - 1 } with s the unique chunk that chunk i resolves to (d_canon[i] - id_base is its local index).
 * Fails with HMSE_E_INVAL when a chunk is empty or longer than 65536 bytes, a compressed chunk is longer than
 * 65535 bytes, or the store exceeds 2 TiB.  Synchronises `stream`. */
int hmse_index_build(hmse_ctx* ctx, const uint8_t* d_digests, const int64_t* d_canon, uint64_t id_base,
                     const uint64_t* d_cuts, uint64_t start0, uint64_t n, const uint64_t* d_select, uint64_t m,
                     const uint64_t* d_offsets, uint8_t* d_index, uint8_t* d_pointers, void* stream);
/* The same records when L4 stores some first-occurrence chunks as deltas (single GPU: canon and base are local
 * indices).  d_select / d_offsets describe the m chunks in the chunk store (first occurrences that keep no delta);
 * chunk c keeps a delta iff d_delta_off[c+1] > d_delta_off[c] (the outputs of hmse_delta_encode).  Writes the delta
 * store: one `struct DeltaChunk` (README.md:2182-2189) per kept delta in chunk order, { u32 base = ChunkIndex entry
 * number of the base chunk (the spec's "LBA lookup" goes through that entry), u16 base raw length - 1, u16 delta
 * length, delta bytes }.  A pointer record whose position (lba * 512 + offset) is >= the chunk store size addresses
 * the DeltaChunk at (position - store size) in the delta store.  Reference counts include one reference per delta on
 * its base.  *delta_store_bytes (host) = bytes written; on HMSE_E_CAPACITY the required delta_store_cap. */
int hmse_index_build_l4(hmse_ctx* ctx, const uint8_t* d_digests, const int64_t* d_canon, const uint64_t* d_cuts,
                        uint64_t start0, uint64_t n, const uint64_t* d_select, uint64_t m, const uint64_t* d_offsets,
                        const int64_t* d_base, const uint64_t* d_delta_off, const uint8_t* d_delta, uint8_t* d_index,
                        uint8_t* d_pointers, uint8_t* d_delta_store, uint64_t delta_store_cap, uint64_t* delta_store_bytes,
                        void* stream);
/* d_dst[d_dst_off[i] : d_dst_off[i+1]) = d_src[d_src_off[i] : + the same length) for i < n (d_dst_off has n+1
 * entries, d_src_off n; d_src needs 4 readable bytes after its last segment). */
int hmse_segment_copy(hmse_ctx* ctx, const uint8_t* d_src, const uint64_t* d_src_off, uint8_t* d_dst,
                      const uint64_t* d_dst_off, uint64_t n, void* stream);

/* ---- Random-access reads: byte ranges of an archive's raw stream, many per call, planned on the device
 *      (the spec's read path, README.md:1617-1675, from pointer records to chunks, for ranges instead of whole
 *      streams).  An archive is opened once (hmse_read_open derives a device layout the caller owns) and read many
 *      times; the library keeps no per-archive state, so one ctx serves any number of open archives. ---------------- */

/* Bytes of the device layout buffer for an archive of n chunks, m stored chunks and n_delta DeltaChunk records. */
uint64_t hmse_read_layout_bytes(uint64_t n, uint64_t m, uint64_t n_delta);

/* Checks the records of an archive on the device and derives what reads need into d_layout (8-byte aligned,
 * layout_bytes >= hmse_read_layout_bytes(n, m, n_delta)): the raw offset of every chunk, the stored slot or DeltaChunk
 * record of every chunk, the store position and raw length of every stored chunk, the base, lengths and position of
 * every record, and the Adler-32 of the dictionary.  d_index = m 40-byte ChunkIndex entries (4-byte aligned),
 * d_pointers = n 8-byte pointer records (8-byte aligned), n_delta == 0: no delta store.  Fails with HMSE_E_INVAL, the
 * failed check named, when (1) the index entries do not tile the store, (2) a pointer below store_bytes does not
 * address the start of a stored chunk, (3) a pointer at or above store_bytes has no delta store, or its record header
 * or delta bytes lie outside it, or its base slot is >= m, (4) two references to one stored chunk or one record
 * disagree on its raw length (a record's base length counts as a reference to its base), (5) a stored chunk has no
 * known raw length, (6) the raw lengths do not add up to raw_bytes.  Synchronises `stream`. */
int hmse_read_open(hmse_ctx* ctx, const uint8_t* d_index, uint64_t m, const uint8_t* d_pointers, uint64_t n,
                   uint64_t store_bytes, const uint8_t* d_delta_store, uint64_t delta_store_bytes, uint64_t n_delta,
                   uint64_t raw_bytes, const uint8_t* d_zdict, uint32_t dict_len,
                   void* d_layout, uint64_t layout_bytes, void* stream);

/* R ranges d_ranges[r] = {offset, length} of the raw stream -> d_out[d_out_off[r] : d_out_off[r+1]) (d_out_off written,
 * packed in request order).  n, m, n_delta: those given to hmse_read_open for d_layout (a mismatch is HMSE_E_INVAL).
 * d_store / d_delta_store / d_zdict: the buffers the layout was opened on; the stores need 16 readable bytes after
 * their end.  Ranges may be empty, overlap, repeat and come in any order.  A range past raw_bytes (or one whose
 * offset + length overflows) fails the call with HMSE_E_INVAL before anything is written.  *total (host) = bytes of
 * all ranges; on HMSE_E_CAPACITY it holds the out_cap needed and nothing is written.  Every stored chunk and
 * DeltaChunk record the batch needs is inflated / applied exactly once, whatever the number of ranges that touch it.
 * d_status[r] = 0, else the hmse_inflate code (1-6) of a stored chunk the range needs, or 16 + the hmse_delta_apply
 * code (1-5) of a delta it needs (the largest code when several fail); a failed range never causes writes outside its
 * own output range, and ranges that need no damaged chunk are correct.  *n_bad (host) = ranges with a non-zero
 * status.  stats4 (host, may be null) = {streams inflated, deltas applied, raw bytes inflated, pieces}.  Two host
 * round trips (the sizes, then n_bad); the number of kernels does not depend on R, n or the ranges.  Synchronises
 * `stream`. */
int hmse_read(hmse_ctx* ctx, const void* d_layout, uint64_t n, uint64_t m, uint64_t n_delta, const uint8_t* d_store,
              const uint8_t* d_delta_store, const uint8_t* d_zdict, uint32_t dict_len, const uint64_t* d_ranges,
              uint64_t R, uint8_t* d_out, uint64_t out_cap, uint64_t* d_out_off, uint64_t* total, uint32_t* d_status,
              uint64_t* n_bad, uint64_t* stats4, void* stream);

/* ---- Compose: files of several opened archives merged or subset into one archive, on the device.  The output is the
 *      archive one ingest of the selected files, in order, would have written when the sources keep no deltas: stored
 *      chunks numbered by first reference, equal SHA-256 digests stored once across sources.  The library keeps no
 *      per-archive state: every source comes with the layout hmse_read_open wrote for it. ------------------------------- */

/* One source: the buffers an archive was opened on (hmse_read_open) and its dims.  d_delta_store may be null when
 * n_delta == 0.  The stores need 4 readable bytes after their end. */
typedef struct hmse_compose_src {
    const void* d_layout;         /* written by hmse_read_open for these buffers and dims */
    const uint8_t* d_index;       /* m 40-byte ChunkIndex entries (4-byte aligned) */
    const uint8_t* d_pointers;    /* n 8-byte pointer records */
    const uint8_t* d_store;       /* chunk store */
    const uint8_t* d_delta_store; /* DeltaChunk records */
    uint64_t n, m, n_delta;
} hmse_compose_src;

/* srcs[n_src] (host): the sources.  d_runs[n_runs][3] (device, u64) = {source, first chunk, chunk count}: the output
 * stream is the runs' chunks back to back, n_out chunks in all (the counts must add up to n_out, n_out <= 2^32 - 2).
 * Outputs (device, caller-owned): d_pointers[n_out] (8-byte aligned) = one pointer record per output chunk, raw length
 * copied from the source pointer; d_index[index_cap] (4-byte aligned) = one ChunkIndex entry per kept stored chunk;
 * d_store[store_cap] = their zlib streams, copied byte for byte; d_delta_store[delta_cap] = the DeltaChunk records.
 * Rule: a stored chunk is kept when an output chunk references it, directly or as the base of a referenced DeltaChunk
 * record; its key is the output position of its first reference (a record's reference to its base counts at the
 * record's chunk).  Kept chunks with equal digests (their sources' index entries) are one chunk: the smaller key wins,
 * references to the other are remapped.  Kept chunks are numbered and packed in key order; records, identified by
 * (source, record), are written once each, numbered by first reference, their base remapped and the rest copied.
 * DeltaChunk records are not deduplicated across sources (the container stores no digest for them).  Refcounts: one
 * per pointer to the slot and one per written record on its base, saturating at 65535.
 * out6 (host) = {n_out, stored chunks referenced (before the digest dedup), stored chunks kept, store bytes, records,
 * delta-store bytes}.  HMSE_E_INVAL, before anything is written: a layout that does not match its source's dims,
 * sources whose dictionaries differ in length or Adler-32, a run outside its source, counts that do not add up to
 * n_out, or an output whose chunk store plus delta store reaches 2 TiB.  HMSE_E_CAPACITY: out6 holds the sizes
 * needed and nothing is written.  hmse_compose uses hmse_dedup's table: it ends a streaming dedup session.  Two host
 * round trips (the sizes, then an error word); the number of kernels does not depend on n_src, n_runs or the sizes.
 * Synchronises `stream`. */
int hmse_compose(hmse_ctx* ctx, const hmse_compose_src* srcs, uint32_t n_src, const uint64_t* d_runs, uint64_t n_runs,
                 uint64_t n_out, uint8_t* d_pointers, uint8_t* d_index, uint64_t index_cap, uint8_t* d_store,
                 uint64_t store_cap, uint8_t* d_delta_store, uint64_t delta_cap, uint64_t* out6, void* stream);

/* ---- Compression against an opened archive: a new snapshot that is mostly in an archive already costs the DEFLATE of
 *      what the archive lacks.  The library keeps no per-archive state: the archive comes as an hmse_compose_src
 *      (the layout hmse_read_open wrote and its buffers), and its digest table is rebuilt on every call. ---------------- */

/* hmse_compress with one more input, the archive `src`, and the SHA-256 of every chunk: d_digests[i][32] (device, 4-byte
 * aligned) for chunk i.  For stream k (chunk i = d_select[k], or k when d_select is NULL):
 *  - known: the smallest source slot whose index entry holds the digest of chunk i also holds a chunk of i's raw length
 *    (the layout's ulen).  Stream k is then the source's stream of that slot, copied byte for byte from src->d_store.
 *    DeltaChunk targets have no index entry and are never known.
 *  - novel: every other stream is compressed exactly as hmse_compress compresses it.
 * d_out, d_offsets[m+1], *total, the sizes-only call (d_out == NULL, out_cap == 0) and HMSE_E_CAPACITY follow
 * hmse_compress, in selection order; in both cases the plan and the compressed novel streams stay in ctx until the next
 * hmse_compress / hmse_compress_known, and hmse_compress_known_pack writes them - no chunk is compressed twice.
 * The output equals hmse_compress's byte for byte whenever the source's streams were written by this encoder at the same
 * level with the same dictionary (every archive that hmse_index_build or hmse_compose wrote from ingests at that level).
 * The container does not record the level: streams of another level are copied as they are - valid streams of the same
 * chunks that inflate correctly, but not the bytes hmse_compress would write.
 * d_known[m] (device, may be NULL) = the source slot stream k was copied from, or -1 when it was compressed.
 * stats4 (host, may be NULL) = {streams copied, bytes copied, streams compressed, raw bytes compressed}.
 * HMSE_E_INVAL before anything is written: a layout that was not opened for src's n, m, n_delta, a dictionary whose length
 * or Adler-32 differs from the source's, null or misaligned buffers (d_cuts, d_select, d_offsets, d_known 8-byte aligned;
 * d_data as for hmse_compress).  The digest table has a scratch slot of its own: a streaming dedup session
 * (hmse_dedup_begin / append) survives the call; its build is also recorded as HMSE_T_DEDUP.  One host round trip besides those of hmse_compress (the checks and
 * counts); the kernels of the lookup and the merge do not depend on m or on the source.  Synchronises `stream`. */
int hmse_compress_known(hmse_ctx* ctx, const hmse_compose_src* src, const uint8_t* d_data, uint64_t start0,
                        const uint64_t* d_cuts, const uint8_t* d_digests, const uint64_t* d_select, uint64_t m,
                        const uint8_t* d_zdict, uint32_t dict_len, int level, uint8_t* d_out, uint64_t out_cap,
                        uint64_t* d_offsets, uint64_t* total, int64_t* d_known, uint64_t* stats4, void* stream);
/* Writes the m streams planned by the last hmse_compress_known on ctx (same d_offsets) into d_out[0 : total). */
int hmse_compress_known_pack(hmse_ctx* ctx, const uint64_t* d_offsets, uint64_t m, uint8_t* d_out, uint64_t out_cap,
                             void* stream);

/* ---- L4 similarity: replaces minhash_compute (README.md:2578-2597) and LSH banding
 *      (README.md:2231-2235). -------------------------------------------------------------- */

/* d_sig[j][n_perm]: running minimum (from 0xFFFFFFFF) of MurmurHash3_x86_32(4-byte shingle,
 * d_seeds[p]) over every byte offset of chunk j.  n_perm must be a multiple of 32, <= 256. */
int hmse_minhash(hmse_ctx* ctx, const uint8_t* d_data, uint64_t start0, const uint64_t* d_cuts,
                 uint64_t n_chunks, const uint32_t* d_seeds, uint32_t n_perm, uint32_t* d_sig,
                 void* stream);
/* The same for the m chunks d_select[0..m) only: d_sig[k][n_perm] = signature of chunk d_select[k] (the spec computes
 * MinHash only for chunks that passed exact dedup, README.md:1553-1556). */
int hmse_minhash_select(hmse_ctx* ctx, const uint8_t* d_data, uint64_t start0, const uint64_t* d_cuts,
                        const uint64_t* d_select, uint64_t m, const uint32_t* d_seeds, uint32_t n_perm, uint32_t* d_sig,
                        void* stream);
/* d_keys[j][bands] = FNV-1a-64 of the band's rows*4 little-endian signature bytes. */
int hmse_lsh_keys(hmse_ctx* ctx, const uint32_t* d_sig, uint64_t n, uint32_t bands, uint32_t rows,
                  uint64_t* d_keys, void* stream);
/* All n*bands triples (band, key, id_base + j) sorted by (band, key, id). */
int hmse_lsh_buckets(hmse_ctx* ctx, const uint64_t* d_keys, uint64_t n, uint32_t bands,
                     uint64_t id_base, uint32_t* d_band, uint64_t* d_key, uint64_t* d_id, void* stream);

/* ---- L4 delta coding: replaces the "probe LSH index -> compute binary delta -> store if <= 20 %" step
 *      (README.md:1328, 1555-1570) and the xdelta3 encode / patch calls of Appendix A (README.md:2160-2198).
 *      The spec gives no byte format (xdelta3 / bsdiff are named, neither is vendored); the format is the COPY/ADD
 *      op list of the spec's example (README.md:1402-1412) as oracle/deltacode.py defines it:
 *        delta = op* ; op = varint(len << 1 | kind) ; kind 0 ADD: len literal bytes ; kind 1 COPY:
 *        varint(zigzag(q - expect)), target += base[q : q + len], expect = q + len (0 at the start) ;
 *        varint = unsigned LEB128.  Chunks and bases longer than 32768 bytes are never delta-coded. ------- */

/* Base selection over the sorted triples of hmse_lsh_buckets (n chunks, bands <= 32, ids id_base..id_base+n-1):
 * head(i, b) = first chunk with d_is_first set of the bucket chunk i falls in for band b (only chunks that passed exact
 * dedup enter the index); votes(i, j) = bands whose head is j < i;
 * root(i) = d_is_first[i] and no j reaches min_votes; d_base[i] = the root with the most votes >= min_votes
 * (ties to the smaller index) as a LOCAL index, or -1 (also for duplicates).  Bases are roots: no chains. */
int hmse_delta_bases(hmse_ctx* ctx, const uint32_t* d_band, const uint64_t* d_key, const uint64_t* d_id, uint64_t n,
                     uint32_t bands, uint64_t id_base, const uint8_t* d_is_first, uint32_t min_votes, int64_t* d_base,
                     void* stream);
/* The pieces of hmse_delta_bases for a stream sharded over several GPUs (ids are then GLOBAL ids of the first
 * occurrences of the whole stream, README.md:1556-1559 "probe LSH index -> return base chunk" is a global lookup):
 * hmse_delta_heads: d_heads[(id - id_base) * bands + band] = first id of the bucket, over sorted triples of n chunks
 *   (d_is_first may be null = every chunk is a first occurrence) - run by the band owners after hmse_lsh_exchange;
 * hmse_delta_votes pass 0: d_root_local[i] = no earlier head of chunk id_base + i reaches min_votes;
 *   pass 1: d_base[i] = best-voted earlier head h with d_root_all[h] set (an id in the heads' id space), or -1.
 *   d_heads[n][bands] belongs to this rank's chunks; d_root_all covers every id (all ranks' pass-0 results gathered). */
int hmse_delta_heads(hmse_ctx* ctx, const uint32_t* d_band, const uint64_t* d_key, const uint64_t* d_id, uint64_t n,
                     uint32_t bands, uint64_t id_base, const uint8_t* d_is_first, uint32_t* d_heads, void* stream);
int hmse_delta_votes(hmse_ctx* ctx, const uint32_t* d_heads, uint64_t n, uint32_t bands, uint64_t id_base, uint32_t min_votes,
                     int pass, uint8_t* d_root_local, const uint8_t* d_root_all, int64_t* d_base, void* stream);
/* hmse_delta_encode with bases that are not chunks of d_data: d_base[i] >= n names external base d_base[i] - n, the bytes
 * d_ext_data[d_ext_off[e] : d_ext_off[e + 1]) (8-byte aligned buffer, 16 readable bytes after the last base) - chunks of
 * another shard fetched beforehand.  Everything else as hmse_delta_encode. */
int hmse_delta_encode_ext(hmse_ctx* ctx, const uint8_t* d_data, uint64_t start0, const uint64_t* d_cuts, uint64_t n,
                          int64_t* d_base, const uint8_t* d_ext_data, const uint64_t* d_ext_off, uint64_t n_ext,
                          uint8_t* d_out, uint64_t out_cap, uint64_t* d_offsets, uint64_t* total, void* stream);
/* For every chunk i with d_base[i] >= 0: the delta of chunk i against chunk d_base[i] (greedy walk over 8-byte
 * seeds of a 16384-bucket index of the base that keeps the smallest position per bucket; backward then forward
 * extension), kept iff 5 * bytes <= chunk length; otherwise d_base[i] is reset to -1.  The kept deltas are packed
 * in chunk order into d_out; d_offsets[n+1] bound them (empty for chunks without a delta); *total (host) =
 * d_offsets[n].  On HMSE_E_CAPACITY *total holds the required out_cap (sum of len / 5 over the candidates always
 * suffices).  d_data: 16-byte aligned, 16 readable bytes after the last chunk.  Synchronises `stream`. */
int hmse_delta_encode(hmse_ctx* ctx, const uint8_t* d_data, uint64_t start0, const uint64_t* d_cuts, uint64_t n,
                      int64_t* d_base, uint8_t* d_out, uint64_t out_cap, uint64_t* d_offsets, uint64_t* total,
                      void* stream);
/* Read path (README.md:2191-2198 "apply patch to decompressed base"): delta j = d_delta[d_delta_off[j] :
 * d_delta_off[j+1]) applied to the raw base d_base[d_base_off[j] : + d_base_len[j]) yields
 * d_out[d_out_off[j] : d_out_off[j+1]).  base_bytes = size of d_base (a base range outside it is status 3).
 * d_status[j] = 0, or 1 bad varint, 2 bad op length or offsets that run backwards, 3 copy outside the
 * base, 4 literals past the end of the delta, 5 trailing bytes; a bad delta never reads or writes outside its ranges.
 * *n_bad (may be null) = number of non-zero statuses (synchronises `stream`). */
int hmse_delta_apply(hmse_ctx* ctx, const uint8_t* d_delta, const uint64_t* d_delta_off, uint64_t m,
                     const uint8_t* d_base, uint64_t base_bytes, const uint64_t* d_base_off, const uint32_t* d_base_len,
                     uint8_t* d_out, const uint64_t* d_out_off, uint32_t* d_status, uint64_t* n_bad, void* stream);

/* ---- Synthetic corpus (bench/test input, not part of the reference path): renders bytes
 *      [byte_off, byte_off + n) of the procedural wiki stream defined in oracle/corpus.py. ---- */
typedef struct hmse_corpus_cfg {
    uint32_t seed;
    uint32_t dup_thr;
    uint32_t near_thr;
    uint32_t n_lex; /* lexicon entries */
    uint32_t pick_tries; /* attempts of a copy article to find an earlier article of the unique class (0 = 4) */
} hmse_corpus_cfg;
/* d_art_len[n_articles] (u32) = byte length of each article first_article.. */
int hmse_corpus_lengths(hmse_ctx* ctx, const hmse_corpus_cfg* cfg, const uint32_t* d_lex_off,
                        uint64_t first_article, uint64_t n_articles, uint32_t* d_art_len, void* stream);
/* d_art_off[n_articles+1] = exclusive prefix sum of lengths (stream offset of each article).
 * Writes stream bytes [byte_off, byte_off+n) to d_out. */
int hmse_corpus_render(hmse_ctx* ctx, const hmse_corpus_cfg* cfg, const uint8_t* d_lex_blob,
                       const uint32_t* d_lex_off, uint64_t first_article, uint64_t n_articles,
                       const uint64_t* d_art_off, uint64_t byte_off, uint64_t n, uint8_t* d_out,
                       void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HMSE_H */
