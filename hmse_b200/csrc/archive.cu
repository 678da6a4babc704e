// archive.cu - the on-disk records of the spec built on the device: the 40-byte packed `ChunkIndex` entry
// (README.md:1264-1269: sha256[32], lba u32, length u16, refcount u16) for every stored (first-occurrence)
// chunk, and the 8-byte pointer record "(LBA + offset)" (README.md:1312) for every chunk of the stream in
// order; and the inverse for the read path, the copy of inflated unique chunks back into stream order
// (README.md:1617-1675).  Layout conventions of this container (hmse_b200/archive.py, oracle/archive.py):
//   store position of unique chunk k   = offsets[k] bytes into the chunk store (the blob of hmse_compress)
//   ChunkIndex.lba                     = position >> 9 (512-byte sectors), .length = compressed bytes,
//                                        .refcount = chunks of the stream that resolve to it (saturating)
//   pointer record                     = { u32 lba, u16 position & 511, u16 raw length - 1 }
#include "ctx.cuh"

namespace {

__global__ void slot_of_kernel(const uint64_t* __restrict__ select, uint64_t m, uint64_t n, uint32_t* __restrict__ slot_of,
                               unsigned int* __restrict__ err) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= m) return;
    if (select[k] < n) slot_of[select[k]] = (uint32_t)k;
    else atomicOr(err, 16u);
}

__global__ void pointer_kernel(const int64_t* __restrict__ canon, uint64_t id_base, const uint64_t* __restrict__ cuts,
                               uint64_t start0, uint64_t n, const uint32_t* __restrict__ slot_of,
                               const uint64_t* __restrict__ offsets, uint32_t* __restrict__ refcount,
                               uint2* __restrict__ pointers, unsigned int* __restrict__ err) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    // canon is a global id: a chunk whose first occurrence lies in another shard (canon < id_base or >= id_base + n) has no
    // record in this shard's store - reported, never dereferenced
    const uint64_t c = (uint64_t)canon[i] - id_base;
    const uint32_t s = c < n ? slot_of[c] : 0xFFFFFFFFu;
    if (s == 0xFFFFFFFFu) {
        atomicOr(err, 4u);
        pointers[i] = make_uint2(0xFFFFFFFFu, 0xFFFFFFFFu);
        return;
    }
    atomicAdd(&refcount[s], 1u);
    const uint64_t pos = offsets[s];
    const uint64_t raw = cuts[i] - (i ? cuts[i - 1] : start0);
    if ((pos >> 9) > 0xFFFFFFFFull || raw == 0 || raw > 65536) atomicOr(err, 1u);
    pointers[i] = make_uint2((uint32_t)(pos >> 9), (uint32_t)(pos & 511) | ((uint32_t)((raw - 1) & 0xFFFF) << 16));
}

__global__ void index_kernel(const uint8_t* __restrict__ digests, const uint64_t* __restrict__ select, uint64_t m,
                             const uint64_t* __restrict__ offsets, const uint32_t* __restrict__ refcount,
                             uint8_t* __restrict__ index, unsigned int* __restrict__ err) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= m) return;
    const uint32_t* dg = reinterpret_cast<const uint32_t*>(digests + select[k] * 32);
    uint32_t* e = reinterpret_cast<uint32_t*>(index + k * 40);   // 40-byte entries stay 4-byte aligned
#pragma unroll
    for (int q = 0; q < 8; q++) e[q] = dg[q];
    const uint64_t pos = offsets[k], len = offsets[k + 1] - pos;
    if (len > 0xFFFF) atomicOr(err, 2u);
    const uint32_t rc = refcount[k] > 0xFFFFu ? 0xFFFFu : refcount[k];
    e[8] = (uint32_t)(pos >> 9);
    e[9] = (uint32_t)(len & 0xFFFF) | (rc << 16);
}

// dst[dst_off[i] .. dst_off[i+1]) = src[src_off[i] .. + the same length): one CTA per segment at a time.  GATHER: src_off[i]
// is the segment's own source address (segments from several buffers), src is unused.
template <bool GATHER>
__global__ void __launch_bounds__(256) segment_copy_kernel(const uint8_t* __restrict__ src, const uint64_t* __restrict__ src_off,
                                                           uint8_t* __restrict__ dst, const uint64_t* __restrict__ dst_off,
                                                           uint64_t n) {
    for (uint64_t i = blockIdx.x; i < n; i += gridDim.x) {
        const uint8_t* s = GATHER ? reinterpret_cast<const uint8_t*>(src_off[i]) : src + src_off[i];
        uint8_t* d = dst + dst_off[i];
        const uint64_t len = dst_off[i + 1] - dst_off[i];
        // head bytes until d is 4-aligned, then words assembled from the (arbitrarily aligned) source
        uint64_t head = (4 - ((uintptr_t)d & 3)) & 3;
        if (head > len) head = len;
        if (threadIdx.x < head) d[threadIdx.x] = s[threadIdx.x];
        const uint64_t body = (len - head) >> 2;
        const uint8_t* sb = s + head;
        const uint32_t kmis = (uint32_t)((uintptr_t)sb & 3);
        const uint32_t* ws = reinterpret_cast<const uint32_t*>(sb - kmis);
        uint32_t* wd = reinterpret_cast<uint32_t*>(d + head);
        for (uint64_t w = threadIdx.x; w < body; w += 256) {
            const uint32_t lo = ws[w], hi = kmis ? ws[w + 1] : 0u;
            wd[w] = __funnelshift_r(lo, hi, kmis * 8);
        }
        const uint64_t done = head + (body << 2);
        if (threadIdx.x < len - done) d[done + threadIdx.x] = s[done + threadIdx.x];
    }
}

// ---- L4: the same records when some first-occurrence chunks are stored as deltas (README.md:2182-2189) ----------------

// flag[c] = 1 when chunk c keeps a delta (u64, scanned into the rank of its DeltaChunk record)
__global__ void delta_flag_kernel(const uint64_t* __restrict__ delta_off, uint64_t n, uint64_t* __restrict__ flag) {
    const uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c < n) flag[c] = delta_off[c + 1] > delta_off[c];
}

__global__ void pointer_l4_kernel(const int64_t* __restrict__ canon, const uint64_t* __restrict__ cuts, uint64_t start0, uint64_t n,
                                  const uint32_t* __restrict__ slot_of, const uint64_t* __restrict__ offsets,
                                  const int64_t* __restrict__ base, const uint64_t* __restrict__ delta_off,
                                  const uint64_t* __restrict__ rank, uint64_t store_bytes, uint32_t* __restrict__ refcount,
                                  uint2* __restrict__ pointers, unsigned int* __restrict__ err) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t c = (uint64_t)canon[i];
    if (c >= n) { atomicOr(err, 4u); pointers[i] = make_uint2(0xFFFFFFFFu, 0xFFFFFFFFu); return; }
    uint64_t pos;
    if (delta_off[c + 1] > delta_off[c]) {
        pos = store_bytes + 8 * rank[c] + delta_off[c];
        if (i == c) {  // the delta itself holds one reference on its base
            const int64_t b = base[c];
            if (b < 0 || (uint64_t)b >= n || slot_of[b] == 0xFFFFFFFFu) atomicOr(err, 4u);
            else atomicAdd(&refcount[slot_of[b]], 1u);
        }
    } else {
        const uint32_t s = slot_of[c];
        if (s == 0xFFFFFFFFu) { atomicOr(err, 4u); return; }
        atomicAdd(&refcount[s], 1u);
        pos = offsets[s];
    }
    const uint64_t raw = cuts[i] - (i ? cuts[i - 1] : start0);
    if ((pos >> 9) > 0xFFFFFFFFull || raw == 0 || raw > 65536) atomicOr(err, 1u);
    pointers[i] = make_uint2((uint32_t)(pos >> 9), (uint32_t)(pos & 511) | ((uint32_t)((raw - 1) & 0xFFFF) << 16));
}

// One warp per chunk; chunks that keep a delta write { u32 base slot, u16 base raw length - 1, u16 delta length, data }.
__global__ void __launch_bounds__(256) delta_record_kernel(const int64_t* __restrict__ base, const uint64_t* __restrict__ delta_off,
                                                           const uint8_t* __restrict__ delta, const uint64_t* __restrict__ rank,
                                                           const uint64_t* __restrict__ cuts, uint64_t start0, uint64_t n,
                                                           const uint32_t* __restrict__ slot_of, uint8_t* __restrict__ out,
                                                           unsigned int* __restrict__ err) {
    const uint64_t c = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31;
    if (c >= n) return;
    const uint64_t d0 = delta_off[c], dl = delta_off[c + 1] - d0;
    if (dl == 0) return;
    const int64_t b = base[c];
    if (b < 0 || (uint64_t)b >= n) return;  // flagged by pointer_l4_kernel
    const uint64_t braw = cuts[b] - (b ? cuts[b - 1] : start0);
    if (dl > 0xFFFF || braw == 0 || braw > 65536) atomicOr(err, 8u);
    uint8_t* o = out + 8 * rank[c] + d0;
    if (lane < 8) {
        const uint32_t slot = slot_of[b];
        const uint32_t hi = (uint32_t)((braw - 1) & 0xFFFF) | ((uint32_t)(dl & 0xFFFF) << 16);
        o[lane] = (uint8_t)((lane < 4 ? slot >> (8 * lane) : hi >> (8 * (lane - 4))) & 0xFF);
    }
    for (uint64_t k = lane; k < dl; k += 32) o[8 + k] = delta[d0 + k];
}

}  // namespace

HMSE_API int hmse_index_build_l4(hmse_ctx* ctx, const uint8_t* d_digests, const int64_t* d_canon, const uint64_t* d_cuts,
                                 uint64_t start0, uint64_t n, const uint64_t* d_select, uint64_t m, const uint64_t* d_offsets,
                                 const int64_t* d_base, const uint64_t* d_delta_off, const uint8_t* d_delta, uint8_t* d_index,
                                 uint8_t* d_pointers, uint8_t* d_delta_store, uint64_t delta_store_cap,
                                 uint64_t* delta_store_bytes, void* stream) {
    if (!ctx) return HMSE_E_INVAL;
    cudaStream_t st = (cudaStream_t)stream;
    if (delta_store_bytes) *delta_store_bytes = 0;
    if (n == 0) return HMSE_OK;
    if (!d_digests || !d_canon || !d_cuts || !d_offsets || !d_index || !d_pointers || !d_base || !d_delta_off ||
        !delta_store_bytes || (m && !d_select))
        HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_index_build_l4: null pointer");
    if (n > 0xFFFFFFFEull) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_index_build_l4: n exceeds 2^32 - 2");
    if (((uintptr_t)d_index & 3) || ((uintptr_t)d_pointers & 7) || ((uintptr_t)d_digests & 3))
        HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_index_build_l4: d_index / d_digests must be 4-byte, d_pointers 8-byte aligned");
    // misc: [rank u64 n+1][slot_of u32 n][refcount u32 m+1][err u32][store_bytes u64 via offsets[m]]
    HMSE_SCRATCH(ctx, misc, uint64_t*, SLOT_ARCHIVE_MISC, (n + 2) * 8 + (n + m + 4) * 4);
    uint64_t* rank = misc;
    uint32_t* slot_of = reinterpret_cast<uint32_t*>(misc + n + 2);
    uint32_t* refcount = slot_of + n;
    unsigned int* err = refcount + m;
    HMSE_CUDA(ctx, cudaMemsetAsync(slot_of, 0xFF, n * 4, st));
    HMSE_CUDA(ctx, cudaMemsetAsync(refcount, 0, (m + 1) * 4, st));
    KL(ctx);
    delta_flag_kernel<<<(unsigned)div_up64(n, 256), 256, 0, st>>>(d_delta_off, n, rank);
    HMSE_LAUNCH_CHECK(ctx);
    if (int rc = hmse_exclusive_scan_u64(ctx, rank, rank, n, rank + n, st)) return rc;
    // host needs: number of delta records, delta bytes, store bytes
    if (int rc = hmse_mail(ctx, 0, rank + n, 2, st)) return rc;
    if (int rc = hmse_mail(ctx, 2, d_delta_off + n, 2, st)) return rc;
    if (int rc = hmse_mail(ctx, 4, d_offsets + m, 2, st)) return rc;
    HMSE_CUDA(ctx, cudaStreamSynchronize(st));
    const uint64_t n_delta = ctx->pinned[0], delta_bytes = ctx->pinned[1], store_bytes = ctx->pinned[2];
    *delta_store_bytes = 8 * n_delta + delta_bytes;
    if (*delta_store_bytes > delta_store_cap)
        HMSE_FAIL(ctx, HMSE_E_CAPACITY, "hmse_index_build_l4: delta_store_cap %llu < %llu", (unsigned long long)delta_store_cap,
                  (unsigned long long)*delta_store_bytes);
    if (n_delta && (!d_delta || !d_delta_store)) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_index_build_l4: null delta buffers");
    if (m) {
        KL(ctx);
        slot_of_kernel<<<(unsigned)div_up64(m, 256), 256, 0, st>>>(d_select, m, n, slot_of, err);
    }
    KL(ctx);
    pointer_l4_kernel<<<(unsigned)div_up64(n, 256), 256, 0, st>>>(d_canon, d_cuts, start0, n, slot_of, d_offsets, d_base, d_delta_off,
                                                                  rank, store_bytes, refcount, reinterpret_cast<uint2*>(d_pointers),
                                                                  err);
    if (m) {
        KL(ctx);
        index_kernel<<<(unsigned)div_up64(m, 256), 256, 0, st>>>(d_digests, d_select, m, d_offsets, refcount, d_index, err);
    }
    if (n_delta) {
        KL(ctx);
        delta_record_kernel<<<(unsigned)div_up64(n * 32, 256), 256, 0, st>>>(d_base, d_delta_off, d_delta, rank, d_cuts, start0, n,
                                                                             slot_of, d_delta_store, err);
    }
    HMSE_LAUNCH_CHECK(ctx);
    if (int mrc = hmse_mail(ctx, 0, err, 1, st)) return mrc;
    HMSE_CUDA(ctx, cudaStreamSynchronize(st));
    const uint32_t e = (uint32_t)ctx->pinned[0];
    if (e & 1) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_index_build_l4: a chunk is empty or longer than 65536 bytes, or the store exceeds 2 TiB");
    if (e & 2) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_index_build_l4: a compressed chunk is longer than 65535 bytes");
    if (e & 4) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_index_build_l4: a chunk resolves to a chunk that is neither stored nor a delta, or a delta's base is not stored");
    if (e & 8) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_index_build_l4: a delta is longer than 65535 bytes or its base longer than 65536");
    if (e & 16) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_index_build_l4: d_select holds an index >= n");
    return HMSE_OK;
}

HMSE_API int hmse_index_build(hmse_ctx* ctx, const uint8_t* d_digests, const int64_t* d_canon, uint64_t id_base,
                              const uint64_t* d_cuts, uint64_t start0, uint64_t n, const uint64_t* d_select, uint64_t m,
                              const uint64_t* d_offsets, uint8_t* d_index, uint8_t* d_pointers, void* stream) {
    if (!ctx) return HMSE_E_INVAL;
    cudaStream_t st = (cudaStream_t)stream;
    if (n == 0) return HMSE_OK;
    if (!d_digests || !d_canon || !d_cuts || !d_select || !d_offsets || !d_index || !d_pointers)
        HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_index_build: null pointer");
    if (n > 0xFFFFFFFFull) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_index_build: n exceeds 2^32");
    if (((uintptr_t)d_index & 3) || ((uintptr_t)d_pointers & 7) || ((uintptr_t)d_digests & 3))
        HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_index_build: d_index / d_digests must be 4-byte, d_pointers 8-byte aligned");
    // misc: [slot_of u32 n][refcount u32 m][err u32]
    HMSE_SCRATCH(ctx, misc, uint32_t*, SLOT_ARCHIVE_MISC, (n + m + 4) * 4);
    uint32_t* slot_of = misc;
    uint32_t* refcount = misc + n;
    unsigned int* err = refcount + m;
    HMSE_CUDA(ctx, cudaMemsetAsync(slot_of, 0xFF, n * 4, st));
    HMSE_CUDA(ctx, cudaMemsetAsync(refcount, 0, (m + 1) * 4, st));
    KL(ctx);
    slot_of_kernel<<<(unsigned)div_up64(m, 256), 256, 0, st>>>(d_select, m, n, slot_of, err);
    KL(ctx);
    pointer_kernel<<<(unsigned)div_up64(n, 256), 256, 0, st>>>(d_canon, id_base, d_cuts, start0, n, slot_of, d_offsets, refcount,
                                                               reinterpret_cast<uint2*>(d_pointers), err);
    KL(ctx);
    index_kernel<<<(unsigned)div_up64(m, 256), 256, 0, st>>>(d_digests, d_select, m, d_offsets, refcount, d_index, err);
    HMSE_LAUNCH_CHECK(ctx);
    if (int mrc = hmse_mail(ctx, 0, err, 1, st)) return mrc;
    HMSE_CUDA(ctx, cudaStreamSynchronize(st));
    const uint32_t e = (uint32_t)ctx->pinned[0];
    if (e & 1) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_index_build: a chunk is empty or longer than 65536 bytes, or the store exceeds 2 TiB");
    if (e & 2) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_index_build: a compressed chunk is longer than 65535 bytes");
    if (e & 4)
        HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_index_build: a chunk resolves (canon) to a chunk outside [id_base, id_base + n) or to one "
                                     "that is not in d_select - cross-shard duplicates have no record in a per-shard archive");
    if (e & 16) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_index_build: d_select holds an index >= n");
    return HMSE_OK;
}

HMSE_API int hmse_segment_copy(hmse_ctx* ctx, const uint8_t* d_src, const uint64_t* d_src_off, uint8_t* d_dst,
                               const uint64_t* d_dst_off, uint64_t n, void* stream) {
    if (!ctx) return HMSE_E_INVAL;
    if (n == 0) return HMSE_OK;
    if (!d_src || !d_src_off || !d_dst || !d_dst_off) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_segment_copy: null pointer");
    const uint64_t cap = (uint64_t)ctx->sm_count * 16;
    KL(ctx);
    segment_copy_kernel<false><<<(unsigned)(n < cap ? n : cap), 256, 0, (cudaStream_t)stream>>>(d_src, d_src_off, d_dst, d_dst_off, n);
    HMSE_LAUNCH_CHECK(ctx);
    return HMSE_OK;
}

int hmse_segment_gather(hmse_ctx* ctx, const uint64_t* d_src_addr, uint8_t* d_dst, const uint64_t* d_dst_off, uint64_t n,
                        cudaStream_t stream) {
    const uint64_t cap = (uint64_t)ctx->sm_count * 16;
    KL(ctx);   // launched for n == 0 too, so that a caller's kernel count does not depend on n
    segment_copy_kernel<true><<<(unsigned)(n == 0 ? 1 : n < cap ? n : cap), 256, 0, stream>>>(nullptr, d_src_addr, d_dst, d_dst_off, n);
    HMSE_LAUNCH_CHECK(ctx);
    return HMSE_OK;
}
