// dedup.cu - L3 exact dedup: the ChunkIndex lookup/insert rule (spec: README.md:1264-1269,
// 1288-1292, 1542-1551) as a GPU open-addressing table keyed by the digest.  The first chunk
// (smallest index in stream order) with a digest is the stored instance; every later one maps
// to it.  Slots hold chunk indices, not digests: keys are compared by reading the caller's
// digest array, so the table is 4 bytes per slot at load factor <= 0.5.
//
// insert : linear probing; empty slot -> CAS(my index); same digest -> atomicMin(my index);
//          other digest -> next slot.  No deletions, so probe sequences are stable.
// lookup : probe until the slot's digest equals mine; the slot value is canon.
//
// Multi-GPU (north_star: "hash table partitioned by digest prefix with NCCL all-to-all"):
// hmse_dedup_partition groups 40-byte records {digest, gid} by owner = le32(digest) % world;
// the host exchanges them (torch.distributed all_to_all_single over NCCL); the owner runs the
// same table over its records (arrival order = gid order), and the reply is scattered back.
#include "ctx.cuh"

namespace {

constexpr uint32_t EMPTY = 0xFFFFFFFFu;

struct Key {
    uint64_t a, b, c, d;
};

__device__ __forceinline__ Key load_key(const uint8_t* __restrict__ base, uint64_t stride, uint64_t i) {
    const uint64_t* p = reinterpret_cast<const uint64_t*>(base + i * stride);
    Key k;
    k.a = p[0];
    k.b = p[1];
    k.c = p[2];
    k.d = p[3];
    return k;
}
__device__ __forceinline__ bool same(const Key& x, const Key& y) {
    return x.a == y.a && x.b == y.b && x.c == y.c && x.d == y.d;
}
// Table position from digest bytes 8..15 (bytes 0..3 choose the owner GPU in the sharded path).
__device__ __forceinline__ uint64_t slot_of(const Key& k, uint64_t mask) {
    uint64_t h = k.b * 0x9E3779B97F4A7C15ull;
    return (h >> 20) & mask;
}

// Inserts keys i0 .. n-1 (earlier indices may already be in the table: streaming append); n_dev (device, may be null)
// lowers n to a count only the device knows.
__global__ void dedup_insert_kernel(const uint8_t* __restrict__ keys, uint64_t stride, uint64_t i0, uint64_t n,
                                    const uint64_t* __restrict__ n_dev, uint32_t* __restrict__ table, uint64_t mask) {
    uint64_t i = i0 + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || (n_dev && i >= *n_dev)) return;
    const Key me = load_key(keys, stride, i);
    uint64_t pos = slot_of(me, mask);
    for (;;) {
        uint32_t cur = table[pos];
        if (cur == EMPTY) {
            cur = atomicCAS(&table[pos], EMPTY, (uint32_t)i);
            if (cur == EMPTY) return;
        }
        if (same(load_key(keys, stride, cur), me)) {
            atomicMin(&table[pos], (uint32_t)i);
            return;
        }
        pos = (pos + 1) & mask;
    }
}

// Looks up keys i0 .. n-1; outputs are indexed from i0 (canon[i - i0] holds the absolute index).
__global__ void dedup_lookup_kernel(const uint8_t* __restrict__ keys, uint64_t stride, uint64_t i0, uint64_t n,
                                    const uint64_t* __restrict__ n_dev, const uint32_t* __restrict__ table, uint64_t mask,
                                    int64_t* __restrict__ canon, uint8_t* __restrict__ is_first, uint64_t* __restrict__ canon_gid) {
    uint64_t i = i0 + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || (n_dev && i >= *n_dev)) return;
    const Key me = load_key(keys, stride, i);
    uint64_t pos = slot_of(me, mask);
    for (;;) {
        uint32_t cur = table[pos];
        if (cur != EMPTY && same(load_key(keys, stride, cur), me)) {
            if (canon) canon[i - i0] = (int64_t)cur;
            if (is_first) is_first[i - i0] = cur == (uint32_t)i;
            if (canon_gid) canon_gid[i - i0] = *reinterpret_cast<const uint64_t*>(keys + (uint64_t)cur * stride + 32);
            return;
        }
        pos = (pos + 1) & mask;
    }
}

// ---- partition by owner ------------------------------------------------------------------
__global__ void owner_hist_kernel(const uint8_t* __restrict__ digests, uint64_t n, uint32_t world,
                                  unsigned long long* __restrict__ hist) {
    extern __shared__ unsigned int sh[];
    for (unsigned w = threadIdx.x; w < world; w += blockDim.x) sh[w] = 0;
    __syncthreads();
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        uint32_t p = *reinterpret_cast<const uint32_t*>(digests + i * 32);
        atomicAdd(&sh[p % world], 1u);
    }
    __syncthreads();
    for (unsigned w = threadIdx.x; w < world; w += blockDim.x)
        if (sh[w]) atomicAdd(&hist[w], (unsigned long long)sh[w]);
}

// Stable placement is not required (the owner orders by gid through atomicMin), so records take
// the next free place in their owner's range.
__global__ void owner_scatter_kernel(const uint8_t* __restrict__ digests, uint64_t n, uint64_t id_base, uint32_t world,
                                     const uint64_t* __restrict__ offs, unsigned long long* __restrict__ cursor,
                                     uint8_t* __restrict__ records, uint32_t* __restrict__ perm) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t* d = reinterpret_cast<const uint64_t*>(digests + i * 32);
    uint32_t owner = (uint32_t)d[0] % world;
    uint64_t k = offs[owner] + atomicAdd(&cursor[owner], 1ull);
    uint64_t* r = reinterpret_cast<uint64_t*>(records + k * 40);
    r[0] = d[0];
    r[1] = d[1];
    r[2] = d[2];
    r[3] = d[3];
    r[4] = id_base + i;
    perm[k] = (uint32_t)i;
}

__global__ void scatter_reply_kernel(const uint64_t* __restrict__ reply, const uint32_t* __restrict__ perm, uint64_t n,
                                     uint64_t id_base, int64_t* __restrict__ canon, uint8_t* __restrict__ is_first) {
    uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    uint32_t i = perm[k];
    uint64_t g = reply[k];
    canon[i] = (int64_t)g;
    if (is_first) is_first[i] = g == id_base + i;
}

// The owner must see equal digests resolve to the smallest GID, but records from different
// senders arrive grouped by sender, not sorted by gid, and table slots order by record index.
// Senders own disjoint ascending gid ranges and are concatenated in rank order, and within a
// sender the scatter above is unordered - so the table is keyed on record index and a second
// pass reduces to the minimum gid among equal digests.
__global__ void min_gid_kernel(const uint8_t* __restrict__ records, uint64_t m, const uint32_t* __restrict__ table,
                               uint64_t mask, unsigned long long* __restrict__ min_gid) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const Key me = load_key(records, 40, i);
    uint64_t pos = slot_of(me, mask);
    for (;;) {
        uint32_t cur = table[pos];
        if (cur != EMPTY && same(load_key(records, 40, cur), me)) {
            atomicMin(&min_gid[cur], *reinterpret_cast<const unsigned long long*>(records + i * 40 + 32));
            return;
        }
        pos = (pos + 1) & mask;
    }
}
__global__ void read_gid_kernel(const uint8_t* __restrict__ records, uint64_t m, const uint32_t* __restrict__ table,
                                uint64_t mask, const unsigned long long* __restrict__ min_gid,
                                uint64_t* __restrict__ canon_gid) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const Key me = load_key(records, 40, i);
    uint64_t pos = slot_of(me, mask);
    for (;;) {
        uint32_t cur = table[pos];
        if (cur != EMPTY && same(load_key(records, 40, cur), me)) {
            canon_gid[i] = min_gid[cur];
            return;
        }
        pos = (pos + 1) & mask;
    }
}

__global__ void flags_to_u64_kernel(const uint8_t* __restrict__ flags, uint64_t n, uint64_t* __restrict__ out) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = flags[i] ? 1ull : 0ull;
}
__global__ void select_scatter_kernel(const uint8_t* __restrict__ flags, const uint64_t* __restrict__ pos, uint64_t n,
                                      uint64_t cap, uint64_t* __restrict__ select) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && flags[i] && pos[i] < cap) select[pos[i]] = i;
}

}  // namespace

int hmse_dedup_table(hmse_ctx* ctx, const uint8_t* keys, uint64_t stride, uint64_t n, const uint64_t* d_n, int64_t* canon,
                     uint8_t* is_first, uint64_t* canon_gid, int slot, cudaStream_t st) {
    if (n >= 0x7FFFFFFFull) HMSE_FAIL(ctx, HMSE_E_INVAL, "dedup: more than 2^31-1 chunks per table");
    uint64_t cap = 1024;
    while (cap < 2 * n) cap <<= 1;
    HMSE_SCRATCH(ctx, table, uint32_t*, slot, cap * sizeof(uint32_t));
    HMSE_CUDA(ctx, cudaMemsetAsync(table, 0xFF, cap * sizeof(uint32_t), st));
    if (slot == SLOT_DEDUP_TABLE) ctx->dedup_cap = 0;   // the one-shot table replaces a streaming one
    const unsigned grid = (unsigned)div_up64(n, 256);
    HT_BEGIN(ctx, HT_DEDUP, st);
    KL(ctx);
    dedup_insert_kernel<<<grid, 256, 0, st>>>(keys, stride, 0, n, d_n, table, cap - 1);
    KL(ctx);
    dedup_lookup_kernel<<<grid, 256, 0, st>>>(keys, stride, 0, n, d_n, table, cap - 1, canon, is_first, canon_gid);
    HMSE_LAUNCH_CHECK(ctx);
    HT_END(ctx, HT_DEDUP, st);
    return HMSE_OK;
}

HMSE_API int hmse_dedup_select(hmse_ctx* ctx, const uint8_t* d_is_first, uint64_t n, uint64_t* d_select, uint64_t cap,
                               uint64_t* m, void* stream) {
    if (!ctx) return HMSE_E_INVAL;
    cudaStream_t st = (cudaStream_t)stream;
    if (!m) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_dedup_select: m is null");
    *m = 0;
    if (n == 0) return HMSE_OK;
    if (!d_is_first) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_dedup_select: null pointer");
    HMSE_SCRATCH(ctx, tmp, uint64_t*, SLOT_DEDUP_MISC, (n + 2) * 8);
    const unsigned grid = (unsigned)div_up64(n, 256);
    KL(ctx);
    flags_to_u64_kernel<<<grid, 256, 0, st>>>(d_is_first, n, tmp);
    HMSE_LAUNCH_CHECK(ctx);
    int rc = hmse_exclusive_scan_u64(ctx, tmp, tmp, n, tmp + n, st);
    if (rc) return rc;
    if (d_select && cap) {
        KL(ctx);
        select_scatter_kernel<<<grid, 256, 0, st>>>(d_is_first, tmp, n, cap, d_select);
        HMSE_LAUNCH_CHECK(ctx);
    }
    if (int mrc = hmse_mail(ctx, 0, tmp + n, 2, st)) return mrc;
    HMSE_CUDA(ctx, cudaStreamSynchronize(st));
    *m = ctx->pinned[0];
    if (!d_select || *m > cap)
        HMSE_FAIL(ctx, HMSE_E_CAPACITY, "d_select capacity %llu < %llu", (unsigned long long)cap, (unsigned long long)*m);
    return HMSE_OK;
}

HMSE_API int hmse_dedup(hmse_ctx* ctx, const uint8_t* d_digests, uint64_t n, int64_t* d_canon, uint8_t* d_is_first,
                          void* stream) {
    if (!ctx) return HMSE_E_INVAL;
    if (n == 0) return HMSE_OK;
    if (!d_digests || !d_canon) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_dedup: null pointer");
    if ((uintptr_t)d_digests & 7) HMSE_FAIL(ctx, HMSE_E_INVAL, "d_digests must be 8-byte aligned");
    return hmse_dedup_table(ctx, d_digests, 32, n, nullptr, d_canon, d_is_first, nullptr, SLOT_DEDUP_TABLE, (cudaStream_t)stream);
}

HMSE_API int hmse_dedup_begin(hmse_ctx* ctx, uint64_t max_chunks, void* stream) {
    if (!ctx) return HMSE_E_INVAL;
    if (max_chunks >= 0x7FFFFFFFull) HMSE_FAIL(ctx, HMSE_E_INVAL, "dedup: more than 2^31-1 chunks per table");
    uint64_t cap = 1024;
    while (cap < 2 * max_chunks) cap <<= 1;
    HMSE_SCRATCH(ctx, table, uint32_t*, SLOT_DEDUP_TABLE, cap * sizeof(uint32_t));
    HMSE_CUDA(ctx, cudaMemsetAsync(table, 0xFF, cap * sizeof(uint32_t), (cudaStream_t)stream));
    ctx->dedup_cap = cap;
    ctx->dedup_n = 0;
    return HMSE_OK;
}

HMSE_API int hmse_dedup_append(hmse_ctx* ctx, const uint8_t* d_digests_all, uint64_t n_prev, uint64_t n_new,
                                 int64_t* d_canon, uint8_t* d_is_first, void* stream) {
    if (!ctx) return HMSE_E_INVAL;
    cudaStream_t st = (cudaStream_t)stream;
    if (!ctx->dedup_cap) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_dedup_append: call hmse_dedup_begin first");
    if (n_prev != ctx->dedup_n) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_dedup_append: n_prev %llu != %llu chunks appended so far",
                                          (unsigned long long)n_prev, (unsigned long long)ctx->dedup_n);
    if (2 * (n_prev + n_new) > ctx->dedup_cap)
        HMSE_FAIL(ctx, HMSE_E_CAPACITY, "hmse_dedup_append: table sized for %llu chunks", (unsigned long long)(ctx->dedup_cap / 2));
    if (n_new == 0) return HMSE_OK;
    if (!d_digests_all || !d_canon) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_dedup_append: null pointer");
    if ((uintptr_t)d_digests_all & 7) HMSE_FAIL(ctx, HMSE_E_INVAL, "d_digests_all must be 8-byte aligned");
    uint32_t* table = (uint32_t*)ctx->slot[SLOT_DEDUP_TABLE];
    const unsigned grid = (unsigned)div_up64(n_new, 256);
    const uint64_t n = n_prev + n_new;
    HT_BEGIN(ctx, HT_DEDUP, st);
    KL(ctx);
    dedup_insert_kernel<<<grid, 256, 0, st>>>(d_digests_all, 32, n_prev, n, nullptr, table, ctx->dedup_cap - 1);
    KL(ctx);
    dedup_lookup_kernel<<<grid, 256, 0, st>>>(d_digests_all, 32, n_prev, n, nullptr, table, ctx->dedup_cap - 1, d_canon, d_is_first,
                                              nullptr);
    HMSE_LAUNCH_CHECK(ctx);
    HT_END(ctx, HT_DEDUP, st);
    ctx->dedup_n = n;
    return HMSE_OK;
}

int hmse_dedup_partition_dev(hmse_ctx* ctx, const uint8_t* d_digests, uint64_t n, uint64_t id_base, uint32_t world,
                             uint8_t* d_records, uint32_t* d_perm, uint64_t* d_counts, cudaStream_t st) {
    if (world == 0 || world > 512) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_dedup_partition: bad world");
    if (n > 0xFFFFFFFFull) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_dedup_partition: n exceeds 2^32");
    // misc: [hist world][offs world][cursor world]
    HMSE_SCRATCH(ctx, misc, uint64_t*, SLOT_DEDUP_MISC, 3 * (size_t)world * 8);
    HMSE_CUDA(ctx, cudaMemsetAsync(misc, 0, 3 * (size_t)world * 8, st));
    if (n) {
        if (!d_digests || !d_records || !d_perm) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_dedup_partition: null pointer");
        const unsigned grid = (unsigned)div_up64(n, 256);
        KL(ctx);
        owner_hist_kernel<<<grid, 256, world * sizeof(unsigned int), st>>>(d_digests, n, world, (unsigned long long*)misc);
        HMSE_LAUNCH_CHECK(ctx);
        int rc = hmse_exclusive_scan_u64(ctx, misc, misc + world, world, nullptr, st);
        if (rc) return rc;
        KL(ctx);
        owner_scatter_kernel<<<grid, 256, 0, st>>>(d_digests, n, id_base, world, misc + world,
                                                   (unsigned long long*)(misc + 2 * world), d_records, d_perm);
        HMSE_LAUNCH_CHECK(ctx);
    }
    if (d_counts) HMSE_CUDA(ctx, cudaMemcpyAsync(d_counts, misc, (size_t)world * 8, cudaMemcpyDeviceToDevice, st));
    return HMSE_OK;
}

HMSE_API int hmse_dedup_partition(hmse_ctx* ctx, const uint8_t* d_digests, uint64_t n, uint64_t id_base,
                                    uint32_t world, uint8_t* d_records, uint32_t* d_perm, uint64_t* counts,
                                    void* stream) {
    if (!ctx) return HMSE_E_INVAL;
    cudaStream_t st = (cudaStream_t)stream;
    if (world == 0 || world > 512 || !counts) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_dedup_partition: bad world/counts");
    for (uint32_t w = 0; w < world; w++) counts[w] = 0;
    if (n == 0) return HMSE_OK;
    if (int rc = hmse_dedup_partition_dev(ctx, d_digests, n, id_base, world, d_records, d_perm, nullptr, st)) return rc;
    if (int mrc = hmse_mail(ctx, 0, ctx->slot[SLOT_DEDUP_MISC], world * 2, st)) return mrc;
    HMSE_CUDA(ctx, cudaStreamSynchronize(st));
    for (uint32_t w = 0; w < world; w++) counts[w] = ctx->pinned[w];
    return HMSE_OK;
}

HMSE_API int hmse_dedup_records(hmse_ctx* ctx, const uint8_t* d_records, uint64_t m, uint64_t* d_canon_gid,
                                  void* stream) {
    if (!ctx) return HMSE_E_INVAL;
    cudaStream_t st = (cudaStream_t)stream;
    if (m == 0) return HMSE_OK;
    if (!d_records || !d_canon_gid) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_dedup_records: null pointer");
    if ((uintptr_t)d_records & 7) HMSE_FAIL(ctx, HMSE_E_INVAL, "d_records must be 8-byte aligned");
    if (m >= 0x7FFFFFFFull) HMSE_FAIL(ctx, HMSE_E_INVAL, "dedup: more than 2^31-1 records per table");
    uint64_t cap = 1024;
    while (cap < 2 * m) cap <<= 1;
    // its own slot: a streaming session (hmse_dedup_begin / append) on the same ctx keeps its table
    HMSE_SCRATCH(ctx, table, uint32_t*, SLOT_DEDUP_OWNER, cap * sizeof(uint32_t) + m * sizeof(uint64_t));
    unsigned long long* min_gid = (unsigned long long*)(table + cap);
    HMSE_CUDA(ctx, cudaMemsetAsync(table, 0xFF, cap * sizeof(uint32_t) + m * sizeof(uint64_t), st));
    const unsigned grid = (unsigned)div_up64(m, 256);
    HT_BEGIN(ctx, HT_DEDUP, st);
    KL(ctx);
    dedup_insert_kernel<<<grid, 256, 0, st>>>(d_records, 40, 0, m, nullptr, table, cap - 1);
    KL(ctx);
    min_gid_kernel<<<grid, 256, 0, st>>>(d_records, m, table, cap - 1, min_gid);
    KL(ctx);
    read_gid_kernel<<<grid, 256, 0, st>>>(d_records, m, table, cap - 1, min_gid, d_canon_gid);
    HMSE_LAUNCH_CHECK(ctx);
    HT_END(ctx, HT_DEDUP, st);
    return HMSE_OK;
}

HMSE_API int hmse_dedup_scatter(hmse_ctx* ctx, const uint64_t* d_reply, const uint32_t* d_perm, uint64_t n,
                                  uint64_t id_base, int64_t* d_canon, uint8_t* d_is_first, void* stream) {
    if (!ctx) return HMSE_E_INVAL;
    if (n == 0) return HMSE_OK;
    if (!d_reply || !d_perm || !d_canon) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_dedup_scatter: null pointer");
    KL(ctx);
    scatter_reply_kernel<<<(unsigned)div_up64(n, 256), 256, 0, (cudaStream_t)stream>>>(d_reply, d_perm, n, id_base,
                                                                                      d_canon, d_is_first);
    HMSE_LAUNCH_CHECK(ctx);
    return HMSE_OK;
}
