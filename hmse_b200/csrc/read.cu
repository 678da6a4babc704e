// read.cu - random-access reads of an archive (K12): byte ranges of the raw stream, many per call, planned on the device.
// The spec's read path goes from one pointer record to one chunk (README.md:1617-1675); a storage read path serves byte
// ranges, usually many at once.  hmse_read_open checks an archive's records once and derives a device layout (owned by
// the caller, so one ctx serves any number of open archives); hmse_read then turns a batch of ranges into the pieces
// {chunk, offset in chunk, length, destination} they cover, inflates every stored chunk and applies every DeltaChunk
// record the batch needs exactly once (K9 inflate_kernel in place in the chunk store, K11 delta_apply_kernel), and
// copies the pieces out with K8 segment_copy_kernel.  Container layout: hmse_b200/archive.py; device layout: layout.cuh.
#include "layout.cuh"

namespace {

using namespace layout;

enum OpenErr : unsigned long long {
    OE_TILE = 1,      // (1) the index entries do not tile the store
    OE_POINTER = 2,   // (2) a pointer below store_bytes does not address the start of a stored chunk
    OE_DELTA = 4,     // (3) a delta pointer without a delta store, a record outside it, or a base slot >= m
    OE_LENGTH = 8,    // (4) references to one stored chunk or one record disagree on its raw length
    OE_UNKNOWN = 16,  // (5) a stored chunk without a known raw length
    OE_SUM = 32       // (6) the raw lengths do not add up to raw_bytes
};

// first k in [0, len) with a[k] >= x (len if none)
__device__ __forceinline__ uint64_t lower_bound(const uint64_t* a, uint64_t len, uint64_t x) {
    uint64_t lo = 0, hi = len;
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if (a[mid] < x) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// The first reference to a length sets it; a later one must agree.
__device__ __forceinline__ bool claim_len(uint64_t* p, uint64_t v) {
    const unsigned long long old = atomicCAS(reinterpret_cast<unsigned long long*>(p), 0ull, (unsigned long long)v);
    return old == 0ull || old == v;
}

__device__ __forceinline__ void set_err(unsigned long long* err, unsigned long long bit) { atomicOr(err, bit); }

// ---- hmse_read_open ---------------------------------------------------------------------------------------------------

__global__ void open_index_kernel(const uint8_t* __restrict__ index, uint64_t m, uint64_t* __restrict__ upos) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < m) upos[k] = reinterpret_cast<const uint32_t*>(index + k * 40)[9] & 0xFFFFu;   // compressed length
}

// check (1): every entry's lba is its running position >> 9
__global__ void open_tile_kernel(const uint8_t* __restrict__ index, uint64_t m, const uint64_t* __restrict__ upos,
                                 unsigned long long* __restrict__ err) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < m && (upos[k] >> 9) != reinterpret_cast<const uint32_t*>(index + k * 40)[8]) set_err(err, OE_TILE);
}

// checks (2), (3) store side, (4) direct references: stored slot of every chunk, record flags over delta-store positions
__global__ void open_pointer_kernel(const uint2* __restrict__ ptrs, uint64_t n, Layout L, uint64_t m, uint64_t store_bytes,
                                    uint64_t dsb, uint64_t n_delta, uint64_t* __restrict__ flag,
                                    unsigned long long* __restrict__ err) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint2 p = ptrs[i];
    const uint64_t pos = (uint64_t)p.x * 512 + (p.y & 0xFFFFu), raw = (uint64_t)(p.y >> 16) + 1;
    L.chunk_off[i] = raw;
    uint64_t ref = 0;
    if (pos < store_bytes) {
        const uint64_t s = lower_bound(L.upos, m, pos);
        if (s >= m || L.upos[s] != pos) set_err(err, OE_POINTER);
        else {
            ref = s;
            if (!claim_len(&L.ulen[s], raw)) set_err(err, OE_LENGTH);
        }
    } else {
        const uint64_t dp = pos - store_bytes;
        if (!n_delta || dp + 8 > dsb) set_err(err, OE_DELTA);
        else {
            flag[dp] = 1;
            ref = REF_DELTA | dp;   // position for now; open_record_kernel turns it into the record number
        }
    }
    L.chunk_ref[i] = ref;
}

// checks (3) record side and (4) through records: record numbers = rank of the position among referenced positions
__global__ void open_record_kernel(const uint2* __restrict__ ptrs, uint64_t n, Layout L, uint64_t m, uint64_t dsb,
                                   const uint8_t* __restrict__ ds, const uint64_t* __restrict__ rank,
                                   unsigned long long* __restrict__ err) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t ref = L.chunk_ref[i];
    if (!(ref & REF_DELTA)) return;
    const uint64_t dp = ref & ~REF_DELTA, r = rank[dp];
    L.chunk_ref[i] = REF_DELTA | r;
    const uint8_t* h = ds + dp;   // { u32 base slot, u16 base raw length - 1, u16 delta length }, any alignment
    const uint64_t bslot = (uint64_t)h[0] | ((uint64_t)h[1] << 8) | ((uint64_t)h[2] << 16) | ((uint64_t)h[3] << 24);
    const uint64_t blen = ((uint64_t)h[4] | ((uint64_t)h[5] << 8)) + 1, dlen = (uint64_t)h[6] | ((uint64_t)h[7] << 8);
    L.rpos[r] = dp;
    L.rbase[r] = bslot;
    L.rblen[r] = blen;
    L.rdlen[r] = dlen;
    const uint2 p = ptrs[i];
    if (!claim_len(&L.rtraw[r], (uint64_t)(p.y >> 16) + 1)) set_err(err, OE_LENGTH);
    if (bslot >= m || dp + 8 + dlen > dsb) set_err(err, OE_DELTA);
    else if (!claim_len(&L.ulen[bslot], blen)) set_err(err, OE_LENGTH);
}

// checks (5), (6), the rest of (1); the header
__global__ void open_final_kernel(Layout L, uint64_t n, uint64_t m, uint64_t n_delta, uint64_t store_bytes, uint64_t dsb,
                                  uint64_t raw_bytes, uint32_t dict_len, uint32_t dict_adler, const uint64_t* __restrict__ rank,
                                  unsigned long long* __restrict__ err) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < m && L.ulen[k] == 0) set_err(err, OE_UNKNOWN);
    if (k == 0) {
        if (L.upos[m] != store_bytes) set_err(err, OE_TILE);
        if (L.chunk_off[n] != raw_bytes) set_err(err, OE_SUM);
        uint64_t* h = L.hdr;
        h[0] = n;
        h[1] = m;
        h[2] = n_delta ? n : 0;
        h[3] = store_bytes;
        h[4] = dsb;
        h[5] = raw_bytes;
        h[6] = dict_len;
        h[7] = dict_adler;
        h[8] = n_delta ? rank[dsb] : 0;
        h[9] = n_delta;
        h[10] = LAYOUT_MAGIC;
    }
}

// ---- hmse_read --------------------------------------------------------------------------------------------------------

struct Plan {
    uint64_t* olen;    // [R+1] range lengths -> output offsets
    uint64_t* c0;      // [R]   first chunk of every range
    uint64_t* poff;    // [R+1] piece counts -> first piece of every range
    uint64_t* mku;     // [m+1] stored slot needed -> its rank among the needed slots
    uint64_t* ofu;     // [m+1] raw length if needed -> its offset in the inflated buffer
    uint64_t* mkr;     // [rc+1] record needed -> rank
    uint64_t* otr;     // [rc+1] target length if needed -> offset behind the inflated stored chunks
    uint64_t* odr;     // [rc+1] delta length if needed -> offset in the gathered delta bytes
    unsigned long long* flags;   // [0] a range past raw_bytes, [1] the layout does not match the dims given
};

// step 1: range checks; a layout that was not opened for these dims stops the batch before anything is read from it
__global__ void read_range_kernel(const uint64_t* __restrict__ ranges, uint64_t R, const uint64_t* __restrict__ hdr, uint64_t n,
                                  uint64_t m, uint64_t n_delta, Plan P) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r == 0 && (hdr[10] != LAYOUT_MAGIC || hdr[0] != n || hdr[1] != m || hdr[9] != n_delta)) set_err(P.flags + 1, 1);
    if (r >= R) return;
    const uint64_t raw = hdr[5], off = ranges[2 * r], len = ranges[2 * r + 1];
    const bool bad = len > raw || off > raw - len;   // also catches offset + length wrapping around 2^64
    if (bad) set_err(P.flags, 1);
    P.olen[r] = bad ? 0 : len;
}

// step 2: first and last chunk of every range (upper bound over chunk_off: the chunk that contains the byte)
__global__ void read_locate_kernel(const uint64_t* __restrict__ ranges, uint64_t R, Layout L, uint64_t n, Plan P) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R || P.flags[1]) return;
    const uint64_t off = ranges[2 * r], len = P.olen[r + 1] - P.olen[r];   // olen holds the scanned offsets by now
    uint64_t first = 0, cnt = 0;
    if (len) {
        first = upper_bound(L.chunk_off, n + 1, off) - 1;
        const uint64_t last = upper_bound(L.chunk_off, n + 1, off + len - 1) - 1;
        cnt = last - first + 1;
    }
    P.c0[r] = first;
    P.poff[r] = cnt;
}

// piece p -> (range, chunk)
__device__ __forceinline__ void piece_of(const Plan& P, uint64_t R, uint64_t p, uint64_t& r, uint64_t& c) {
    r = upper_bound(P.poff, R + 1, p) - 1;
    c = P.c0[r] + (p - P.poff[r]);
}

// step 3: mark what every piece needs: its stored slot, or its record and the record's base slot
__global__ void read_mark_kernel(uint64_t R, Layout L, uint64_t m, uint64_t rc, Plan P) {
    if (P.flags[1]) return;
    const uint64_t np = P.poff[R];
    for (uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; p < np; p += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t r, c;
        piece_of(P, R, p, r, c);
        const uint64_t ref = L.chunk_ref[c];
        if (ref & REF_DELTA) {
            const uint64_t rec = ref & ~REF_DELTA;
            P.mkr[rec] = 1;
            P.mku[L.rbase[rec]] = 1;
        } else {
            P.mku[ref] = 1;
        }
    }
}

// step 4: the lengths of what is needed, scanned next into offsets
__global__ void read_values_kernel(Layout L, uint64_t m, uint64_t rc, Plan P) {
    if (P.flags[1]) return;
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < m) P.ofu[k] = P.mku[k] ? L.ulen[k] : 0;
    if (k < rc) {
        P.otr[k] = P.mkr[k] ? L.rtraw[k] : 0;
        P.odr[k] = P.mkr[k] ? L.rdlen[k] : 0;
    }
}

__global__ void read_sizes_kernel(const Plan P, uint64_t R, uint64_t m, uint64_t rc, const uint64_t* __restrict__ hdr,
                                  uint64_t* __restrict__ mail) {
    if (threadIdx.x != 0) return;
    const bool ok = !P.flags[1];
    mail[0] = P.flags[0];
    mail[1] = P.flags[1];
    mail[2] = P.olen[R];
    mail[3] = ok ? P.poff[R] : 0;
    mail[4] = ok ? P.mku[m] : 0;
    mail[5] = ok ? P.ofu[m] : 0;
    mail[6] = ok ? P.mkr[rc] : 0;
    mail[7] = ok ? P.otr[rc] : 0;
    mail[8] = ok ? P.odr[rc] : 0;
    mail[9] = hdr[7];
}

struct Work {
    uint64_t *ib, *ie, *uo;               // needed stored chunks: stream range in the store, output offsets [Ku+1]
    uint64_t *dsrc, *ddst, *bo, *to;      // needed records: delta bytes in the delta store / gathered [Kr+1], base offset,
                                          // target offsets [Kr+1] (behind the stored chunks)
    uint64_t *psrc, *pdst;                // pieces: source in the inflated buffer, destination in d_out [np+1]
    uint32_t *ust, *rst, *bl;             // inflate statuses, delta statuses, base lengths
    unsigned long long* bad;
};

// compaction of the marks into need lists (step 4, after the sizes are known)
__global__ void read_compact_kernel(Layout L, uint64_t m, uint64_t rc, Plan P, Work W, uint64_t Ku, uint64_t U, uint64_t Kr,
                                    uint64_t T, uint64_t Dl) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < m && P.mku[k + 1] != P.mku[k]) {
        const uint64_t j = P.mku[k];
        W.ib[j] = L.upos[k];
        W.ie[j] = L.upos[k + 1];
        W.uo[j] = P.ofu[k];
    }
    if (k < rc && P.mkr[k + 1] != P.mkr[k]) {
        const uint64_t j = P.mkr[k];
        W.dsrc[j] = L.rpos[k] + 8;
        W.ddst[j] = P.odr[k];
        W.bo[j] = P.ofu[L.rbase[k]];
        W.bl[j] = (uint32_t)L.rblen[k];
        W.to[j] = U + P.otr[k];
    }
    if (k == 0) {
        W.uo[Ku] = U;
        W.ddst[Kr] = Dl;
        W.to[Kr] = U + T;
    }
}

// steps 8-9: source and destination of every piece, and the statuses of what it needed folded into its range
__global__ void read_piece_kernel(const uint64_t* __restrict__ ranges, uint64_t R, Layout L, Plan P, Work W, uint64_t np,
                                  uint64_t total, uint32_t* __restrict__ status) {
    for (uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; p < np; p += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t r, c;
        piece_of(P, R, p, r, c);
        const uint64_t off = ranges[2 * r], cs = L.chunk_off[c];
        const uint64_t a = cs > off ? cs : off;
        const uint64_t ref = L.chunk_ref[c];
        uint64_t src;
        uint32_t code;
        if (ref & REF_DELTA) {
            const uint64_t rec = ref & ~REF_DELTA, j = P.mkr[rec];
            src = W.to[j];
            const uint32_t ds = W.rst[j], bs = W.ust[P.mku[L.rbase[rec]]];
            code = ds ? 16 + ds : bs;
        } else {
            const uint64_t j = P.mku[ref];
            src = W.uo[j];
            code = W.ust[j];
        }
        W.psrc[p] = src + (a - cs);
        W.pdst[p] = P.olen[r] + (a - off);
        if (code) atomicMax(status + r, code);
        if (p == 0) W.pdst[np] = total;
    }
}

__global__ void read_count_kernel(const uint32_t* __restrict__ status, uint64_t R, unsigned long long* __restrict__ bad) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool b = i < R && status[i] != 0;
    const uint32_t c = __popc(__ballot_sync(0xffffffffu, b));
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(bad, (unsigned long long)c);
}

unsigned grid_of(uint64_t n, uint64_t cap) {
    const uint64_t g = div_up64(n, 256);
    return (unsigned)(g == 0 ? 1 : (g < cap ? g : cap));
}

}  // namespace

HMSE_API uint64_t hmse_read_layout_bytes(uint64_t n, uint64_t m, uint64_t n_delta) { return 8 * layout_words(n, m, n_delta); }

HMSE_API int hmse_read_open(hmse_ctx* ctx, const uint8_t* d_index, uint64_t m, const uint8_t* d_pointers, uint64_t n,
                            uint64_t store_bytes, const uint8_t* d_delta_store, uint64_t delta_store_bytes, uint64_t n_delta,
                            uint64_t raw_bytes, const uint8_t* d_zdict, uint32_t dict_len, void* d_layout, uint64_t layout_bytes,
                            void* stream) {
    if (!ctx) return HMSE_E_INVAL;
    cudaStream_t st = (cudaStream_t)stream;
    if (!d_layout || (m && !d_index) || (n && !d_pointers) || (n_delta && !d_delta_store) || (dict_len && !d_zdict))
        HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_read_open: null pointer");
    if (((uintptr_t)d_layout & 7) || ((uintptr_t)d_pointers & 7) || ((uintptr_t)d_index & 3))
        HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_read_open: d_layout / d_pointers must be 8-byte, d_index 4-byte aligned");
    if (layout_bytes < hmse_read_layout_bytes(n, m, n_delta))
        HMSE_FAIL(ctx, HMSE_E_CAPACITY, "hmse_read_open: layout_bytes %llu < %llu", (unsigned long long)layout_bytes,
                  (unsigned long long)hmse_read_layout_bytes(n, m, n_delta));
    if (dict_len > 32768) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_read_open: dict_len must be <= 32768");
    if (!n_delta) delta_store_bytes = 0;
    uint32_t dict_adler = 0;
    if (dict_len) {   // once per archive: hmse_read finds the DICTID in the layout
        static thread_local uint8_t tmp[32768];
        HMSE_CUDA(ctx, cudaMemcpyAsync(tmp, d_zdict, dict_len, cudaMemcpyDeviceToHost, st));
        HMSE_CUDA(ctx, cudaStreamSynchronize(st));
        dict_adler = hmse_adler32_host(tmp, dict_len);
    }
    const Layout L = layout_of(d_layout, n, m, n_delta);
    const uint64_t rc = n_delta ? n : 0;
    // misc: [err][record flags over delta-store positions, scanned into record numbers: dsb + 1]
    HMSE_SCRATCH(ctx, misc, uint64_t*, SLOT_READ_OPEN, 8 * (delta_store_bytes + 2));
    unsigned long long* err = reinterpret_cast<unsigned long long*>(misc);
    uint64_t* flag = misc + 1;
    HMSE_CUDA(ctx, cudaMemsetAsync(misc, 0, 8 * (delta_store_bytes + 2), st));
    HMSE_CUDA(ctx, cudaMemsetAsync(L.ulen, 0, 8 * m, st));
    if (rc) HMSE_CUDA(ctx, cudaMemsetAsync(L.rtraw, 0, 8 * rc, st));
    KL(ctx);
    open_index_kernel<<<grid_of(m, ~0u), 256, 0, st>>>(d_index, m, L.upos);
    HMSE_LAUNCH_CHECK(ctx);
    if (int rc2 = hmse_exclusive_scan_u64(ctx, L.upos, L.upos, m, L.upos + m, st)) return rc2;
    KL(ctx);
    open_tile_kernel<<<grid_of(m, ~0u), 256, 0, st>>>(d_index, m, L.upos, err);
    KL(ctx);
    open_pointer_kernel<<<grid_of(n, ~0u), 256, 0, st>>>(reinterpret_cast<const uint2*>(d_pointers), n, L, m, store_bytes,
                                                         delta_store_bytes, n_delta, flag, err);
    HMSE_LAUNCH_CHECK(ctx);
    if (n_delta) {
        if (int rc2 = hmse_exclusive_scan_u64(ctx, flag, flag, delta_store_bytes, flag + delta_store_bytes, st)) return rc2;
        KL(ctx);
        open_record_kernel<<<grid_of(n, ~0u), 256, 0, st>>>(reinterpret_cast<const uint2*>(d_pointers), n, L, m, delta_store_bytes,
                                                            d_delta_store, flag, err);
        HMSE_LAUNCH_CHECK(ctx);
    }
    if (int rc2 = hmse_exclusive_scan_u64(ctx, L.chunk_off, L.chunk_off, n, L.chunk_off + n, st)) return rc2;
    KL(ctx);
    open_final_kernel<<<grid_of(m, ~0u), 256, 0, st>>>(L, n, m, n_delta, store_bytes, delta_store_bytes, raw_bytes, dict_len,
                                                       dict_adler, flag, err);
    HMSE_LAUNCH_CHECK(ctx);
    if (int mrc = hmse_mail(ctx, 0, err, 2, st)) return mrc;
    HMSE_CUDA(ctx, cudaStreamSynchronize(st));
    const uint64_t e = ctx->pinned[0];
    if (e & OE_TILE) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_read_open: index entries do not tile the chunk store");
    if (e & OE_POINTER) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_read_open: a pointer record does not address a stored chunk");
    if (e & OE_DELTA)
        HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_read_open: a pointer record addresses a delta store this archive does not have, or a "
                                     "DeltaChunk record is damaged (outside the delta store, or its base slot >= m)");
    if (e & OE_LENGTH) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_read_open: pointer records disagree about a chunk's length");
    if (e & OE_UNKNOWN) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_read_open: a stored chunk has no known raw length");
    if (e & OE_SUM) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_read_open: pointer records do not add up to the stream length");
    return HMSE_OK;
}

HMSE_API int hmse_read(hmse_ctx* ctx, const void* d_layout, uint64_t n, uint64_t m, uint64_t n_delta, const uint8_t* d_store,
                       const uint8_t* d_delta_store, const uint8_t* d_zdict, uint32_t dict_len, const uint64_t* d_ranges,
                       uint64_t R, uint8_t* d_out, uint64_t out_cap, uint64_t* d_out_off, uint64_t* total, uint32_t* d_status,
                       uint64_t* n_bad, uint64_t* stats4, void* stream) {
    if (!ctx) return HMSE_E_INVAL;
    cudaStream_t st = (cudaStream_t)stream;
    if (total) *total = 0;
    if (n_bad) *n_bad = 0;
    if (stats4)
        for (int q = 0; q < 4; q++) stats4[q] = 0;
    if (!d_layout || !total || !d_out_off || (R && (!d_ranges || !d_status)) || (m && !d_store) || (n_delta && !d_delta_store) ||
        (dict_len && !d_zdict) || (out_cap && !d_out))
        HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_read: null pointer");
    if (((uintptr_t)d_layout & 7) || ((uintptr_t)d_ranges & 7)) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_read: d_layout / d_ranges must be 8-byte aligned");
    if (dict_len > 32768) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_read: dict_len must be <= 32768");
    const uint64_t rc = n_delta ? n : 0;
    const Layout L = layout_of(const_cast<void*>(d_layout), n, m, n_delta);
    const uint64_t cap = (uint64_t)ctx->sm_count * 8;
    // ---- steps 1-4 on the device, sized by R and the archive (never by the pieces) ----
    const uint64_t plan_words = (R + 1) + R + (R + 1) + 2 * (m + 1) + 3 * (rc + 1) + 2;
    HMSE_SCRATCH(ctx, pw, uint64_t*, SLOT_READ_PLAN, 8 * plan_words);
    Plan P;
    P.olen = pw;
    P.c0 = P.olen + R + 1;
    P.poff = P.c0 + R;
    P.mku = P.poff + R + 1;
    P.ofu = P.mku + m + 1;
    P.mkr = P.ofu + m + 1;
    P.otr = P.mkr + rc + 1;
    P.odr = P.otr + rc + 1;
    P.flags = reinterpret_cast<unsigned long long*>(P.odr + rc + 1);
    HMSE_CUDA(ctx, cudaMemsetAsync(P.mku, 0, 8 * (m + 1), st));
    HMSE_CUDA(ctx, cudaMemsetAsync(P.mkr, 0, 8 * (rc + 1), st));
    HMSE_CUDA(ctx, cudaMemsetAsync(P.flags, 0, 16, st));
    HT_BEGIN(ctx, HT_READ_PLAN, st);
    KL(ctx);
    read_range_kernel<<<grid_of(R, ~0u), 256, 0, st>>>(d_ranges, R, L.hdr, n, m, n_delta, P);
    HMSE_LAUNCH_CHECK(ctx);
    if (int e = hmse_exclusive_scan_u64(ctx, P.olen, P.olen, R, P.olen + R, st)) return e;
    KL(ctx);
    read_locate_kernel<<<grid_of(R, ~0u), 256, 0, st>>>(d_ranges, R, L, n, P);
    HMSE_LAUNCH_CHECK(ctx);
    if (int e = hmse_exclusive_scan_u64(ctx, P.poff, P.poff, R, P.poff + R, st)) return e;
    KL(ctx);
    read_mark_kernel<<<(unsigned)cap, 256, 0, st>>>(R, L, m, rc, P);
    KL(ctx);
    read_values_kernel<<<grid_of(m > rc ? m : rc, ~0u), 256, 0, st>>>(L, m, rc, P);
    HMSE_LAUNCH_CHECK(ctx);
    if (int e = hmse_exclusive_scan_u64(ctx, P.mku, P.mku, m, P.mku + m, st)) return e;
    if (int e = hmse_exclusive_scan_u64(ctx, P.ofu, P.ofu, m, P.ofu + m, st)) return e;
    if (int e = hmse_exclusive_scan_u64(ctx, P.mkr, P.mkr, rc, P.mkr + rc, st)) return e;
    if (int e = hmse_exclusive_scan_u64(ctx, P.otr, P.otr, rc, P.otr + rc, st)) return e;
    if (int e = hmse_exclusive_scan_u64(ctx, P.odr, P.odr, rc, P.odr + rc, st)) return e;
    HT_END(ctx, HT_READ_PLAN, st);
    // ---- step 5: one mailbox read of the sizes ----
    KL(ctx);
    read_sizes_kernel<<<1, 32, 0, st>>>(P, R, m, rc, L.hdr, ctx->pinned_dev);
    HMSE_LAUNCH_CHECK(ctx);
    HMSE_CUDA(ctx, cudaStreamSynchronize(st));
    const uint64_t* mb = ctx->pinned;
    if (mb[1]) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_read: d_layout was not opened (hmse_read_open) for an archive of these n, m, n_delta");
    if (mb[0]) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_read: a range runs past raw_bytes (or its offset + length overflows)");
    const uint64_t tot = mb[2], np = mb[3], Ku = mb[4], U = mb[5], Kr = mb[6], T = mb[7], Dl = mb[8];
    const uint32_t dict_adler = (uint32_t)mb[9];
    *total = tot;
    if (tot > out_cap)
        HMSE_FAIL(ctx, HMSE_E_CAPACITY, "hmse_read: out_cap %llu < %llu", (unsigned long long)out_cap, (unsigned long long)tot);
    if (Ku >= 0xFFFFFFFFull) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_read: too many stored chunks in one batch");
    if (stats4) {
        stats4[0] = Ku;
        stats4[1] = Kr;
        stats4[2] = U;
        stats4[3] = np;
    }
    HMSE_CUDA(ctx, cudaMemcpyAsync(d_out_off, P.olen, 8 * (R + 1), cudaMemcpyDeviceToDevice, st));
    if (R) HMSE_CUDA(ctx, cudaMemsetAsync(d_status, 0, 4 * R, st));
    // ---- scratch that follows the batch: need lists, pieces, the inflated chunks ----
    const uint64_t work_words = 2 * Ku + (Ku + 1) + Kr + (Kr + 1) + Kr + (Kr + 1) + np + (np + 1) + div_up64(4 * (Ku + 2 * Kr), 8) + 2;
    HMSE_SCRATCH(ctx, ww, uint64_t*, SLOT_READ_WORK, 8 * work_words);
    Work W;
    W.ib = ww;
    W.ie = W.ib + Ku;
    W.uo = W.ie + Ku;
    W.dsrc = W.uo + Ku + 1;
    W.ddst = W.dsrc + Kr;
    W.bo = W.ddst + Kr + 1;
    W.to = W.bo + Kr;
    W.psrc = W.to + Kr + 1;
    W.pdst = W.psrc + np;
    W.bad = reinterpret_cast<unsigned long long*>(W.pdst + np + 1);
    W.ust = reinterpret_cast<uint32_t*>(W.bad + 2);
    W.rst = W.ust + Ku;
    W.bl = W.rst + Kr;
    const uint64_t data_bytes = ((U + T + 15) & ~15ull) + Dl + 64;   // inflated chunks, delta targets, gathered delta bytes
    HMSE_SCRATCH(ctx, data, uint8_t*, SLOT_READ_DATA, data_bytes);
    uint8_t* dbuf = data + ((U + T + 15) & ~15ull);
    HMSE_CUDA(ctx, cudaMemsetAsync(W.bad, 0, 8, st));
    if (Ku || Kr) {
        KL(ctx);
        read_compact_kernel<<<grid_of(m > rc ? m : rc, ~0u), 256, 0, st>>>(L, m, rc, P, W, Ku, U, Kr, T, Dl);
        HMSE_LAUNCH_CHECK(ctx);
    }
    // ---- steps 6-7: the stored chunks inflate in place in the store; the deltas are gathered, then applied ----
    if (int e = hmse_inflate_ranges(ctx, d_store, W.ib, W.ie, Ku, d_zdict, dict_len, dict_adler, data, W.uo, W.ust, st)) return e;
    if (Kr) {
        HT_BEGIN(ctx, HT_DELTA, st);
        if (int e = hmse_segment_copy(ctx, d_delta_store, W.dsrc, dbuf, W.ddst, Kr, stream)) return e;
        if (int e = hmse_delta_apply(ctx, dbuf, W.ddst, Kr, data, U, W.bo, W.bl, data, W.to, W.rst, nullptr, stream)) return e;
        HT_END(ctx, HT_DELTA, st);
    }
    // ---- steps 8-9: the pieces, and the statuses per range ----
    HT_BEGIN(ctx, HT_READ_COPY, st);
    if (np) {
        KL(ctx);
        read_piece_kernel<<<grid_of(np, cap), 256, 0, st>>>(d_ranges, R, L, P, W, np, tot, d_status);
        HMSE_LAUNCH_CHECK(ctx);
        if (int e = hmse_segment_copy(ctx, data, W.psrc, d_out, W.pdst, np, stream)) return e;
    }
    HT_END(ctx, HT_READ_COPY, st);
    KL(ctx);
    read_count_kernel<<<grid_of(R, ~0u), 256, 0, st>>>(d_status, R, W.bad);
    HMSE_LAUNCH_CHECK(ctx);
    if (int e = hmse_mail(ctx, 0, W.bad, 2, st)) return e;
    HMSE_CUDA(ctx, cudaStreamSynchronize(st));
    if (n_bad) *n_bad = ctx->pinned[0];
    return HMSE_OK;
}
