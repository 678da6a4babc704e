// layout.cuh - the device layout of an opened archive (hmse_read_open writes it; hmse_read and hmse_compose read it).
//
// Layout (u64 words; n chunks, m stored chunks, rc = n_delta ? n : 0 record slots - at most one record per chunk):
//   hdr[16]          n, m, rc, store_bytes, delta_store_bytes, raw_bytes, dict_len, dict_adler, records, n_delta, magic
//   chunk_off[n+1]   raw offset of every chunk (exclusive scan of the pointer records' raw lengths), chunk_off[n] = raw
//   chunk_ref[n]     stored slot of the chunk, or REF_DELTA | its record number
//   upos[m+1]        store position of every stored chunk (running sum of the index lengths), upos[m] = store_bytes
//   ulen[m]          raw length of every stored chunk
//   rpos, rbase, rblen, rdlen, rtraw [rc]   per record: delta-store position, base slot, base raw length, delta length,
//                                           target raw length (records are numbered in delta-store order)
#pragma once
#include "ctx.cuh"

namespace layout {

constexpr uint64_t REF_DELTA = 1ull << 63;
constexpr uint64_t LAYOUT_MAGIC = 0x314C445245534D48ull;   // "HMSERDL1"
constexpr int HDR_WORDS = 16;

struct Layout {
    uint64_t *hdr, *chunk_off, *chunk_ref, *upos, *ulen, *rpos, *rbase, *rblen, *rdlen, *rtraw;
};

inline uint64_t layout_words(uint64_t n, uint64_t m, uint64_t n_delta) {
    const uint64_t rc = n_delta ? n : 0;
    return HDR_WORDS + (n + 1) + n + (m + 1) + m + 5 * rc;
}

__host__ __device__ inline Layout layout_of(void* base, uint64_t n, uint64_t m, uint64_t n_delta) {
    const uint64_t rc = n_delta ? n : 0;
    Layout L;
    L.hdr = (uint64_t*)base;
    L.chunk_off = L.hdr + HDR_WORDS;
    L.chunk_ref = L.chunk_off + n + 1;
    L.upos = L.chunk_ref + n;
    L.ulen = L.upos + m + 1;
    L.rpos = L.ulen + m;
    L.rbase = L.rpos + rc;
    L.rblen = L.rbase + rc;
    L.rdlen = L.rblen + rc;
    L.rtraw = L.rdlen + rc;
    return L;
}

// first k in [0, len) with a[k] > x (len if none)
__device__ __forceinline__ uint64_t upper_bound(const uint64_t* a, uint64_t len, uint64_t x) {
    uint64_t lo = 0, hi = len;
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if (a[mid] <= x) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

}  // namespace layout
