// known.cu - hmse_compress against an opened archive (K14): the selected chunks whose digest and raw length the archive
// already holds take its stream byte for byte, and only the others are compressed.  A stream depends only on its chunk,
// the dictionary and the level, so the output is hmse_compress's whenever the archive's streams came from this encoder
// at the same level and dictionary.  The archive comes as the layout hmse_read_open wrote (layout.cuh): the library
// keeps no per-archive state, and the digest table is rebuilt on every call.  The rule is stated in include/hmse.h
// (hmse_compress_known) and DESIGN.md section 4, K14.
//
// Scratch (SLOT_KNOWN, u64 words; M source slots, S selected chunks):
//   hdr[8]    [0] error flags, [1..4] stats4, [5] novel streams (scan total)
//   addr      [S]            device address of every output stream: in the source store or in the compression stage
//   keys      [(M + S) * 4]  the source's index digests, then the selected chunks' digests (32-byte keys)
//   canon     [M + S]        first key with the same digest
//   kslot     [S]            source slot copied for stream k, or -1
//   nov       [S + 1]        novel flags, scanned into novel positions
//   nsel      [S]            the novel chunks (the select list handed to hmse_compress)
//   noff      [S + 1]        stream offsets of the compressed novel chunks
// The plan (addr, and the staged novel streams) stays until the next hmse_compress: hmse_compress_known_pack gathers it.
#include "layout.cuh"

namespace {

using namespace layout;

enum KnownErr : unsigned long long {
    KE_LAYOUT = 1,   // a layout that was not opened for the given dims
    KE_DICT = 2      // a dictionary that differs from the archive's in length or Adler-32
};

struct Plan {
    Layout L;
    const uint8_t *index, *store;
    uint64_t n, m, n_delta;
    unsigned long long* hdr;
    uint8_t* keys;
    int64_t *canon, *kslot;
    uint64_t *nov, *nsel, *noff, *addr;
};

__device__ __forceinline__ uint64_t chunk_len(const uint64_t* __restrict__ cuts, uint64_t start0, uint64_t i) {
    return cuts[i] - (i ? cuts[i - 1] : start0);
}

// step 1: the layout against its dims, the dictionary (length and Adler-32) against the layout's header words 6 and 7
__global__ void __launch_bounds__(256) known_check_kernel(Plan P, const uint8_t* __restrict__ dict, uint32_t dict_len) {
    __shared__ uint64_t s_a[256], s_b[256];
    uint64_t a = 0, b = 0;
    for (uint32_t i = threadIdx.x; i < dict_len; i += 256) {
        a += dict[i];
        b += (uint64_t)(dict_len - i) * dict[i];
    }
    s_a[threadIdx.x] = a;
    s_b[threadIdx.x] = b;
    __syncthreads();
    if (threadIdx.x) return;
    for (int i = 1; i < 256; i++) {
        a += s_a[i];
        b += s_b[i];
    }
    const uint64_t adler = ((((uint64_t)dict_len + b) % 65521u) << 16) | ((1 + a) % 65521u);
    const uint64_t* h = P.L.hdr;
    if (h[10] != LAYOUT_MAGIC || h[0] != P.n || h[1] != P.m || h[9] != P.n_delta) atomicOr(P.hdr, KE_LAYOUT);
    else if (h[6] != dict_len || (dict_len && h[7] != adler)) atomicOr(P.hdr, KE_DICT);
}

// step 1: the keys - M index digests (40-byte entries), then the S selected chunks' digests
__global__ void known_keys_kernel(Plan P, const uint8_t* __restrict__ digests, const uint64_t* __restrict__ select, uint64_t S) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= P.m + S) return;
    const uint32_t* src = t < P.m ? reinterpret_cast<const uint32_t*>(P.index + t * 40)
                                  : reinterpret_cast<const uint32_t*>(digests + 32 * (select ? select[t - P.m] : t - P.m));
    uint32_t* d = reinterpret_cast<uint32_t*>(P.keys + t * 32);
#pragma unroll
    for (int q = 0; q < 8; q++) d[q] = src[q];
}

// step 3: stream k is known when the smallest source slot with its digest holds a chunk of its raw length
__global__ void known_decide_kernel(Plan P, const uint64_t* __restrict__ cuts, uint64_t start0, const uint64_t* __restrict__ select,
                                    uint64_t S) {
    if (P.hdr[0]) return;
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint64_t copied = 0, cbytes = 0, novel = 0, nbytes = 0;
    if (k < S) {
        const uint64_t len = chunk_len(cuts, start0, select ? select[k] : k);
        const uint64_t c = (uint64_t)P.canon[P.m + k];
        const bool known = c < P.m && P.L.ulen[c] == len;
        P.kslot[k] = known ? (int64_t)c : -1;
        P.nov[k] = !known;
        if (known) {
            copied = 1;
            cbytes = P.L.upos[c + 1] - P.L.upos[c];
        } else {
            novel = 1;
            nbytes = len;
        }
    }
    // one atomic per warp and counter
    for (int o = 16; o; o >>= 1) {
        copied += __shfl_down_sync(0xFFFFFFFFu, copied, o);
        cbytes += __shfl_down_sync(0xFFFFFFFFu, cbytes, o);
        novel += __shfl_down_sync(0xFFFFFFFFu, novel, o);
        nbytes += __shfl_down_sync(0xFFFFFFFFu, nbytes, o);
    }
    if ((threadIdx.x & 31) == 0 && (copied | novel)) {
        atomicAdd(P.hdr + 1, (unsigned long long)copied);
        atomicAdd(P.hdr + 2, (unsigned long long)cbytes);
        atomicAdd(P.hdr + 3, (unsigned long long)novel);
        atomicAdd(P.hdr + 4, (unsigned long long)nbytes);
    }
}

// step 3: the novel select list, in selection order
__global__ void known_novel_kernel(Plan P, const uint64_t* __restrict__ select, uint64_t S) {
    if (P.hdr[0]) return;
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < S && P.kslot[k] < 0) P.nsel[P.nov[k]] = select ? select[k] : k;
}

// step 5: every stream's length (into d_offsets, scanned next) and address; d_known
__global__ void known_merge_kernel(Plan P, uint64_t S, const uint8_t* __restrict__ stage, const uint64_t* __restrict__ slot_off,
                                   uint64_t* __restrict__ offsets, int64_t* __restrict__ known) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= S) return;
    const int64_t c = P.kslot[k];
    if (c >= 0) {
        offsets[k] = P.L.upos[c + 1] - P.L.upos[c];
        P.addr[k] = (uint64_t)(uintptr_t)(P.store + P.L.upos[c]);
    } else {
        const uint64_t j = P.nov[k];
        offsets[k] = P.noff[j + 1] - P.noff[j];
        P.addr[k] = (uint64_t)(uintptr_t)(stage + slot_off[j]);
    }
    if (known) known[k] = c;
}

unsigned grid_of(uint64_t n) {
    const uint64_t g = div_up64(n, 256);
    return (unsigned)(g == 0 ? 1 : g);
}

}  // namespace

// step 6: every stream gathered into d_out, from the source store or from the stage
static int known_gather(hmse_ctx* ctx, const uint64_t* d_offsets, uint64_t m, uint8_t* d_out, uint64_t out_cap, cudaStream_t st) {
    if (!ctx->known_valid || m != ctx->known_m)
        HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compress_known_pack: no planned result of %llu streams (call hmse_compress_known first)",
                  (unsigned long long)m);
    if (m == 0) return HMSE_OK;
    if (!d_offsets || !d_out) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compress_known_pack: null pointer");
    if (ctx->known_total > out_cap)
        HMSE_FAIL(ctx, HMSE_E_CAPACITY, "d_out capacity %llu < %llu bytes", (unsigned long long)out_cap,
                  (unsigned long long)ctx->known_total);
    HT_BEGIN(ctx, HT_PACK, st);
    if (int e = hmse_segment_gather(ctx, (const uint64_t*)ctx->slot[SLOT_KNOWN] + 8, d_out, d_offsets, m, st)) return e;
    HT_END(ctx, HT_PACK, st);
    return HMSE_OK;
}

HMSE_API int hmse_compress_known_pack(hmse_ctx* ctx, const uint64_t* d_offsets, uint64_t m, uint8_t* d_out, uint64_t out_cap,
                                      void* stream) {
    if (!ctx) return HMSE_E_INVAL;
    return known_gather(ctx, d_offsets, m, d_out, out_cap, (cudaStream_t)stream);
}

HMSE_API int hmse_compress_known(hmse_ctx* ctx, const hmse_compose_src* src, const uint8_t* d_data, uint64_t start0,
                                 const uint64_t* d_cuts, const uint8_t* d_digests, const uint64_t* d_select, uint64_t m,
                                 const uint8_t* d_zdict, uint32_t dict_len, int level, uint8_t* d_out, uint64_t out_cap,
                                 uint64_t* d_offsets, uint64_t* total, int64_t* d_known, uint64_t* stats4, void* stream) {
    if (!ctx) return HMSE_E_INVAL;
    cudaStream_t st = (cudaStream_t)stream;
    if (!total || !d_offsets || !src) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compress_known: src / total / d_offsets is null");
    *total = 0;
    if (stats4)
        for (int q = 0; q < 4; q++) stats4[q] = 0;
    ctx->known_valid = 0;
    if (dict_len > 32768) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compress_known: dict_len must be <= 32768");
    if (dict_len && !d_zdict) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compress_known: d_zdict is null");
    if (m >= 0xFFFFFFFFull) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compress_known: too many chunks in one call");
    if (m && (!d_data || !d_cuts || !d_digests)) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compress_known: null pointer");
    if (((uintptr_t)d_data & 3) || ((uintptr_t)d_digests & 3) || ((uintptr_t)d_cuts & 7) || ((uintptr_t)d_select & 7) ||
        ((uintptr_t)d_offsets & 7) || ((uintptr_t)d_known & 7))
        HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compress_known: d_data / d_digests must be 4-byte, d_cuts / d_select / d_offsets / "
                                     "d_known 8-byte aligned");
    if (!src->d_layout || (src->m && (!src->d_index || !src->d_store)) || ((uintptr_t)src->d_layout & 7) ||
        ((uintptr_t)src->d_index & 3))
        HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compress_known: source: null or misaligned buffer");
    const uint64_t M = src->m, S = m;
    const uint64_t words = 8 + S + 4 * (M + S) + (M + S) + S + (S + 1) + S + (S + 1);
    HMSE_SCRATCH(ctx, w, uint64_t*, SLOT_KNOWN, 8 * words);
    Plan P;
    P.L = layout_of(const_cast<void*>(src->d_layout), src->n, M, src->n_delta);
    P.index = src->d_index;
    P.store = src->d_store;
    P.n = src->n;
    P.m = M;
    P.n_delta = src->n_delta;
    P.hdr = reinterpret_cast<unsigned long long*>(w);
    P.addr = w + 8;
    P.keys = reinterpret_cast<uint8_t*>(P.addr + S);
    P.canon = reinterpret_cast<int64_t*>(P.keys) + 4 * (M + S);
    P.kslot = P.canon + (M + S);
    P.nov = reinterpret_cast<uint64_t*>(P.kslot + S);
    P.nsel = P.nov + S + 1;
    P.noff = P.nsel + S;
    HMSE_CUDA(ctx, cudaMemsetAsync(w, 0, 64, st));
    // ---- steps 1-3: checks, keys, the digest table, known / novel, one mailbox read ----
    HT_BEGIN(ctx, HT_KNOWN, st);
    KL(ctx);
    known_check_kernel<<<1, 256, 0, st>>>(P, d_zdict, dict_len);
    KL(ctx);
    known_keys_kernel<<<grid_of(M + S), 256, 0, st>>>(P, d_digests, d_select, S);
    HMSE_LAUNCH_CHECK(ctx);
    if (int e = hmse_dedup_table(ctx, P.keys, 32, M + S, nullptr, P.canon, nullptr, nullptr, SLOT_KNOWN_TABLE, st)) return e;
    KL(ctx);
    known_decide_kernel<<<grid_of(S), 256, 0, st>>>(P, d_cuts, start0, d_select, S);
    HMSE_LAUNCH_CHECK(ctx);
    if (int e = hmse_exclusive_scan_u64(ctx, P.nov, P.nov, S, reinterpret_cast<uint64_t*>(P.hdr) + 5, st)) return e;
    KL(ctx);
    known_novel_kernel<<<grid_of(S), 256, 0, st>>>(P, d_select, S);
    HMSE_LAUNCH_CHECK(ctx);
    HT_END(ctx, HT_KNOWN, st);
    if (int e = hmse_mail(ctx, 0, P.hdr, 12, st)) return e;
    HMSE_CUDA(ctx, cudaStreamSynchronize(st));
    uint64_t h[6];
    for (int q = 0; q < 6; q++) h[q] = ctx->pinned[q];
    if (h[0] & KE_LAYOUT) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compress_known: the layout was not opened (hmse_read_open) for the source's n, m, n_delta");
    if (h[0] & KE_DICT) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compress_known: the dictionary differs from the source's");
    if (stats4)
        for (int q = 0; q < 4; q++) stats4[q] = h[1 + q];
    const uint64_t n_nov = h[5];
    // ---- step 4: the novel chunks, compressed and staged (hmse_compress: HMSE_T_DEFLATE) ----
    uint64_t nov_total = 0;
    if (int e = hmse_compress(ctx, d_data, start0, d_cuts, P.nsel, n_nov, d_zdict, dict_len, level, nullptr, 0, P.noff, &nov_total, stream))
        return e;
    if (n_nov == 0) {   // hmse_compress of no chunk returns before it counts: hmse_compress_stats must show nothing parsed
        memset(ctx->stat, 0, sizeof(ctx->stat));
        ctx->pev_n = 0;
    }
    const uint8_t* stage = nullptr;
    const uint64_t* slot_off = nullptr;
    if (int e = hmse_compress_staged(ctx, n_nov, &stage, &slot_off)) return e;
    // ---- step 5: lengths scanned into d_offsets, addresses ----
    HT_BEGIN(ctx, HT_KNOWN_MERGE, st);
    KL(ctx);
    known_merge_kernel<<<grid_of(S), 256, 0, st>>>(P, S, stage, slot_off, d_offsets, d_known);
    HMSE_LAUNCH_CHECK(ctx);
    if (int e = hmse_exclusive_scan_u64(ctx, d_offsets, d_offsets, S, d_offsets + S, st)) return e;
    HT_END(ctx, HT_KNOWN_MERGE, st);
    // the total needs no round trip: the copied bytes came with the mailbox, the compressed ones from hmse_compress
    ctx->known_m = S;
    ctx->known_total = h[2] + nov_total;
    ctx->known_valid = 1;
    *total = ctx->known_total;
    if (!d_out && out_cap == 0) return HMSE_OK;   // sizes only
    if (!d_out || *total > out_cap)
        HMSE_FAIL(ctx, HMSE_E_CAPACITY, "d_out capacity %llu < %llu bytes", (unsigned long long)out_cap, (unsigned long long)*total);
    if (int e = known_gather(ctx, d_offsets, S, d_out, out_cap, st)) return e;
    HMSE_CUDA(ctx, cudaStreamSynchronize(st));
    return HMSE_OK;
}
