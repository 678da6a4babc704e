// compose.cu - one archive from the files of several opened archives (K13): merge, subset, reorder and repeat on the
// device, with stored chunks deduplicated across sources by the digests their index entries hold.  Compressed streams
// and DeltaChunk records move byte for byte (a stream depends only on its chunk, the dictionary and the level); only
// the records are rewritten.  Sources come as the layouts hmse_read_open wrote (layout.cuh): the library keeps no
// per-archive state.  The rule is stated in include/hmse.h (hmse_compose) and DESIGN.md section 4, K13.
//
// Global spaces: stored slot g = sbase[s] + slot of source s, record g = rbase[s] + record of source s (rc record slots
// per source, layout.cuh).  Keys are output positions, so "first reference" is an atomicMin and key order needs no
// sort: a position holds one reference, so stored keys are unique, and record keys are unique.
#include "layout.cuh"

namespace {

using namespace layout;

constexpr uint64_t NO_KEY = ~0ull;

enum ComposeErr : unsigned long long {
    CE_RUN = 1,      // a run names a source that does not exist or chunks outside its source
    CE_LAYOUT = 2,   // a layout that was not opened for its source's dims
    CE_DICT = 4,     // dictionaries that differ in length or Adler-32
    CE_COUNT = 8     // run counts that do not add up to n_out
};

struct Src {
    Layout L;
    const uint8_t *index, *ptrs, *store, *dstore;
    uint64_t n, m, n_delta;
};

struct Work {
    const Src* src;
    const uint64_t *sbase, *rbase;   // [n_src + 1] first global stored slot / record of every source
    uint32_t n_src;
    unsigned long long* flags;       // [0] ComposeErr, [1] an invariant of the record writers broken
    uint64_t* run_off;               // [n_runs + 1] run counts -> first output position of every run
    uint64_t *ukey, *rkey;           // [SM], [SR] first-reference position of every stored slot / record (NO_KEY: none)
    uint64_t *uflag, *rflag;         // [n_out + 1] a stored key / record key at this position -> candidate number
    uint8_t* dig;                    // [KU][32] digests of the stored candidates, key order
    uint64_t *clen, *usrc;           // [KU] compressed length and source address of every stored candidate
    int64_t* canon;                  // [KU] first candidate with the same digest
    uint8_t* is_first;               // [KU]
    uint64_t *krank, *uoff;          // [KU + 1] kept flags -> new slot numbers; kept lengths -> output store offsets
    unsigned long long* refc;        // [KU] reference count of every new slot
    uint64_t *rcand, *rsrc, *roff;   // [KR] global record of every record candidate, its source address; [KR + 1] offsets
};

// output position p -> (source, chunk of the source)
__device__ __forceinline__ void chunk_of(const Work& W, const uint64_t* __restrict__ runs, uint64_t n_runs, uint64_t p,
                                         uint64_t& s, uint64_t& i) {
    const uint64_t r = upper_bound(W.run_off, n_runs + 1, p) - 1;
    s = runs[3 * r];
    i = runs[3 * r + 1] + (p - W.run_off[r]);
}

// step 1: every source's layout against its dims and source 0's dictionary; every run inside its source
__global__ void compose_check_kernel(Work W, const uint64_t* __restrict__ runs, uint64_t n_runs) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < W.n_src) {
        const Src& S = W.src[t];
        const uint64_t* h = S.L.hdr;
        if (h[10] != LAYOUT_MAGIC || h[0] != S.n || h[1] != S.m || h[9] != S.n_delta) atomicOr(W.flags, CE_LAYOUT);
        else if (h[6] != W.src[0].L.hdr[6] || h[7] != W.src[0].L.hdr[7]) atomicOr(W.flags, CE_DICT);
    }
    if (t < n_runs) {
        const uint64_t s = runs[3 * t], first = runs[3 * t + 1], cnt = runs[3 * t + 2];
        const bool ok = s < W.n_src && cnt <= W.src[s < W.n_src ? s : 0].n && first <= W.src[s < W.n_src ? s : 0].n - cnt;
        if (!ok) atomicOr(W.flags, CE_RUN);
        W.run_off[t] = ok ? cnt : 0;
    }
}

__device__ __forceinline__ bool stopped(const Work& W, uint64_t n_runs, uint64_t n_out) {
    return W.flags[0] || W.run_off[n_runs] != n_out;
}

// step 2: first reference of every stored slot and record (a record's reference to its base counts at its chunk)
__global__ void compose_key_kernel(Work W, const uint64_t* __restrict__ runs, uint64_t n_runs, uint64_t n_out) {
    if (stopped(W, n_runs, n_out)) {
        if (blockIdx.x == 0 && threadIdx.x == 0 && W.run_off[n_runs] != n_out) atomicOr(W.flags, CE_COUNT);
        return;
    }
    for (uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n_out; p += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t s, i;
        chunk_of(W, runs, n_runs, p, s, i);
        const Layout& L = W.src[s].L;
        const uint64_t ref = L.chunk_ref[i];
        unsigned long long* uk = reinterpret_cast<unsigned long long*>(W.ukey + W.sbase[s]);
        if (ref & REF_DELTA) {
            const uint64_t rec = ref & ~REF_DELTA;
            atomicMin(reinterpret_cast<unsigned long long*>(W.rkey + W.rbase[s] + rec), (unsigned long long)p);
            atomicMin(uk + L.rbase[rec], (unsigned long long)p);
        } else {
            atomicMin(uk + ref, (unsigned long long)p);
        }
    }
}

// step 3a: flag every key's position (scanned next into candidate numbers in key order)
__global__ void compose_flag_kernel(Work W, uint64_t SM, uint64_t SR) {
    if (W.flags[0]) return;
    const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g < SM && W.ukey[g] != NO_KEY) W.uflag[W.ukey[g]] = 1;
    if (g < SR && W.rkey[g] != NO_KEY) W.rflag[W.rkey[g]] = 1;
}

// step 3b / 4: the candidate lists - digests, stream lengths and addresses of the stored chunks, the records
__global__ void compose_cand_kernel(Work W, uint64_t SM, uint64_t SR) {
    if (W.flags[0]) return;
    const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g < SM && W.ukey[g] != NO_KEY) {
        const uint64_t k = W.uflag[W.ukey[g]];
        const uint64_t s = upper_bound(W.sbase, W.n_src + 1, g) - 1, slot = g - W.sbase[s];
        const Src& S = W.src[s];
        const uint32_t* e = reinterpret_cast<const uint32_t*>(S.index + slot * 40);
        uint32_t* d = reinterpret_cast<uint32_t*>(W.dig + k * 32);
#pragma unroll
        for (int q = 0; q < 8; q++) d[q] = e[q];
        W.clen[k] = S.L.upos[slot + 1] - S.L.upos[slot];
        W.usrc[k] = (uint64_t)(uintptr_t)(S.store + S.L.upos[slot]);
    }
    if (g < SR && W.rkey[g] != NO_KEY) {
        const uint64_t j = W.rflag[W.rkey[g]];
        const uint64_t s = upper_bound(W.rbase, W.n_src + 1, g) - 1, rec = g - W.rbase[s];
        const Src& S = W.src[s];
        W.rcand[j] = g;
        W.rsrc[j] = (uint64_t)(uintptr_t)(S.dstore + S.L.rpos[rec]);
        W.roff[j] = 8 + S.L.rdlen[rec];
    }
}

// step 5: a candidate is kept when it is the first with its digest
__global__ void compose_keep_kernel(Work W, uint64_t KU) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= KU) return;
    W.krank[k] = W.is_first[k];
    W.uoff[k] = W.is_first[k] ? W.clen[k] : 0;
}

__global__ void compose_sizes_kernel(Work W, uint64_t n_runs, uint64_t n_out, uint64_t KU, uint64_t KR, uint64_t* __restrict__ mail) {
    if (threadIdx.x != 0) return;
    mail[0] = W.flags[0];
    mail[1] = W.uflag[n_out];
    mail[2] = W.krank[KU];
    mail[3] = W.uoff[KU];
    mail[4] = W.rflag[n_out];
    mail[5] = W.roff[KR];
}

// step 7: the pointer records, and one reference per pointer on its new slot
__global__ void compose_pointer_kernel(Work W, const uint64_t* __restrict__ runs, uint64_t n_runs, uint64_t n_out,
                                       uint64_t store_bytes, uint2* __restrict__ out) {
    for (uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n_out; p += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t s, i;
        chunk_of(W, runs, n_runs, p, s, i);
        const Src& S = W.src[s];
        const uint64_t ref = S.L.chunk_ref[i];
        uint64_t pos;
        if (ref & REF_DELTA) {
            pos = store_bytes + W.roff[W.rflag[W.rkey[W.rbase[s] + (ref & ~REF_DELTA)]]];
        } else {
            const uint64_t c = (uint64_t)W.canon[W.uflag[W.ukey[W.sbase[s] + ref]]];
            pos = W.uoff[c];
            atomicAdd(W.refc + W.krank[c], 1ull);
        }
        const uint32_t raw16 = reinterpret_cast<const uint2*>(S.ptrs)[i].y & 0xFFFF0000u;
        out[p] = make_uint2((uint32_t)(pos >> 9), (uint32_t)(pos & 511) | raw16);
    }
}

// step 7: every record's base slot remapped (the rest of the record was copied), one reference on that slot
__global__ void compose_record_kernel(Work W, uint64_t Kr, uint64_t kept, uint8_t* __restrict__ ds) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= Kr) return;
    const uint64_t g = W.rcand[j];
    const uint64_t s = upper_bound(W.rbase, W.n_src + 1, g) - 1, rec = g - W.rbase[s];
    const uint64_t key = W.ukey[W.sbase[s] + W.src[s].L.rbase[rec]];
    const uint64_t ns = key == NO_KEY ? kept : W.krank[W.canon[W.uflag[key]]];
    if (ns >= kept) {   // the base of a referenced record always has a key
        atomicOr(W.flags + 1, 1ull);
        return;
    }
    atomicAdd(W.refc + ns, 1ull);
    uint8_t* h = ds + W.roff[j];
#pragma unroll
    for (int q = 0; q < 4; q++) h[q] = (uint8_t)(ns >> (8 * q));
}

// step 7: the index entries of the kept chunks, with their reference counts
__global__ void compose_index_kernel(Work W, uint64_t Kc, uint8_t* __restrict__ index) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= Kc || !W.is_first[k]) return;
    const uint64_t ns = W.krank[k], pos = W.uoff[k];
    const uint32_t* d = reinterpret_cast<const uint32_t*>(W.dig + k * 32);
    uint32_t* e = reinterpret_cast<uint32_t*>(index + ns * 40);
#pragma unroll
    for (int q = 0; q < 8; q++) e[q] = d[q];
    const unsigned long long rc = W.refc[ns] > 0xFFFFull ? 0xFFFFull : W.refc[ns];
    e[8] = (uint32_t)(pos >> 9);
    e[9] = (uint32_t)(W.clen[k] & 0xFFFF) | ((uint32_t)rc << 16);
}

unsigned grid_of(uint64_t n, uint64_t cap) {
    const uint64_t g = div_up64(n, 256);
    return (unsigned)(g == 0 ? 1 : (g < cap ? g : cap));
}

}  // namespace

HMSE_API int hmse_compose(hmse_ctx* ctx, const hmse_compose_src* srcs, uint32_t n_src, const uint64_t* d_runs, uint64_t n_runs,
                          uint64_t n_out, uint8_t* d_pointers, uint8_t* d_index, uint64_t index_cap, uint8_t* d_store,
                          uint64_t store_cap, uint8_t* d_delta_store, uint64_t delta_cap, uint64_t* out6, void* stream) {
    if (!ctx) return HMSE_E_INVAL;
    cudaStream_t st = (cudaStream_t)stream;
    if (!out6) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compose: out6 is null");
    for (int q = 0; q < 6; q++) out6[q] = 0;
    if (n_out > 0xFFFFFFFEull) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compose: n_out exceeds 2^32 - 2 chunks");
    if (n_out && (!n_src || !srcs || !d_runs || !n_runs || !d_pointers))
        HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compose: null pointer, or no source or run for n_out chunks");
    if (((uintptr_t)d_pointers & 7) || ((uintptr_t)d_index & 3) || ((uintptr_t)d_runs & 7))
        HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compose: d_pointers / d_runs must be 8-byte, d_index 4-byte aligned");
    // the source table, with the first global stored slot and record of every source
    const size_t src_words = div_up64(sizeof(Src) * n_src, 8);
    const size_t table_bytes = 8 * (src_words + 2 * (n_src + 1));
    Src* hs = (Src*)calloc(1, table_bytes);
    if (!hs) HMSE_FAIL(ctx, HMSE_E_NOMEM, "hmse_compose: host allocation failed");
    uint64_t* hb = reinterpret_cast<uint64_t*>(hs) + src_words;   // sbase[n_src + 1], rbase[n_src + 1]
    uint64_t SM = 0, SR = 0;
    for (uint32_t s = 0; s < n_src; s++) {
        const hmse_compose_src& c = srcs[s];
        if (!c.d_layout || (c.m && (!c.d_index || !c.d_store)) || (c.n && !c.d_pointers) || (c.n_delta && !c.d_delta_store) ||
            ((uintptr_t)c.d_layout & 7) || ((uintptr_t)c.d_pointers & 7) || ((uintptr_t)c.d_index & 3)) {
            free(hs);
            HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compose: source %u: null or misaligned buffer", s);
        }
        hs[s].L = layout_of(const_cast<void*>(c.d_layout), c.n, c.m, c.n_delta);
        hs[s].index = c.d_index;
        hs[s].ptrs = c.d_pointers;
        hs[s].store = c.d_store;
        hs[s].dstore = c.d_delta_store;
        hs[s].n = c.n;
        hs[s].m = c.m;
        hs[s].n_delta = c.n_delta;
        hb[s] = SM;
        hb[n_src + 1 + s] = SR;
        SM += c.m;
        SR += c.n_delta ? c.n : 0;
    }
    hb[n_src] = SM;
    hb[2 * n_src + 1] = SR;
    // candidates are bounded by the slots and records of the sources and by the output's chunks
    const uint64_t KU = (SM < n_out ? SM : n_out) + 1, KR = (SR < n_out ? SR : n_out) + 1;
    // scratch (u64 words): [src][sbase rbase][run_off][ukey rkey][flags uflag rflag clen refc roff is_first][dig][usrc canon
    // krank uoff][rcand rsrc]
    const uint64_t zero_words = 2 + 2 * (n_out + 1) + 2 * KU + (KR + 1) + div_up64(KU, 8);
    const uint64_t words = src_words + 2 * (n_src + 1) + (n_runs + 1) + SM + SR + zero_words + 4 * KU + 4 * KU + 2 + 2 * KR;
    uint64_t* w = (uint64_t*)hmse_scratch(ctx, SLOT_COMPOSE, 8 * words);
    if (!w) {
        free(hs);
        return HMSE_E_NOMEM;
    }
    Work W;
    W.src = reinterpret_cast<const Src*>(w);
    uint64_t* q = w + src_words;
    W.sbase = q;
    W.rbase = q + n_src + 1;
    W.n_src = n_src;
    q += 2 * (n_src + 1);
    W.run_off = q;
    q += n_runs + 1;
    W.ukey = q;
    W.rkey = q + SM;
    q += SM + SR;
    uint64_t* zero = q;
    W.flags = reinterpret_cast<unsigned long long*>(q);
    W.uflag = q + 2;
    W.rflag = W.uflag + n_out + 1;
    W.clen = W.rflag + n_out + 1;
    W.refc = reinterpret_cast<unsigned long long*>(W.clen + KU);
    W.roff = W.clen + 2 * KU;
    W.is_first = reinterpret_cast<uint8_t*>(W.roff + KR + 1);
    q += zero_words;
    W.dig = reinterpret_cast<uint8_t*>(q);
    q += 4 * KU;
    W.usrc = q;
    W.canon = reinterpret_cast<int64_t*>(q + KU);
    W.krank = q + 2 * KU;
    W.uoff = W.krank + KU + 1;
    q += 4 * KU + 2;
    W.rcand = q;
    W.rsrc = q + KR;
    // from pageable memory: the copy has taken the bytes when it returns, so the host table can go
    const cudaError_t ce = cudaMemcpyAsync(w, hs, table_bytes, cudaMemcpyHostToDevice, st);
    free(hs);
    HMSE_CUDA(ctx, ce);
    HMSE_CUDA(ctx, cudaMemsetAsync(W.ukey, 0xFF, 8 * (SM + SR), st));
    HMSE_CUDA(ctx, cudaMemsetAsync(zero, 0, 8 * zero_words, st));
    const uint64_t cap = (uint64_t)ctx->sm_count * 8;
    HT_BEGIN(ctx, HT_COMPOSE, st);
    // ---- steps 1-5 ----
    KL(ctx);
    compose_check_kernel<<<grid_of(n_runs > n_src ? n_runs : n_src, ~0u), 256, 0, st>>>(W, d_runs, n_runs);
    HMSE_LAUNCH_CHECK(ctx);
    if (int e = hmse_exclusive_scan_u64(ctx, W.run_off, W.run_off, n_runs, W.run_off + n_runs, st)) return e;
    KL(ctx);
    compose_key_kernel<<<grid_of(n_out, cap), 256, 0, st>>>(W, d_runs, n_runs, n_out);
    KL(ctx);
    compose_flag_kernel<<<grid_of(SM > SR ? SM : SR, ~0u), 256, 0, st>>>(W, SM, SR);
    HMSE_LAUNCH_CHECK(ctx);
    if (int e = hmse_exclusive_scan_u64(ctx, W.uflag, W.uflag, n_out, W.uflag + n_out, st)) return e;
    if (int e = hmse_exclusive_scan_u64(ctx, W.rflag, W.rflag, n_out, W.rflag + n_out, st)) return e;
    KL(ctx);
    compose_cand_kernel<<<grid_of(SM > SR ? SM : SR, ~0u), 256, 0, st>>>(W, SM, SR);
    HMSE_LAUNCH_CHECK(ctx);
    if (int e = hmse_dedup_table(ctx, W.dig, 32, KU, W.uflag + n_out, W.canon, W.is_first, nullptr, SLOT_DEDUP_TABLE, st)) return e;
    KL(ctx);
    compose_keep_kernel<<<grid_of(KU, ~0u), 256, 0, st>>>(W, KU);
    HMSE_LAUNCH_CHECK(ctx);
    if (int e = hmse_exclusive_scan_u64(ctx, W.krank, W.krank, KU, W.krank + KU, st)) return e;
    if (int e = hmse_exclusive_scan_u64(ctx, W.uoff, W.uoff, KU, W.uoff + KU, st)) return e;
    if (int e = hmse_exclusive_scan_u64(ctx, W.roff, W.roff, KR, W.roff + KR, st)) return e;
    // ---- one mailbox read of the sizes ----
    KL(ctx);
    compose_sizes_kernel<<<1, 32, 0, st>>>(W, n_runs, n_out, KU, KR, ctx->pinned_dev);
    HMSE_LAUNCH_CHECK(ctx);
    HMSE_CUDA(ctx, cudaStreamSynchronize(st));
    const uint64_t* mb = ctx->pinned;
    const uint64_t err = mb[0], Kc = mb[1], kept = mb[2], sb = mb[3], Kr = mb[4], dsb = mb[5];
    if (err & CE_LAYOUT) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compose: a layout was not opened (hmse_read_open) for its source's n, m, n_delta");
    if (err & CE_DICT) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compose: the sources' dictionaries differ");
    if (err & CE_RUN) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compose: a run lies outside its source");
    if (err & CE_COUNT) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compose: the run counts do not add up to n_out");
    if (sb + dsb >= (1ull << 41)) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compose: the chunk store plus the delta store reach 2 TiB");
    out6[0] = n_out;
    out6[1] = Kc;
    out6[2] = kept;
    out6[3] = sb;
    out6[4] = Kr;
    out6[5] = dsb;
    if (kept > index_cap || sb > store_cap || dsb > delta_cap)
        HMSE_FAIL(ctx, HMSE_E_CAPACITY, "hmse_compose: needs index_cap %llu, store_cap %llu, delta_cap %llu", (unsigned long long)kept,
                  (unsigned long long)sb, (unsigned long long)dsb);
    if ((kept && (!d_index || !d_store)) || (Kr && !d_delta_store)) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compose: null output buffer");
    // ---- step 6: the streams and records gathered from their sources ----
    if (int e = hmse_segment_gather(ctx, W.usrc, d_store, W.uoff, Kc, st)) return e;
    if (int e = hmse_segment_gather(ctx, W.rsrc, d_delta_store, W.roff, Kr, st)) return e;
    // ---- step 7: the records ----
    KL(ctx);
    compose_pointer_kernel<<<grid_of(n_out, cap), 256, 0, st>>>(W, d_runs, n_runs, n_out, sb, reinterpret_cast<uint2*>(d_pointers));
    KL(ctx);
    compose_record_kernel<<<grid_of(Kr, ~0u), 256, 0, st>>>(W, Kr, kept, d_delta_store);
    KL(ctx);
    compose_index_kernel<<<grid_of(Kc, ~0u), 256, 0, st>>>(W, Kc, d_index);
    HMSE_LAUNCH_CHECK(ctx);
    HT_END(ctx, HT_COMPOSE, st);
    if (int e = hmse_mail(ctx, 0, W.flags + 1, 2, st)) return e;
    HMSE_CUDA(ctx, cudaStreamSynchronize(st));
    if (ctx->pinned[0]) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_compose: a DeltaChunk record's base has no kept slot");
    return HMSE_OK;
}
