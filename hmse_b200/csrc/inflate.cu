// inflate.cu - the read path's decoder (spec: README.md:1617-1675, the skeleton's mz_inflate round trip at
// README.md:2397-2400): every zlib stream produced by hmse_compress (or by stock zlib with a 32 KiB window and
// the same preset dictionary) back into raw chunk bytes, checked against the stream's own Adler-32 trailer.
//
// A DEFLATE stream is a serial bit string, so the parallelism is across streams: one WARP per stream.
// All 32 lanes carry the same bit-reader state and decode the same symbol (warp-uniform control flow, the
// loads are broadcasts); what the lanes share out is the work a symbol causes - the copy of a match (up to
// 258 bytes, lane i takes bytes i, i+32, ...), the construction of the decoding tables of a dynamic block, and
// the final Adler-32 of the output.  Tables per warp in shared memory: a 10-bit direct lookup for the
// literal/length code and an 8-bit one for the distance code; longer codes fall back to the canonical
// count/first-code walk.
#include "ctx.cuh"

namespace {

constexpr int IW = 8;              // warps (streams in flight) per CTA
constexpr int LBITS = 10, DBITS = 8;
constexpr uint32_t MAXL = 288, MAXD = 32;

enum InfStatus : uint32_t {
    INF_OK = 0,
    INF_BAD_HEADER = 1,     // CMF/FLG check, method, window, FDICT without/with a dictionary, DICTID mismatch
    INF_BAD_BLOCK = 2,      // reserved block type, stored length check, bad code lengths
    INF_BAD_CODE = 3,       // undecodable symbol or a distance beyond the window / dictionary
    INF_OVERRUN = 4,        // more output than the expected length, or input exhausted
    INF_LENGTH = 5,         // stream ended with fewer bytes than expected
    INF_ADLER = 6           // Adler-32 trailer does not match the output
};

struct Tables {
    uint16_t lit[1 << LBITS];     // (symbol << 4) | code length, 0 = longer than LBITS (or unused)
    uint16_t dist[1 << DBITS];
    uint16_t lsym[MAXL], dsym[MAXD];   // symbols ordered by (length, symbol): the canonical order
    uint16_t lcount[16], dcount[16];   // codes per length
    uint8_t lens[MAXL + MAXD + 32];    // code lengths of the current block; while a dynamic header is read: the
                                       // code-length code's own lengths in [0, 19), the vectors behind them from 32 on
    uint16_t cl_tab[128];              // 7-bit lookup of the code-length code
};

struct BitReader {
    const uint8_t* p;     // next unread byte
    const uint8_t* end;
    uint64_t buf;
    uint32_t cnt;         // valid bits in buf
    uint32_t over;        // bits consumed past the end of the input (error)
    __device__ __forceinline__ void init(const uint8_t* b, const uint8_t* e) {
        p = b;
        end = e;
        buf = 0;
        cnt = 0;
        over = 0;
    }
    __device__ __forceinline__ void refill() {   // keep >= 32 bits (zeros past the end)
        while (cnt <= 32) {
            uint32_t v = 0;
            if (p + 4 <= end) {
                v = (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
                p += 4;
                buf |= (uint64_t)v << cnt;
                cnt += 32;
            } else {
                if (p < end) v = *p;
                else over += 8;
                p++;
                buf |= (uint64_t)v << cnt;
                cnt += 8;
            }
        }
    }
    __device__ __forceinline__ uint32_t peek(uint32_t n) const { return (uint32_t)buf & ((1u << n) - 1); }
    __device__ __forceinline__ void drop(uint32_t n) {
        buf >>= n;
        cnt -= n;
    }
    __device__ __forceinline__ uint32_t bits(uint32_t n) {   // n <= 16
        refill();
        const uint32_t v = peek(n);
        drop(n);
        return v;
    }
    // bytes consumed so far, counting only whole bytes still in the buffer as unread
    __device__ __forceinline__ const uint8_t* byte_pos() const { return p - (cnt >> 3); }
};

__device__ __forceinline__ uint32_t rev_bits(uint32_t code, uint32_t len) { return __brev(code) >> (32 - len); }

// Builds the direct lookup + canonical arrays of one code from lens[0..n).  Collective over the warp.
// Accepts exactly the length sets zlib's inflate_table accepts: a complete code, a code with no symbols at all (a
// symbol read from it is then an error), or - except for the code-length code (cl_code) - a single code of length 1.
// Returns false on an over-subscribed or any other incomplete set.
__device__ bool build_table(const uint8_t* lens, uint32_t n, uint16_t* tab, uint32_t tbits, uint16_t* sym, uint16_t* count,
                            bool cl_code, unsigned lane) {
    for (uint32_t i = lane; i < (1u << tbits); i += 32) tab[i] = 0;
    if (lane < 16) count[lane] = 0;
    __syncwarp();
    for (uint32_t i = lane; i < n; i += 32)
        if (lens[i]) atomicAdd(reinterpret_cast<unsigned int*>(count) + (lens[i] >> 1), 1u << (16 * (lens[i] & 1)));
    __syncwarp();
    // first code and first index of every length (every lane computes them: 15 steps)
    uint32_t first[16], offs[16];
    uint32_t code = 0, idx = 0, max_len = 0;
    int left = 1;
    bool over = false;
    first[0] = offs[0] = 0;
#pragma unroll
    for (int l = 1; l < 16; l++) {
        const uint32_t c = count[l];
        left = (left << 1) - (int)c;
        if (left < 0) over = true;
        first[l] = code;
        offs[l] = idx;
        code = (code + c) << 1;
        idx += c;
        if (c) max_len = l;
    }
    if (over) return false;
    if (left > 0 && max_len != 0 && (cl_code || max_len != 1)) return false;   // incomplete
    // rank of a symbol inside its length class = symbols of the same length before it: chunks of 32 in order
    uint32_t seen[16];
#pragma unroll
    for (int l = 0; l < 16; l++) seen[l] = 0;
    const uint32_t lt = (1u << lane) - 1;
    for (uint32_t base = 0; base < n; base += 32) {
        const uint32_t s = base + lane;
        const uint32_t l = s < n ? lens[s] : 0u;
        const uint32_t peers = __match_any_sync(0xffffffffu, l ? l : 100u + lane);
        const uint32_t rank = __popc(peers & lt);
        uint32_t before = 0, c_first = 0, c_offs = 0;
#pragma unroll
        for (int q = 1; q < 16; q++) {   // register arrays: select by comparison, no dynamic indexing
            const uint32_t cnt_q = __popc(__ballot_sync(0xffffffffu, l == (uint32_t)q));
            if (l == (uint32_t)q) {
                before = seen[q];
                c_first = first[q];
                c_offs = offs[q];
            }
            seen[q] += cnt_q;
        }
        if (l) {
            const uint32_t k = before + rank;
            sym[c_offs + k] = (uint16_t)s;
            if (l <= tbits) {
                const uint32_t r = rev_bits(c_first + k, l);
                const uint16_t e = (uint16_t)((s << 4) | l);
                for (uint32_t x = r; x < (1u << tbits); x += 1u << l) tab[x] = e;
            }
        }
    }
    __syncwarp();
    return true;
}

// Decodes one symbol: direct lookup, else the canonical walk over lengths tbits+1 .. 15.  Warp-uniform.
// Returns 0xFFFF on an invalid code.
__device__ __forceinline__ uint32_t decode_sym(BitReader& br, const uint16_t* tab, uint32_t tbits, const uint16_t* sym,
                                               const uint16_t* count) {
    br.refill();
    const uint32_t e = tab[br.peek(tbits)];
    if (e) {
        br.drop(e & 15);
        return e >> 4;
    }
    // slow path: bit by bit (MSB-first code value), as in the reference decoder of RFC 1951 section 3.2.2
    uint32_t code = 0, first = 0, index = 0;
    uint64_t b = br.buf;
    for (uint32_t len = 1; len < 16; len++) {
        code |= (uint32_t)b & 1;
        b >>= 1;
        const uint32_t c = count[len];
        if (code < first + c) {
            br.drop(len);
            return sym[index + (code - first)];
        }
        index += c;
        first = (first + c) << 1;
        code <<= 1;
    }
    return 0xFFFFu;
}

__constant__ uint16_t c_lbase[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
__constant__ uint8_t c_lext[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
__constant__ uint16_t c_dbase[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
__constant__ uint8_t c_dext[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
__constant__ uint8_t c_clorder[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

struct InfArgs {
    const uint8_t* blob;
    const uint64_t* offs;       // [m+1]; with offs_end: [m], stream j = blob[offs[j] : offs_end[j])
    const uint64_t* offs_end;   // null: stream j = blob[offs[j] : offs[j+1])
    uint64_t m;
    const uint8_t* dict;
    uint32_t dict_len, dict_adler;
    uint8_t* out;
    const uint64_t* out_offs;   // [m+1]
    uint32_t* status;           // [m]
    unsigned int* counter;
};

__global__ void __launch_bounds__(IW * 32) inflate_kernel(InfArgs a) {
    __shared__ Tables s_tab[IW];
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    Tables& T = s_tab[warp];
    for (;;) {
        uint64_t j = 0;
        if (lane == 0) j = atomicAdd(a.counter, 1u);
        j = __shfl_sync(0xffffffffu, j, 0);
        if (j >= a.m) break;
        // the offsets come from the caller (an archive that may be damaged): a stream or an output range that runs
        // backwards, or an output range beyond 32 bits, is reported and nothing is read or written for it
        const uint64_t o0 = a.offs[j], o1 = a.offs_end ? a.offs_end[j] : a.offs[j + 1], q0 = a.out_offs[j], q1 = a.out_offs[j + 1];
        if (o1 < o0 || q1 < q0 || q1 - q0 > 0xFFFFFFFFull) {
            if (lane == 0) a.status[j] = o1 < o0 ? INF_BAD_HEADER : INF_OVERRUN;
            continue;
        }
        const uint8_t* in = a.blob + o0;
        const uint8_t* in_end = a.blob + o1;
        uint8_t* out = a.out + q0;
        const uint32_t out_len = (uint32_t)(q1 - q0);
        uint32_t status = INF_OK;
        uint32_t pos = 0;
        BitReader br;
        // ---- zlib header (RFC 1950) ----
        const uint32_t hdr_need = a.dict_len ? 6u : 2u;
        if ((uint64_t)(in_end - in) < hdr_need + 4u) {
            status = INF_BAD_HEADER;
        } else {
            const uint32_t cmf = in[0], flg = in[1];
            const bool fdict = (flg & 0x20u) != 0;
            if ((cmf & 15u) != 8u || (cmf >> 4) > 7u || ((cmf << 8) | flg) % 31u != 0 || fdict != (a.dict_len != 0)) {
                status = INF_BAD_HEADER;
            } else if (fdict) {
                const uint32_t id = ((uint32_t)in[2] << 24) | ((uint32_t)in[3] << 16) | ((uint32_t)in[4] << 8) | in[5];
                if (id != a.dict_adler) status = INF_BAD_HEADER;
            }
        }
        br.init(in + hdr_need, in_end);
        // ---- DEFLATE blocks (RFC 1951) ----
        bool last = false;
        while (status == INF_OK && !last) {
            last = br.bits(1) != 0;
            const uint32_t type = br.bits(2);
            if (type == 0) {   // stored: skip to a byte boundary, LEN / NLEN, raw bytes
                br.drop(br.cnt & 7);
                br.refill();
                const uint32_t len = br.peek(16);
                br.drop(16);
                br.refill();
                const uint32_t nlen = br.peek(16);
                br.drop(16);
                if ((len ^ nlen) != 0xFFFFu) {
                    status = INF_BAD_BLOCK;
                    break;
                }
                const uint8_t* src = br.byte_pos();
                if (src + len > in_end || pos + len > out_len) {
                    status = INF_OVERRUN;
                    break;
                }
                for (uint32_t i = lane; i < len; i += 32) out[pos + i] = src[i];
                pos += len;
                br.init(src + len, in_end);
                __syncwarp();
                continue;
            }
            if (type == 3) {
                status = INF_BAD_BLOCK;
                break;
            }
            uint32_t nlit = 288, ndist = 32;
            if (type == 1) {   // fixed code
                for (uint32_t i = lane; i < 288; i += 32) T.lens[i] = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : 8;
                T.lens[288 + lane] = 5;   // 32 five-bit distance codes (30 and 31 never occur in valid data)
                __syncwarp();
            } else {           // dynamic code: code-length code, then the two length vectors
                nlit = br.bits(5) + 257;
                ndist = br.bits(5) + 1;
                const uint32_t ncl = br.bits(4) + 4;
                if (nlit > 286 || ndist > 30) {
                    status = INF_BAD_BLOCK;
                    break;
                }
                uint32_t my_cl = 0;   // lane i holds the length of code-length symbol i (i < 19)
                for (uint32_t i = 0; i < ncl; i++) {
                    const uint32_t v = br.bits(3);
                    if (lane == c_clorder[i]) my_cl = v;
                }
                __syncwarp();
                if (lane < 19) T.lens[lane] = (uint8_t)my_cl;
                __syncwarp();
                uint16_t* clsym = T.lsym;   // scratch: rebuilt below
                if (!build_table(T.lens, 19, T.cl_tab, 7, clsym, T.lcount, true, lane)) {
                    status = INF_BAD_BLOCK;
                    break;
                }
                // the lengths themselves: serial in the bit stream, identical in every lane
                uint32_t i = 0, prev = 0;
                const uint32_t total = nlit + ndist;
                uint8_t* dst = T.lens + 32;   // decode behind the code-length code's own lengths, move down afterwards
                while (i < total) {
                    const uint32_t s = decode_sym(br, T.cl_tab, 7, clsym, T.lcount);
                    if (s < 16) {
                        if (lane == 0) dst[i] = (uint8_t)s;
                        prev = s;
                        i++;
                        continue;
                    }
                    uint32_t rep, val = 0;
                    if (s == 16) {
                        if (i == 0) {
                            status = INF_BAD_BLOCK;
                            break;
                        }
                        val = prev;
                        rep = 3 + br.bits(2);
                    } else if (s == 17) {
                        rep = 3 + br.bits(3);
                    } else if (s == 18) {
                        rep = 11 + br.bits(7);
                    } else {
                        status = INF_BAD_CODE;
                        break;
                    }
                    if (i + rep > total) {
                        status = INF_BAD_BLOCK;
                        break;
                    }
                    if (lane < rep) dst[i + lane] = (uint8_t)val;        // rep <= 138: up to five strides of 32
                    for (uint32_t q = lane + 32; q < rep; q += 32) dst[i + q] = (uint8_t)val;
                    if (s != 16) prev = 0;
                    i += rep;
                }
                if (status != INF_OK) break;
                __syncwarp();
                // lay the two vectors out at lens[0..288) and lens[288..320)
                uint8_t mine[10];
#pragma unroll
                for (int q = 0; q < 10; q++) {
                    const uint32_t x = lane + 32 * q;
                    uint8_t v = 0;
                    if (x < 288) v = x < nlit ? dst[x] : 0;
                    else if (x < 320) v = (x - 288) < ndist ? dst[nlit + (x - 288)] : 0;
                    mine[q] = v;
                }
                __syncwarp();
#pragma unroll
                for (int q = 0; q < 10; q++) T.lens[lane + 32 * q] = mine[q];
                __syncwarp();
                if (T.lens[256] == 0) {   // no end-of-block code
                    status = INF_BAD_BLOCK;
                    break;
                }
            }
            if (!build_table(T.lens, 288, T.lit, LBITS, T.lsym, T.lcount, false, lane) ||
                !build_table(T.lens + 288, 32, T.dist, DBITS, T.dsym, T.dcount, false, lane)) {
                status = INF_BAD_BLOCK;
                break;
            }
            // ---- symbols ----
            for (;;) {
                const uint32_t s = decode_sym(br, T.lit, LBITS, T.lsym, T.lcount);
                if (s < 256) {
                    if (pos >= out_len) {
                        status = INF_OVERRUN;
                        break;
                    }
                    if (lane == 0) out[pos] = (uint8_t)s;
                    pos++;
                    continue;
                }
                if (s == 256) break;
                if (s > 285) {
                    status = INF_BAD_CODE;
                    break;
                }
                const uint32_t li = s - 257;
                const uint32_t len = c_lbase[li] + br.bits(c_lext[li]);
                const uint32_t ds = decode_sym(br, T.dist, DBITS, T.dsym, T.dcount);
                if (ds > 29) {
                    status = INF_BAD_CODE;
                    break;
                }
                const uint32_t dist = c_dbase[ds] + br.bits(c_dext[ds]);
                if (dist > pos + a.dict_len) {
                    status = INF_BAD_CODE;
                    break;
                }
                if (pos + len > out_len) {
                    status = INF_OVERRUN;
                    break;
                }
                __syncwarp();   // earlier literal / match stores of other lanes are visible to the loads below
                // byte i of the match comes from i mod dist behind the start (overlapping copies repeat)
                for (uint32_t i = lane; i < len; i += 32) {
                    const uint32_t back = i < dist ? i : i % dist;
                    const int32_t sp = (int32_t)(pos + back) - (int32_t)dist;
                    out[pos + i] = sp >= 0 ? out[sp] : a.dict[(int32_t)a.dict_len + sp];
                }
                pos += len;
                __syncwarp();
            }
            if (br.over) status = INF_OVERRUN;
        }
        // ---- trailer: Adler-32 of the output, big endian, after the last block (byte aligned) ----
        if (status == INF_OK && pos != out_len) status = INF_LENGTH;
        if (status == INF_OK) {
            br.drop(br.cnt & 7);
            const uint8_t* tr = br.byte_pos();
            if (tr + 4 != in_end) {
                status = tr + 4 > in_end ? INF_OVERRUN : INF_LENGTH;
            } else {
                __syncwarp();
                uint32_t sa = 0, sb = 0;   // per-lane partial sums over bytes lane, lane+32, ...; reduce mod 65521 often enough
                uint32_t pending = 0;
                for (uint32_t i = lane; i < out_len; i += 32) {
                    const uint32_t b = out[i];
                    sa += b;
                    sb += ((out_len - i) % 65521u) * b % 65521u;
                    if (++pending == 4096) {
                        sa %= 65521u;
                        sb %= 65521u;
                        pending = 0;
                    }
                }
                sa %= 65521u;
                sb %= 65521u;
#pragma unroll
                for (int o = 16; o; o >>= 1) {
                    sa += __shfl_xor_sync(0xffffffffu, sa, o);
                    sb += __shfl_xor_sync(0xffffffffu, sb, o);
                }
                const uint32_t A = (1u + sa) % 65521u, B = (out_len % 65521u + sb) % 65521u;
                const uint32_t want = ((uint32_t)tr[0] << 24) | ((uint32_t)tr[1] << 16) | ((uint32_t)tr[2] << 8) | tr[3];
                if (((B << 16) | A) != want) status = INF_ADLER;
            }
        }
        if (lane == 0) a.status[j] = status;
        __syncwarp();
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

__global__ void count_bad_kernel(const uint32_t* __restrict__ status, uint64_t m, unsigned long long* __restrict__ bad) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool b = i < m && status[i] != 0;
    const uint32_t n = __popc(__ballot_sync(0xffffffffu, b));
    if ((threadIdx.x & 31) == 0 && n) atomicAdd(bad, (unsigned long long)n);
}

}  // namespace

// Streams j = d_blob[d_begin[j] : d_end[j]) (d_end null: d_begin[j+1]), the DICTID given by the caller; no host round
// trip.  hmse_read inflates the stored chunks it needs in place in the chunk store through this form.
int hmse_inflate_ranges(hmse_ctx* ctx, const uint8_t* d_blob, const uint64_t* d_begin, const uint64_t* d_end, uint64_t m,
                        const uint8_t* d_zdict, uint32_t dict_len, uint32_t dict_adler, uint8_t* d_out,
                        const uint64_t* d_out_offsets, uint32_t* d_status, cudaStream_t st) {
    if (m == 0) return HMSE_OK;
    HMSE_SCRATCH(ctx, misc, unsigned long long*, SLOT_INFLATE_MISC, 64);
    HMSE_CUDA(ctx, cudaMemsetAsync(misc, 0, 64, st));
    InfArgs a;
    a.blob = d_blob;
    a.offs = d_begin;
    a.offs_end = d_end;
    a.m = m;
    a.dict = d_zdict;
    a.dict_len = dict_len;
    a.dict_adler = dict_adler;
    a.out = d_out;
    a.out_offs = d_out_offsets;
    a.status = d_status;
    a.counter = (unsigned int*)(misc + 1);
    const uint64_t want = div_up64(m, IW);
    const uint64_t cap = (uint64_t)ctx->sm_count * 8;
    HT_BEGIN(ctx, HT_INFLATE, st);
    KL(ctx);
    inflate_kernel<<<(unsigned)(want < cap ? want : cap), IW * 32, 0, st>>>(a);
    HMSE_LAUNCH_CHECK(ctx);
    HT_END(ctx, HT_INFLATE, st);
    return HMSE_OK;
}

uint32_t hmse_adler32_host(const uint8_t* d, size_t n) { return host_adler32(d, n); }

HMSE_API int hmse_inflate(hmse_ctx* ctx, const uint8_t* d_blob, const uint64_t* d_offsets, uint64_t m, const uint8_t* d_zdict,
                          uint32_t dict_len, uint8_t* d_out, const uint64_t* d_out_offsets, uint32_t* d_status,
                          uint64_t* n_bad, void* stream) {
    if (!ctx) return HMSE_E_INVAL;
    cudaStream_t st = (cudaStream_t)stream;
    if (n_bad) *n_bad = 0;
    if (m == 0) return HMSE_OK;
    if (!d_blob || !d_offsets || !d_out_offsets || !d_status || !d_out) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_inflate: null pointer");
    if (dict_len > 32768) HMSE_FAIL(ctx, HMSE_E_INVAL, "dict_len must be <= 32768");
    if (dict_len && !d_zdict) HMSE_FAIL(ctx, HMSE_E_INVAL, "d_zdict is null");
    if (m >= 0xFFFFFFFFull) HMSE_FAIL(ctx, HMSE_E_INVAL, "too many streams in one call");
    uint32_t dict_adler = 0;
    if (dict_len) {   // DICTID of the header = Adler-32 of the dictionary (a 32 KiB one-off per call)
        static thread_local uint8_t tmp[32768];
        HMSE_CUDA(ctx, cudaMemcpyAsync(tmp, d_zdict, dict_len, cudaMemcpyDeviceToHost, st));
        HMSE_CUDA(ctx, cudaStreamSynchronize(st));
        dict_adler = host_adler32(tmp, dict_len);
    }
    if (int rc = hmse_inflate_ranges(ctx, d_blob, d_offsets, nullptr, m, d_zdict, dict_len, dict_adler, d_out, d_out_offsets,
                                     d_status, st))
        return rc;
    if (n_bad) {
        HMSE_SCRATCH(ctx, misc, unsigned long long*, SLOT_INFLATE_MISC, 64);
        KL(ctx);
        count_bad_kernel<<<(unsigned)div_up64(m, 256), 256, 0, st>>>(d_status, m, misc);
        HMSE_LAUNCH_CHECK(ctx);
        if (int mrc = hmse_mail(ctx, 0, misc, 2, st)) return mrc;
        HMSE_CUDA(ctx, cudaStreamSynchronize(st));
        *n_bad = ctx->pinned[0];
    }
    return HMSE_OK;
}
