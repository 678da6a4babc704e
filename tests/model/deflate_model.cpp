// deflate_model.cpp - sequential CPU model of the GPU DEFLATE encoder (hmse_b200/csrc/deflate.cu).
// TEST INFRASTRUCTURE: compiled with g++ by tests/model/build.py; shares deflate_core.h with the
// kernel so the Huffman / header / symbol-map logic is validated against stock zlib on the CPU.
// Never loaded by the product package.
//
// model_compress       one zlib stream of one block (chunks of at most 32 KiB: parse_kernel's size classes)
// model_compress_long  one zlib stream of 32 KiB blocks (longer chunks: long_dict_kernel / encode_long_kernel /
//                      stored_kernel)
// With mode 2, prev0 1 and the own-candidate count of the size class (2 / 3 / 4; 4 in every block of a long chunk) the
// streams are the kernel's byte for byte (tests/test_gpu_deflate_exact.py).
#include <stdint.h>
#include <string.h>

#include <vector>

#include "../../hmse_b200/csrc/deflate_core.h"

using namespace dfl;

struct Params {
    int hash_bytes;   // 3 or 4
    int chain_own;    // max own-chunk candidates examined
    int chain_dict;   // max dictionary candidates examined
    int lazy;         // 0 greedy, 1 zlib-style lazy
    int too_far;      // drop length-3 matches farther than this (0 = keep)
    int dict_hash_bits;  // buckets of the dictionary index (the own-chunk index uses HASH_BITS)
    int mode;         // 0: every position extends its candidates; 1: run heads only + prefix max (skip a pair
                      // only when the previous position examined its predecessor); 2: same, unconditional skip
    int min_len;      // shortest match emitted (0 -> hash_bytes)
    int hist;         // the first `hist` bytes are history only: searched, not emitted (multi-block chunks)
    int prev0;        // run-head test of modes 1-3 at position 0 of either side: 0 no byte precedes it (such a pair is
                      // always a head); 1 the kernel's sentinels - 0xFE precedes the chunk (CHUNK_PREV0), 0xFF the
                      // dictionary (DICT_PREV0), so a pair is no head when the other side's previous byte equals it
};

constexpr uint32_t CHUNK_PREV0 = 0xFEu, DICT_PREV0 = 0xFFu;   // the kernel's values (csrc/deflate.cu)
constexpr uint32_t LONG_BLOCK = 32768, LONG_MAX_BLOCKS = 2048, STORED_MAX = 65535;

static inline uint32_t rd(const uint8_t* p, int nb) {
    uint32_t v = p[0] | (p[1] << 8) | (p[2] << 16);
    if (nb == 4) v |= (uint32_t)p[3] << 24;
    return v;
}

static uint32_t adler32(const uint8_t* d, uint64_t n) {
    uint32_t a = 1, b = 0;
    for (uint64_t i = 0; i < n; i++) {
        a = (a + d[i]) % 65521;
        b = (b + a) % 65521;
    }
    return (b << 16) | a;
}

// One parsed block: tokens (literal: byte; match: 1<<31 | len<<16 | (dist-1)) and their symbol counts (EOB included).
struct Parsed {
    std::vector<uint32_t> tok;
    uint32_t lit_freq[288], dist_freq[32];
    uint32_t n_match;
};

// Match search + lazy parse of data[0..n) with dict[0..dict_len) in front of it.
static void parse_block(const uint8_t* data, uint32_t n, const uint8_t* dict, uint32_t dict_len, const Params* pr,
                        Parsed& ps, uint32_t* stats) {
    const int HB = pr->hash_bytes;
    const int DB = pr->dict_hash_bits ? pr->dict_hash_bits : HASH_BITS;
    auto dhash = [&](uint32_t v) { return (v * 0x9E3779B1u) >> (32 - DB); };
    std::vector<std::vector<uint32_t>> own(NBUCKET), dic((size_t)1 << DB);
    for (uint32_t j = 0; j + HB <= dict_len; j++) dic[dhash(rd(dict + j, HB))].push_back(j);
    std::vector<uint16_t> mlen(n + 1, 0), mdist(n + 1, 0);
    if (!pr->mode) {
        for (uint32_t p = 0; p < n; p++) {
            uint32_t best = 0, bdist = 0;
            if (p + HB <= n) {
                const uint32_t maxl = n - p < MAX_MATCH ? n - p : MAX_MATCH;
                const uint32_t h = hash4(rd(data + p, HB));
                auto& ob = own[h];
                int ex = 0;
                for (int i = (int)ob.size() - 1; i >= 0 && ex < pr->chain_own; i--, ex++) {
                    uint32_t q = ob[i], l = 0;
                    if (p - q > WSIZE) break;
                    while (l < maxl && data[q + l] == data[p + l]) l++;
                    if (l > best) { best = l; bdist = p - q; }
                    if (best >= (uint32_t)NICE_LENGTH || best == maxl) break;
                }
                auto& db = dic[dhash(rd(data + p, HB))];
                ex = 0;
                if (best < (uint32_t)NICE_LENGTH && best < maxl)
                    for (int i = (int)db.size() - 1; i >= 0 && ex < pr->chain_dict; i--, ex++) {
                        uint32_t j = db[i], l = 0;
                        uint32_t dist = p + dict_len - j;
                        if (dist > WSIZE) break;
                        uint32_t lim = dict_len - j < maxl ? dict_len - j : maxl;  // matches do not cross into the chunk
                        while (l < lim && dict[j + l] == data[p + l]) l++;
                        if (l > best) { best = l; bdist = dist; }
                        if (best >= (uint32_t)NICE_LENGTH || best == maxl) break;
                    }
                ob.push_back(p);
            }
            if (best < (uint32_t)MIN_MATCH) best = 0;
            if (best == 3 && pr->too_far && bdist > (uint32_t)pr->too_far) best = 0;
            mlen[p] = (uint16_t)best;
            mdist[p] = (uint16_t)(bdist - (best ? 1 : 0));  // stored as dist-1 so 32768 fits
        }
    } else {
        // Run formulation: a verified pair (p, source s) whose preceding bytes differ starts a run that ends at
        // `end`; every position inside it has a match of length end - p at the same distance, so
        // best[p] = (prefix max of run ends over start positions) - p.  The head test comes first: only heads are
        // extended to their end (non-heads only as far as the statistics count them, 258 bytes).
        std::vector<uint32_t> prev_own, prev_dic, cur_own, cur_dic;
        bool prev_sat = false, cur_sat = false;  // mode 3: a candidate list was cut short by its cap
        uint64_t key_run = 0;  // end << 16 | (65535 - (dist-1))
        uint64_t n_pairs = 0, n_heads = 0, steps_all = 0, steps_head = 0;
        const uint32_t minl = pr->min_len ? pr->min_len : HB;
        // the byte before data[x] / dict[x] as the run-head test sees it (x == 0: a sentinel, or none)
        const bool sent = pr->prev0 != 0;
        auto before_data = [&](uint32_t x) { return x ? (uint32_t)data[x - 1] : CHUNK_PREV0; };
        auto before_dict = [&](uint32_t x) { return x ? (uint32_t)dict[x - 1] : DICT_PREV0; };
        for (uint32_t p = 0; p < n; p++) {
            cur_own.clear();
            cur_dic.clear();
            cur_sat = false;
            if (p + HB <= n) {
                const uint32_t v = rd(data + p, HB);
                auto& ob = own[hash4(v)];
                if ((int)ob.size() > pr->chain_own || (int)dic[dhash(v)].size() > pr->chain_dict) cur_sat = true;
                int ex = 0;
                for (int i = (int)ob.size() - 1; i >= 0 && ex < pr->chain_own; i--, ex++) {
                    const uint32_t q = ob[i];
                    if (p - q > WSIZE) break;
                    cur_own.push_back(q);
                    if (rd(data + q, HB) != v) continue;
                    n_pairs++;
                    bool inh = sent ? before_data(p) == before_data(q) : p >= 1 && q >= 1 && data[p - 1] == data[q - 1];
                    if (inh && pr->mode == 1) {
                        bool found = false;
                        for (uint32_t x : prev_own) found |= x == q - 1;
                        inh = found;
                    }
                    if (inh && pr->mode == 3) inh = !prev_sat;
                    const uint32_t cap = inh ? (stats ? (uint32_t)MAX_MATCH : 0u) : n - p;
                    uint32_t l = 0;
                    while (l < cap && p + l < n && data[q + l] == data[p + l]) l++;
                    steps_all += ((l < 258 ? l : 258) + 7) / 8;
                    if (inh) continue;
                    n_heads++;
                    steps_head += (l + 7) / 8;
                    const uint64_t key = ((uint64_t)(p + l) << 16) | (65535 - (p - q - 1));
                    if (key > key_run) key_run = key;
                }
                auto& db = dic[dhash(v)];
                ex = 0;
                for (int i = (int)db.size() - 1; i >= 0 && ex < pr->chain_dict; i--, ex++) {
                    const uint32_t j = db[i];
                    const uint32_t dist = p + dict_len - j;
                    if (dist > WSIZE) break;
                    cur_dic.push_back(j);
                    if (rd(dict + j, HB) != v) continue;
                    n_pairs++;
                    bool inh = sent ? before_data(p) == before_dict(j) : p >= 1 && j >= 1 && data[p - 1] == dict[j - 1];
                    if (inh && pr->mode == 1) {
                        bool found = false;
                        for (uint32_t x : prev_dic) found |= x == j - 1;
                        inh = found;
                    }
                    if (inh && pr->mode == 3) inh = !prev_sat;
                    const uint32_t cap = inh ? (stats ? (uint32_t)MAX_MATCH : 0u) : n - p;
                    uint32_t l = 0;
                    while (l < cap && p + l < n && j + l < dict_len && dict[j + l] == data[p + l]) l++;
                    steps_all += ((l < 258 ? l : 258) + 7) / 8;
                    if (inh) continue;
                    n_heads++;
                    steps_head += (l + 7) / 8;
                    const uint64_t key = ((uint64_t)(p + l) << 16) | (65535 - (dist - 1));
                    if (key > key_run) key_run = key;
                }
                ob.push_back(p);
            }
            prev_own.swap(cur_own);
            prev_dic.swap(cur_dic);
            prev_sat = cur_sat;
            const uint32_t end = (uint32_t)(key_run >> 16);
            if (end >= p + minl) {
                const uint32_t L = end - p < (uint32_t)MAX_MATCH ? end - p : (uint32_t)MAX_MATCH;
                const uint32_t d1 = 65535 - (uint32_t)(key_run & 0xffff);
                if (!(L == 3 && pr->too_far && d1 + 1 > (uint32_t)pr->too_far)) {
                    mlen[p] = (uint16_t)L;
                    mdist[p] = (uint16_t)d1;
                }
            }
        }
        if (stats) { stats[4] = (uint32_t)n_pairs; stats[5] = (uint32_t)n_heads; stats[6] = (uint32_t)steps_all; stats[7] = (uint32_t)steps_head; }
    }
    // parse
    ps.tok.clear();
    memset(ps.lit_freq, 0, sizeof ps.lit_freq);
    memset(ps.dist_freq, 0, sizeof ps.dist_freq);
    ps.n_match = 0;
    uint32_t p = (uint32_t)pr->hist;
    while (p < n) {
        uint32_t L = mlen[p];
        bool lit = L < 3;
        if (!lit && pr->lazy && L < (uint32_t)MAX_LAZY && p + 1 < n && mlen[p + 1] > L) lit = true;
        if (lit) {
            ps.tok.push_back(data[p]);
            ps.lit_freq[data[p]]++;
            p++;
        } else {
            ps.tok.push_back(0x80000000u | (L << 16) | mdist[p]);
            uint32_t s, eb, ev;
            len_sym(L, s, eb, ev);
            ps.lit_freq[s]++;
            dist_sym((uint32_t)mdist[p] + 1, s, eb, ev);
            ps.dist_freq[s]++;
            p += L;
            ps.n_match++;
        }
    }
    ps.lit_freq[EOB]++;
}

// Fixed and dynamic cost of a parsed block (header, tokens and end-of-block, in bits) and the dynamic header.
struct Plan {
    DynHeader h;
    uint64_t dyn_bits, fix_bits;
};

static void plan_block(const Parsed& ps, Plan& pl) {
    HuffWork hw;
    uint32_t lf[288], df[32];
    memcpy(lf, ps.lit_freq, sizeof lf);
    memcpy(df, ps.dist_freq, sizeof df);
    pl.dyn_bits = plan_dynamic_header(lf, df, pl.h, hw);
    pl.fix_bits = 3;
    for (int s = 0; s < NLIT; s++) {
        pl.dyn_bits += (uint64_t)ps.lit_freq[s] * (pl.h.lit_lens[s] + (s > 256 ? lsym_extra(s) : 0));
        pl.fix_bits += (uint64_t)ps.lit_freq[s] * (fixed_lit_len(s) + (s > 256 ? lsym_extra(s) : 0));
    }
    for (int s = 0; s < NDIST; s++) {
        pl.dyn_bits += (uint64_t)ps.dist_freq[s] * (pl.h.dist_lens[s] + dsym_extra(s));
        pl.fix_bits += (uint64_t)ps.dist_freq[s] * (5 + dsym_extra(s));
    }
}

// One coded block (mode 1 fixed, 2 dynamic) appended to bw.
static void write_block(const Parsed& ps, const Plan& pl, int mode, int bfinal, BitWriter& bw) {
    uint32_t lc[288], dc[32];
    if (mode == 2) {
        write_dynamic_header(pl.h, bw, bfinal);
        assign_codes(pl.h.lit_lens, NLIT, lc);
        assign_codes(pl.h.dist_lens, NDIST, dc);
    } else {
        bw.put((uint32_t)bfinal, 1);
        bw.put(1, 2);
        for (int s = 0; s < 288; s++) lc[s] = fixed_lit_code(s);
        for (int s = 0; s < 30; s++) dc[s] = fixed_dist_code(s);
    }
    for (uint32_t t : ps.tok) {
        if (!(t >> 31)) {
            bw.put(lc[t] & 0xffff, lc[t] >> 16);
        } else {
            uint32_t L = (t >> 16) & 0x7fff, D = (t & 0xffff) + 1, s, eb, ev;
            len_sym(L, s, eb, ev);
            bw.put(lc[s] & 0xffff, lc[s] >> 16);
            bw.put(ev, eb);
            dist_sym(D, s, eb, ev);
            bw.put(dc[s] & 0xffff, dc[s] >> 16);
            bw.put(ev, eb);
        }
    }
    bw.put(lc[EOB] & 0xffff, lc[EOB] >> 16);
}

static uint64_t zlib_head(uint8_t* out, const uint8_t* dict, uint32_t dict_len) {
    zlib_header(dict_len != 0, out[0], out[1]);
    if (!dict_len) return 2;
    const uint32_t a = adler32(dict, dict_len);
    out[2] = a >> 24; out[3] = a >> 16; out[4] = a >> 8; out[5] = a;
    return 6;
}

static void put_adler(uint8_t* t, const uint8_t* data, uint64_t n) {
    const uint32_t a = adler32(data, n);
    t[0] = a >> 24; t[1] = a >> 16; t[2] = a >> 8; t[3] = a;
}

extern "C" int64_t model_compress(const uint8_t* data, uint32_t n, const uint8_t* dict, uint32_t dict_len,
                                  const Params* pr, uint8_t* out, uint64_t cap, uint32_t* stats) {
    Parsed ps;
    parse_block(data, n, dict, dict_len, pr, ps, stats);
    Plan pl;
    plan_block(ps, pl);
    const uint64_t stored_bytes = (uint64_t)n + 5;  // n <= 65535 in the model
    const uint64_t hdr = 2 + (dict_len ? 4 : 0);
    uint64_t best_bits = pl.dyn_bits < pl.fix_bits ? pl.dyn_bits : pl.fix_bits;
    uint64_t body = (best_bits + 7) / 8;
    int mode = pl.dyn_bits < pl.fix_bits ? 2 : 1;
    if (stored_bytes <= body) { mode = 0; body = stored_bytes; }
    uint64_t total = hdr + body + 4;
    if (stats) { stats[0] = (uint32_t)ps.tok.size(); stats[1] = ps.n_match; stats[2] = (uint32_t)mode; stats[3] = pl.h.bits; }
    if (total > cap) return -(int64_t)total;
    memset(out, 0, total);
    zlib_head(out, dict, dict_len);
    if (mode == 0) {
        uint8_t* o = out + hdr;
        o[0] = 1;
        o[1] = n & 0xff; o[2] = n >> 8; o[3] = ~n & 0xff; o[4] = (~n >> 8) & 0xff;
        memcpy(o + 5, data, n);
    } else {
        BitWriter bw;
        bw.buf = out + hdr;
        bw.bitpos = 0;
        write_block(ps, pl, mode, 1, bw);
        bw.finish();
        if ((bw.bitpos + 7) / 8 != body) return -1000000 - (int64_t)bw.bitpos;
    }
    put_adler(out + hdr + body, data, n);
    return (int64_t)total;
}

// Chunks longer than 32 KiB, as hmse_compress strings them together: blocks of LONG_BLOCK input bytes; block 0 searches
// the preset dictionary, block b >= 1 the whole block b - 1 in its place (indexed on positions j + 4 <= LONG_BLOCK,
// matches do not run out of it); every block is parsed with the caller's Params (the kernel: 4 own candidates, whatever
// the block's length) and is fixed or dynamic by exact cost, never stored on its own; BFINAL on the last block only.
// The stream is stored blocks of up to 65535 bytes instead when the coded body is not smaller than theirs, at level 0,
// and for more than LONG_MAX_BLOCKS blocks.  One Adler-32 over the whole chunk.
extern "C" int64_t model_compress_long(const uint8_t* data, uint64_t n, const uint8_t* dict, uint32_t dict_len,
                                       const Params* pr, int level, uint8_t* out, uint64_t cap) {
    const uint64_t nblk = (n + LONG_BLOCK - 1) / LONG_BLOCK;
    const uint64_t hdr = 2 + (dict_len ? 4 : 0);
    const uint64_t n_stored = n / STORED_MAX + 1;   // the last stored block is empty when n % 65535 == 0
    const uint64_t stored_body = n + 5 * n_stored;
    std::vector<Parsed> ps;
    std::vector<Plan> pl;
    uint64_t body = stored_body;
    bool coded = false;
    if (level != 0 && nblk <= LONG_MAX_BLOCKS) {
        ps.resize(nblk);
        pl.resize(nblk);
        uint64_t bits = 0;
        for (uint64_t b = 0; b < nblk; b++) {
            const uint64_t off = b * LONG_BLOCK;
            const uint32_t len = (uint32_t)(n - off < LONG_BLOCK ? n - off : LONG_BLOCK);
            if (b) parse_block(data + off, len, data + off - LONG_BLOCK, LONG_BLOCK, pr, ps[b], nullptr);
            else parse_block(data, len, dict, dict_len, pr, ps[b], nullptr);
            plan_block(ps[b], pl[b]);
            bits += pl[b].dyn_bits < pl[b].fix_bits ? pl[b].dyn_bits : pl[b].fix_bits;
        }
        if ((bits + 7) / 8 < stored_body) {
            body = (bits + 7) / 8;
            coded = true;
        }
    }
    const uint64_t total = hdr + body + 4;
    if (total > cap) return -(int64_t)total;
    memset(out, 0, total);
    zlib_head(out, dict, dict_len);
    uint8_t* o = out + hdr;
    if (coded) {
        BitWriter bw;
        bw.buf = o;
        bw.bitpos = 0;
        for (uint64_t b = 0; b < nblk; b++)
            write_block(ps[b], pl[b], pl[b].dyn_bits < pl[b].fix_bits ? 2 : 1, b + 1 == nblk, bw);
        bw.finish();
        if ((bw.bitpos + 7) / 8 != body) return -1000000 - (int64_t)bw.bitpos;
    } else {
        for (uint64_t b = 0; b < n_stored; b++) {
            const uint64_t off = b * STORED_MAX;
            const uint32_t bl = (uint32_t)(n - off < STORED_MAX ? n - off : STORED_MAX);
            uint8_t* h = o + off + 5 * b;
            h[0] = b + 1 == n_stored;
            h[1] = bl & 0xff; h[2] = bl >> 8; h[3] = ~bl & 0xff; h[4] = (~bl >> 8) & 0xff;
            memcpy(h + 5, data + off, bl);
        }
    }
    put_adler(o + body, data, n);
    return (int64_t)total;
}
