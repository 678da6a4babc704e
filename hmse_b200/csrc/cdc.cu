// cdc.cu - L2 content-defined chunking: FastCDC (Gear hash + normalised chunking), bit-exact
// against the sequential algorithm (spec: README.md:289, 1202-1256, 2434-2514; algorithm per the
// paper the spec cites at README.md:2753-2755; restated in oracle/cdc.py).
//
// K1 gear_scan     reads the stream ONCE.  A 64-bit Gear hash is the sum of the table entries of the trailing 64
//                  bytes, so a thread can start anywhere after a 64-byte warm-up and then roll on for as long
//                  as it likes: a thread owns up to 32 consecutive 128-byte runs of the stream and emits one
//                  MaskS bit and one MaskL bit per byte.  A tile (one run of each of the 256 threads, 32 KB)
//                  arrives by ONE tensor-map TMA copy into a SWIZZLE_128B box, counted on an mbarrier; the
//                  Gear table is replicated sixteen times so that the lookups are bank-conflict free
//                  (gear_scan_tma_kernel; the earlier forms of the kernel stay selectable, see hmse_chunk_scan).
// K2 resolve       sequential FastCDC resets fp at start+min, so next_cut(s) is a pure
//                  function of s: partial-window positions (64 bytes after the skip) are
//                  recomputed with a warp scan, the rest is a find-first-set over the
//                  bitmaps.  Segments of the stream are walked speculatively by one warp
//                  each from a guessed entry; fix-up rounds re-walk from the true entry until
//                  the chain merges with the speculative one (chains converge in a few
//                  chunks); rounds repeat until no segment exit changes.  The same mechanism
//                  stitches byte-range shards across GPUs (hmse_chunk_resolve with `entry`).
#include <cuda.h>   // CUtensorMap types only: the encoder is looked up at run time (cudaGetDriverEntryPoint), no -lcuda
#include <stdlib.h>

#include "ctx.cuh"

namespace {

struct CdcDev {
    uint64_t gear[256];
    uint64_t ms, ml, mc;
    uint32_t mn, av, mx, pad;
};

// ------------------------------------------------------------------------------------------
// K1: gear scan
// ------------------------------------------------------------------------------------------
constexpr int K1_THREADS = 256;
constexpr int K1_RUN = 128;                     // bytes rolled per thread per tile (+64 of warm-up)
constexpr int K1_TILE = K1_THREADS * K1_RUN;    // 32 KiB
constexpr int K1_SLOT = K1_RUN + 16;            // padded slot stride: LDS.128 conflict-free
constexpr int K1_STAGE = (K1_THREADS + 1) * K1_SLOT;  // slot 0 carries the 64-byte halo
// gear_scan_kernel, the tile-at-a-time form (HMSE_SCAN_VARIANT 0-2, and the fallback without a tensor-map encoder): every
// thread rolls ONE 128-byte run of a contiguous 32 KiB tile after re-hashing the 64 bytes before it; the tile is staged by
// one 128-byte bulk copy per thread into slots padded to 144 bytes (LDS.128 conflict free).
// REP > 1 keeps REP copies of the Gear table, one per bank pair (row e = the copies of entry e, lane l reads copy l & 15), so
// that the data-dependent 8-byte lookups of a half-warp never share a bank: with ONE table sixteen random entries fall
// into sixteen bank pairs about three deep, and at five to six shared-memory wavefronts per byte and warp the lookups,
// not the arithmetic, bounded the kernel (measured: see hmse_chunk_scan).
template <int STAGES, int REP>
struct K1Cfg {
    static constexpr int CTAS = (STAGES == 1 || REP == 1) ? 3 : 2;   // resident CTAs per SM (shared memory bounds it)
    static constexpr size_t SMEM = (size_t)STAGES * K1_STAGE + (size_t)REP * 256 * 8 + 64;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// 1-D bulk async copy global -> shared (TMA engine), completion counted on an mbarrier.
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// Gear[byte K of W] for this lane.  REP == 1: one table.  REP == 16: lane l reads copy l & 15, entry e of copy c at
// word 16 e + c, so the 16 lanes of a half-warp hit 16 different bank pairs whatever bytes they hold; the byte is
// pulled out by one PRMT and scaled and added to the lane's base by one IMAD (the fma pipe is idle in this kernel).
template <int REP, int K>
__device__ __forceinline__ uint64_t gear_at(const uint64_t* sg, uint32_t sgl, uint32_t stride, uint32_t W) {
    if constexpr (REP == 1) {
        return sg[K == 3 ? (W >> 24) : ((W >> (8 * K)) & 0xffu)];
    } else {
        uint32_t lo, hi;
        const uint32_t a = __byte_perm(W, 0, 0x4440 + K) * stride + sgl;
        asm("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(lo), "=r"(hi) : "r"(a));
        return ((uint64_t)hi << 32) | lo;
    }
}

#define GEAR_HIT(FP, BITPOS)                                         \
    if (((FP) & mc) == 0) {                                          \
        if (((FP) & ms) == 0) sb |= 1ull << (BITPOS);                \
        if (((FP) & ml) == 0) lb |= 1ull << (BITPOS);                \
    }

#define GEAR_WORD(W, B0)                                             \
    {                                                                \
        const uint64_t f0 = (fp << 1) + gear_at<REP, 0>(sg, sgl, stride, (W));   \
        const uint64_t f1 = (f0 << 1) + gear_at<REP, 1>(sg, sgl, stride, (W));   \
        const uint64_t f2 = (f1 << 1) + gear_at<REP, 2>(sg, sgl, stride, (W));   \
        fp = (f2 << 1) + gear_at<REP, 3>(sg, sgl, stride, (W));      \
        GEAR_HIT(f0, (B0)) GEAR_HIT(f1, (B0) + 1) GEAR_HIT(f2, (B0) + 2) GEAR_HIT(fp, (B0) + 3) \
    }

#define WARM_WORD(W)                                                 \
    fp = (fp << 1) + gear_at<REP, 0>(sg, sgl, stride, (W));          \
    fp = (fp << 1) + gear_at<REP, 1>(sg, sgl, stride, (W));          \
    fp = (fp << 1) + gear_at<REP, 2>(sg, sgl, stride, (W));          \
    fp = (fp << 1) + gear_at<REP, 3>(sg, sgl, stride, (W));

template <int STAGES, int REP>
__global__ void __launch_bounds__(K1_THREADS, (K1Cfg<STAGES, REP>::CTAS))
gear_scan_kernel(const uint8_t* __restrict__ data, uint64_t n, uint64_t n_tiles, const CdcDev* __restrict__ cfg,
                 uint64_t* __restrict__ bitS, uint64_t* __restrict__ bitL, uint32_t stride) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* stage0 = smem;
    uint64_t* sg_all = reinterpret_cast<uint64_t*>(smem + (size_t)STAGES * K1_STAGE);
    uint64_t* bars = sg_all + REP * 256;  // STAGES barriers
    const unsigned t = threadIdx.x;

    {
        const uint64_t g = cfg->gear[t];
#pragma unroll
        for (int c = 0; c < REP; c++) sg_all[t * REP + c] = g;
    }
    // sg[b * REP] = this lane's copy of entry b (its own bank pair when REP == 16)
    const uint64_t* sg = sg_all + (REP > 1 ? (t & (REP - 1)) : 0);
    const uint32_t sgl = smem_u32(sg);   // (stride = 8 * REP bytes between entries: a kernel argument, so that it stays an IMAD)
    const uint64_t ms = cfg->ms, ml = cfg->ml, mc = cfg->mc;
    if (t == 0) {
        for (int s = 0; s < STAGES; s++) mbar_init(&bars[s], K1_THREADS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    const uint64_t n_pad = (n + 15) & ~15ull;  // copies are 16-byte granular (d_data is 16-aligned)

    auto issue = [&](uint64_t tile, int s) {
        uint8_t* st = stage0 + (size_t)s * K1_STAGE;
        const uint64_t tile_base = tile * (uint64_t)K1_TILE;
        const uint64_t pos = tile_base + (uint64_t)t * K1_RUN;
        uint32_t bytes = 0;
        if (pos < n_pad) {
            uint64_t left = n_pad - pos;
            bytes = left < K1_RUN ? (uint32_t)left : (uint32_t)K1_RUN;
        }
        uint32_t halo = (t == 0 && tile_base >= 64) ? 64u : 0u;
        mbar_arrive_tx(&bars[s], bytes + halo);
        if (bytes) bulk_g2s(st + (size_t)(t + 1) * K1_SLOT, data + pos, bytes, &bars[s]);
        if (halo) bulk_g2s(st + (K1_SLOT - 16 - 64), data + tile_base - 64, 64, &bars[s]);
    };

    uint64_t tile = blockIdx.x;
    if (STAGES == 2 && tile < n_tiles) issue(tile, 0);
    for (uint32_t it = 0; tile < n_tiles; it++, tile += gridDim.x) {
        int s = 0;
        if (STAGES == 2) {
            s = it & 1;
            const uint64_t next = tile + gridDim.x;
            if (next < n_tiles) issue(next, s ^ 1);
            mbar_wait(&bars[s], (it >> 1) & 1);
        } else {
            issue(tile, 0);                 // one buffer: the other CTAs of the SM compute while this copy is in flight
            mbar_wait(&bars[0], it & 1);
        }

        const uint8_t* st = stage0 + (size_t)s * K1_STAGE;
        const uint64_t pos = tile * (uint64_t)K1_TILE + (uint64_t)t * K1_RUN;
        uint64_t sw[K1_RUN / 64] = {0, 0}, lw[K1_RUN / 64] = {0, 0};
        static_assert(K1_RUN == 128, "two 64-bit words per mask per thread");
        if (pos < n) {
            uint64_t fp = 0;
            if (pos >= 64) {
                // warm-up: the 64 bytes before the run are the tail of the previous slot
                const uint4* wp = reinterpret_cast<const uint4*>(st + (size_t)t * K1_SLOT + (K1_RUN - 64));
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    uint4 v = wp[q];
                    WARM_WORD(v.x) WARM_WORD(v.y) WARM_WORD(v.z) WARM_WORD(v.w)
                }
            }
            const uint4* rp = reinterpret_cast<const uint4*>(st + (size_t)(t + 1) * K1_SLOT);
#pragma unroll
            for (int w = 0; w < K1_RUN / 64; w++) {
                uint64_t sb = 0, lb = 0;
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    uint4 v = rp[w * 4 + q];
                    GEAR_WORD(v.x, q * 16)
                    GEAR_WORD(v.y, q * 16 + 4)
                    GEAR_WORD(v.z, q * 16 + 8)
                    GEAR_WORD(v.w, q * 16 + 12)
                }
                sw[w] = sb;
                lw[w] = lb;
            }
            // positions >= n (stale bytes in the slot) never become candidates
            const uint64_t left = n - pos;
            if (left < K1_RUN) {
#pragma unroll
                for (int w = 0; w < K1_RUN / 64; w++) {
                    uint64_t keep = left >= 64ull * (w + 1) ? ~0ull : (left <= 64ull * w ? 0ull : ((1ull << (left - 64 * w)) - 1));
                    sw[w] &= keep;
                    lw[w] &= keep;
                }
            }
        }
        // 2 words per mask per thread: lanes are contiguous -> 512 B coalesced per warp
        const uint64_t wbase = pos >> 6;
        uint4* os = reinterpret_cast<uint4*>(bitS + wbase);
        uint4* ol = reinterpret_cast<uint4*>(bitL + wbase);
        os[0] = make_uint4((uint32_t)sw[0], (uint32_t)(sw[0] >> 32), (uint32_t)sw[1], (uint32_t)(sw[1] >> 32));
        ol[0] = make_uint4((uint32_t)lw[0], (uint32_t)(lw[0] >> 32), (uint32_t)lw[1], (uint32_t)(lw[1] >> 32));
        __syncthreads();  // everyone is done reading stage s before it is refilled
    }
}

// The same scan with runs that CONTINUE across tiles (HMSE_SCAN_VARIANT=3 / 4, experimental): a thread owns `tpt`
// consecutive 128-byte runs of the stream (a region of 256 * tpt * 128 bytes per CTA trip) and carries its hash from one
// to the next, so the 64-byte warm-up is paid once per tpt runs instead of once per run (a third of all hashing
// otherwise).  A thread reads only its own bytes, so the slots of a warp are nobody else's business: no __syncthreads in
// the loop.  The warm-up bytes come straight from global memory (four 16-byte loads per region and thread).  Bitmaps
// and cut lists are the same bit for bit: the hash at a position is the sum of the trailing 64 bytes' table entries
// whatever came before.
// Staging.  BULK: one 128-byte bulk-async (TMA) copy per thread and tile, counted on the CTA's mbarrier - ptxas
//   serialises the 32 copies of a warp (UBLKCP takes uniform registers: an ELECT / R2UR / UBLKCP loop of ~8
//   instructions per lane, a sixth of the kernel's instructions).  !BULK: 16-byte cp.async (LDGSTS) copies - the eight
//   lanes of a group fetch ONE lane's 128-byte line per instruction (whole sectors, a conflict-free 128-byte write),
//   eight instructions a tile; completion per warp (wait_group + __syncwarp), and every lane prefetches its next line
//   into L2 while the current one is hashed.
__device__ __forceinline__ void cp_async16(void* dst, const void* src, uint32_t src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(dst)), "l"(src), "r"(src_bytes) : "memory");
}

template <bool BULK>
__global__ void __launch_bounds__(K1_THREADS, 3)
gear_scan_cont_kernel(const uint8_t* __restrict__ data, uint64_t n, uint64_t byte0, uint64_t n_regions, uint32_t tpt, uint64_t words,
                      const CdcDev* __restrict__ cfg, uint64_t* __restrict__ bitS, uint64_t* __restrict__ bitL, uint32_t stride) {
    constexpr int REP = 16;
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* stage0 = smem;
    uint64_t* sg_all = reinterpret_cast<uint64_t*>(smem + (size_t)K1_STAGE);
    uint64_t* bars = sg_all + REP * 256;
    const unsigned t = threadIdx.x, lane = t & 31;
    {
        const uint64_t g = cfg->gear[t];
#pragma unroll
        for (int c = 0; c < REP; c++) sg_all[t * REP + c] = g;
    }
    const uint64_t* sg = sg_all + (t & (REP - 1));
    const uint32_t sgl = smem_u32(sg);
    const uint64_t ms = cfg->ms, ml = cfg->ml, mc = cfg->mc;
    if (BULK && t == 0) {
        mbar_init(&bars[0], K1_THREADS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const uint64_t n_pad = (n + 15) & ~15ull;
    const uint64_t span = (uint64_t)tpt * K1_RUN;   // bytes of one thread per region
    uint8_t* slot = stage0 + (size_t)(t + 1) * K1_SLOT;
    uint32_t it = 0;
    for (uint64_t region = blockIdx.x; region < n_regions; region += gridDim.x) {
        const uint64_t region_base = byte0 + region * (span * K1_THREADS);   // (byte0: the kernel may cover a tail of the stream only)
        const uint64_t my_base = region_base + (uint64_t)t * span;
        uint64_t fp = 0;
        if (my_base >= 64 && my_base < n) {   // the 64 bytes before the first run (my_base is a multiple of 128: aligned)
            const uint4* wp = reinterpret_cast<const uint4*>(data + my_base - 64);
            uint4 wv[4];
#pragma unroll
            for (int q = 0; q < 4; q++) wv[q] = __ldg(wp + q);
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const uint4 v = wv[q];
                WARM_WORD(v.x) WARM_WORD(v.y) WARM_WORD(v.z) WARM_WORD(v.w)
            }
        }
        for (uint32_t i = 0; i < tpt; i++, it++) {
            const uint64_t pos = my_base + (uint64_t)i * K1_RUN;
            if constexpr (BULK) {
                uint32_t bytes = 0;
                if (pos < n_pad) {
                    const uint64_t left = n_pad - pos;
                    bytes = left < K1_RUN ? (uint32_t)left : (uint32_t)K1_RUN;
                }
                // (a thread that is past its wait of trip `it` has seen every thread arrive for it: nobody is a whole
                //  phase ahead, and the slot is read by its owner only)
                mbar_arrive_tx(&bars[0], bytes);
                if (bytes) bulk_g2s(slot, data + pos, bytes, &bars[0]);
                mbar_wait(&bars[0], it & 1);
            } else {
                // lane l = 8 g + c copies 16-byte chunk c of the line of lane 8 g + k, k = 0 .. 7
                const uint32_t c16 = (lane & 7u) * 16u;
                const uint64_t grp_pos = pos - (uint64_t)(lane & 7u) * span + c16;       // chunk c of lane 8 g
                uint8_t* grp_slot = slot - (size_t)(lane & 7u) * K1_SLOT + c16;
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    const uint64_t sp = grp_pos + (uint64_t)k * span;
                    const bool in = sp < n_pad;   // chunks are 16-byte granular and so is n_pad: all or nothing
                    cp_async16(grp_slot + (size_t)k * K1_SLOT, data + (in ? sp : 0), in ? 16u : 0u);
                }
                asm volatile("cp.async.commit_group;" ::: "memory");
                if (i + 1 < tpt && pos + K1_RUN < n_pad) asm volatile("prefetch.global.L2 [%0];" ::"l"(data + pos + K1_RUN));
                asm volatile("cp.async.wait_group 0;" ::: "memory");
                __syncwarp();
            }
            uint64_t sw[2] = {0, 0}, lw[2] = {0, 0};
            if (pos < n) {
                const uint4* rp = reinterpret_cast<const uint4*>(slot);
#pragma unroll
                for (int w = 0; w < 2; w++) {
                    uint64_t sb = 0, lb = 0;
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        const uint4 v = rp[w * 4 + q];
                        GEAR_WORD(v.x, q * 16)
                        GEAR_WORD(v.y, q * 16 + 4)
                        GEAR_WORD(v.z, q * 16 + 8)
                        GEAR_WORD(v.w, q * 16 + 12)
                    }
                    sw[w] = sb;
                    lw[w] = lb;
                }
                const uint64_t left = n - pos;   // positions >= n (stale bytes in the slot) never become candidates
                if (left < K1_RUN) {
#pragma unroll
                    for (int w = 0; w < 2; w++) {
                        const uint64_t keep = left >= 64ull * (w + 1) ? ~0ull : (left <= 64ull * w ? 0ull : ((1ull << (left - 64 * w)) - 1));
                        sw[w] &= keep;
                        lw[w] &= keep;
                    }
                }
            }
            const uint64_t wbase = pos >> 6;   // even: one 16-byte store per mask (a region may end past the bitmaps)
            if (wbase < words) {
                *reinterpret_cast<uint4*>(bitS + wbase) = make_uint4((uint32_t)sw[0], (uint32_t)(sw[0] >> 32), (uint32_t)sw[1], (uint32_t)(sw[1] >> 32));
                *reinterpret_cast<uint4*>(bitL + wbase) = make_uint4((uint32_t)lw[0], (uint32_t)(lw[0] >> 32), (uint32_t)lw[1], (uint32_t)(lw[1] >> 32));
            }
            if constexpr (!BULK) __syncwarp();   // the slots of this warp are refilled by its other lanes
        }
    }
}

// HMSE_SCAN_VARIANT=5 (experimental): the continuing runs staged by ONE tensor-map TMA copy per tile and CTA.  The
// stream is described to the TMA unit as a 3-D tensor {byte in a thread's span, thread (256), region}; tile i of a
// region is the box {128 bytes, 256 threads, 1} at {128 i, 0, region}: 256 rows of 128 bytes, one per thread, 32 KB,
// fetched by a single cp.async.bulk.tensor issued by one thread - no per-thread copies, no staging instructions at all.
// SWIZZLE_128B lays the box out densely and XORs the 16-byte chunk index with the row index (mod 8), so that the eight
// lanes of a quarter-warp, which read the same chunk of eight consecutive rows, hit eight different bank groups.
// Only whole regions go through this kernel; the tail of the stream is scanned by gear_scan_cont_kernel from byte0.
__global__ void __launch_bounds__(K1_THREADS, 3)
gear_scan_tma_kernel(const __grid_constant__ CUtensorMap tmap, const uint8_t* __restrict__ data, uint64_t n_regions, uint32_t tpt,
                     const CdcDev* __restrict__ cfg, uint64_t* __restrict__ bitS, uint64_t* __restrict__ bitL, uint32_t stride) {
    constexpr int REP = 16;
    extern __shared__ __align__(128) uint8_t smem_raw[];
    // the swizzled box needs a 1024-byte aligned home (the launch asks for 1 KB more than the layout needs)
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* stage = smem;                                                  // 256 rows x 128 bytes
    uint64_t* sg_all = reinterpret_cast<uint64_t*>(smem + K1_TILE);         // 32 KB table
    uint64_t* bar = sg_all + REP * 256;
    const unsigned t = threadIdx.x;
    {
        const uint64_t g = cfg->gear[t];
#pragma unroll
        for (int c = 0; c < REP; c++) sg_all[t * REP + c] = g;
    }
    const uint64_t* sg = sg_all + (t & (REP - 1));
    const uint32_t sgl = smem_u32(sg);
    const uint64_t ms = cfg->ms, ml = cfg->ml, mc = cfg->mc;
    if (t == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const uint64_t span = (uint64_t)tpt * K1_RUN;
    // row t, chunk q of the box lives at t * 128 + ((q ^ (t & 7)) << 4)
    const uint8_t* row = stage + (((size_t)t * 128u) ^ ((t & 7u) << 4));
    uint32_t it = 0;
    for (uint64_t region = blockIdx.x; region < n_regions; region += gridDim.x) {
        const uint64_t my_base = region * (span * K1_THREADS) + (uint64_t)t * span;
        uint64_t fp = 0;
        if (my_base >= 64) {
            const uint4* wp = reinterpret_cast<const uint4*>(data + my_base - 64);
            uint4 wv[4];
#pragma unroll
            for (int q = 0; q < 4; q++) wv[q] = __ldg(wp + q);
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const uint4 v = wv[q];
                WARM_WORD(v.x) WARM_WORD(v.y) WARM_WORD(v.z) WARM_WORD(v.w)
            }
        }
        for (uint32_t i = 0; i < tpt; i++, it++) {
            if (t == 0) {
                mbar_arrive_tx(bar, (uint32_t)K1_TILE);
                asm volatile(
                    "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
                        smem_u32(stage)),
                    "l"(&tmap), "r"((int)(i * K1_RUN)), "r"(0), "r"((int)region), "r"(smem_u32(bar))
                    : "memory");
            }
            mbar_wait(bar, it & 1);
            uint64_t sw[2], lw[2];
#pragma unroll
            for (int w = 0; w < 2; w++) {
                uint64_t sb = 0, lb = 0;
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    const uint4 v = *reinterpret_cast<const uint4*>(reinterpret_cast<uintptr_t>(row) ^ (uintptr_t)((w * 4 + q) << 4));
                    GEAR_WORD(v.x, q * 16)
                    GEAR_WORD(v.y, q * 16 + 4)
                    GEAR_WORD(v.z, q * 16 + 8)
                    GEAR_WORD(v.w, q * 16 + 12)
                }
                sw[w] = sb;
                lw[w] = lb;
            }
            const uint64_t wbase = (my_base + (uint64_t)i * K1_RUN) >> 6;
            *reinterpret_cast<uint4*>(bitS + wbase) = make_uint4((uint32_t)sw[0], (uint32_t)(sw[0] >> 32), (uint32_t)sw[1], (uint32_t)(sw[1] >> 32));
            *reinterpret_cast<uint4*>(bitL + wbase) = make_uint4((uint32_t)lw[0], (uint32_t)(lw[0] >> 32), (uint32_t)lw[1], (uint32_t)(lw[1] >> 32));
            __syncthreads();   // every row has been read: the next box may land
        }
    }
}

typedef CUresult (*TmapEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
TmapEncodeFn tmap_encoder() {
    static TmapEncodeFn fn = nullptr;
    static bool looked = false;
    if (!looked) {
        looked = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = (TmapEncodeFn)p;
    }
    return fn;
}

// ------------------------------------------------------------------------------------------
// K2: resolve
// ------------------------------------------------------------------------------------------
// The resolve walks a table of segments.  A segment owns the chunk starts in [start, end) and never cuts past file_end.
// A head segment knows its entry (segment 0: ResolveArgs::entry, any other head: its start, the first byte of a file);
// every other segment speculates from its start and is fixed up from its predecessor's exit.  The single stream
// (hmse_chunk_resolve) is one file whose only head is segment 0; hmse_chunk_files makes one head per non-empty file.
// A cut decision for a chunk starting at s reads no byte before s (the bitmaps only from s + min_size + 64 on, and a bit
// depends on the 64 bytes ending at its position), so one scan of the whole buffer serves every file in it.
struct SegDesc {
    uint64_t start;     // cuts are stored relative to it
    uint64_t end;       // chunk starts >= end belong to the next segment
    uint64_t file_end;  // end of the bytes the chain may use (file end, or the available bytes of a shard)
    uint64_t list;      // first entry of its spec / pre lists
    uint32_t cap;       // entries of each list
    uint32_t head;
};
// Starts in [start, end) lie at least min_size apart, so a segment holds at most end/mn - start/mn + 1 of them.  A file
// table gives segment k cap = end/mn - start/mn + 2 entries at list = start/mn + 2 k (consecutive lists never overlap,
// the total is n/mn + 2 n_seg: scratch follows the bytes, not the file count); the implicit table of one stream gives
// every segment seg_len/mn + 2 entries at k (seg_len/mn + 2).

struct SegMeta {
    uint64_t spec_entry;  // start the speculative chain was walked from
    uint64_t cur_entry;   // start the current (pre + spec tail) list is valid for
    uint64_t spec_exit;   // first chunk start >= seg_end on the speculative chain
    uint64_t exit[2];     // double-buffered exit of the current list
    uint32_t spec_cnt, pre_cnt, spec_skip, pad;
};

struct ResolveArgs {
    const uint8_t* data;
    const uint64_t* bitS;
    const uint64_t* bitL;
    const CdcDev* cfg;
    const SegDesc* seg;   // the file table (kernels <true>); the <false> kernels use the implicit table of one stream
    uint64_t n_seg;
    uint64_t seg_len, n_own, n_avail, stride;   // (the implicit table)
    uint32_t* spec;   // speculative cut lists, relative to the segment start, at seg[k].list
    uint32_t* pre;    // fix-up cut lists, same layout
    SegMeta* meta;
    uint64_t entry;   // where the chain of segment 0 starts
};

__device__ __forceinline__ uint64_t find_first(const uint64_t* __restrict__ bits, uint64_t lo, uint64_t hi,
                                               unsigned lane) {
    const uint64_t w0 = lo >> 6, w1 = (hi - 1) >> 6;
    for (uint64_t wb = w0; wb <= w1; wb += 32) {
        const uint64_t w = wb + lane;
        uint64_t v = w <= w1 ? __ldg(bits + w) : 0ull;
        if (w == w0) v &= ~0ull << (lo & 63);
        if (w == w1) {
            unsigned r = (unsigned)((hi - 1) & 63);
            if (r != 63) v &= (1ull << (r + 1)) - 1;
        }
        unsigned b = __ballot_sync(0xffffffffu, v != 0);
        if (b) {
            int src = __ffs(b) - 1;
            uint64_t vv = __shfl_sync(0xffffffffu, v, src);
            return ((wb + src) << 6) + (uint64_t)(__ffsll((long long)vv) - 1);
        }
    }
    return ~0ull;
}

// One application of FastCDC Algorithm 1 to the chunk starting at s of a stream that ends at fe (warp-cooperative,
// all lanes return the same value).  sg = gear table in shared memory.
__device__ __forceinline__ uint64_t next_cut_warp(const ResolveArgs& a, const uint64_t* sg, uint64_t ms, uint64_t ml,
                                                  uint32_t mn, uint32_t av, uint32_t mx, uint64_t fe, uint64_t s, unsigned lane) {
    const uint64_t rem = fe - s;
    if (rem <= mn) return fe;
    const uint64_t end = s + (rem < mx ? rem : (uint64_t)mx);
    const uint64_t normal = s + ((end - s) < av ? (end - s) : (uint64_t)av);
    const uint64_t base = s + mn;
    // (1) the 64 positions after the skip see a partial window (fp was reset to 0 at base)
    const uint64_t q0 = base + lane, q1 = q0 + 32;
    uint64_t f0 = q0 < end ? sg[a.data[q0]] : 0ull;
    uint64_t f1 = q1 < end ? sg[a.data[q1]] : 0ull;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint64_t t0 = __shfl_up_sync(0xffffffffu, f0, o);
        uint64_t t1 = __shfl_up_sync(0xffffffffu, f1, o);
        if (lane >= (unsigned)o) {
            f0 += t0 << o;
            f1 += t1 << o;
        }
    }
    const uint64_t tot0 = __shfl_sync(0xffffffffu, f0, 31);
    f1 += tot0 << (lane + 1);
    bool h0 = q0 < end && (f0 & (q0 < normal ? ms : ml)) == 0;
    bool h1 = q1 < end && (f1 & (q1 < normal ? ms : ml)) == 0;
    unsigned b0 = __ballot_sync(0xffffffffu, h0);
    if (b0) return base + (uint64_t)(__ffs(b0) - 1);
    unsigned b1 = __ballot_sync(0xffffffffu, h1);
    if (b1) return base + 32 + (uint64_t)(__ffs(b1) - 1);
    // (2) full-window positions: first MaskS candidate before `normal`, else first MaskL before `end`
    const uint64_t lo = base + 64;
    if (lo < normal) {
        uint64_t c = find_first(a.bitS, lo, normal, lane);
        if (c != ~0ull) return c;
    }
    const uint64_t lo2 = lo > normal ? lo : normal;
    if (lo2 < end) {
        uint64_t c = find_first(a.bitL, lo2, end, lane);
        if (c != ~0ull) return c;
    }
    return end;
}

constexpr int K2_THREADS = 128;

// Segment k.  TABLE: the file table.  Otherwise the implicit table of one stream, from the kernel parameters (no table
// load, no registers for the bounds): segments of seg_len bytes over [0, n_own), every chain may read up to n_avail,
// segment 0 is the only head.
template <bool TABLE>
__device__ __forceinline__ SegDesc seg_at(const ResolveArgs& a, uint64_t k) {
    if constexpr (TABLE) return a.seg[k];
    SegDesc g;
    g.start = k * a.seg_len;
    g.end = g.start + a.seg_len < a.n_own ? g.start + a.seg_len : a.n_own;
    g.file_end = a.n_avail;
    g.list = k * a.stride;
    g.cap = (uint32_t)a.stride;
    g.head = k == 0;
    return g;
}

__device__ __forceinline__ void load_gear(uint64_t* sg, const CdcDev* cfg) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) sg[i] = cfg->gear[i];
    __syncthreads();
}

template <bool TABLE>
__global__ void __launch_bounds__(K2_THREADS) resolve_spec_kernel(ResolveArgs a) {
    __shared__ uint64_t sg[256];
    load_gear(sg, a.cfg);
    const unsigned lane = threadIdx.x & 31;
    const uint64_t k = (uint64_t)blockIdx.x * (K2_THREADS / 32) + (threadIdx.x >> 5);
    if (k >= a.n_seg) return;
    const SegDesc g = seg_at<TABLE>(a, k);
    uint64_t s = k == 0 ? a.entry : g.start;
    const uint64_t ms = a.cfg->ms, ml = a.cfg->ml;
    const uint32_t mn = a.cfg->mn, av = a.cfg->av, mx = a.cfg->mx;
    const uint32_t cap = g.cap;
    uint32_t* spec = a.spec + g.list;
    const uint64_t s0 = s;
    uint32_t cnt = 0;
    while (s < g.end) {
        uint64_t c = next_cut_warp(a, sg, ms, ml, mn, av, mx, g.file_end, s, lane);
        if (lane == 0 && cnt < cap) spec[cnt] = (uint32_t)(c - g.start);
        cnt++;
        s = c;
    }
    if (lane == 0) {
        SegMeta m;
        m.spec_entry = s0;
        m.cur_entry = s0;
        m.spec_exit = s;
        m.exit[0] = s;
        m.exit[1] = s;
        m.spec_cnt = cnt;
        m.pre_cnt = 0;
        m.spec_skip = 0;
        m.pad = 0;
        a.meta[k] = m;
    }
}

// One fix-up round: a continuation segment re-enters at its predecessor's exit[in] (a head at its own entry) and walks
// until its chain merges with the speculative chain or leaves the segment.
template <bool TABLE>
__global__ void __launch_bounds__(K2_THREADS) resolve_fix_kernel(ResolveArgs a, int in, uint32_t* changed) {
    __shared__ uint64_t sg[256];
    load_gear(sg, a.cfg);
    const unsigned lane = threadIdx.x & 31;
    const uint64_t k = (uint64_t)blockIdx.x * (K2_THREADS / 32) + (threadIdx.x >> 5);
    if (k >= a.n_seg) return;
    const int out = in ^ 1;
    SegMeta* m = a.meta + k;
    const SegDesc g = seg_at<TABLE>(a, k);
    const uint64_t e = g.head ? (k == 0 ? a.entry : g.start) : a.meta[k - 1].exit[in];
    const uint64_t old_exit = m->exit[in];
    if (e == m->cur_entry) {
        if (lane == 0) m->exit[out] = old_exit;
        return;
    }
    const uint64_t ms = a.cfg->ms, ml = a.cfg->ml;
    const uint32_t mn = a.cfg->mn, av = a.cfg->av, mx = a.cfg->mx;
    const uint32_t cap = g.cap;
    const uint32_t* spec = a.spec + g.list;
    uint32_t* pre = a.pre + g.list;
    const uint64_t spec_entry = m->spec_entry;
    const uint32_t spec_cnt = m->spec_cnt;
    uint64_t s = e;
    uint32_t pc = 0, si = 0;
    bool merged = false;
    // chunk starts on the speculative chain: start(0) = spec_entry, start(i) = seg_start + spec[i-1]
    uint64_t sstart = spec_entry;
    while (s < g.end) {
        while (si < spec_cnt && sstart < s) {
            sstart = g.start + spec[si];
            si++;
        }
        // si == number of spec cuts consumed; sstart is start(si) when si < spec_cnt or the spec exit
        if (sstart == s && si < spec_cnt) {
            merged = true;
            break;
        }
        uint64_t c = next_cut_warp(a, sg, ms, ml, mn, av, mx, g.file_end, s, lane);
        if (lane == 0 && pc < cap) pre[pc] = (uint32_t)(c - g.start);
        pc++;
        s = c;
    }
    const uint64_t new_exit = merged ? m->spec_exit : s;
    __syncwarp();
    if (lane == 0) {
        m->cur_entry = e;
        m->pre_cnt = pc;
        m->spec_skip = merged ? si : spec_cnt;
        m->exit[out] = new_exit;
        if (new_exit != old_exit) atomicOr(changed, 1u);
    }
}

__global__ void seg_counts_kernel(const SegMeta* __restrict__ meta, uint64_t n_seg, uint64_t* __restrict__ counts) {
    uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n_seg) counts[k] = (uint64_t)meta[k].pre_cnt + meta[k].spec_cnt - meta[k].spec_skip;
}

template <bool TABLE>
__global__ void __launch_bounds__(K2_THREADS)
seg_gather_kernel(ResolveArgs a, const uint64_t* __restrict__ offs, uint64_t cap, uint64_t* __restrict__ cuts) {
    const unsigned lane = threadIdx.x & 31;
    const uint64_t k = (uint64_t)blockIdx.x * (K2_THREADS / 32) + (threadIdx.x >> 5);
    if (k >= a.n_seg) return;
    const SegMeta m = a.meta[k];
    const SegDesc g = seg_at<TABLE>(a, k);
    const uint64_t seg_start = g.start, list = g.list;
    const uint32_t* spec = a.spec + list;
    const uint32_t* pre = a.pre + list;
    const uint64_t o = offs[k];
    const uint32_t cnt = m.pre_cnt + m.spec_cnt - m.spec_skip;
    for (uint32_t i = lane; i < cnt; i += 32) {
        uint32_t rel = i < m.pre_cnt ? pre[i] : spec[m.spec_skip + (i - m.pre_cnt)];
        if (o + i < cap) cuts[o + i] = seg_start + rel;
    }
}

// File table, step 1 (one thread per offset i <= n_files): off[0] == 0, off never decreases, off[n_files] == n; nseg[f] =
// segments of file f (0 for an empty file, and for any file whose offsets are bad: *bad is then set).
__global__ void file_count_kernel(const uint64_t* __restrict__ off, uint64_t n_files, uint64_t n, uint64_t seg_len,
                                  uint64_t* __restrict__ nseg, uint32_t* __restrict__ bad) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n_files) return;
    const uint64_t hi = off[i];
    const uint64_t lo = i ? off[i - 1] : 0;
    const bool ok = hi <= n && lo <= hi && (i || hi == 0) && (i < n_files || hi == n);
    if (!ok) atomicOr(bad, 1u);
    if (i) nseg[i - 1] = ok ? (hi - lo + seg_len - 1) / seg_len : 0;
}

// File table, step 2 (one thread per segment): first[f] = index of file f's first segment (exclusive scan of nseg), so
// segment k belongs to the last file f with first[f] <= k (files before it with the same first[] are empty).
__global__ void file_table_kernel(const uint64_t* __restrict__ off, const uint64_t* __restrict__ first, uint64_t n_files,
                                  uint64_t n_seg, uint64_t seg_len, uint32_t mn, SegDesc* __restrict__ seg) {
    const uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_seg) return;
    uint64_t lo = 0, hi = n_files - 1;   // invariant: first[lo] <= k (first[0] == 0), answer in [lo, hi]
    while (lo < hi) {
        const uint64_t mid = lo + (hi - lo + 1) / 2;
        if (__ldg(first + mid) <= k) lo = mid;
        else hi = mid - 1;
    }
    const uint64_t j = k - first[lo];
    const uint64_t fe = off[lo + 1];
    SegDesc g;
    g.start = off[lo] + j * seg_len;
    g.end = g.start + seg_len < fe ? g.start + seg_len : fe;
    g.file_end = fe;
    g.list = g.start / mn + 2 * k;
    g.cap = (uint32_t)(g.end / mn - g.start / mn + 2);
    g.head = j == 0;
    seg[k] = g;
}

// file_chunk[f] = index of file f's first chunk = chunk offset of its head segment; an empty file shares the index of
// the next non-empty one (or the total); file_chunk[n_files] = total.
__global__ void file_chunk_kernel(const uint64_t* __restrict__ first, const uint64_t* __restrict__ offs, uint64_t n_files,
                                  uint64_t n_seg, const uint64_t* __restrict__ total, uint64_t* __restrict__ file_chunk) {
    const uint64_t f = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f > n_files) return;
    const uint64_t s = f < n_files ? first[f] : n_seg;
    file_chunk[f] = s < n_seg ? offs[s] : (n_seg ? *total : 0);
}

// Bytes per resolve segment: a warp walks at most this many bytes before a fix-up round.
uint64_t resolve_seg_len(const hmse_cdc_cfg& c) {
    const uint64_t len = 8ull * c.max_size;
    return len < (256u << 10) ? (256u << 10) : len;
}

// Scratch of a resolve over n_seg segments whose last one ends at last_end: lists in SLOT_CDC_SEG, and in SLOT_CDC_META
// [SegMeta n_seg][SegDesc n_seg][counts u64 n_seg][offs u64 n_seg][tail: changed flag u32, total u64, ...].
struct ResolveScratch {
    ResolveArgs a;
    SegDesc* seg;
    uint64_t *counts, *offs, *tail;
};

int resolve_scratch(hmse_ctx* ctx, uint64_t n_seg, uint64_t last_end, const uint8_t* d_data, uint64_t n_avail,
                    uint64_t entry, bool file_table, ResolveScratch* r) {
    const uint64_t mn = ctx->cdc_cfg.min_size, stride = resolve_seg_len(ctx->cdc_cfg) / mn + 2;
    const uint64_t list_entries = file_table ? last_end / mn + 2 * n_seg : n_seg * stride;
    HMSE_SCRATCH(ctx, lists, uint32_t*, SLOT_CDC_SEG, 2 * list_entries * sizeof(uint32_t));
    const size_t meta_bytes = n_seg * (sizeof(SegMeta) + sizeof(SegDesc)) + 2 * n_seg * sizeof(uint64_t) + 64;
    HMSE_SCRATCH(ctx, meta_raw, uint8_t*, SLOT_CDC_META, meta_bytes);
    const uint64_t n_tiles = div_up64(n_avail, K1_TILE);
    const uint64_t words = (n_tiles ? n_tiles : 1) * (K1_TILE / 64);
    ResolveArgs& a = r->a;
    a.data = d_data;
    a.bitS = (const uint64_t*)ctx->slot[SLOT_CDC_BITS];
    a.bitL = a.bitS + words;
    a.cfg = (const CdcDev*)ctx->slot[SLOT_CDC_CFG];
    a.meta = (SegMeta*)meta_raw;
    r->seg = (SegDesc*)(meta_raw + n_seg * sizeof(SegMeta));
    a.seg = file_table ? r->seg : nullptr;
    a.n_seg = n_seg;
    a.seg_len = resolve_seg_len(ctx->cdc_cfg);
    a.n_own = last_end;
    a.n_avail = n_avail;
    a.stride = stride;
    a.spec = lists;
    a.pre = lists + list_entries;
    a.entry = entry;
    r->counts = (uint64_t*)(meta_raw + n_seg * (sizeof(SegMeta) + sizeof(SegDesc)));
    r->offs = r->counts + n_seg;
    r->tail = r->offs + n_seg;
    return HMSE_OK;
}

// Speculative walk (fresh) or the exits of the previous call, fix-up rounds until no exit changes (one host round trip
// each), then counts, their scan (total in tail[1]) and the gather into d_cuts[cap].  Leaves the round count and the
// parity of the final exits in ctx->cdc_rounds; *in_out = that parity.
int resolve_run(hmse_ctx* ctx, const ResolveScratch& r, bool fresh, uint64_t* d_cuts, uint64_t cap, int* in_out,
                cudaStream_t st) {
    const ResolveArgs& a = r.a;
    const unsigned wgrid = (unsigned)div_up64(a.n_seg, K2_THREADS / 32);
    int in = 0;
    int rounds = 0;
    if (fresh) {
        KL(ctx);
        if (a.seg) resolve_spec_kernel<true><<<wgrid, K2_THREADS, 0, st>>>(a);
        else resolve_spec_kernel<false><<<wgrid, K2_THREADS, 0, st>>>(a);
        HMSE_LAUNCH_CHECK(ctx);
    } else {
        in = ctx->cdc_rounds & 1;  // parity the previous call's final exits live in
    }
    volatile uint64_t* mail = ctx->pinned;
    for (;;) {
        HMSE_CUDA(ctx, cudaMemsetAsync(r.tail, 0, 8, st));
        KL(ctx);
        if (a.seg) resolve_fix_kernel<true><<<wgrid, K2_THREADS, 0, st>>>(a, in, (uint32_t*)r.tail);
        else resolve_fix_kernel<false><<<wgrid, K2_THREADS, 0, st>>>(a, in, (uint32_t*)r.tail);
        HMSE_LAUNCH_CHECK(ctx);
        if (int mrc = hmse_mail(ctx, 0, r.tail, 2, st)) return mrc;
        HMSE_CUDA(ctx, cudaStreamSynchronize(st));
        in ^= 1;
        rounds++;
        if ((uint32_t)mail[0] == 0) break;
        if ((uint64_t)rounds > a.n_seg + 2) HMSE_FAIL(ctx, HMSE_E_CUDA, "resolve did not converge");
    }
    ctx->cdc_rounds = (rounds << 1) | in;  // low bit: parity the final exits live in
    *in_out = in;

    KL(ctx);
    seg_counts_kernel<<<(unsigned)div_up64(a.n_seg, 256), 256, 0, st>>>(a.meta, a.n_seg, r.counts);
    HMSE_LAUNCH_CHECK(ctx);
    int rc = hmse_exclusive_scan_u64(ctx, r.counts, r.offs, a.n_seg, r.tail + 1, st);
    if (rc) return rc;
    if (d_cuts && cap) {
        KL(ctx);
        if (a.seg) seg_gather_kernel<true><<<wgrid, K2_THREADS, 0, st>>>(a, r.offs, cap, d_cuts);
        else seg_gather_kernel<false><<<wgrid, K2_THREADS, 0, st>>>(a, r.offs, cap, d_cuts);
        HMSE_LAUNCH_CHECK(ctx);
    }
    return HMSE_OK;
}

int upload_cfg(hmse_ctx* ctx, const hmse_cdc_cfg* cfg, cudaStream_t st) {
    if (!cfg) HMSE_FAIL(ctx, HMSE_E_INVAL, "cdc cfg is null");
    if (!(cfg->min_size >= 64 && cfg->min_size <= cfg->avg_size && cfg->avg_size <= cfg->max_size &&
          cfg->max_size <= (1u << 20)))
        HMSE_FAIL(ctx, HMSE_E_INVAL, "need 64 <= min <= avg <= max <= 1 MiB");
    if (cfg->mask_s == 0 || cfg->mask_l == 0) HMSE_FAIL(ctx, HMSE_E_INVAL, "masks must be non-zero");
    HMSE_SCRATCH(ctx, dev, CdcDev*, SLOT_CDC_CFG, sizeof(CdcDev));
    if (ctx->cdc_cfg_valid && memcmp(&ctx->cdc_cfg, cfg, sizeof(*cfg)) == 0) return HMSE_OK;
    CdcDev* h = reinterpret_cast<CdcDev*>(ctx->pinned);  // 2096 bytes < 4 KiB mailbox
    HMSE_CUDA(ctx, cudaStreamSynchronize(st));           // mailbox may still be in flight
    memcpy(h->gear, cfg->gear, sizeof(h->gear));
    h->ms = cfg->mask_s;
    h->ml = cfg->mask_l;
    h->mc = cfg->mask_s & cfg->mask_l;
    h->mn = cfg->min_size;
    h->av = cfg->avg_size;
    h->mx = cfg->max_size;
    h->pad = 0;
    HMSE_CUDA(ctx, cudaMemcpyAsync(dev, h, sizeof(CdcDev), cudaMemcpyHostToDevice, st));
    HMSE_CUDA(ctx, cudaStreamSynchronize(st));
    ctx->cdc_cfg = *cfg;
    ctx->cdc_cfg_valid = 1;
    ctx->cdc_have_scan = 0;
    ctx->res_valid = 0;
    return HMSE_OK;
}

}  // namespace

HMSE_API int hmse_chunk_scan(hmse_ctx* ctx, const uint8_t* d_data, uint64_t n_avail, const hmse_cdc_cfg* cfg,
                               void* stream) {
    if (!ctx) return HMSE_E_INVAL;
    cudaStream_t st = (cudaStream_t)stream;
    if (n_avail && !d_data) HMSE_FAIL(ctx, HMSE_E_INVAL, "d_data is null");
    if ((uintptr_t)d_data & 15) HMSE_FAIL(ctx, HMSE_E_INVAL, "d_data must be 16-byte aligned");
    int rc = upload_cfg(ctx, cfg, st);
    if (rc) return rc;
    ctx->cdc_have_scan = 0;
    ctx->res_valid = 0;
    ctx->cdc_n_avail = n_avail;
    const uint64_t n_tiles = div_up64(n_avail, K1_TILE);
    const uint64_t words = (n_tiles ? n_tiles : 1) * (K1_TILE / 64);
    HMSE_SCRATCH(ctx, bits, uint64_t*, SLOT_CDC_BITS, 2 * words * sizeof(uint64_t));
    if (n_tiles) {
        // variant 5 (default): gear_scan_tma_kernel - runs that continue across tiles, staged by one tensor-map TMA copy
        // per tile and CTA into a hardware-swizzled box - plus gear_scan_cont_kernel for the tail of the stream.
        // HMSE_SCAN_VARIANT (read at every call) selects the measured alternatives, all bit-equal (tools/scan_check.py,
        // tools/scan_variants.py; B200, 4 GB of text, profiles/r02P_*, r02Q_*, r02R_scan_check.txt):
        //   5  continuing runs, tensor-map TMA                                         1834 GB/s  (10 GB: 1899)
        //   4  continuing runs, 16-byte cp.async copies (eight lanes per line)         1711
        //   3  continuing runs, one bulk copy per thread (32 serialised UBLKCPs a warp) 1549
        //   1  a warm-up per tile, one bulk copy per thread, 16-fold table, 3 CTAs     1410  (the fallback when the driver
        //      has no cuTensorMapEncodeTiled)
        //   2  as 1 with two staging buffers, 2 CTAs                                   1233
        //   0  as 2 with ONE table (the round-1 kernel), 3 CTAs                         1212
        // Measured on top of 1 and dropped: one branch per four positions (1310: it trades branches for ALU-pipe work) and
        // the hash update on the fma pipe (mad.wide + mad: 1269, ptxas splits the 64-bit addend off again).
        const char* ve = getenv("HMSE_SCAN_VARIANT");
        int variant = ve ? atoi(ve) : 5;
        if (variant < 0 || variant > 5) variant = 5;
        if (variant == 5 && !tmap_encoder()) variant = 1;
        const CdcDev* dc = (const CdcDev*)ctx->slot[SLOT_CDC_CFG];
        HT_BEGIN(ctx, HT_SCAN, st);
        KL(ctx);
#define K1_LAUNCH(ST, RP)                                                                                                     \
    {                                                                                                                         \
        HMSE_CUDA(ctx, cudaFuncSetAttribute(gear_scan_kernel<ST, RP>, cudaFuncAttributeMaxDynamicSharedMemorySize,             \
                                            (int)K1Cfg<ST, RP>::SMEM));                                                       \
        const uint64_t resident = (uint64_t)ctx->sm_count * K1Cfg<ST, RP>::CTAS;                                              \
        const uint64_t grid = n_tiles < resident ? n_tiles : resident;                                                        \
        gear_scan_kernel<ST, RP><<<(unsigned)grid, K1_THREADS, K1Cfg<ST, RP>::SMEM, st>>>(d_data, n_avail, n_tiles, dc, bits, \
                                                                                          bits + words, 8u * RP);                      \
    }
        if (variant == 0) K1_LAUNCH(2, 1)
        else if (variant == 2) K1_LAUNCH(2, 16)
        else if (variant == 3 || variant == 4) {
            // runs of up to 32 tiles per thread, as long as every resident CTA still gets four regions or more
            const uint64_t resident = (uint64_t)ctx->sm_count * 3;
            uint32_t tpt = 32;
            while (tpt > 1 && div_up64(n_avail, (uint64_t)tpt * K1_TILE) < 4 * resident) tpt >>= 1;
            const uint64_t n_regions = div_up64(n_avail, (uint64_t)tpt * K1_TILE);
            const unsigned grid = (unsigned)(n_regions < resident ? n_regions : resident);
            if (variant == 3) {
                HMSE_CUDA(ctx, cudaFuncSetAttribute(gear_scan_cont_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                    (int)K1Cfg<1, 16>::SMEM));
                gear_scan_cont_kernel<true><<<grid, K1_THREADS, K1Cfg<1, 16>::SMEM, st>>>(d_data, n_avail, 0, n_regions, tpt, words, dc,
                                                                                           bits, bits + words, 8u * 16);
            } else {
                HMSE_CUDA(ctx, cudaFuncSetAttribute(gear_scan_cont_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                    (int)K1Cfg<1, 16>::SMEM));
                gear_scan_cont_kernel<false><<<grid, K1_THREADS, K1Cfg<1, 16>::SMEM, st>>>(d_data, n_avail, 0, n_regions, tpt, words, dc,
                                                                                            bits, bits + words, 8u * 16);
            }
        } else if (variant == 5) {
            const uint64_t resident = (uint64_t)ctx->sm_count * 3;
            uint32_t tpt = 32;
            while (tpt > 1 && n_avail / ((uint64_t)tpt * K1_TILE) < 4 * resident) tpt >>= 1;
            const uint64_t region_bytes = (uint64_t)tpt * K1_TILE, span = (uint64_t)tpt * K1_RUN;
            const uint64_t n_full = n_avail / region_bytes;   // whole regions: every byte the TMA touches lies inside the buffer
            TmapEncodeFn enc = tmap_encoder();
            if (n_full) {
                CUtensorMap tm;
                const cuuint64_t gdim[3] = {span, (cuuint64_t)K1_THREADS, n_full};
                const cuuint64_t gstr[2] = {span, span * K1_THREADS};
                const cuuint32_t box[3] = {(cuuint32_t)K1_RUN, (cuuint32_t)K1_THREADS, 1};
                const cuuint32_t estr[3] = {1, 1, 1};
                const CUresult r = enc(&tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, (void*)d_data, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                       CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
                if (r != CUDA_SUCCESS) HMSE_FAIL(ctx, HMSE_E_CUDA, "cuTensorMapEncodeTiled failed: %d", (int)r);
                const int sm5 = K1_TILE + 16 * 256 * 8 + 64 + 1024;
                HMSE_CUDA(ctx, cudaFuncSetAttribute(gear_scan_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, sm5));
                gear_scan_tma_kernel<<<(unsigned)(n_full < resident ? n_full : resident), K1_THREADS, sm5, st>>>(tm, d_data, n_full, tpt, dc, bits,
                                                                                                              bits + words, 8u * 16);
            }
            const uint64_t byte0 = n_full * region_bytes;
            if (byte0 < n_avail) {
                if (n_full) KL(ctx);
                const uint64_t n_tail = div_up64(n_avail - byte0, K1_TILE);
                HMSE_CUDA(ctx, cudaFuncSetAttribute(gear_scan_cont_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                    (int)K1Cfg<1, 16>::SMEM));
                gear_scan_cont_kernel<true><<<(unsigned)(n_tail < resident ? n_tail : resident), K1_THREADS, K1Cfg<1, 16>::SMEM, st>>>(
                    d_data, n_avail, byte0, n_tail, 1, words, dc, bits, bits + words, 8u * 16);
            }
        } else K1_LAUNCH(1, 16)
#undef K1_LAUNCH
        HMSE_LAUNCH_CHECK(ctx);
        HT_END(ctx, HT_SCAN, st);
    }
    ctx->cdc_have_scan = 1;
    return HMSE_OK;
}

HMSE_API int hmse_chunk_resolve(hmse_ctx* ctx, const uint8_t* d_data, uint64_t n_own, uint64_t n_avail, int eof,
                                  uint64_t entry, uint64_t* d_cuts, uint64_t cap, uint64_t* n_cuts,
                                  uint64_t* exit_off, void* stream) {
    if (!ctx) return HMSE_E_INVAL;
    cudaStream_t st = (cudaStream_t)stream;
    if (!ctx->cdc_have_scan || ctx->cdc_n_avail != n_avail)
        HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_chunk_resolve: no matching hmse_chunk_scan");
    if (!n_cuts) HMSE_FAIL(ctx, HMSE_E_INVAL, "n_cuts is null");
    const hmse_cdc_cfg& c = ctx->cdc_cfg;
    if (eof) n_own = n_avail;
    if (!eof && n_avail < n_own + c.max_size)
        HMSE_FAIL(ctx, HMSE_E_INVAL, "non-final shard needs max_size bytes of look-ahead");
    *n_cuts = 0;
    if (exit_off) *exit_off = entry;
    if (n_own == 0 || entry >= n_own) return HMSE_OK;

    const uint64_t seg_len = resolve_seg_len(c);
    if (entry >= seg_len) HMSE_FAIL(ctx, HMSE_E_INVAL, "entry must lie in the first segment");
    const uint64_t n_seg = div_up64(n_own, seg_len);
    ResolveScratch r;
    if (int rc = resolve_scratch(ctx, n_seg, n_own, d_data, n_avail, entry, false, &r)) return rc;
    // the segment records of the previous call are reused when they belong to the same shard geometry (incremental
    // re-resolve with another entry); hmse_chunk_scan and hmse_chunk_files clear res_valid
    const bool fresh = !(ctx->res_valid && ctx->res_n_own == n_own && ctx->res_eof == eof && ctx->seg_len == seg_len &&
                         ctx->n_seg == n_seg);
    HT_BEGIN(ctx, HT_RESOLVE, st);
    ctx->res_valid = 0;
    int in = 0;
    if (int rc = resolve_run(ctx, r, fresh, d_cuts, cap, &in, st)) return rc;
    ctx->res_valid = 1;
    ctx->res_n_own = n_own;
    ctx->res_eof = eof;
    ctx->seg_len = seg_len;
    ctx->n_seg = n_seg;
    HT_END(ctx, HT_RESOLVE, st);
    volatile uint64_t* mail = ctx->pinned;
    if (int mrc = hmse_mail(ctx, 0, r.tail + 1, 2, st)) return mrc;
    if (int mrc = hmse_mail(ctx, 2, &r.a.meta[n_seg - 1].exit[in], 2, st)) return mrc;
    HMSE_CUDA(ctx, cudaStreamSynchronize(st));
    *n_cuts = mail[0];
    if (exit_off) *exit_off = mail[1];
    if (!d_cuts || mail[0] > cap)
        HMSE_FAIL(ctx, HMSE_E_CAPACITY, "d_cuts capacity %llu < %llu cuts", (unsigned long long)cap,
                  (unsigned long long)mail[0]);
    return HMSE_OK;
}

HMSE_API int hmse_chunk_files(hmse_ctx* ctx, const uint8_t* d_data, uint64_t n, const uint64_t* d_file_off, uint64_t n_files,
                              const hmse_cdc_cfg* cfg, uint64_t* d_cuts, uint64_t cap, uint64_t* n_cuts,
                              uint64_t* d_file_chunk, void* stream) {
    if (!ctx) return HMSE_E_INVAL;
    cudaStream_t st = (cudaStream_t)stream;
    if (!n_cuts || !d_file_off || !d_file_chunk) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_chunk_files: null pointer");
    *n_cuts = 0;
    if (int rc = hmse_chunk_scan(ctx, d_data, n, cfg, stream)) return rc;   // (clears res_valid)
    const hmse_cdc_cfg& c = ctx->cdc_cfg;
    const uint64_t seg_len = resolve_seg_len(c);
    // [first u64 n_files][bad u32 | n_seg u64 | ...]
    HMSE_SCRATCH(ctx, files, uint64_t*, SLOT_CDC_FILES, n_files * sizeof(uint64_t) + 64);
    uint64_t* ftail = files + n_files;
    volatile uint64_t* mail = ctx->pinned;
    HT_BEGIN(ctx, HT_RESOLVE, st);
    HMSE_CUDA(ctx, cudaMemsetAsync(ftail, 0, 16, st));
    KL(ctx);
    file_count_kernel<<<(unsigned)div_up64(n_files + 1, 256), 256, 0, st>>>(d_file_off, n_files, n, seg_len, files,
                                                                            (uint32_t*)ftail);
    HMSE_LAUNCH_CHECK(ctx);
    if (int rc = hmse_exclusive_scan_u64(ctx, files, files, n_files, ftail + 1, st)) return rc;
    if (int mrc = hmse_mail(ctx, 0, ftail, 4, st)) return mrc;
    HMSE_CUDA(ctx, cudaStreamSynchronize(st));
    if ((uint32_t)mail[0])
        HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_chunk_files: file offsets must start at 0, never decrease and end at n = %llu",
                  (unsigned long long)n);
    const uint64_t n_seg = mail[1];
    ResolveScratch r;
    if (int rc = resolve_scratch(ctx, n_seg, n, d_data, n, 0, true, &r)) return rc;
    int in = 0;
    if (n_seg) {
        KL(ctx);
        file_table_kernel<<<(unsigned)div_up64(n_seg, 256), 256, 0, st>>>(d_file_off, files, n_files, n_seg, seg_len,
                                                                         c.min_size, r.seg);
        HMSE_LAUNCH_CHECK(ctx);
        if (int rc = resolve_run(ctx, r, true, d_cuts, cap, &in, st)) return rc;
    } else {
        HMSE_CUDA(ctx, cudaMemsetAsync(r.tail + 1, 0, 8, st));
        ctx->cdc_rounds = 0;
    }
    KL(ctx);
    file_chunk_kernel<<<(unsigned)div_up64(n_files + 1, 256), 256, 0, st>>>(files, r.offs, n_files, n_seg, r.tail + 1,
                                                                            d_file_chunk);
    HMSE_LAUNCH_CHECK(ctx);
    HT_END(ctx, HT_RESOLVE, st);
    if (int mrc = hmse_mail(ctx, 0, r.tail + 1, 2, st)) return mrc;
    HMSE_CUDA(ctx, cudaStreamSynchronize(st));
    *n_cuts = mail[0];
    if (mail[0] > cap || (mail[0] && !d_cuts))
        HMSE_FAIL(ctx, HMSE_E_CAPACITY, "d_cuts capacity %llu < %llu cuts", (unsigned long long)cap,
                  (unsigned long long)mail[0]);
    return HMSE_OK;
}

HMSE_API int hmse_chunk_candidates(hmse_ctx* ctx, uint64_t* d_bits_s, uint64_t* d_bits_l, uint64_t n_words,
                                   void* stream) {
    if (!ctx) return HMSE_E_INVAL;
    if (!ctx->cdc_have_scan) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_chunk_candidates: no scan");
    const uint64_t n_tiles = div_up64(ctx->cdc_n_avail, K1_TILE);
    const uint64_t words = (n_tiles ? n_tiles : 1) * (K1_TILE / 64);
    if (n_words > words) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_chunk_candidates: n_words exceeds the scanned range");
    const uint64_t* bits = (const uint64_t*)ctx->slot[SLOT_CDC_BITS];
    HMSE_CUDA(ctx, cudaMemcpyAsync(d_bits_s, bits, n_words * 8, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    HMSE_CUDA(ctx, cudaMemcpyAsync(d_bits_l, bits + words, n_words * 8, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return HMSE_OK;
}

HMSE_API int hmse_chunk_last_rounds(hmse_ctx* ctx) { return ctx ? (ctx->cdc_rounds >> 1) : 0; }

HMSE_API int hmse_chunk(hmse_ctx* ctx, const uint8_t* d_data, uint64_t n, const hmse_cdc_cfg* cfg, uint64_t* d_cuts,
                          uint64_t cap, uint64_t* n_cuts, void* stream) {
    int rc = hmse_chunk_scan(ctx, d_data, n, cfg, stream);
    if (rc) return rc;
    return hmse_chunk_resolve(ctx, d_data, n, n, 1, 0, d_cuts, cap, n_cuts, nullptr, stream);
}
