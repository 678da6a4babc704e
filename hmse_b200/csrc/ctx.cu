// ctx.cu - context lifetime and scratch management for libhmse_b200.so.
#include <stdlib.h>

#include <new>

#include "ctx.cuh"

HMSE_API int hmse_abi_version(void) { return HMSE_ABI_VERSION; }

HMSE_API int hmse_create(int device, hmse_ctx** out) {
    if (!out) return HMSE_E_INVAL;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) return HMSE_E_CUDA;
    if (cudaSetDevice(device) != cudaSuccess) return HMSE_E_CUDA;
    hmse_ctx* c = new (std::nothrow) hmse_ctx();
    if (!c) return HMSE_E_NOMEM;
    memset(c, 0, sizeof(*c));
    c->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) {
        delete c;
        return HMSE_E_CUDA;
    }
    c->sm_count = prop.multiProcessorCount;
    if (cudaHostAlloc((void**)&c->pinned, HMSE_MAILBOX_BYTES, cudaHostAllocMapped) != cudaSuccess ||
        cudaHostGetDevicePointer((void**)&c->pinned_dev, c->pinned, 0) != cudaSuccess) {
        delete c;
        return HMSE_E_CUDA;
    }
    for (int i = 0; i < 2 * HT_EVENT_PAIRS; i++)
        if (cudaEventCreate(&c->ev[i]) != cudaSuccess) {
            delete c;
            return HMSE_E_CUDA;
        }
    for (int i = 0; i < 2 * HMSE_PARSE_EVENTS; i++)
        if (cudaEventCreate(&c->pev[i]) != cudaSuccess) {
            delete c;
            return HMSE_E_CUDA;
        }
    *out = c;
    return HMSE_OK;
}

HMSE_API void hmse_destroy(hmse_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    hmse_comm_destroy(ctx);
    for (int i = 0; i < SLOT_COUNT; i++)
        if (ctx->slot[i]) cudaFree(ctx->slot_base[i]);
    for (int i = 0; i < 2 * HT_EVENT_PAIRS; i++)
        if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    for (int i = 0; i < 2 * HMSE_PARSE_EVENTS; i++)
        if (ctx->pev[i]) cudaEventDestroy(ctx->pev[i]);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    free(ctx->dict_host);
    delete ctx;
}

HMSE_API const char* hmse_last_error(hmse_ctx* ctx) { return ctx ? ctx->err : "null ctx"; }

HMSE_API uint64_t hmse_scratch_bytes(hmse_ctx* ctx) {
    uint64_t s = 0;
    if (ctx)
        for (int i = 0; i < SLOT_COUNT; i++) s += ctx->slot_bytes[i];
    return s;
}

// HMSE_GUARD=1 (checked mode of the test suite; compute-sanitizer is closed on the B200 pool): every scratch slot is
// surrounded by two 4 KiB bands of 0xA5 that hmse_guard_check compares - a kernel that writes outside its scratch slot is
// caught at the end of the test that ran it.
constexpr size_t GUARD_BYTES = 4096;
static int guard_mode() {
    static int g = -1;
    if (g < 0) {
        const char* e = getenv("HMSE_GUARD");
        g = (e && *e && *e != '0') ? 1 : 0;
    }
    return g;
}

void* hmse_scratch(hmse_ctx* ctx, int slot, size_t bytes) {
    if (bytes == 0) bytes = 256;
    if (ctx->slot_bytes[slot] >= bytes) return ctx->slot[slot];
    if (ctx->slot[slot]) {
        cudaFree(ctx->slot_base[slot]);
        ctx->slot[slot] = ctx->slot_base[slot] = nullptr;
        ctx->slot_bytes[slot] = 0;
    }
    const size_t G = guard_mode() ? GUARD_BYTES : 0;
    // checked mode: no headroom, so that the band starts right behind the bytes the caller asked for (rounded to 256)
    size_t want = G ? bytes : bytes + bytes / 8;  // headroom so slowly growing inputs do not thrash
    want = (want + 255) & ~(size_t)255;
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, want + 2 * G);
    if (e != cudaSuccess) {
        cudaGetLastError();
        want = (bytes + 255) & ~(size_t)255;
        e = cudaMalloc(&p, want + 2 * G);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        snprintf(ctx->err, sizeof(ctx->err), "scratch slot %d: cudaMalloc(%zu) failed: %s", slot, want,
                 cudaGetErrorString(e));
        return nullptr;
    }
    if (G) {
        cudaMemset(p, 0xA5, G);
        cudaMemset((uint8_t*)p + G + want, 0xA5, G);
    }
    ctx->slot_base[slot] = p;
    ctx->slot[slot] = (uint8_t*)p + G;
    ctx->slot_bytes[slot] = want;
    return ctx->slot[slot];
}

HMSE_API int hmse_guard_check(hmse_ctx* ctx) {
    if (!ctx) return HMSE_E_INVAL;
    if (!guard_mode()) HMSE_FAIL(ctx, HMSE_E_INVAL, "hmse_guard_check: the library runs without guard bands (set HMSE_GUARD=1 before loading it)");
    HMSE_CUDA(ctx, cudaDeviceSynchronize());
    static thread_local uint8_t host[2 * GUARD_BYTES];
    for (int s = 0; s < SLOT_COUNT; s++) {
        if (!ctx->slot[s]) continue;
        uint8_t* base = (uint8_t*)ctx->slot_base[s];
        HMSE_CUDA(ctx, cudaMemcpy(host, base, GUARD_BYTES, cudaMemcpyDeviceToHost));
        HMSE_CUDA(ctx, cudaMemcpy(host + GUARD_BYTES, base + GUARD_BYTES + ctx->slot_bytes[s], GUARD_BYTES, cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < 2 * GUARD_BYTES; i++)
            if (host[i] != 0xA5)
                HMSE_FAIL(ctx, HMSE_E_INVAL, "scratch slot %d (%zu bytes): guard band overwritten %s the slot, byte %zu of the band", s,
                          ctx->slot_bytes[s], i < GUARD_BYTES ? "BEFORE" : "BEHIND", i % GUARD_BYTES);
    }
    return HMSE_OK;
}

namespace {
__global__ void mail_kernel(uint32_t* __restrict__ dst, const uint32_t* __restrict__ src, uint32_t n32) {
    for (uint32_t i = threadIdx.x; i < n32; i += blockDim.x) dst[i] = src[i];
}
}  // namespace

int hmse_mail(hmse_ctx* ctx, uint32_t word32, const void* d_src, uint32_t n32, cudaStream_t stream) {
    if ((size_t)(word32 + n32) * 4 > HMSE_MAILBOX_BYTES) HMSE_FAIL(ctx, HMSE_E_INVAL, "mailbox overflow");
    KL(ctx);
    mail_kernel<<<1, 32, 0, stream>>>(reinterpret_cast<uint32_t*>(ctx->pinned_dev) + word32,
                                      reinterpret_cast<const uint32_t*>(d_src), n32);
    HMSE_LAUNCH_CHECK(ctx);
    return HMSE_OK;
}

HMSE_API int hmse_timing(hmse_ctx* ctx, int enable) {
    if (!ctx) return HMSE_E_INVAL;
    ctx->timing = enable;
    memset(ctx->ev_set, 0, sizeof(ctx->ev_set));
    return HMSE_OK;
}

HMSE_API int hmse_timing_ms(hmse_ctx* ctx, int id, float* ms) {
    if (!ctx || !ms || id < 0 || id >= HT_COUNT) return HMSE_E_INVAL;
    *ms = 0.f;
    if (!ctx->ev_set[id]) HMSE_FAIL(ctx, HMSE_E_INVAL, "timer %d has not been recorded", id);
    HMSE_CUDA(ctx, cudaEventSynchronize(ctx->ev[2 * id + 1]));
    HMSE_CUDA(ctx, cudaEventElapsedTime(ms, ctx->ev[2 * id], ctx->ev[2 * id + 1]));
    if (id == HT_KNOWN && ctx->ev_set[HT_KNOWN_MERGE]) {
        float merge = 0.f;
        HMSE_CUDA(ctx, cudaEventSynchronize(ctx->ev[2 * HT_KNOWN_MERGE + 1]));
        HMSE_CUDA(ctx, cudaEventElapsedTime(&merge, ctx->ev[2 * HT_KNOWN_MERGE], ctx->ev[2 * HT_KNOWN_MERGE + 1]));
        *ms += merge;
    }
    return HMSE_OK;
}

HMSE_API uint64_t hmse_launch_count(hmse_ctx* ctx) { return ctx ? ctx->launches : 0; }

HMSE_API int hmse_compress_stats(hmse_ctx* ctx, uint64_t* out4, float* parse_ms_sum, uint32_t* parse_ms_n) {
    if (!ctx || !out4) return HMSE_E_INVAL;
    for (int i = 0; i < 4; i++) out4[i] = ctx->stat[i];
    float sum = 0.f;
    uint32_t n = 0;
    for (uint32_t i = 0; i < ctx->pev_n && i < (uint32_t)HMSE_PARSE_EVENTS; i++) {
        float ms = 0.f;
        if (cudaEventSynchronize(ctx->pev[2 * i + 1]) != cudaSuccess ||
            cudaEventElapsedTime(&ms, ctx->pev[2 * i], ctx->pev[2 * i + 1]) != cudaSuccess)
            HMSE_FAIL(ctx, HMSE_E_CUDA, "parse launch %u: event read failed", i);
        sum += ms;
        n++;
    }
    if (parse_ms_sum) *parse_ms_sum = sum;
    if (parse_ms_n) *parse_ms_n = n;
    return HMSE_OK;
}
