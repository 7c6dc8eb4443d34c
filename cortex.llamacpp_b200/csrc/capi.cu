// capi.cu -- the C ABI declared in include/ggml_b200.h: device discovery, contexts, memory, events.
// (Compute entry points live in graph.cu.)  Mirrors the host-side responsibilities of
// ggml-cuda.cu:514-1112 (buffers) and :2338-2431, :2790-2813, :3287-3315 (backend, events) without
// memory pools or per-device stream arrays: one stream per context, plain cudaMalloc buffers owned by
// the ggml buffer objects above us, and a few growable scratch areas per context.
#include "common.cuh"
#include <stdarg.h>
#include <mutex>

static thread_local char g_err[512] = "";

void b200_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    if (getenv("GGML_B200_DEBUG")) fprintf(stderr, "[ggml-b200] error: %s\n", g_err);
}

void graph_cache_free(b200_ctx *ctx);   // graph.cu

void *b200_ctx::get_scratch(int slot, size_t size) {
    if (size <= scratch_size[slot]) return scratch[slot];
    if (capturing) { b200_set_error("scratch growth during graph capture"); return nullptr; }
    size_t want = size + size / 4;
    want = (want + 255) & ~(size_t)255;
    cudaStreamSynchronize(stream);
    // captured cudaGraphExec entries have the OLD scratch pointers baked into their kernel nodes: a replay after this
    // reallocation would read and write freed memory.  Drop every captured graph (they are re-captured on the next
    // sightings); scratch growth is rare (sizes grow by 25% and the large areas are allocated at their upper bound).
    graph_cache_free(this);
    if (scratch[slot]) cudaFree(scratch[slot]);
    scratch[slot] = nullptr; scratch_size[slot] = 0;
    void *p = nullptr;
    const cudaError_t me = cudaMalloc(&p, want);
    if (me != cudaSuccess) {
        int cur = -1;
        cudaGetDevice(&cur);
        cudaGetLastError();
        b200_set_error("scratch alloc of %zu bytes failed on device %d (current %d): %s", want, device, cur, cudaGetErrorString(me));
        return nullptr;
    }
    scratch[slot] = p; scratch_size[slot] = want;
    return p;
}

struct b200_event { int device; cudaEvent_t ev; };

extern "C" {

int b200_abi_version(void) { return B200_ABI_VERSION; }

const char *b200_last_error(void) { return g_err; }

int b200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    int usable = 0;
    for (int i = 0; i < n; i++) {
        cudaDeviceProp p;
        if (cudaGetDeviceProperties(&p, i) == cudaSuccess && p.major == 10) usable++;
        else break;     // we only drive a homogeneous prefix of sm_100 devices
    }
    return usable;
}

int b200_device_info(int device, char *name, size_t name_len, size_t *free_bytes, size_t *total_bytes, int *sm_count, int *cc_major,
                     int *cc_minor) {
    cudaDeviceProp p;
    CUDA_TRY(cudaGetDeviceProperties(&p, device));
    if (name && name_len) snprintf(name, name_len, "%s", p.name);
    if (free_bytes || total_bytes) {
        CUDA_TRY(cudaSetDevice(device));
        size_t f = 0, t = 0;
        CUDA_TRY(cudaMemGetInfo(&f, &t));
        if (free_bytes) *free_bytes = f;
        if (total_bytes) *total_bytes = t;
    }
    if (sm_count) *sm_count = p.multiProcessorCount;
    if (cc_major) *cc_major = p.major;
    if (cc_minor) *cc_minor = p.minor;
    return B200_OK;
}

b200_ctx *b200_ctx_create(int device) {
    if (device < 0 || device >= b200_device_count()) { b200_set_error("no sm_100 device %d", device); return nullptr; }
    if (cudaSetDevice(device) != cudaSuccess) { b200_set_error("cudaSetDevice(%d) failed", device); return nullptr; }
    b200_ctx *ctx = new b200_ctx();
    ctx->device = device;
    cudaDeviceProp p;
    cudaGetDeviceProperties(&p, device);
    ctx->sm_count = p.multiProcessorCount;
    ctx->smem_optin = p.sharedMemPerBlockOptin;
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
        b200_set_error("stream create failed");
        delete ctx;
        return nullptr;
    }
    if (const char *e = getenv("GGML_B200_GRAPHS")) ctx->opt_cuda_graphs = atoi(e);
    if (const char *e = getenv("GGML_B200_FUSION")) ctx->opt_fusion = atoi(e);
    if (const char *e = getenv("GGML_B200_PDL")) ctx->opt_pdl = atoi(e);
    if (const char *e = getenv("GGML_B200_FFN_PAIR")) ctx->opt_ffn_pair = atoi(e);
    if (const char *e = getenv("GGML_B200_FA_EXACT")) ctx->opt_cpu_exact = atoi(e);
    if (const char *e = getenv("GGML_B200_CPU_EXACT")) ctx->opt_cpu_exact = atoi(e);
    return ctx;
}

void b200_ctx_destroy(b200_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    graph_cache_free(ctx);
    b200_comm_destroy(ctx);
    for (int i = 0; i < 16; i++) {
        if (ctx->split_join[i]) cudaEventDestroy(ctx->split_join[i]);
        if (ctx->split_peer[i]) { b200_ctx_destroy(ctx->split_peer[i]); cudaSetDevice(ctx->device); }
    }
    if (ctx->split_fork) cudaEventDestroy(ctx->split_fork);
    for (int i = 0; i < SCRATCH_COUNT; i++) if (ctx->scratch[i]) cudaFree(ctx->scratch[i]);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
}

int b200_ctx_device(const b200_ctx *ctx) { return ctx->device; }
void *b200_ctx_stream(const b200_ctx *ctx) { return (void *)ctx->stream; }
int64_t b200_kernel_launches(const b200_ctx *ctx) { return ctx->launches; }

int b200_synchronize(b200_ctx *ctx) {
    CUDA_TRY(cudaSetDevice(ctx->device));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return comm_check(ctx);          // a tensor-parallel step whose all-reduce lost a peer fails here instead of returning garbage sums
}

int b200_set_option(b200_ctx *ctx, const char *key, int value) {
    std::string k(key);
    int *slot = k == "fusion" ? &ctx->opt_fusion : k == "pdl" ? &ctx->opt_pdl : k == "l2_prefetch" ? &ctx->opt_l2_prefetch :
                k == "debug_skip" ? &ctx->opt_debug_skip : (k == "fa_exact" || k == "cpu_exact") ? &ctx->opt_cpu_exact :
                k == "ffn_pair" ? &ctx->opt_ffn_pair : nullptr;
    if (k == "cuda_graphs") ctx->opt_cuda_graphs = value;
    else if (slot) {
        if (*slot != value) {                 // captured graphs bake these options in: drop them
            cudaSetDevice(ctx->device);
            cudaStreamSynchronize(ctx->stream);
            graph_cache_free(ctx);
        }
        *slot = value;
    }
    else { b200_set_error("unknown option %s", key); return B200_ERR_UNSUPPORTED; }
    return B200_OK;
}

int b200_debug_set_prof(b200_ctx *ctx, void *buf) { ctx->prof_buf = buf; return B200_OK; }

// ---- memory ----
void *b200_malloc(int device, size_t size) {
    if (cudaSetDevice(device) != cudaSuccess) return nullptr;
    void *p = nullptr;
    if (cudaMalloc(&p, size ? size : 1) != cudaSuccess) {
        cudaGetLastError();   // clear; caller handles NULL (ggml-cuda.cu:654-660)
        b200_set_error("cudaMalloc(%zu) failed on device %d", size, device);
        return nullptr;
    }
    return p;
}
void b200_free(int device, void *ptr) {
    if (!ptr) return;
    cudaSetDevice(device);
    cudaFree(ptr);
}
void *b200_host_malloc(size_t size) {
    void *p = nullptr;
    if (cudaMallocHost(&p, size ? size : 1) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void b200_host_free(void *ptr) { if (ptr) cudaFreeHost(ptr); }

int b200_memset(int device, void *dst, int value, size_t size) {
    CUDA_TRY(cudaSetDevice(device));
    CUDA_TRY(cudaMemset(dst, value, size));
    CUDA_TRY(cudaDeviceSynchronize());
    return B200_OK;
}
int b200_memcpy_h2d(int device, void *dst, const void *src, size_t size) {
    CUDA_TRY(cudaSetDevice(device));
    CUDA_TRY(cudaMemcpy(dst, src, size, cudaMemcpyHostToDevice));
    return B200_OK;
}
int b200_memcpy_d2h(int device, void *dst, const void *src, size_t size) {
    CUDA_TRY(cudaSetDevice(device));
    CUDA_TRY(cudaMemcpy(dst, src, size, cudaMemcpyDeviceToHost));
    return B200_OK;
}
int b200_memcpy_d2d(int dst_device, void *dst, int src_device, const void *src, size_t size) {
    CUDA_TRY(cudaSetDevice(dst_device));
    if (dst_device == src_device) CUDA_TRY(cudaMemcpy(dst, src, size, cudaMemcpyDeviceToDevice));
    else CUDA_TRY(cudaMemcpyPeer(dst, dst_device, src, src_device, size));
    CUDA_TRY(cudaDeviceSynchronize());
    return B200_OK;
}
int b200_memcpy_h2d_async(b200_ctx *ctx, void *dst, const void *src, size_t size) {
    CUDA_TRY(cudaSetDevice(ctx->device));
    CUDA_TRY(cudaMemcpyAsync(dst, src, size, cudaMemcpyHostToDevice, ctx->stream));
    return B200_OK;
}
int b200_memcpy_d2h_async(b200_ctx *ctx, void *dst, const void *src, size_t size) {
    CUDA_TRY(cudaSetDevice(ctx->device));
    CUDA_TRY(cudaMemcpyAsync(dst, src, size, cudaMemcpyDeviceToHost, ctx->stream));
    return B200_OK;
}
int b200_memcpy_d2d_async(b200_ctx *ctx, void *dst, int src_device, const void *src, size_t size) {
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (src_device == ctx->device) CUDA_TRY(cudaMemcpyAsync(dst, src, size, cudaMemcpyDeviceToDevice, ctx->stream));
    else CUDA_TRY(cudaMemcpyPeerAsync(dst, ctx->device, src, src_device, size, ctx->stream));
    return B200_OK;
}

// The streaming GEMV reads whole 16-byte lines and may touch up to 15 bytes past the last weight row
// (and the misalignment of the first); every quantised tensor therefore gets 128 bytes of tail padding.
size_t b200_alloc_size(int32_t type, const int64_t ne[4], size_t nbytes) {
    (void)ne;
    if (b200_type_is_quant(type)) return ((nbytes + 127) & ~(size_t)127) + 128;
    return nbytes;
}

// ---- events ----
b200_event *b200_event_create(int device) {
    if (cudaSetDevice(device) != cudaSuccess) return nullptr;
    b200_event *e = new b200_event();
    e->device = device;
    if (cudaEventCreate(&e->ev) != cudaSuccess) { delete e; return nullptr; }
    return e;
}
void b200_event_destroy(b200_event *e) {
    if (!e) return;
    cudaSetDevice(e->device);
    cudaEventDestroy(e->ev);
    delete e;
}
int b200_event_record(b200_ctx *ctx, b200_event *e) {
    CUDA_TRY(cudaSetDevice(ctx->device));
    CUDA_TRY(cudaEventRecord(e->ev, ctx->stream));
    return B200_OK;
}
int b200_event_wait(b200_ctx *ctx, b200_event *e) {
    CUDA_TRY(cudaSetDevice(ctx->device));
    CUDA_TRY(cudaStreamWaitEvent(ctx->stream, e->ev, 0));
    return B200_OK;
}
int b200_event_synchronize(b200_event *e) {
    CUDA_TRY(cudaSetDevice(e->device));
    CUDA_TRY(cudaEventSynchronize(e->ev));
    return B200_OK;
}
float b200_event_elapsed_ms(b200_event *a, b200_event *b) {
    float ms = -1.0f;
    if (cudaEventElapsedTime(&ms, a->ev, b->ev) != cudaSuccess) { cudaGetLastError(); return -1.0f; }
    return ms;
}

}  // extern "C"
