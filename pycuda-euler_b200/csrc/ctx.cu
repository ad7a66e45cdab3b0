// ctx.cu -- context, error reporting, grow-only device buffers.
#include <stdarg.h>
#include <stdlib.h>

#include "common.cuh"
#include "scan.cuh"

void pipeline_destroy(Pipeline *p);

int euler_fail(euler_ctx *ctx, int code, const char *fmt, ...)
{
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf;
    return code;
}

int dev_reserve(euler_ctx *ctx, DevBuf &b, size_t bytes)
{
    if (bytes <= b.cap && b.p) return EULER_OK;
    if (b.p) {
        cudaStreamSynchronize(ctx->stream);
        cudaFree(b.p);
        b.p = nullptr;
        b.cap = 0;
    }
    size_t want = bytes + bytes / 8 + 256;  // slack so small growth does not reallocate
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e != cudaSuccess) {
        want = bytes + 256;
        e = cudaMalloc(&b.p, want);
    }
    if (e != cudaSuccess) {
        b.p = nullptr;
        return euler_fail(ctx, EULER_ERR_NOMEM, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
    }
    b.cap = want;
    return EULER_OK;
}

void dev_free(DevBuf &b)
{
    if (b.p) cudaFree(b.p);
    b.p = nullptr;
    b.cap = 0;
}

int scan_state_reserve(euler_ctx *ctx, u64 ntiles, ScanState **state, u64 **counter)
{
    EULER_TRY(dev_reserve(ctx, ctx->scan_state, (ntiles + 1) * sizeof(ScanState)));
    *state = (ScanState *)ctx->scan_state.p;
    *counter = (u64 *)(*state + ntiles);
    return EULER_OK;
}

extern "C" {

int euler_version(void) { return 101; }

int euler_ctx_create(int device, euler_ctx **out)
{
    if (!out) return EULER_ERR_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return EULER_ERR_NOGPU;  // no CPU fallback
    if (device < 0 || device >= ndev) return EULER_ERR_ARG;
    if (cudaSetDevice(device) != cudaSuccess) return EULER_ERR_CUDA;
    euler_ctx *ctx = new euler_ctx();
    ctx->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) {
        ctx->num_sms = prop.multiProcessorCount;
        ctx->l2_bytes = (size_t)prop.l2CacheSize;
        ctx->persist_max = (size_t)prop.persistingL2CacheMaxSize;
        ctx->window_max = (size_t)prop.accessPolicyMaxWindowSize;
        // the persisting-L2 set-aside is only carved out on request: measured on B200 it slows every
        // other kernel more than it helps the table (EULER_B200_L2_PERSIST=1 to try it)
        const char *pe = getenv("EULER_B200_L2_PERSIST");
        if (pe && atoi(pe) == 1 && ctx->persist_max) cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, ctx->persist_max);
        else ctx->persist_max = 0;
    }
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return EULER_ERR_CUDA; }
    ctx->own_stream = true;
    if (cudaMallocHost((void **)&ctx->h_pinned, EULER_PINNED_WORDS * sizeof(u64)) != cudaSuccess) { delete ctx; return EULER_ERR_NOMEM; }
    for (int i = 0; i < 8; i++) cudaEventCreate(&ctx->ev[i]);
    // keep stream-ordered temporaries cached between calls
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        unsigned long long thr = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    *out = ctx;
    return EULER_OK;
}

void euler_ctx_destroy(euler_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    if (ctx->pipe) pipeline_destroy(ctx->pipe);
    dev_free(ctx->scan_state);
    dev_free(ctx->cg_buf);
    dev_free(ctx->text_buf);
    for (int i = 0; i < 8; i++) if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    if (ctx->h_pinned) cudaFreeHost(ctx->h_pinned);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char *euler_last_error(const euler_ctx *ctx) { return ctx ? ctx->err.c_str() : "no context (no CUDA device?)"; }

int euler_ctx_set_stream(euler_ctx *ctx, void *cuda_stream)
{
    if (!ctx) return EULER_ERR_ARG;
    if (ctx->own_stream && ctx->stream) {
        cudaStreamSynchronize(ctx->stream);
        cudaStreamDestroy(ctx->stream);
    }
    ctx->stream = (cudaStream_t)cuda_stream;
    ctx->own_stream = false;
    return EULER_OK;
}

int euler_ctx_sync(euler_ctx *ctx)
{
    if (!ctx) return EULER_ERR_ARG;
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return EULER_OK;
}

}  // extern "C"
