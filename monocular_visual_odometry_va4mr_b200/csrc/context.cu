// Context, buffer pool and error plumbing of libb200vo.so.
#include "internal.cuh"
#include "tma.cuh"
#include <cmath>
#include <cstdarg>

int vo_set_err(b200vo_ctx* ctx, int code, const char* fmt, ...)
{
    if (ctx) {
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(ctx->err, sizeof(ctx->err), fmt, ap);
        va_end(ap);
    }
    return code;
}

int vo_cuda_fail(b200vo_ctx* ctx, cudaError_t e, const char* what)
{
    vo_set_err(ctx, (int)e, "CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
    return (int)e > 0 ? (int)e : 1;
}

int vo_reserve(b200vo_ctx* ctx, DevBuf& b, size_t bytes)
{
    if (bytes <= b.cap) return 0;
    if (b.p) {
        VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        VO_CUDA(ctx, cudaFree(b.p));
        b.p = nullptr;
        b.cap = 0;
    }
    size_t cap = vo_align(bytes + bytes / 4, 4096);
    VO_CUDA(ctx, cudaMalloc(&b.p, cap));
    b.cap = cap;
    return 0;
}

int vo_reserve_pinned(b200vo_ctx* ctx, size_t bytes)
{
    if (bytes <= ctx->h_pin_cap) return 0;
    if (ctx->h_pin) {
        VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        VO_CUDA(ctx, cudaFreeHost(ctx->h_pin));
        ctx->h_pin = nullptr;
        ctx->h_pin_cap = 0;
    }
    size_t cap = vo_align(bytes + bytes / 4, 4096);
    VO_CUDA(ctx, cudaMallocHost(&ctx->h_pin, cap));
    ctx->h_pin_cap = cap;
    return 0;
}

bool vo_intrinsics_valid(const double K[9])
{
    if (!K) return false;
    const bool focal = std::isfinite(K[0]) && K[0] > 0 && std::isfinite(K[4]) && K[4] > 0;
    const bool centre = std::isfinite(K[2]) && std::isfinite(K[5]);
    const bool zeros = K[1] == 0 && K[3] == 0 && K[6] == 0 && K[7] == 0 && K[8] == 1;
    return focal && centre && zeros;
}

void vo_intrinsics_row(VoIntrinsics& r, const double K[9], double emat_thr)
{
    r = VoIntrinsics{};
    r.fx = K[0]; r.fy = K[4]; r.cx = K[2]; r.cy = K[5];
    for (int k = 0; k < 9; ++k) r.K[k] = K[k];
    const double Ki[9] = {1.0 / K[0], 0, -K[2] / K[0], 0, 1.0 / K[4], -K[5] / K[4], 0, 0, 1};
    for (int k = 0; k < 9; ++k) r.Ki[k] = Ki[k];
    const double t = emat_thr / ((r.fx + r.fy) / 2);
    r.emat_thr_sq = (float)(t * t);
}

int vo_intrinsics_uniform(b200vo_ctx* ctx, const double K[9], double emat_thr, int n, const VoIntrinsics** d_rows)
{
    std::vector<VoIntrinsics> h(n > 0 ? n : 1);
    vo_intrinsics_row(h[0], K, emat_thr);
    for (size_t s = 1; s < h.size(); ++s) h[s] = h[0];
    VO_TRY(vo_reserve(ctx, ctx->d_intr, h.size() * sizeof(VoIntrinsics)));
    VO_CUDA(ctx, cudaMemcpyAsync(ctx->d_intr.p, h.data(), h.size() * sizeof(VoIntrinsics), cudaMemcpyHostToDevice, ctx->stream));
    *d_rows = (const VoIntrinsics*)ctx->d_intr.p;
    return 0;
}

int vo_check_seqs(b200vo_ctx* ctx, int batch, int n_seq, const int32_t* seqs)
{
    if (n_seq < 1 || n_seq > batch) return vo_set_err(ctx, B200VO_E_BADARG, "n_seq = %d is outside [1, batch = %d]", n_seq, batch);
    if (!seqs) return vo_set_err(ctx, B200VO_E_BADARG, "null array");
    std::vector<char> seen(batch, 0);
    for (int k = 0; k < n_seq; ++k) {
        if (seqs[k] < 0 || seqs[k] >= batch)
            return vo_set_err(ctx, B200VO_E_BADARG, "seqs[%d] = %d is outside [0, batch = %d)", k, seqs[k], batch);
        if (seen[seqs[k]]++) return vo_set_err(ctx, B200VO_E_BADARG, "sequence %d is listed twice", seqs[k]);
    }
    return 0;
}

extern "C" int b200vo_version(int* sm_arch)
{
    if (sm_arch) *sm_arch = 100;
    return 100;  // 1.00
}

extern "C" int b200vo_create(int device, b200vo_ctx** out)
{
    if (!out) return B200VO_E_BADARG;
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev <= 0) return 100;  // no CUDA device: fail loudly, no CPU fallback
    if (device < 0 || device >= ndev) return B200VO_E_BADARG;
    b200vo_ctx* ctx = new b200vo_ctx();
    ctx->device = device;
    if ((e = cudaSetDevice(device)) != cudaSuccess) { delete ctx; return (int)e; }
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) { delete ctx; return (int)e; }
    if (prop.major != 10) {  // sm_100a cubins only
        delete ctx;
        return 101;
    }
    ctx->num_sms = prop.multiProcessorCount;
    if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) { delete ctx; return (int)e; }
    cudaEventCreate(&ctx->ev0);
    cudaEventCreate(&ctx->ev1);
    *out = ctx;
    return 0;
}

extern "C" void b200vo_destroy(b200vo_ctx* ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (auto& b : ctx->d_stage_img) if (b.p) cudaFree(b.p);
    for (auto& b : ctx->d_scratch) if (b.p) cudaFree(b.p);
    for (auto& s : ctx->slots) if (s.slab.p) cudaFree(s.slab.p);
    if (ctx->d_rng.p) cudaFree(ctx->d_rng.p);
    if (ctx->d_intr.p) cudaFree(ctx->d_intr.p);
    if (ctx->d_mask.p) cudaFree(ctx->d_mask.p);
    if (ctx->d_undist.p) cudaFree(ctx->d_undist.p);
    if (ctx->d_sift.p) cudaFree(ctx->d_sift.p);
    for (DevBuf* b : {&ctx->d_sift_out[0], &ctx->d_sift_out[1], &ctx->d_sift_sort}) if (b->p) cudaFree(b->p);
    if (ctx->d_klt_queue.p) cudaFree(ctx->d_klt_queue.p);
    if (ctx->h_pin) cudaFreeHost(ctx->h_pin);
    cudaEventDestroy(ctx->ev0);
    cudaEventDestroy(ctx->ev1);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
}

extern "C" const char* b200vo_last_error(b200vo_ctx* ctx) { return ctx ? ctx->err : "null ctx"; }
extern "C" long long b200vo_launch_count(b200vo_ctx* ctx) { return ctx ? ctx->launches : 0; }
extern "C" float b200vo_last_gpu_ms(b200vo_ctx* ctx) { return ctx ? ctx->last_ms : 0.f; }
extern "C" void* b200vo_stream(b200vo_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

extern "C" int b200vo_sync(b200vo_ctx* ctx)
{
    if (!ctx) return B200VO_E_BADARG;
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int vo_encode_tiled(b200vo_ctx* ctx, CUtensorMap* map, CUtensorMapDataType dtype, int rank, void* gptr,
                    const cuuint64_t* dims, const cuuint64_t* strides_bytes, const cuuint32_t* box,
                    CUtensorMapSwizzle swizzle)
{
    if (!ctx->encode_tiled) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
        if (e != cudaSuccess || !fn || qres != cudaDriverEntryPointSuccess)
            return vo_set_err(ctx, 200, "cuTensorMapEncodeTiled entry point unavailable");
        ctx->encode_tiled = fn;
    }
    const cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = ((EncodeTiledFn)ctx->encode_tiled)(map, dtype, (cuuint32_t)rank, gptr, dims, strides_bytes, box, estr,
                                                    CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return vo_set_err(ctx, 201, "cuTensorMapEncodeTiled failed (%d)", (int)r);
    return 0;
}
