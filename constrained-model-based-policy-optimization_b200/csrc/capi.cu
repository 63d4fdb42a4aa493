// Context, error reporting, scratch management and weight upload of libcmbpo_b200.so.
#include <stdarg.h>
#include <string.h>

#include "common.cuh"

static thread_local char g_err[1024] = "";

void cmbpo_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" const char* cmbpo_last_error(void) { return g_err; }
extern "C" int cmbpo_abi_version(void) { return CMBPO_ABI_VERSION; }

int cmbpo_ws_get(cmbpo_ctx* ctx, int slot, size_t bytes, void** out) {
    Workspace& w = ctx->ws[slot];
    if (bytes > w.bytes) {
        if (w.ptr) {
            CUDA_TRY(cudaStreamSynchronize(ctx->stream));
            CUDA_TRY(cudaFree(w.ptr));
            w.ptr = nullptr; w.bytes = 0;
        }
        size_t want = bytes + bytes / 8 + 256;
        CUDA_TRY(cudaMalloc(&w.ptr, want));
        w.bytes = want;
    }
    *out = w.ptr;
    return 0;
}

extern "C" int cmbpo_ctx_create(int device, cmbpo_ctx** out) {
    CMBPO_CHECK(out, "null output pointer");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    CMBPO_CHECK(e == cudaSuccess && n > 0, "no CUDA device available (%s): this library has no CPU fallback",
                cudaGetErrorString(e));
    CMBPO_CHECK(device >= 0 && device < n, "device %d out of range (%d devices)", device, n);
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    CMBPO_CHECK(prop.major == 10, "device %d is sm_%d%d; this library is built for sm_100a (B200) only",
                device, prop.major, prop.minor);
    cmbpo_ctx* ctx = new cmbpo_ctx();
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->stream = nullptr;
    *out = ctx;
    return 0;
}

void net_free(Net& n) {
    for (int l = 0; l < CMBPO_MAX_LAYERS; ++l) {
        if (n.W[l]) cudaFree(n.W[l]);
        if (n.b[l]) cudaFree(n.b[l]);
    }
    float* ptrs[] = {n.mu_in, n.sig_in, n.mu_out, n.sig_out, n.l2s_out, n.tc_bias};
    for (float* p : ptrs) if (p) cudaFree(p);
    if (n.elite) cudaFree(n.elite);
    for (int i = 0; i < 3; ++i) if (n.tc_pack[i]) cudaFree(n.tc_pack[i]);
    n = Net();
}

extern "C" int cmbpo_ctx_destroy(cmbpo_ctx* ctx) {
    if (!ctx) return 0;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    for (int w = 0; w < CMBPO_NET_COUNT; ++w) train_free(ctx, w);
    for (Net& n : ctx->nets) net_free(n);
    net_free(ctx->polnet);
    if (ctx->log_std) cudaFree(ctx->log_std);
    for (Workspace& w : ctx->ws) if (w.ptr) cudaFree(w.ptr);
    if (ctx->host_n) cudaFreeHost(ctx->host_n);
    for (cudaEvent_t e : ctx->n_ev) if (e) cudaEventDestroy(e);
    delete ctx;
    return 0;
}

extern "C" int cmbpo_ctx_set_stream(cmbpo_ctx* ctx, void* s) {
    CMBPO_CHECK(ctx, "null context");
    ctx->stream = (cudaStream_t)s;
    return 0;
}

extern "C" int cmbpo_ctx_synchronize(cmbpo_ctx* ctx) {
    CMBPO_CHECK(ctx, "null context");
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" int64_t cmbpo_ctx_launch_count(cmbpo_ctx* ctx) { return ctx ? ctx->launches : 0; }

extern "C" int cmbpo_ctx_profile(cmbpo_ctx* ctx, int enable) {
    CMBPO_CHECK(ctx, "null context");
    ctx->profile = enable != 0;
    return 0;
}

extern "C" int cmbpo_ctx_profile_read(cmbpo_ctx* ctx, int slot, double* total_ms, int64_t* launches,
                                      int reset) {
    CMBPO_CHECK(ctx && slot >= 0 && slot < CMBPO_PROF_SLOTS, "bad arguments");
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    ProfSlot& p = ctx->prof[slot];
    double ms = 0;
    for (size_t i = 0; i < p.used; ++i) {
        float t = 0;
        CUDA_TRY(cudaEventElapsedTime(&t, p.start[i], p.stop[i]));
        ms += t;
    }
    if (total_ms) *total_ms = ms;
    if (launches) *launches = (int64_t)p.used;
    if (reset) p.used = 0;
    return 0;
}

// sigma = max(sqrt(var), 1e-2) (pens/utils.py:156); l2s = 2*log(sigma) (pens/utils.py:187)
__global__ void prep_scaler_kernel(const float* var, int n, float* sig, float* l2s) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float s = fmaxf(sqrtf(var[i]), 1e-2f);
    sig[i] = s;
    if (l2s) l2s[i] = __fmul_rn(2.0f, logf(s));
}

static int upload(cmbpo_ctx* ctx, const float* src, size_t n, bool on_device, float** dst) {
    CUDA_TRY(cudaMalloc(dst, n * sizeof(float)));
    CUDA_TRY(cudaMemcpyAsync(*dst, src, n * sizeof(float),
                             on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, ctx->stream));
    return 0;
}

extern "C" int cmbpo_net_set_weights(cmbpo_ctx* ctx, int which, int E, int n_layers, const int* dims,
                                     const float* const* W, const float* const* b, const int* acts,
                                     const float* mu_in, const float* var_in, const float* mu_out,
                                     const float* var_out, int probabilistic, const int* elite_inds,
                                     int n_elite, int on_device) {
    CMBPO_CHECK(ctx && which >= 0 && which < CMBPO_NET_COUNT, "bad arguments");
    CMBPO_CHECK(E >= 1 && n_layers >= 1 && n_layers <= CMBPO_MAX_LAYERS, "bad network shape");
    CMBPO_CHECK((mu_in == nullptr) == (var_in == nullptr) && (mu_out == nullptr) == (var_out == nullptr),
                "scaler mean and variance must be given together");
    CUDA_TRY(cudaSetDevice(ctx->device));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    Net& n = ctx->nets[which];
    train_free(ctx, which);                  // a new set of variables: the optimiser state goes with the old one
    net_free(n);
    n.E = E; n.n_layers = n_layers; n.probabilistic = probabilistic != 0;
    for (int l = 0; l <= n_layers; ++l) n.dims[l] = dims[l];
    const int last = dims[n_layers];
    CMBPO_CHECK(!probabilistic || last % 2 == 0, "probabilistic net needs an even output width");
    n.D = probabilistic ? last / 2 : last;
    const bool dev = on_device != 0;
    for (int l = 0; l < n_layers; ++l) {
        n.acts[l] = acts[l];
        if (upload(ctx, W[l], (size_t)E * dims[l] * dims[l + 1], dev, &n.W[l])) return 1;
        if (upload(ctx, b[l], (size_t)E * dims[l + 1], dev, &n.b[l])) return 1;
    }
    if (mu_in) {
        float* var;
        n.has_in = true;
        if (upload(ctx, mu_in, dims[0], dev, &n.mu_in)) return 1;
        if (upload(ctx, var_in, dims[0], dev, &var)) return 1;
        CUDA_TRY(cudaMalloc(&n.sig_in, dims[0] * sizeof(float)));
        prep_scaler_kernel<<<cdiv(dims[0], 128), 128, 0, ctx->stream>>>(var, dims[0], n.sig_in, nullptr);
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        cudaFree(var);
    }
    if (mu_out) {
        float* var;
        n.has_out = true;
        if (upload(ctx, mu_out, n.D, dev, &n.mu_out)) return 1;
        if (upload(ctx, var_out, n.D, dev, &var)) return 1;
        CUDA_TRY(cudaMalloc(&n.sig_out, n.D * sizeof(float)));
        CUDA_TRY(cudaMalloc(&n.l2s_out, n.D * sizeof(float)));
        prep_scaler_kernel<<<cdiv(n.D, 128), 128, 0, ctx->stream>>>(var, n.D, n.sig_out, n.l2s_out);
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        cudaFree(var);
    }
    n.n_elite = n_elite;
    if (n_elite > 0) {
        for (int i = 0; i < n_elite; ++i)
            CMBPO_CHECK(elite_inds[i] >= 0 && elite_inds[i] < E, "elite index %d out of range", elite_inds[i]);
        CUDA_TRY(cudaMalloc(&n.elite, n_elite * sizeof(int)));
        CUDA_TRY(cudaMemcpyAsync(n.elite, elite_inds, n_elite * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    }
    n.loaded = true;
    if (ens_tc_supported(n) && ens_tc_prepare(ctx, n)) return 1;
    if (which != CMBPO_NET_DYN && policy_pack_build(ctx)) return 1;
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" int cmbpo_actor_set_log_std(cmbpo_ctx* ctx, const float* log_std, int A, int on_device) {
    CMBPO_CHECK(ctx && log_std && A > 0, "bad arguments");
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (ctx->log_std) { CUDA_TRY(cudaFree(ctx->log_std)); ctx->log_std = nullptr; }
    if (upload(ctx, log_std, A, on_device != 0, &ctx->log_std)) return 1;
    ctx->A = A;
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return 0;
}
