// localBA entry points of the C ABI: single window, batch of windows, and the multi-GPU solve whose per-iteration
// exchange of the reduced camera system goes through PEER MEMORY over NVLink inside the solve kernel (ba_lm.cu) -
// no NCCL call, no host round trip between LM iterations.
//
// Reference behaviour replaced: Optimizer::localBA's solve sections (/root/reference/src/optimizer.cpp:436-735);
// the multi-GPU split is BASELINE.json configs[4] (SURVEY.md 8e): landmarks (with all their observations) are
// partitioned over the ranks, every rank holds all keyframe poses, the partial reduced systems are summed every LM
// iteration and every rank solves the identical system (identical decisions, no broadcast).
#include "ba_lm.cuh"

#include <stdlib.h>
#include <string.h>

using namespace balm;

ov2_status ov2_localba_solve_legacy(ov2_ctx* ctx, const ov2_ba_problem* pb, const ov2_ba_opts* opts, ov2_ba_result* res,
                                    uint8_t* outlier_out);

struct ov2_ba_comm {
    ov2_ctx* ctx = nullptr;
    int rank = 0, world = 1;
    void* mine = nullptr;                 // exported buffer (XB_BYTES)
    void* base[MAX_RANKS] = {nullptr};    // every rank's buffer as mapped here
    bool opened[MAX_RANKS] = {false};     // mapped through cudaIpcOpenMemHandle (must be closed)
    bool connected = false;
    unsigned long long seq = 0;           // launches so far: epochs of launch k start at k << 20
};

static int* stop_flag_of(ov2_ctx* ctx) {
    // one int of mapped pinned host memory per context: signalStopLocalBA writes it from another host thread, the
    // solve kernel polls it before the refinement (optimizer.cpp:603-604)
    if (!ctx->ba_stop) {
        if (cudaHostAlloc((void**)&ctx->ba_stop, sizeof(int), cudaHostAllocMapped) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        *ctx->ba_stop = 0;
    }
    return ctx->ba_stop;
}

extern "C" ov2_status ov2_localba_request_stop(ov2_ctx* ctx, int stop) {
    if (!ctx) return OV2_ERR_INVALID;
    int* f = stop_flag_of(ctx);
    if (!f) return ov2_fail(ctx, OV2_ERR_NOMEM, "ov2_localba_request_stop: cudaHostAlloc");
    *reinterpret_cast<volatile int*>(f) = stop ? 1 : 0;
    return OV2_OK;
}

static const int* stop_flag_dev(ov2_ctx* ctx) {
    int* f = stop_flag_of(ctx);
    if (!f) return nullptr;
    int* d = nullptr;
    if (cudaHostGetDevicePointer((void**)&d, f, 0) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return d;
}

static_assert(MAX_VAR_CAMS == OV2_BA_SMALL_MAX_OPT_KEYFRAMES && MAX_CAMS == OV2_BA_SMALL_MAX_KEYFRAMES,
              "the published small-window limits are ba_lm_kernel's");

// Number of optimised (non-constant) keyframes of a window; pose_const may be device memory when pose is.
static int optimised_keyframes(const ov2_ba_problem* pb) {
    if (!pb->pose_const || pb->ncam <= 0) return 0;
    std::vector<uint8_t> h;
    const uint8_t* pc = pb->pose_const;
    if (ov2_is_device_ptr(pb->pose) && ov2_is_device_ptr(pc)) {
        h.resize(pb->ncam);
        if (cudaMemcpy(h.data(), pc, pb->ncam, cudaMemcpyDeviceToHost) != cudaSuccess) { cudaGetLastError(); return 0; }
        pc = h.data();
    }
    int ncv = 0;
    for (int c = 0; c < pb->ncam; ++c) ncv += pc[c] ? 0 : 1;
    return ncv;
}

extern "C" ov2_status ov2_localba_solve(ov2_ctx* ctx, const ov2_ba_problem* pb, const ov2_ba_opts* opts,
                                        ov2_ba_result* res, uint8_t* outlier_out) {
    if (!ctx || !pb || !opts || !res) return ov2_fail(ctx, OV2_ERR_INVALID, "ov2_localba_solve: bad arguments");
    const char* e = getenv("OV2_BA_LEGACY");
    const bool legacy = e && atoi(e) != 0;
    // more than 64 optimised keyframes: the large-window solve (ba_large.cu); smaller windows are routed as before
    if (!legacy && pb->ncam > MAX_VAR_CAMS && optimised_keyframes(pb) > MAX_VAR_CAMS)
        return balm_solve_large(ctx, pb, opts, res, outlier_out, stop_flag_dev(ctx));
    if (legacy || pb->ncam > MAX_CAMS) return ov2_localba_solve_legacy(ctx, pb, opts, res, outlier_out);
    memset(res, 0, sizeof(*res));
    if (pb->nobs == 0) return OV2_OK;
    uint8_t* outs[1] = {outlier_out};
    return balm_solve(ctx, 1, pb, opts, res, outs, nullptr, stop_flag_dev(ctx));
}

extern "C" ov2_status ov2_localba_solve_batch(ov2_ctx* ctx, int nprob, const ov2_ba_problem* pbs, const ov2_ba_opts* opts,
                                              ov2_ba_result* results, uint8_t* const* outlier_outs) {
    if (!ctx || nprob < 0 || (nprob > 0 && (!pbs || !opts || !results))) return ov2_fail(ctx, OV2_ERR_INVALID, "ov2_localba_solve_batch: bad arguments");
    if (nprob == 0) return OV2_OK;
    return balm_solve(ctx, nprob, pbs, opts, results, outlier_outs, nullptr, nullptr);
}

// ------------------------------------------------------------------ multi-GPU communicator (peer memory)
extern "C" ov2_status ov2_ba_comm_create(ov2_ctx* ctx, int rank, int world, ov2_ba_comm** out) {
    if (!ctx || !out || world < 1 || world > MAX_RANKS || rank < 0 || rank >= world)
        return ov2_fail(ctx, OV2_ERR_INVALID, "ov2_ba_comm_create: bad arguments (at most 8 ranks)");
    *out = nullptr;
    OV2_CUDA(ctx, cudaSetDevice(ctx->device));
    ov2_ba_comm* c = new ov2_ba_comm();
    c->ctx = ctx; c->rank = rank; c->world = world;
    cudaError_t e = cudaMalloc(&c->mine, XB_BYTES);
    if (e != cudaSuccess) { delete c; return ov2_fail(ctx, OV2_ERR_NOMEM, "ov2_ba_comm_create: cudaMalloc", e); }
    e = cudaMemset(c->mine, 0, XB_BYTES);
    if (e != cudaSuccess) { cudaFree(c->mine); delete c; return ov2_fail(ctx, OV2_ERR_CUDA, "ov2_ba_comm_create: cudaMemset", e); }
    c->base[rank] = c->mine;
    *out = c;
    return OV2_OK;
}

extern "C" ov2_status ov2_ba_comm_handle(ov2_ba_comm* c, void* handle_out, size_t handle_bytes) {
    if (!c || !handle_out || handle_bytes < sizeof(cudaIpcMemHandle_t)) return OV2_ERR_INVALID;
    cudaIpcMemHandle_t h;
    OV2_CUDA(c->ctx, cudaSetDevice(c->ctx->device));
    OV2_CUDA(c->ctx, cudaIpcGetMemHandle(&h, c->mine));
    memset(handle_out, 0, handle_bytes);
    memcpy(handle_out, &h, sizeof(h));
    return OV2_OK;
}

extern "C" ov2_status ov2_ba_comm_connect(ov2_ba_comm* c, const void* handles, size_t handle_stride) {
    if (!c || !handles || handle_stride < sizeof(cudaIpcMemHandle_t)) return OV2_ERR_INVALID;
    OV2_CUDA(c->ctx, cudaSetDevice(c->ctx->device));
    for (int r = 0; r < c->world; ++r) {
        if (r == c->rank) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, (const char*)handles + (size_t)r * handle_stride, sizeof(h));
        void* p = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) return ov2_fail(c->ctx, OV2_ERR_CUDA, "ov2_ba_comm_connect: cudaIpcOpenMemHandle (peer access between the GPUs needed)", e);
        c->base[r] = p;
        c->opened[r] = true;
    }
    c->connected = true;
    return OV2_OK;
}

// ranks that live in ONE process (tests; a multi-GPU process): the buffers are used directly
extern "C" ov2_status ov2_ba_comm_connect_local(ov2_ba_comm* c, ov2_ba_comm* const* all) {
    if (!c || !all) return OV2_ERR_INVALID;
    for (int r = 0; r < c->world; ++r) {
        if (!all[r] || all[r]->world != c->world || all[r]->rank != r) return ov2_fail(c->ctx, OV2_ERR_INVALID, "ov2_ba_comm_connect_local: inconsistent communicators");
        if (all[r]->ctx->device != c->ctx->device) {
            int can = 0;
            cudaDeviceCanAccessPeer(&can, c->ctx->device, all[r]->ctx->device);
            if (!can) return ov2_fail(c->ctx, OV2_ERR_CUDA, "ov2_ba_comm_connect_local: no peer access between the devices");
            cudaSetDevice(c->ctx->device);
            cudaError_t e = cudaDeviceEnablePeerAccess(all[r]->ctx->device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return ov2_fail(c->ctx, OV2_ERR_CUDA, "cudaDeviceEnablePeerAccess", e);
            cudaGetLastError();
        }
        c->base[r] = all[r]->mine;
    }
    c->connected = true;
    return OV2_OK;
}

extern "C" void ov2_ba_comm_destroy(ov2_ba_comm* c) {
    if (!c) return;
    cudaSetDevice(c->ctx->device);
    cudaStreamSynchronize(c->ctx->stream);
    for (int r = 0; r < c->world; ++r)
        if (c->opened[r] && c->base[r]) cudaIpcCloseMemHandle(c->base[r]);
    if (c->mine) cudaFree(c->mine);
    delete c;
}

// Every rank calls this with ITS shard (collective: the kernels of all ranks synchronise with each other through the
// exported buffers, so all ranks must call it the same number of times, in the same order).
extern "C" ov2_status ov2_localba_solve_p2p(ov2_ctx* ctx, ov2_ba_comm* comm, const ov2_ba_problem* pb, const ov2_ba_opts* opts,
                                            ov2_ba_result* res, uint8_t* outlier_out) {
    if (!ctx || !comm || !pb || !opts || !res || comm->ctx != ctx) return ov2_fail(ctx, OV2_ERR_INVALID, "ov2_localba_solve_p2p: bad arguments");
    if (comm->world > 1 && !comm->connected) return ov2_fail(ctx, OV2_ERR_INVALID, "ov2_localba_solve_p2p: communicator not connected");
    Peers X;
    memset(&X, 0, sizeof(X));
    X.world = comm->world; X.rank = comm->rank;
    X.epoch0 = (++comm->seq) << 20;
    for (int r = 0; r < comm->world; ++r) X.base[r] = comm->base[r];
    uint8_t* outs[1] = {outlier_out};
    return balm_solve(ctx, 1, pb, opts, res, outs, comm->world > 1 ? &X : nullptr, nullptr);
}
