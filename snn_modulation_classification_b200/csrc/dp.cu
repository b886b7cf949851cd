// Data-parallel window driver: the T-loop of train.py:249-251 over a batch SHARD, with the local-layer gradients averaged over
// the ranks by raw NCCL all-reduces on a side stream (SURVEY.md section 8e; the reference has no multi-GPU code).
//
// One process per GPU.  Every rank holds identical weights and its own B/world samples; a layer's gradients
// (gW, gb[, gWout, gbout]) live back to back in one flat bucket.  Per timestep and layer:
//
//     main stream:  [wait reduced(l)] -> Adam on the averaged bucket (identical on every rank) -> forward -> backward (grads -> bucket)
//                   -> record grads(l)
//     side stream:  wait grads(l) -> ncclAllReduce(bucket l, avg) -> record reduced(l)
//
// so the collective of layer l overlaps the forward/backward of the other layers and is only waited for right before layer
// l's next forward.  Everything is enqueued from this one C loop: no per-timestep Python, no host synchronisation.
// The communicator is created with a small maxCTAs: NCCL's CTAs otherwise take SMs away from the 148-CTA persistent kernels
// (whose CTAs need a whole SM each), which then run a second wave.
//
// NCCL is not linked: the library is dlopen'ed (the copy torch already loaded, path passed in by the host), so the
// single-GPU path keeps depending on cudart only.
#include <dlfcn.h>
#include <string.h>

#include <nccl.h>

#include "common.cuh"

namespace dcll {

// defined in wgrad.cu / net.cu
int launch_bucket_adam(const dcll_conv_layer *L, dcll_train_args *a, const float *bucket, cudaStream_t st, dcll_optim *opt);
int dp_step_fwd(dcll_conv_layer *L, const void *x, const float *target, int loss_kind, int32_t *clout, cudaStream_t st,
                const dcll_conv_layer *next, bool trace_done, int spike_io, int layer);
int dp_step_bwd(dcll_conv_layer *L, dcll_train_args *a, cudaStream_t st, int layer);
int dp_check_opt(const dcll_optim *opt, int n_layers);
int dp_check(const dcll_conv_layer *layers, const dcll_train_args *train, int n_layers);

struct NcclApi {
    void *handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRankConfig)(ncclComm_t *, int, ncclUniqueId, int, ncclConfig_t *) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
};

static int load_nccl(const char *path, NcclApi *api) {
    const char *cands[] = {path, "libnccl.so.2", "libnccl.so"};
    for (const char *c : cands) {
        if (!c || !c[0]) continue;
        api->handle = dlopen(c, RTLD_NOW | RTLD_GLOBAL);
        if (api->handle) break;
    }
    DCLL_REQUIRE(api->handle, DCLL_EINVAL, "dcll_dp: cannot dlopen NCCL (%s): %s", path ? path : "libnccl.so.2", dlerror());
#define SYM(field, name)                                                                       \
    api->field = reinterpret_cast<decltype(api->field)>(dlsym(api->handle, name));             \
    DCLL_REQUIRE(api->field, DCLL_EINVAL, "dcll_dp: symbol %s missing in the NCCL library", name)
    SYM(GetUniqueId, "ncclGetUniqueId");
    SYM(CommInitRankConfig, "ncclCommInitRankConfig");
    SYM(CommDestroy, "ncclCommDestroy");
    SYM(AllReduce, "ncclAllReduce");
    SYM(GetErrorString, "ncclGetErrorString");
#undef SYM
    return DCLL_OK;
}

}  // namespace dcll

using namespace dcll;

struct dcll_dp {
    NcclApi api;
    ncclComm_t comm = nullptr;
    cudaStream_t side = nullptr;
    cudaEvent_t ev_grad[16], ev_red[16];
    int rank = 0, world = 1, max_ctas = 0;
};

#define DCLL_NCCL_OK(dp, expr)                                                                         \
    do {                                                                                               \
        ncclResult_t _r = (expr);                                                                      \
        if (_r != ncclSuccess) {                                                                       \
            ::dcll::set_error("%s failed: %s", #expr, (dp)->api.GetErrorString(_r));                   \
            return DCLL_ECUDA;                                                                         \
        }                                                                                              \
    } while (0)

extern "C" __attribute__((visibility("default"))) int dcll_dp_unique_id(const char *nccl_lib, void *id128) {
    DCLL_REQUIRE(id128, DCLL_EINVAL, "dcll_dp_unique_id: null output");
    NcclApi api;
    int rc = load_nccl(nccl_lib, &api);
    if (rc != DCLL_OK) return rc;
    ncclUniqueId id;
    ncclResult_t r = api.GetUniqueId(&id);
    DCLL_REQUIRE(r == ncclSuccess, DCLL_ECUDA, "ncclGetUniqueId failed: %s", api.GetErrorString(r));
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    memcpy(id128, &id, 128);
    return DCLL_OK;
}

extern "C" __attribute__((visibility("default"))) int dcll_dp_create(const char *nccl_lib, const void *id128, int rank, int world, int max_ctas,
                                                                      dcll_dp **out) {
    DCLL_REQUIRE(id128 && out && world >= 1 && rank >= 0 && rank < world, DCLL_EINVAL, "dcll_dp_create: bad arguments");
    dcll_dp *dp = new dcll_dp();
    int rc = load_nccl(nccl_lib, &dp->api);
    if (rc != DCLL_OK) {
        delete dp;
        return rc;
    }
    dp->rank = rank, dp->world = world, dp->max_ctas = max_ctas;
    ncclUniqueId id;
    memcpy(&id, id128, 128);
    ncclConfig_t cfg = NCCL_CONFIG_INITIALIZER;
    cfg.blocking = 1;
    if (max_ctas > 0) cfg.maxCTAs = max_ctas, cfg.minCTAs = 1;
    DCLL_NCCL_OK(dp, dp->api.CommInitRankConfig(&dp->comm, world, id, rank, &cfg));
    int lo = 0, hi = 0;
    DCLL_CUDA_OK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    DCLL_CUDA_OK(cudaStreamCreateWithPriority(&dp->side, cudaStreamNonBlocking, hi));   // collectives first when SMs free up
    for (int i = 0; i < 16; ++i) {
        DCLL_CUDA_OK(cudaEventCreateWithFlags(&dp->ev_grad[i], cudaEventDisableTiming));
        DCLL_CUDA_OK(cudaEventCreateWithFlags(&dp->ev_red[i], cudaEventDisableTiming));
    }
    *out = dp;
    return DCLL_OK;
}

extern "C" __attribute__((visibility("default"))) int dcll_dp_destroy(dcll_dp *dp) {
    if (!dp) return DCLL_OK;
    if (dp->side) cudaStreamSynchronize(dp->side);
    if (dp->comm) dp->api.CommDestroy(dp->comm);
    for (int i = 0; i < 16; ++i) cudaEventDestroy(dp->ev_grad[i]), cudaEventDestroy(dp->ev_red[i]);
    if (dp->side) cudaStreamDestroy(dp->side);
    delete dp;
    return DCLL_OK;
}

// The window of dcll_net_window (net.cu) with the per-layer all-reduce between a layer's backward and its next forward.
// train[l].apply_update must be 0 and train[l].grad_w / grad_b [/ grad_wout / grad_bout] must point, in this order and back to
// back, into bucket[l] (bucket_floats[l] floats in total).  Every rank must make the same call sequence.
extern "C" __attribute__((visibility("default"))) int dcll_net_window_dp(dcll_dp *dp, dcll_conv_layer *layers, dcll_train_args *train, int n_layers,
                                                                          const void *x0, const float *target, int64_t target_t_stride, int T,
                                                                          int burnin, const int32_t *iter0, int32_t *clout,
                                                                          float *const *bucket, const size_t *bucket_floats, void *stream) {
    return dcll_net_window_dp_opt(dp, layers, train, nullptr, n_layers, x0, target, target_t_stride, T, burnin, iter0, clout, bucket,
                                  bucket_floats, stream);
}

// opt: the update rules opt[2l] (train[l].adam_i2h) and opt[2l + 1] (train[l].adam_out), or null (Adam everywhere)
extern "C" __attribute__((visibility("default"))) int dcll_net_window_dp_opt(dcll_dp *dp, dcll_conv_layer *layers, dcll_train_args *train,
                                                                              dcll_optim *opt, int n_layers, const void *x0,
                                                                              const float *target, int64_t target_t_stride, int T,
                                                                              int burnin, const int32_t *iter0, int32_t *clout,
                                                                              float *const *bucket, const size_t *bucket_floats,
                                                                              void *stream) {
    DCLL_REQUIRE(dp && dp->comm && layers && train && n_layers > 0 && n_layers <= 16 && x0 && target && T > 0 && iter0 && bucket && bucket_floats,
                 DCLL_EINVAL, "dcll_net_window_dp: bad arguments");
    set_reserved_sms(0);
    int rc = dp_check(layers, train, n_layers);
    if (rc != DCLL_OK) return rc;
    rc = dp_check_opt(opt, n_layers);
    if (rc != DCLL_OK) return rc;
    for (int l = 0; l < n_layers; ++l) {
        const dcll_conv_layer &L = layers[l];
        const dcll_train_args &a = train[l];
        Geo g = geo_of(&L);
        size_t need = (size_t)g.nW + L.Cout + (L.output_layer ? (size_t)L.K * g.F + L.K : 0);
        DCLL_REQUIRE(!a.apply_update && bucket[l] && bucket_floats[l] == need && a.grad_w == bucket[l] && a.grad_b == bucket[l] + g.nW &&
                         (!L.output_layer || (a.grad_wout == bucket[l] + g.nW + L.Cout && a.grad_bout == a.grad_wout + (size_t)L.K * g.F)),
                     DCLL_EINVAL, "dcll_net_window_dp: layer %d: gradients must lie back to back in the bucket (apply_update = 0)", l);
    }
    cudaStream_t st = (cudaStream_t)stream;
    const dcll_conv_layer &L0 = layers[0];
    const size_t x_stride = L0.x_mode == DCLL_X_CELLS ? (size_t)L0.B * 2 * sizeof(int32_t) : (size_t)L0.B * L0.Cin * L0.H * L0.W * sizeof(float);
    bool pending[16] = {false};
    // while a collective may be running, the persistent kernels leave NCCL's CTAs their SMs (common.cuh: sm_budget)
    auto reserve = [&]() {
        bool any = false;
        for (int l = 0; l < n_layers; ++l) any = any || pending[l];
        // (a single-rank communicator moves nothing: no SMs to leave, and the window then equals dcll_net_window bit for bit)
        set_reserved_sms(any && dp->world > 1 ? (dp->max_ctas > 0 ? dp->max_ctas : 16) : 0);
    };
    auto finish = [&](int l) -> int {
        if (!pending[l]) return DCLL_OK;
        DCLL_CUDA_OK(cudaStreamWaitEvent(st, dp->ev_red[l], 0));
        pending[l] = false;
        reserve();
        return launch_bucket_adam(&layers[l], &train[l], bucket[l], st, opt ? opt + 2 * l : nullptr);
    };
    for (int t = 0; t < T; ++t) {
        const float *tgt = target + (size_t)t * target_t_stride;
        for (int l = 0; l < n_layers; ++l) {
            dcll_conv_layer *L = &layers[l];
            rc = finish(l);                                         // the averaged gradients of timestep t-1 update layer l now
            if (rc != DCLL_OK) return rc;
            const void *x = l == 0 ? (const void *)((const char *)x0 + (size_t)t * x_stride) : (const void *)layers[l - 1].spikes;
            const int it = iter0[l] + t + 1;
            const bool do_train = it >= burnin;
            int32_t *co = clout ? clout + ((size_t)t * n_layers + l) * L->B : nullptr;
            const bool fuse_next = l + 1 < n_layers && tc_trace_fusable(L, &layers[l + 1]);
            const bool trace_done = l > 0 && tc_trace_fusable(&layers[l - 1], L);
            rc = dp_step_fwd(L, x, do_train ? tgt : nullptr, do_train ? train[l].loss_kind : 0, co, st, fuse_next ? &layers[l + 1] : nullptr,
                             trace_done, spike_io_of(layers, l, n_layers, fuse_next, trace_done), l);
            if (rc != DCLL_OK) return rc;
            if (do_train) {
                rc = dp_step_bwd(L, &train[l], st, l);
                if (rc != DCLL_OK) return rc;
                DCLL_CUDA_OK(cudaEventRecord(dp->ev_grad[l], st));
                DCLL_CUDA_OK(cudaStreamWaitEvent(dp->side, dp->ev_grad[l], 0));
                DCLL_NCCL_OK(dp, dp->api.AllReduce(bucket[l], bucket[l], bucket_floats[l], ncclFloat32, ncclAvg, dp->comm, dp->side));
                DCLL_CUDA_OK(cudaEventRecord(dp->ev_red[l], dp->side));
                pending[l] = true;
                reserve();
            }
        }
    }
    for (int l = 0; l < n_layers; ++l) {
        rc = finish(l);
        if (rc != DCLL_OK) break;
    }
    set_reserved_sms(0);
    return rc;
}
