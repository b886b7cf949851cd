// C-ABI glue of libdcll_b200: argument checks, workspace carve-up, the per-layer step entry points and the
// whole-window driver that replaces the Python T-loop of train.py:249-251 / test_radio_ml.py:144-145.
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"

namespace dcll {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

// programmatic dependent launch is on unless DCLL_PDL=0 (read once)
bool pdl_enabled() {
    static int on = -1;
    if (on < 0) {
        const char *e = getenv("DCLL_PDL");
        on = (e && e[0] == '0') ? 0 : 1;
    }
    return on != 0;
}

// ---- launch counter + sampled CUDA-event profile ------------------------------------------------
static int64_t g_launches = 0;
void count_launch(const char *) { ++g_launches; }

static constexpr int PROF_MAX = 4096, PROF_LAYERS = 8;
static int g_prof_every = 0;
static int64_t g_prof_tick = 0;      // layer-steps seen
static bool g_prof_active = false;   // current layer-step is sampled
static int g_prof_n = 0;
static cudaEvent_t g_prof_ev[PROF_MAX][2];
static int g_prof_key[PROF_MAX];
static bool g_prof_init = false;

void prof_begin_layer_step() {
    if (!g_prof_every) { g_prof_active = false; return; }
    g_prof_active = (g_prof_tick++ % g_prof_every) == 0;
}

ProfScope::ProfScope(int kclass, int layer, cudaStream_t st_) : slot(-1), st(st_) {
    if (!g_prof_active || g_prof_n >= PROF_MAX) return;
    if (!g_prof_init) {
        for (int i = 0; i < PROF_MAX; ++i) cudaEventCreate(&g_prof_ev[i][0]), cudaEventCreate(&g_prof_ev[i][1]);
        g_prof_init = true;
    }
    slot = g_prof_n++;
    g_prof_key[slot] = kclass * PROF_LAYERS + (layer < PROF_LAYERS ? layer : PROF_LAYERS - 1);
    cudaEventRecord(g_prof_ev[slot][0], st);
}
ProfScope::~ProfScope() {
    if (slot >= 0) cudaEventRecord(g_prof_ev[slot][1], st);
}

WsLayout ws_layout(const dcll_conv_layer *L) {
    Geo g = geo_of(L);
    WsLayout w;
    // read-out partial blocks: enough CTAs (6 per SM) to hide the load latency of the single-buffered tiles
    w.n_ro = max(1, min(ceil_div(g.F, 64), 148 * 3));
    w.n_ro_tc = readout_tc_blocks(L);
    w.n_split = max(wgrad_splits(L), wgrad_tc_splits(L));   // room for either weight-gradient kernel
    size_t off = 0;
    w.off_ro_part = off;
    off = align_up(off + sizeof(float) * (size_t)max(w.n_ro, w.n_ro_tc) * L->B * g.Ktot, 256);
    w.off_go = off;
    off = align_up(off + sizeof(float) * (size_t)L->B * L->K, 256);
    w.off_go2 = off;
    off = align_up(off + sizeof(float) * (size_t)L->B * L->K, 256);
    w.off_wg_part = off;
    size_t wg_floats = (size_t)w.n_split * (g.nW + L->Cout);
    if (wgrad_tc2_supported(L)) wg_floats = max(wg_floats, wgrad_tc2_partial_floats());   // one compact block per CTA
    off = align_up(off + sizeof(float) * wg_floats, 256);
    w.off_wimg2 = off;
    off = align_up(off + conv_mma2_image_bytes(L), 256);
    w.total = off;
    return w;
}

AdamScalars adam_scalars(const dcll_adam &a, int64_t step_after) {
    // torch/optim/adam.py (_single_tensor_adam), python-float arithmetic
    double bc1 = 1.0 - pow(a.beta1, (double)step_after);
    double bc2 = 1.0 - pow(a.beta2, (double)step_after);
    double step_size = a.lr / bc1;
    AdamScalars s;
    s.wd = (float)a.weight_decay;
    s.beta1 = (float)a.beta1;
    s.one_minus_beta1 = (float)(1.0 - a.beta1);
    s.beta2 = (float)a.beta2;
    s.one_minus_beta2 = (float)(1.0 - a.beta2);
    s.neg_step_size = (float)(-step_size);
    s.bc2_sqrt = (float)sqrt(bc2);
    s.eps = (float)a.eps;
    return s;
}

OptScalars opt_scalars(const dcll_adam &a, const dcll_optim &o, int64_t step_after, float *mu_product) {
    // torch/optim/{adam,adamax,nadam,radam}.py (_single_tensor_*), python-float arithmetic on the float32 step count
    const double t = (double)step_after, lr = a.lr, b1 = a.beta1, b2 = a.beta2, wd = a.weight_decay;
    const bool decoupled = o.kind == DCLL_OPT_ADAMW || ((o.kind == DCLL_OPT_NADAM || o.kind == DCLL_OPT_RADAM) && o.decoupled_wd);
    OptScalars s = {};
    s.kind = o.kind;
    s.decay = (decoupled && wd != 0.0) ? (float)(1.0 - lr * wd) : 1.f;
    s.wd = decoupled ? 0.f : (float)wd;
    s.one_minus_beta1 = (float)(1.0 - b1);
    s.beta2 = (float)b2;
    s.one_minus_beta2 = (float)(1.0 - b2);
    s.eps = (float)a.eps;
    const double bc1 = 1.0 - pow(b1, t), bc2 = 1.0 - pow(b2, t);
    if (o.kind == DCLL_OPT_ADAMW) {
        s.c0 = (float)(-(lr / bc1));
        s.c1 = (float)sqrt(bc2);
    } else if (o.kind == DCLL_OPT_ADAMAX) {
        s.c0 = (float)(-(lr / bc1));
    } else if (o.kind == DCLL_OPT_NADAM) {
        const double mu = b1 * (1.0 - 0.5 * pow(0.96, t * o.momentum_decay));
        const double mu_next = b1 * (1.0 - 0.5 * pow(0.96, (t + 1.0) * o.momentum_decay));
        *mu_product = *mu_product * (float)mu;                    // mu_product *= mu: a float32 tensor times a python float
        const double mp = (double)*mu_product, mp_next = mp * mu_next;
        s.c0 = (float)bc2;
        s.c1 = (float)(-lr * (1.0 - mu) / (1.0 - mp));
        s.c2 = (float)((-lr * mu_next) / (1.0 - mp_next));
    } else {                                                        // DCLL_OPT_RADAM
        const double rho_inf = 2.0 / (1.0 - b2) - 1.0;
        const double rho_t = rho_inf - 2.0 * t * pow(b2, t) / bc2;
        s.rect = rho_t > 5.0;
        s.c0 = (float)bc1;
        s.c1 = (float)lr;
        if (s.rect) {
            s.c2 = (float)pow(bc2, 0.5);
            s.c3 = (float)pow((rho_t - 4.0) * (rho_t - 2.0) * rho_inf / ((rho_inf - 4.0) * (rho_inf - 2.0) * rho_t), 0.5);
        }
    }
    return s;
}

const OptScalars *next_opt_scalars(const dcll_adam &a, dcll_optim *o, OptScalars *buf) {
    if (!opt_active(o)) return nullptr;
    *buf = opt_scalars(a, *o, a.step + 1, &o->mu_product);
    return buf;
}

static int check_opt(const dcll_optim *opt, int n, const char *who) {
    for (int i = 0; opt && i < n; ++i)
        DCLL_REQUIRE(opt[i].kind >= DCLL_OPT_ADAM && opt[i].kind <= DCLL_OPT_RADAM, DCLL_EINVAL, "%s: unknown update rule %d", who,
                     opt[i].kind);
    return DCLL_OK;
}
int dp_check_opt(const dcll_optim *opt, int n_layers) { return check_opt(opt, 2 * n_layers, "dcll_net_window_dp_opt"); }

static int check_layer(const dcll_conv_layer *L, const char *who) {
    DCLL_REQUIRE(L, DCLL_EINVAL, "%s: null layer", who);
    DCLL_REQUIRE(L->B > 0 && L->Cin > 0 && L->H > 0 && L->W > 0 && L->Cout > 0 && L->K > 0, DCLL_EINVAL,
                 "%s: non-positive dimension", who);
    Geo g = geo_of(L);
    DCLL_REQUIRE(g.Hc > 0 && g.Wc > 0, DCLL_EINVAL, "%s: kernel larger than the padded input", who);
    DCLL_REQUIRE(L->poolH >= 1 && L->poolH <= 2 && L->poolW >= 1 && L->poolW <= 2, DCLL_EUNSUPPORTED,
                 "%s: pooling (%d,%d): each axis must be 1 or 2", who, L->poolH, L->poolW);
    DCLL_REQUIRE(g.Hp > 0 && g.Wp > 0, DCLL_EINVAL, "%s: pooled output is empty (%dx%d conv output, pooling (%d,%d))", who,
                 g.Hc, g.Wc, L->poolH, L->poolW);
    DCLL_REQUIRE(L->precision == DCLL_PREC_FP32 || prec_tc(L), DCLL_EINVAL, "%s: unknown precision mode %d",
                 who, L->precision);
    DCLL_REQUIRE(!prec_tc(L) || !tc_supported(L) || (L->weight_mma && L->eps1_mma), DCLL_EINVAL,
                 "%s: the bf16x3 tensor-core conv needs weight_mma and eps1_mma", who);
    DCLL_REQUIRE(L->alpha && L->alphas && L->tau_m && L->tau_s && L->weight && L->weight_t && L->bias && L->wo && L->bo,
                 DCLL_EINVAL, "%s: null parameter pointer", who);
    DCLL_REQUIRE(!L->output_layer || (L->wout && L->bout && L->output), DCLL_EINVAL, "%s: output layer without output_", who);
    DCLL_REQUIRE(L->eps0[0] && L->eps0[1] && L->eps1[0] && L->eps1[1], DCLL_EINVAL, "%s: null state pointer", who);
    DCLL_REQUIRE(!(L->wrp > 0.f) || L->arp, DCLL_EINVAL, "%s: refractory layer without arp state", who);
    DCLL_REQUIRE(L->spikes && L->pv && L->pvoutput, DCLL_EINVAL, "%s: null output pointer", who);
    DCLL_REQUIRE(L->poolH * L->poolW == 1 || L->pool_idx, DCLL_EINVAL, "%s: pooled layer without pool_idx", who);
    DCLL_REQUIRE(L->x_mode == DCLL_X_DENSE || (L->x_mode == DCLL_X_CELLS && L->Cin == 1), DCLL_EINVAL,
                 "%s: cell input needs Cin == 1", who);
    DCLL_REQUIRE(L->workspace && L->workspace_bytes >= ws_layout(L).total, DCLL_EINVAL,
                 "%s: workspace too small (%zu < %zu)", who, L->workspace_bytes, ws_layout(L).total);
    const void *al[] = {L->arp, L->spikes, L->pv, L->pvmem, L->weight_t, L->workspace};
    for (const void *q : al) DCLL_REQUIRE(((uintptr_t)q & 15) == 0, DCLL_EINVAL, "%s: tensor not 16-byte aligned", who);
    return DCLL_OK;
}

static int g_reserved_sms = 0;
int sm_budget() { return 148 - g_reserved_sms; }
void set_reserved_sms(int n) { g_reserved_sms = n < 0 ? 0 : (n > 64 ? 64 : n); }

// in-kernel stopwatch blocks (common.cuh): allocated on first use when DCLL_TIMELINE=1
static unsigned long long *g_timeline = nullptr;
static int g_layer = 0;  // layer index of the step being enqueued (profile key only)
unsigned long long *timeline_buf(int kind) {
    static int on = -1, only_layer = -1;                    // DCLL_TIMELINE_LAYER=l: only launches of layer l write their block
    if (on < 0) {
        const char *e = getenv("DCLL_TIMELINE");
        const char *el = getenv("DCLL_TIMELINE_LAYER");
        only_layer = el ? atoi(el) : -1;
        on = (e && e[0] == '1') ? 1 : 0;
        if (on) {
            const size_t bytes = sizeof(unsigned long long) * TL_KINDS * TL_CTAS * TL_SLOTS;
            if (cudaMalloc(&g_timeline, bytes) != cudaSuccess || cudaMemset(g_timeline, 0, bytes) != cudaSuccess) g_timeline = nullptr, on = 0;
        }
    }
    if (only_layer >= 0 && g_layer != only_layer) return nullptr;
    return (on && kind >= 0 && kind < TL_KINDS) ? g_timeline + (size_t)kind * TL_CTAS * TL_SLOTS : nullptr;
}

int prof_layer() { return g_layer; }

static int step_fwd(dcll_conv_layer *L, const void *x, const float *target, int loss_kind, int32_t *clout, float *loss_out,
                    cudaStream_t st, const dcll_conv_layer *next = nullptr, bool trace_done = false, int spike_io = SPK_WRITE) {
    prof_begin_layer_step();
    int rc;
    {
        ProfScope ps(KC_CONV_FWD, g_layer, st);
        rc = launch_conv_fwd(L, x, st, next, trace_done, spike_io);
    }
    if (rc != DCLL_OK) return rc;
    L->cur ^= 1;
    ProfScope ps(KC_READOUT_FWD, g_layer, st);
    return launch_readout_fwd(L, target, loss_kind, clout, loss_out, st);
}

// opt: the rules of adam_i2h / adam_out, or null (Adam)
static int step_bwd(dcll_conv_layer *L, dcll_train_args *a, cudaStream_t st, dcll_optim *opt = nullptr) {
    int rc;
    OptScalars buf_i2h, buf_out;
    const OptScalars *so_i2h = nullptr, *so_out = nullptr;
    if (a->apply_update && opt) {
        so_i2h = next_opt_scalars(a->adam_i2h, &opt[0], &buf_i2h);
        if (L->output_layer) so_out = next_opt_scalars(a->adam_out, &opt[1], &buf_out);
    }
    {
        ProfScope ps(KC_READOUT_BWD, g_layer, st);
        rc = launch_readout_bwd(L, a, st, so_out);
    }
    if (rc != DCLL_OK) return rc;
    {
        ProfScope ps(KC_WGRAD, g_layer, st);
        rc = launch_wgrad(L, a, st, so_i2h);
    }
    if (rc != DCLL_OK) return rc;
    if (a->apply_update) {
        a->adam_i2h.step += 1;
        if (L->output_layer) a->adam_out.step += 1;
    }
    return DCLL_OK;
}

static int check_train(const dcll_conv_layer *L, const dcll_train_args *a, const char *who) {
    DCLL_REQUIRE(a, DCLL_EINVAL, "%s: null train args", who);
    DCLL_REQUIRE(L->g_u, DCLL_EINVAL, "%s: null g_u scratch", who);
    DCLL_REQUIRE(a->loss_kind >= DCLL_LOSS_SMOOTHL1 && a->loss_kind <= DCLL_LOSS_HINGE, DCLL_EINVAL, "%s: unknown loss", who);
    DCLL_REQUIRE(a->loss_kind != DCLL_LOSS_EXTERNAL || (a->g_o_ext && (!L->output_layer || a->g_o2_ext)), DCLL_EINVAL,
                 "%s: external loss gradient missing", who);
    if (a->apply_update) {
        DCLL_REQUIRE(a->adam_i2h.m_w && a->adam_i2h.v_w && a->adam_i2h.m_b && a->adam_i2h.v_b, DCLL_EINVAL,
                     "%s: null Adam state (i2h)", who);
        DCLL_REQUIRE(!L->output_layer || (a->adam_out.m_w && a->adam_out.v_w && a->adam_out.m_b && a->adam_out.v_b),
                     DCLL_EINVAL, "%s: null Adam state (output_)", who);
    } else {
        DCLL_REQUIRE(a->grad_w && a->grad_b, DCLL_EINVAL, "%s: apply_update == 0 needs gradient buffers", who);
        DCLL_REQUIRE(!L->output_layer || (a->grad_wout && a->grad_bout), DCLL_EINVAL, "%s: needs output_ gradient buffers",
                     who);
    }
    return DCLL_OK;
}

// entry points of the data-parallel driver (dp.cu) into the per-layer steps above
int dp_step_fwd(dcll_conv_layer *L, const void *x, const float *target, int loss_kind, int32_t *clout, cudaStream_t st,
                const dcll_conv_layer *next, bool trace_done, int spike_io, int layer) {
    g_layer = layer;
    return step_fwd(L, x, target, loss_kind, clout, nullptr, st, next, trace_done, spike_io);
}
int dp_step_bwd(dcll_conv_layer *L, dcll_train_args *a, cudaStream_t st, int layer) {
    g_layer = layer;
    return step_bwd(L, a, st);
}
int dp_check(const dcll_conv_layer *layers, const dcll_train_args *train, int n_layers) {
    for (int l = 0; l < n_layers; ++l) {
        int rc = check_layer(&layers[l], "dcll_net_window_dp");
        if (rc != DCLL_OK) return rc;
        rc = check_train(&layers[l], &train[l], "dcll_net_window_dp");
        if (rc != DCLL_OK) return rc;
        DCLL_REQUIRE(train[l].loss_kind != DCLL_LOSS_EXTERNAL, DCLL_EUNSUPPORTED, "dcll_net_window_dp: external loss gradients need the per-step API");
        DCLL_REQUIRE(train[l].adam_i2h.m_w && train[l].adam_i2h.v_w && train[l].adam_i2h.m_b && train[l].adam_i2h.v_b, DCLL_EINVAL,
                     "dcll_net_window_dp: null Adam state (i2h)");
        DCLL_REQUIRE(!layers[l].output_layer || (train[l].adam_out.m_w && train[l].adam_out.v_w && train[l].adam_out.m_b && train[l].adam_out.v_b),
                     DCLL_EINVAL, "dcll_net_window_dp: null Adam state (output_)");
        if (l > 0) {
            Geo gp = geo_of(&layers[l - 1]);
            DCLL_REQUIRE(layers[l].x_mode == DCLL_X_DENSE && layers[l].Cin == layers[l - 1].Cout && layers[l].H == gp.Hp &&
                             layers[l].W == gp.Wp && layers[l].B == layers[0].B,
                         DCLL_EINVAL, "dcll_net_window_dp: layer %d does not chain onto layer %d", l, l - 1);
        }
    }
    return DCLL_OK;
}

__global__ void vote_kernel(const int32_t *__restrict__ clout, int T, int t_stride, int B, int K, int32_t *__restrict__ pred) {
    pdl_entry();
    // Counter(...).most_common(1): highest count, first-seen wins ties (dcll/pytorch_libdcll.py:51)
    int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    int cnt[64], first[64];
    for (int k = 0; k < 64; ++k) cnt[k] = 0, first[k] = 0x7fffffff;
    for (int t = 0; t < T; ++t) {
        int c = clout[(size_t)t * t_stride + b];
        if (c >= 0 && c < K) {
            if (cnt[c] == 0) first[c] = t;
            cnt[c]++;
        }
    }
    int best = 0;
    for (int k = 1; k < K; ++k)
        if (cnt[k] > cnt[best] || (cnt[k] == cnt[best] && first[k] < first[best])) best = k;
    pred[b] = best;
}

__global__ void quantize_kernel(const float *__restrict__ w, int rows, int cols, int8_t *__restrict__ codes,
                                float *__restrict__ scales) {
    pdl_entry();
    // one CTA per output channel: s = max|w| / 127 (1 if the row is all zero), q = clamp(rint(w / s), -127, 127)
    __shared__ float red[32];
    __shared__ float s_scale;
    const int r = blockIdx.x;
    const float *row = w + (size_t)r * cols;
    float m = 0.f;
    for (int i = threadIdx.x; i < cols; i += blockDim.x) m = fmaxf(m, fabsf(row[i]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        float mm = 0.f;
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) mm = fmaxf(mm, red[i]);
        float s = mm > 0.f ? __fdiv_rn(mm, 127.f) : 1.f;
        s_scale = s;
        scales[r] = s;
    }
    __syncthreads();
    const float s = s_scale;
    for (int i = threadIdx.x; i < cols; i += blockDim.x) {
        float q = rintf(__fdiv_rn(row[i], s));
        q = fminf(fmaxf(q, -127.f), 127.f);
        codes[(size_t)r * cols + i] = (int8_t)q;
    }
}

__global__ void dequantize_kernel(const int8_t *__restrict__ codes, const float *__restrict__ scales, int rows, int cols,
                                  float *__restrict__ w) {
    pdl_entry();
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (i >= (size_t)rows * cols) return;
    w[i] = __fmul_rn((float)codes[i], scales[i / cols]);
}

}  // namespace dcll

using namespace dcll;

extern "C" __attribute__((visibility("default"))) int dcll_abi_version(void) { return DCLL_ABI_VERSION; }

extern "C" __attribute__((visibility("default"))) int64_t dcll_launch_count(int reset) {
    int64_t v = g_launches;
    if (reset) g_launches = 0;
    return v;
}

extern "C" __attribute__((visibility("default"))) int dcll_profile_enable(int every_n) {
    DCLL_REQUIRE(every_n >= 0, DCLL_EINVAL, "dcll_profile_enable: every_n must be >= 0");
    g_prof_every = every_n;
    g_prof_tick = 0;
    g_prof_active = false;
    return DCLL_OK;
}

extern "C" __attribute__((visibility("default"))) int dcll_profile_read(double *ms, int64_t *n) {
    DCLL_REQUIRE(ms && n, DCLL_EINVAL, "dcll_profile_read: null output");
    for (int i = 0; i < KC_COUNT * PROF_LAYERS; ++i) ms[i] = 0.0, n[i] = 0;
    for (int i = 0; i < g_prof_n; ++i) {
        DCLL_CUDA_OK(cudaEventSynchronize(g_prof_ev[i][1]));
        float t = 0.f;
        DCLL_CUDA_OK(cudaEventElapsedTime(&t, g_prof_ev[i][0], g_prof_ev[i][1]));
        ms[g_prof_key[i]] += t;
        n[g_prof_key[i]] += 1;
    }
    g_prof_n = 0;
    return DCLL_OK;
}
extern "C" __attribute__((visibility("default"))) int dcll_debug_timeline(uint64_t *out, int n_u64) {
    const int n = TL_KINDS * TL_CTAS * TL_SLOTS;
    DCLL_REQUIRE(out && n_u64 >= n, DCLL_EINVAL, "dcll_debug_timeline: need room for %d values", n);
    timeline_buf(0);
    DCLL_REQUIRE(g_timeline, DCLL_EINVAL, "dcll_debug_timeline: the stopwatch is off (DCLL_TIMELINE=1 before the first launch)");
    DCLL_CUDA_OK(cudaDeviceSynchronize());
    DCLL_CUDA_OK(cudaMemcpy(out, g_timeline, sizeof(uint64_t) * n, cudaMemcpyDeviceToHost));
    return n;
}
extern "C" __attribute__((visibility("default"))) const char *dcll_last_error(void) { return g_err; }
extern "C" __attribute__((visibility("default"))) size_t dcll_sizeof_conv_layer(void) { return sizeof(dcll_conv_layer); }
extern "C" __attribute__((visibility("default"))) size_t dcll_sizeof_train_args(void) { return sizeof(dcll_train_args); }

extern "C" __attribute__((visibility("default"))) size_t dcll_conv_workspace_bytes(const dcll_conv_layer *L) {
    if (!L || L->B <= 0 || L->Cin <= 0 || L->Cout <= 0 || L->K <= 0) return 0;
    return ws_layout(L).total;
}

extern "C" __attribute__((visibility("default"))) int dcll_conv_step_fwd(dcll_conv_layer *L, const void *x, int32_t *clout, void *stream) {
    int rc = check_layer(L, "dcll_conv_step_fwd");
    if (rc != DCLL_OK) return rc;
    DCLL_REQUIRE(x, DCLL_EINVAL, "dcll_conv_step_fwd: null input");
    return step_fwd(L, x, nullptr, 0, clout, nullptr, (cudaStream_t)stream);
}

// bool tc_trace_fusable(L, next) is defined in conv_fwd_tc.cu
extern "C" __attribute__((visibility("default"))) int dcll_conv_chain_fusable(const dcll_conv_layer *L, const dcll_conv_layer *next) {
    return tc_trace_fusable(L, next) ? 1 : 0;
}

extern "C" __attribute__((visibility("default"))) int dcll_conv_step_fwd_chain(dcll_conv_layer *L, const dcll_conv_layer *next, int trace_done,
                                                                                const void *x, int32_t *clout, void *stream) {
    int rc = check_layer(L, "dcll_conv_step_fwd_chain");
    if (rc != DCLL_OK) return rc;
    DCLL_REQUIRE(x, DCLL_EINVAL, "dcll_conv_step_fwd_chain: null input");
    if (next) {
        rc = check_layer(const_cast<dcll_conv_layer *>(next), "dcll_conv_step_fwd_chain (next)");
        if (rc != DCLL_OK) return rc;
        DCLL_REQUIRE(tc_trace_fusable(L, next), DCLL_EINVAL, "dcll_conv_step_fwd_chain: the two layers are not fusable (dcll_conv_chain_fusable)");
    }
    return step_fwd(L, x, nullptr, 0, clout, nullptr, (cudaStream_t)stream, next, trace_done != 0);
}

extern "C" __attribute__((visibility("default"))) int dcll_conv_core_fwd(dcll_conv_layer *L, const void *x, void *stream) {
    DCLL_REQUIRE(L && x, DCLL_EINVAL, "dcll_conv_core_fwd: null argument");
    DCLL_REQUIRE(L->poolH == 1 && L->poolW == 1, DCLL_EINVAL, "dcll_conv_core_fwd: the i2h core has no pooling");
    DCLL_REQUIRE(L->alpha && L->alphas && L->tau_m && L->tau_s && L->weight_t && L->bias && L->eps0[0] && L->eps0[1] &&
                     L->eps1[0] && L->eps1[1] && L->spikes && L->pv && (!(L->wrp > 0.f) || L->arp),
                 DCLL_EINVAL, "dcll_conv_core_fwd: null tensor");
    DCLL_REQUIRE(L->x_mode == DCLL_X_DENSE || L->Cin == 1, DCLL_EINVAL, "dcll_conv_core_fwd: cell input needs Cin == 1");
    int rc = launch_conv_fwd(L, x, (cudaStream_t)stream);
    if (rc == DCLL_OK) L->cur ^= 1;
    return rc;
}

extern "C" __attribute__((visibility("default"))) int dcll_conv_step_bwd_update(dcll_conv_layer *L, dcll_train_args *a, void *stream) {
    return dcll_conv_step_bwd_update_opt(L, a, nullptr, stream);
}

extern "C" __attribute__((visibility("default"))) int dcll_conv_step_bwd_update_opt(dcll_conv_layer *L, dcll_train_args *a, dcll_optim *opt,
                                                                                     void *stream) {
    int rc = check_layer(L, "dcll_conv_step_bwd_update");
    if (rc != DCLL_OK) return rc;
    rc = check_train(L, a, "dcll_conv_step_bwd_update");
    if (rc != DCLL_OK) return rc;
    rc = check_opt(opt, 2, "dcll_conv_step_bwd_update_opt");
    if (rc != DCLL_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (a->loss_kind == DCLL_LOSS_EXTERNAL) {
        WsLayout ws = ws_layout(L);
        char *base = (char *)L->workspace;
        size_t n = sizeof(float) * (size_t)L->B * L->K;
        DCLL_CUDA_OK(cudaMemcpyAsync(base + ws.off_go, a->g_o_ext, n, cudaMemcpyDeviceToDevice, st));
        if (L->output_layer) DCLL_CUDA_OK(cudaMemcpyAsync(base + ws.off_go2, a->g_o2_ext, n, cudaMemcpyDeviceToDevice, st));
    } else {
        DCLL_REQUIRE(a->target, DCLL_EINVAL, "dcll_conv_step_bwd_update: null target");
        if (a->loss_out) DCLL_CUDA_OK(cudaMemsetAsync(a->loss_out, 0, sizeof(float), st));
        rc = launch_loss_grad(L, a->target, a->loss_kind, a->loss_out, st);
        if (rc != DCLL_OK) return rc;
    }
    return step_bwd(L, a, st, opt);
}

// Adam, or the rule of the slot, over flat parameters (w, b) with gradients (gw, gb)
static int flat_update(dcll_adam &a, dcll_optim *o, float *w, const float *gw, size_t nw, float *b, const float *gb, size_t nb,
                       cudaStream_t st) {
    OptScalars buf;
    const OptScalars *so = next_opt_scalars(a, o, &buf);
    const AdamScalars sc = adam_scalars(a, a.step + 1);
    int rc = so ? launch_opt_flat(w, gw, a.m_w, a.v_w, nw, *so, st) : launch_adam_flat(w, gw, a.m_w, a.v_w, nw, sc, st);
    if (rc != DCLL_OK) return rc;
    rc = so ? launch_opt_flat(b, gb, a.m_b, a.v_b, nb, *so, st) : launch_adam_flat(b, gb, a.m_b, a.v_b, nb, sc, st);
    if (rc != DCLL_OK) return rc;
    a.step += 1;
    return DCLL_OK;
}

extern "C" __attribute__((visibility("default"))) int dcll_conv_apply_update(dcll_conv_layer *L, dcll_train_args *a, void *stream) {
    return dcll_conv_apply_update_opt(L, a, nullptr, stream);
}

extern "C" __attribute__((visibility("default"))) int dcll_conv_apply_update_opt(dcll_conv_layer *L, dcll_train_args *a, dcll_optim *opt,
                                                                                  void *stream) {
    int rc = check_layer(L, "dcll_conv_apply_update");
    if (rc != DCLL_OK) return rc;
    DCLL_REQUIRE(a && a->grad_w && a->grad_b, DCLL_EINVAL, "dcll_conv_apply_update: null gradients");
    rc = check_opt(opt, 2, "dcll_conv_apply_update_opt");
    if (rc != DCLL_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    Geo g = geo_of(L);
    rc = flat_update(a->adam_i2h, opt, L->weight, a->grad_w, (size_t)g.nW, L->bias, a->grad_b, (size_t)L->Cout, st);
    if (rc != DCLL_OK) return rc;
    if (L->output_layer) {
        DCLL_REQUIRE(a->grad_wout && a->grad_bout, DCLL_EINVAL, "dcll_conv_apply_update: null output_ gradients");
        rc = flat_update(a->adam_out, opt ? opt + 1 : nullptr, L->wout, a->grad_wout, (size_t)L->K * g.F, L->bout, a->grad_bout,
                         (size_t)L->K, st);
        if (rc != DCLL_OK) return rc;
    }
    return dcll_conv_sync_weights(L, stream);
}

int dcll::dense_flat_update(dcll_adam &a, dcll_optim *o, float *w, const float *gw, size_t nw, float *b, const float *gb, size_t nb,
                      cudaStream_t st) {
    return flat_update(a, o, w, gw, nw, b, gb, nb, st);
}

// 19 equal bins over [0,1], last bin closed on the right (numpy.histogram with bins = linspace(0,1,20)).
// pv sits near 0.5 for most neurons, so almost every element of a warp lands in the same bin: the lanes are grouped with
// match.any and one lane per distinct bin adds the group's population to a warp-private row (a shared atomic per element
// serialised on that one address: 0.21 ms for 134 MB; this form streams at HBM speed).
__global__ void __launch_bounds__(256) activity_hist_kernel(const float *__restrict__ pv, size_t n, int32_t *__restrict__ hist) {
    pdl_entry();
    __shared__ int sh[8][20];                                       // [warp][bin], bin 19 = out of range / padding
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < 8 * 20; i += 256) (&sh[0][0])[i] = 0;
    __syncthreads();
    auto add = [&](float v) {
        const int b = (v >= 0.f && v <= 1.f) ? min((int)(v * 19.f), 18) : 19;
        const unsigned m = __match_any_sync(0xffffffffu, b);
        if (lane == __ffs(m) - 1) atomicAdd(&sh[warp][b], __popc(m));
    };
    const bool vec = (reinterpret_cast<uintptr_t>(pv) & 15) == 0;
    const size_t n4 = vec ? n / 4 : 0;
    // uniform trip count per CTA: every lane takes part in every match
    for (size_t i0 = blockIdx.x * (size_t)256; i0 < n4; i0 += (size_t)gridDim.x * 256) {
        const size_t i = i0 + threadIdx.x;
        float4 v = make_float4(-1.f, -1.f, -1.f, -1.f);
        if (i < n4) v = __ldg(reinterpret_cast<const float4 *>(pv) + i);
        add(v.x), add(v.y), add(v.z), add(v.w);
    }
    for (size_t i0 = 4 * n4 + blockIdx.x * (size_t)256; i0 < n; i0 += (size_t)gridDim.x * 256) {
        const size_t i = i0 + threadIdx.x;
        add(i < n ? pv[i] : -1.f);
    }
    __syncthreads();
    if (threadIdx.x < 19) {
        int c = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) c += sh[w][threadIdx.x];
        if (c) atomicAdd(&hist[threadIdx.x], c);
    }
}

extern "C" __attribute__((visibility("default"))) int dcll_net_window(dcll_conv_layer *layers, dcll_train_args *train, int n_layers,
                                                                       const void *x0, const float *target,
                                                                       int64_t target_t_stride, int T, int train_mode, int burnin,
                                                                       const int32_t *iter0, int32_t *clout, void *stream) {
    return dcll_net_window_stats(layers, train, n_layers, x0, target, target_t_stride, T, train_mode, burnin, iter0, clout, nullptr, 0,
                                 0, stream);
}

extern "C" __attribute__((visibility("default"))) int dcll_net_window_stats(dcll_conv_layer *layers, dcll_train_args *train, int n_layers, const void *x0,
                               const float *target, int64_t target_t_stride, int T, int train_mode, int burnin,
                               const int32_t *iter0, int32_t *clout, int32_t *hist, int hist_every, int hist_cap, void *stream) {
    return dcll_net_window_stats_opt(layers, train, nullptr, n_layers, x0, target, target_t_stride, T, train_mode, burnin, iter0, clout,
                                     hist, hist_every, hist_cap, stream);
}

// opt: the update rules opt[2l] (train[l].adam_i2h) and opt[2l + 1] (train[l].adam_out), or null (Adam everywhere)
extern "C" __attribute__((visibility("default"))) int dcll_net_window_stats_opt(dcll_conv_layer *layers, dcll_train_args *train, dcll_optim *opt,
                               int n_layers, const void *x0, const float *target, int64_t target_t_stride, int T, int train_mode,
                               int burnin, const int32_t *iter0, int32_t *clout, int32_t *hist, int hist_every, int hist_cap,
                               void *stream) {
    DCLL_REQUIRE(layers && n_layers > 0 && x0 && T > 0 && iter0, DCLL_EINVAL, "dcll_net_window: bad arguments");
    DCLL_REQUIRE(!hist || (hist_every > 0 && hist_cap > 0), DCLL_EINVAL, "dcll_net_window: bad histogram arguments");
    int hist_n[16] = {0};
    DCLL_REQUIRE(!hist || n_layers <= 16, DCLL_EINVAL, "dcll_net_window: statistics support at most 16 layers");
    DCLL_REQUIRE(!train_mode || (train && target), DCLL_EINVAL, "dcll_net_window: training needs train args and a target");
    int rc0 = check_opt(opt, 2 * n_layers, "dcll_net_window_stats_opt");
    if (rc0 != DCLL_OK) return rc0;
    for (int l = 0; l < n_layers; ++l) {
        int rc = check_layer(&layers[l], "dcll_net_window");
        if (rc != DCLL_OK) return rc;
        if (train_mode) {
            rc = check_train(&layers[l], &train[l], "dcll_net_window");
            if (rc != DCLL_OK) return rc;
            DCLL_REQUIRE(train[l].apply_update, DCLL_EINVAL, "dcll_net_window: apply_update must be set");
            DCLL_REQUIRE(train[l].loss_kind != DCLL_LOSS_EXTERNAL, DCLL_EUNSUPPORTED,
                         "dcll_net_window: external loss gradients need the per-step API");
        }
        if (l > 0) {
            Geo gp = geo_of(&layers[l - 1]);
            DCLL_REQUIRE(layers[l].x_mode == DCLL_X_DENSE && layers[l].Cin == layers[l - 1].Cout && layers[l].H == gp.Hp &&
                             layers[l].W == gp.Wp && layers[l].B == layers[0].B,
                         DCLL_EINVAL, "dcll_net_window: layer %d does not chain onto layer %d", l, l - 1);
        }
    }
    cudaStream_t st = (cudaStream_t)stream;
    const dcll_conv_layer &L0 = layers[0];
    const size_t x_stride = L0.x_mode == DCLL_X_CELLS ? (size_t)L0.B * 2 * sizeof(int32_t)
                                                      : (size_t)L0.B * L0.Cin * L0.H * L0.W * sizeof(float);
    for (int t = 0; t < T; ++t) {
        const float *tgt = target ? target + (size_t)t * target_t_stride : nullptr;
        for (int l = 0; l < n_layers; ++l) {
            dcll_conv_layer *L = &layers[l];
            g_layer = l;
            const void *x = l == 0 ? (const void *)((const char *)x0 + (size_t)t * x_stride) : (const void *)layers[l - 1].spikes;
            const int it = iter0[l] + t + 1;                       // DCLLBase.forward :656
            const bool do_train = train_mode && it >= burnin;      // train_dcll :692
            int32_t *co = clout ? clout + ((size_t)t * n_layers + l) * L->B : nullptr;
            // the trace update of layer l+1 rides in the epilogue of layer l's tensor-core convolution where that is free
            const bool fuse_next = l + 1 < n_layers && tc_trace_fusable(L, &layers[l + 1]);
            const bool trace_done = l > 0 && tc_trace_fusable(&layers[l - 1], L);
            // the spike tensor of this step is stored only when somebody reads it -- the next layer's own trace pass -- and then as
            // packed bits between two tensor-core layers
            int rc = step_fwd(L, x, do_train ? tgt : nullptr, do_train ? train[l].loss_kind : 0, co, nullptr, st,
                              fuse_next ? &layers[l + 1] : nullptr, trace_done, spike_io_of(layers, l, n_layers, fuse_next, trace_done));
            if (rc != DCLL_OK) return rc;
            if (hist && (it % hist_every) == 0 && hist_n[l] < hist_cap) {          // DCLLBase.forward :658-661
                Geo g = geo_of(L);
                const size_t n = (size_t)L->B * g.F;
                int32_t *dst = hist + ((size_t)l * hist_cap + hist_n[l]++) * 19;
                const int blocks = (int)(n / 1024 / 4 + 1 < 148 * 8 ? n / 1024 / 4 + 1 : 148 * 8);
                launch_k(activity_hist_kernel, blocks, 256, 0, st, L->pv, n, dst);
                DCLL_LAUNCH_OK("activity_hist_kernel");
            }
            if (do_train) {
                rc = step_bwd(L, &train[l], st, opt ? opt + 2 * l : nullptr);
                if (rc != DCLL_OK) return rc;
            }
        }
    }
    return DCLL_OK;
}

extern "C" __attribute__((visibility("default"))) int dcll_vote(const int32_t *clout, int T, int t_stride, int B, int K, int32_t *pred, void *stream) {
    DCLL_REQUIRE(clout && pred && T > 0 && B > 0 && K > 0 && K <= 64, DCLL_EINVAL, "dcll_vote: bad arguments (K <= 64)");
    launch_k(vote_kernel, ceil_div(B, 128), 128, 0, (cudaStream_t)stream, clout, T, t_stride, B, K, pred);
    DCLL_LAUNCH_OK("vote_kernel");
    return DCLL_OK;
}

extern "C" __attribute__((visibility("default"))) int dcll_quantize(const float *w, int rows, int cols, int8_t *codes, float *scales, void *stream) {
    DCLL_REQUIRE(w && codes && scales && rows > 0 && cols > 0, DCLL_EINVAL, "dcll_quantize: bad arguments");
    launch_k(quantize_kernel, rows, 256, 0, (cudaStream_t)stream, w, rows, cols, codes, scales);
    DCLL_LAUNCH_OK("quantize_kernel");
    return DCLL_OK;
}

extern "C" __attribute__((visibility("default"))) int dcll_dequantize(const int8_t *codes, const float *scales, int rows, int cols, float *w, void *stream) {
    DCLL_REQUIRE(w && codes && scales && rows > 0 && cols > 0, DCLL_EINVAL, "dcll_dequantize: bad arguments");
    size_t n = (size_t)rows * cols;
    launch_k(dequantize_kernel, (unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream, codes, scales, rows, cols, w);
    DCLL_LAUNCH_OK("dequantize_kernel");
    return DCLL_OK;
}
