// Shared helpers for libdcll_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/dcll_b200.h"

namespace dcll {

void set_error(const char *fmt, ...);

#define DCLL_REQUIRE(cond, code, ...)              \
    do {                                           \
        if (!(cond)) {                             \
            ::dcll::set_error(__VA_ARGS__);        \
            return (code);                         \
        }                                          \
    } while (0)

#define DCLL_CUDA_OK(expr)                                                                      \
    do {                                                                                        \
        cudaError_t _e = (expr);                                                                \
        if (_e != cudaSuccess) {                                                                \
            ::dcll::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                              __LINE__);                                                        \
            return DCLL_ECUDA;                                                                  \
        }                                                                                       \
    } while (0)

// Kernel classes for the launch counter and the optional CUDA-event profile (dcll_profile_*).
enum KClass { KC_ENCODE = 0, KC_CONV_FWD, KC_READOUT_FWD, KC_READOUT_BWD, KC_WGRAD, KC_ADAM, KC_MISC, KC_TRACE, KC_COUNT };
int prof_layer();   // layer index of the step being enqueued (profile key only)
void count_launch(const char *name);
// RAII: brackets the launches of one kernel class with CUDA events when profiling samples this step.
struct ProfScope {
    int slot;
    cudaStream_t st;
    ProfScope(int kclass, int layer, cudaStream_t st);
    ~ProfScope();
};

#define DCLL_LAUNCH_OK(name)                                                                         \
    do {                                                                                             \
        ::dcll::count_launch(name);                                                                  \
        cudaError_t _e = cudaGetLastError();                                                         \
        if (_e != cudaSuccess) {                                                                     \
            ::dcll::set_error("launch of %s failed: %s", name, cudaGetErrorString(_e));              \
            return DCLL_ECUDA;                                                                       \
        }                                                                                            \
    } while (0)

// ---- programmatic dependent launch (PDL) -------------------------------------------------------------------------------
// Every launch goes through launch_k (cudaLaunchKernelEx + programmaticStreamSerialization) and every kernel starts with
// pdl_entry() = griddepcontrol.wait: the next kernel of the stream is scheduled while the CTAs of the previous one are still
// retiring (implicit trigger at CTA exit), and blocks until that grid has completed and its writes are visible.  Nothing is
// read or written before the wait, so only launch latency and CTA scheduling overlap the previous grid's tail; the dependency
// chain of the stream is unchanged.  The instruction is a no-op for a kernel launched without the attribute (DCLL_PDL=0).
// Measured (B200, profiles/r01_pdl_ab.txt): 16x16 B = 64 training +25 %, B = 1024 +7.6 %, 128x128 B = 64 +1 %.  An explicit
// early trigger (griddepcontrol.launch_dependents at kernel entry) was worse: +16 % at 16x16 B = 64 but -7 % at 128x128,
// where CTAs of up to two later grids sat resident and blocked beside the running one.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_entry() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
#endif
bool pdl_enabled();
template <typename... KArgs, typename... Args>
inline void launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args &&...args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid, cfg.blockDim = block, cfg.dynamicSmemBytes = smem, cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at, cfg.numAttrs = pdl_enabled() ? 1 : 0;
    (void)cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);   // the error is picked up by DCLL_LAUNCH_OK
}

// same, as clusters of two CTAs (CTA pairs for tcgen05 cta_group::2; the grid must be even)
template <typename... KArgs, typename... Args>
inline void launch_k_pair(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args &&...args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid, cfg.blockDim = block, cfg.dynamicSmemBytes = smem, cfg.stream = st;
    cudaLaunchAttribute at[2];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2, at[0].val.clusterDim.y = 1, at[0].val.clusterDim.z = 1;
    at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at, cfg.numAttrs = pdl_enabled() ? 2 : 1;
    (void)cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-DEVICE attribute: set it once per (call site, device), keyed by the
// current device, so that a process which moves on to a second GPU does not get launch failures there.
#define DCLL_SMEM_ATTR(kern, bytes)                                                                              \
    do {                                                                                                         \
        static unsigned long long done_mask_ = 0ull;                                                             \
        int dev_ = 0;                                                                                            \
        DCLL_CUDA_OK(cudaGetDevice(&dev_));                                                                      \
        if (dev_ >= 64 || !((done_mask_ >> dev_) & 1ull)) {                                                      \
            DCLL_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes))); \
            if (dev_ < 64) done_mask_ |= 1ull << dev_;                                                           \
        }                                                                                                        \
    } while (0)

// ---- in-kernel stopwatch (DCLL_TIMELINE=1; debugging aid, off by default) -----------------------------------------------
// The persistent tensor-core kernels accumulate, per CTA, the SM cycles their roles spend waiting on each barrier and in each
// phase into TL_SLOTS 64-bit slots of a per-kernel-kind block; dcll_debug_timeline copies the blocks out (tools/timeline.py).
// The last launch of a kind wins.  timeline_buf returns nullptr when the stopwatch is off: the kernels then skip every clock read.
enum { TL_CONV_MMA32 = 0, TL_CONV_MMA1, TL_CONV_MMA2, TL_WGRAD2, TL_KINDS, TL_SLOTS = 16, TL_CTAS = 148 };
enum { TL_TOTAL = 0, TL_PROLOGUE, TL_ISS_A_FULL, TL_ISS_ACC_EMPTY, TL_ISS_W_FULL, TL_ISS_LOOP, TL_EPI_ACC_FULL, TL_EPI_LOOP, TL_WPROD_EMPTY,
       TL_APROD_EMPTY, TL_FIRST_MMA, TL_DRAIN, TL_EPI_LOADS, TL_T_ENTRY, TL_T_EXIT };   // the last two: %globaltimer (ns)
unsigned long long *timeline_buf(int kind);
#ifdef __CUDACC__
__device__ __forceinline__ unsigned long long gtimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
#define TL_TIMED(on, acc, stmt)                  \
    do {                                         \
        if (on) {                                \
            const long long tl_t0_ = clock64();  \
            stmt;                                \
            (acc) += clock64() - tl_t0_;         \
        } else {                                 \
            stmt;                                \
        }                                        \
    } while (0)
#endif

// SMs the one-CTA-per-SM persistent kernels may fill: all 148, minus the ones the data-parallel driver (dp.cu) leaves to NCCL
// while a collective is in flight.  A persistent grid that finds some SMs taken runs its last CTAs as a second wave (static
// tile striding: up to 2x the kernel time); launching it a few CTAs smaller costs those few CTAs' share instead.
int sm_budget();
void set_reserved_sms(int n);

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// precision modes: does the layer run on the tensor-core kernels at all / with fp16 traces (DCLL_PREC_F16X2, 32-channel input)
static inline bool prec_tc(const dcll_conv_layer *L) { return L->precision == DCLL_PREC_BF16X3 || L->precision == DCLL_PREC_F16X2; }
static inline bool prec_f16(const dcll_conv_layer *L) { return L->precision == DCLL_PREC_F16X2 && L->Cin == 32 && L->w_exp; }
#ifdef __CUDACC__
__host__ __device__ __forceinline__ float pow2i(int e) {             // 2^e as a float, e in [-126, 127]
    const unsigned bits = (unsigned)(e + 127) << 23;
#ifdef __CUDA_ARCH__
    return __uint_as_float(bits);
#else
    float f;
    memcpy(&f, &bits, 4);
    return f;
#endif
}
// exponent k of an fp16 weight image: max |w| * 2^k in [2^7, 2^8) -- 2^8 of headroom below the fp16 maximum
__device__ __forceinline__ int weight_exp_for(float maxabs) {
    if (!(maxabs > 0.f)) return 0;
    const int e = (int)((__float_as_uint(maxabs) >> 23) & 0xff) - 127;     // floor(log2(maxabs)) for normal floats
    const int k = 7 - e;
    return k < -100 ? -100 : (k > 100 ? 100 : k);
}
#endif

// Derived geometry of a layer.
struct Geo {
    int Hc, Wc, Hp, Wp, F, Ktot, CoutPad, nW;
};
static inline Geo geo_of(const dcll_conv_layer *L) {
    Geo g;
    g.Hc = L->H + 2 * L->padH - L->KH + 1;
    g.Wc = L->W + 2 * L->padW - L->KW + 1;
    g.Hp = g.Hc / L->poolH;
    g.Wp = g.Wc / L->poolW;
    g.F = L->Cout * g.Hp * g.Wp;
    g.Ktot = L->K * (L->output_layer ? 2 : 1);
    g.CoutPad = ceil_div(L->Cout, 32) * 32;
    g.nW = L->Cout * L->Cin * L->KH * L->KW;
    return g;
}

// Workspace carve-up (offsets in bytes, 256-B aligned).
struct WsLayout {
    int n_ro;            // read-out partial blocks (FP32 kernel)
    int n_ro_tc;         // read-out partial blocks of the tcgen05 kernel (512 features each)
    int n_split;         // weight-gradient position splits
    size_t off_ro_part;  // float [max(n_ro, n_ro_tc)][B][Ktot]
    size_t off_go;       // float [B][K]   dL/dpvoutput
    size_t off_go2;      // float [B][K]   dL/doutput (output layer)
    size_t off_wg_part;  // float [n_split][nW + Cout]
    size_t off_wimg2;    // bf16 weight image of conv_mma2_kernel (7x7, 32->32 tensor-core layers), else unused
    size_t total;
};
WsLayout ws_layout(const dcll_conv_layer *L);

// Launchers implemented in the individual .cu files (all asynchronous on `st`).
// write_spikes = false (window driver, tensor-core path): nobody reads this step's spike tensor -- the consumer is the trace
// update fused into this launch's epilogue, or there is none (last layer) -- so the epilogue does not store it.
// spike_io: SPK_WRITE as above; SPK_PACKED: the spikes leave as one uint16 word per (sample, 16 channels, position) in the
// same buffer instead of 32 floats per position (window drivers, between two tensor-core layers: the consumer is the next layer's
// trace kernel, which then reads 2 bytes instead of 32 per position and channel group); SPK_X_PACKED: this layer's input is
// such a word array.  The per-step API always moves float spikes.
enum { SPK_WRITE = 1, SPK_PACKED = 2, SPK_X_PACKED = 4 };
bool tc_spikes_packable(const dcll_conv_layer *L, const dcll_conv_layer *next);
static inline int spike_io_of(const dcll_conv_layer *layers, int l, int n_layers, bool fuse_next, bool trace_done) {
    const bool read = l + 1 < n_layers && !fuse_next;
    return (read ? SPK_WRITE : 0) | ((read && tc_spikes_packable(&layers[l], &layers[l + 1])) ? SPK_PACKED : 0) |
           ((l > 0 && !trace_done && tc_spikes_packable(&layers[l - 1], &layers[l])) ? SPK_X_PACKED : 0);
}
int launch_conv_fwd(const dcll_conv_layer *L, const void *x, cudaStream_t st, const dcll_conv_layer *next = nullptr,
                    bool trace_done = false, int spike_io = SPK_WRITE);
// tcgen05, split-bf16 x3.  Window driver only: `next` != null makes the epilogue also apply the NEXT layer's trace update
// (its input is exactly the spike the epilogue thread just produced) and write that layer's operand image;
// `trace_done` says the previous layer already did so for this one.
int launch_conv_fwd_tc(const dcll_conv_layer *L, const void *x, cudaStream_t st, const dcll_conv_layer *next = nullptr,
                       bool trace_done = false, int spike_io = SPK_WRITE);
bool tc_trace_fusable(const dcll_conv_layer *L, const dcll_conv_layer *next);
int launch_weight_mma(const dcll_conv_layer *L, const float *w, cudaStream_t st);
int sync_kernel_weights(const dcll_conv_layer *L, cudaStream_t st);   // weight -> weight_t / weight_mma (quantised or not)
bool tc_supported(const dcll_conv_layer *L);
size_t conv_mma2_image_bytes(const dcll_conv_layer *L);   // 0 when the layer has no conv_mma2 path
int launch_readout_fwd(const dcll_conv_layer *L, const float *target, int loss_kind, int32_t *clout,
                       float *loss_out, cudaStream_t st);
bool readout_tc_supported(const dcll_conv_layer *L);
int readout_tc_blocks(const dcll_conv_layer *L);
int launch_readout_tc(const dcll_conv_layer *L, float *partial, cudaStream_t st);   // tcgen05, split-bf16 x3
int launch_loss_grad(const dcll_conv_layer *L, const float *target, int loss_kind, float *loss_out, cudaStream_t st);
// so_out / so_i2h: the rule of adam_out / adam_i2h when it is not Adam (null: the Adam kernels)
struct OptScalars;
int launch_readout_bwd(const dcll_conv_layer *L, dcll_train_args *a, cudaStream_t st, const OptScalars *so_out = nullptr);
bool readout_bwd_tc_supported(const dcll_conv_layer *L, int hw, int F);                   // readout_bwd_tc.cu (DCLL_RB_TC=1)
int launch_readout_bwd_tc(const dcll_conv_layer *L, const float *g_o, int hw, int F, float g_scale, cudaStream_t st);
int launch_wgrad(const dcll_conv_layer *L, dcll_train_args *a, cudaStream_t st, const OptScalars *so_i2h = nullptr);
int wgrad_splits(const dcll_conv_layer *L);
bool wgrad_tc_supported(const dcll_conv_layer *L);
int wgrad_tc_splits(const dcll_conv_layer *L);
int launch_wgrad_tc(const dcll_conv_layer *L, float *partial, int S, cudaStream_t st);
// row-pair N-concatenation kernel (wgrad_tc2.cu): operands from the eps1 image and from g_u left as bf16 {hi,lo} planes by
// the packed backward read-out; one compact partial block per CTA, reduced by reduce_adam_rp_kernel
bool wgrad_tc2_supported(const dcll_conv_layer *L);
size_t wgrad_tc2_partial_floats();
int launch_wgrad_tc2(const dcll_conv_layer *L, float *partial, int *nA, int *nB, cudaStream_t st);
struct AdamScalars;
int launch_adam_flat(float *w, const float *g, float *m, float *v, size_t n, const AdamScalars &sc, cudaStream_t st);

// Scalars of one Adam step, computed on the host in double exactly as torch does
// (torch/optim/adam.py: bias_correction1/2, step_size, bias_correction2_sqrt).
struct AdamScalars {
    float wd, beta1, one_minus_beta1, beta2, one_minus_beta2, neg_step_size, bc2_sqrt, eps;
};
AdamScalars adam_scalars(const dcll_adam &a, int64_t step_after);

__device__ __forceinline__ void adam_elem(float &w, float g, float &m, float &v, const AdamScalars &s) {
    if (s.wd != 0.f) g = __fmaf_rn(s.wd, w, g);                       // grad.add(param, alpha=wd)
    // exp_avg.lerp_(grad, 1-beta1)
    if (s.one_minus_beta1 < 0.5f) m = __fmaf_rn(s.one_minus_beta1, __fsub_rn(g, m), m);
    else m = __fsub_rn(g, __fmul_rn(__fsub_rn(g, m), __fsub_rn(1.f, s.one_minus_beta1)));
    // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1-beta2)
    v = __fadd_rn(__fmul_rn(v, s.beta2), __fmul_rn(__fmul_rn(s.one_minus_beta2, g), g));
    float denom = __fadd_rn(__fdiv_rn(__fsqrt_rn(v), s.bc2_sqrt), s.eps);
    w = __fadd_rn(w, __fdiv_rn(__fmul_rn(s.neg_step_size, m), denom)); // addcdiv_(m, denom, -step_size)
}

// Scalars of one step of an AdamW / Adamax / NAdam / RAdam rule (dcll_optim), computed on the host in double exactly as torch's
// _single_tensor_<rule> (net.cu: opt_scalars).  Each float is the python float rounded as torch rounds it when it meets a
// float32 tensor.  c0..c3 by kind:
//   ADAMW   -step_size, sqrt(bc2)                   ADAMAX  -lr / bc1
//   NADAM   bc2, addcdiv value of grad, of exp_avg  RADAM   bc1, lr, sqrt(bc2), rect
struct OptScalars {
    int kind;                  // DCLL_OPT_*, never DCLL_OPT_ADAM (that rule runs adam_elem)
    int rect;                  // RAdam: rho_t > 5 (decided on the host, uniform across the launch)
    float decay;               // decoupled weight decay: param.mul_(1 - lr * weight_decay); 1 = none
    float wd;                  // coupled weight decay: grad.add(param, alpha=weight_decay); 0 = none
    float one_minus_beta1, beta2, one_minus_beta2, eps;
    float c0, c1, c2, c3;
};
// step_after: the step count after this update; *mu_product (NAdam) is torch's float32 state, updated in place
OptScalars opt_scalars(const dcll_adam &a, const dcll_optim &o, int64_t step_after, float *mu_product);
// the scalars of slot o's next update (step a.step + 1) in *buf, or null when the slot runs Adam; advances o->mu_product
const OptScalars *next_opt_scalars(const dcll_adam &a, dcll_optim *o, OptScalars *buf);

__device__ __forceinline__ void opt_elem(float &w, float g, float &m, float &v, const OptScalars &s) {
    if (s.decay != 1.f) w = __fmul_rn(w, s.decay);                   // param.mul_(1 - lr * weight_decay)
    if (s.wd != 0.f) g = __fmaf_rn(s.wd, w, g);                       // grad.add(param, alpha=wd)
    // exp_avg.lerp_(grad, 1-beta1), as adam_elem
    if (s.one_minus_beta1 < 0.5f) m = __fmaf_rn(s.one_minus_beta1, __fsub_rn(g, m), m);
    else m = __fsub_rn(g, __fmul_rn(__fsub_rn(g, m), __fsub_rn(1.f, s.one_minus_beta1)));
    if (s.kind == DCLL_OPT_ADAMAX) {
        v = fmaxf(__fmul_rn(v, s.beta2), __fadd_rn(fabsf(g), s.eps));  // maximum(exp_inf.mul_(beta2), grad.abs().add_(eps))
        w = __fadd_rn(w, __fdiv_rn(__fmul_rn(s.c0, m), v));            // addcdiv_(exp_avg, exp_inf, value=-clr)
        return;
    }
    // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1-beta2)
    v = __fadd_rn(__fmul_rn(v, s.beta2), __fmul_rn(__fmul_rn(s.one_minus_beta2, g), g));
    if (s.kind == DCLL_OPT_NADAM) {
        const float denom = __fadd_rn(__fsqrt_rn(__fdiv_rn(v, s.c0)), s.eps);   // exp_avg_sq.div(bc2).sqrt().add_(eps)
        w = __fadd_rn(w, __fdiv_rn(__fmul_rn(s.c1, g), denom));                 // addcdiv_(grad, denom, -lr(1-mu)/(1-mu_product))
        w = __fadd_rn(w, __fdiv_rn(__fmul_rn(s.c2, m), denom));                 // addcdiv_(exp_avg, denom, -lr mu_next/(1-mu_product_next))
    } else if (s.kind == DCLL_OPT_RADAM) {
        float u = __fmul_rn(__fdiv_rn(m, s.c0), s.c1);                          // exp_avg / bc1 * lr
        // * (sqrt(bc2) / (sqrt(v) + eps)) * rect; a python float over a tensor is reciprocal() * float in torch
        if (s.rect) u = __fmul_rn(__fmul_rn(u, __fmul_rn(__frcp_rn(__fadd_rn(__fsqrt_rn(v), s.eps)), s.c2)), s.c3);
        w = __fsub_rn(w, u);                                                    // param.add_(update, alpha=-1)
    } else {                                                                    // DCLL_OPT_ADAMW: Adam after the decay
        const float denom = __fadd_rn(__fdiv_rn(__fsqrt_rn(v), s.c1), s.eps);
        w = __fadd_rn(w, __fdiv_rn(__fmul_rn(s.c0, m), denom));
    }
}

// the element update of a kernel body shared by the Adam kernel and its _opt sibling
__device__ __forceinline__ void elem_update(float &w, float g, float &m, float &v, const AdamScalars &s) { adam_elem(w, g, m, v, s); }
__device__ __forceinline__ void elem_update(float &w, float g, float &m, float &v, const OptScalars &s) { opt_elem(w, g, m, v, s); }
// the rule of an optimizer slot: null or DCLL_OPT_ADAM is Adam (the pre-existing kernels)
static inline bool opt_active(const dcll_optim *o) { return o && o->kind != DCLL_OPT_ADAM; }
int launch_opt_flat(float *w, const float *g, float *m, float *v, size_t n, const OptScalars &sc, cudaStream_t st);
// Adam or the rule o over two flat parameters (weight, bias), then step += 1 (net.cu; the dense layer's update)
int dense_flat_update(dcll_adam &a, dcll_optim *o, float *w, const float *gw, size_t nw, float *b, const float *gb, size_t nb,
                      cudaStream_t st);

__device__ __forceinline__ float sigmoidf_ref(float x) {
    // 1/(1+exp(-x)) with IEEE division: matches torch-CPU sigmoid to ~1 ulp
    return __fdiv_rn(1.f, __fadd_rn(1.f, expf(-x)));
}

// Element-wise losses of a read-out value x against its target y (every kind except DCLL_LOSS_CROSS_ENTROPY).
// d(mean-reduced loss)/dx: torch multiplies by norm = float(1/numel) (float(2/numel) for MSE),
// aten/src/ATen/native/cpu/PointwiseOpsKernel.cpp (smooth_l1_backward, mse_backward).
__device__ __forceinline__ float loss_grad_elem(float x, float y, int kind, int numel) {
    const float d = x - y;
    if (kind == DCLL_LOSS_MSE) return __fmul_rn((float)(2.0 / (double)numel), d);
    const float norm = (float)(1.0 / (double)numel);
    if (kind == DCLL_LOSS_SMOOTHL1) return d < -1.f ? -norm : (d > 1.f ? norm : __fmul_rn(norm, d));
    if (kind == DCLL_LOSS_L1) return d > 0.f ? norm : (d < 0.f ? -norm : 0.f);
    if (kind == DCLL_LOSS_BCE_LOGITS) return __fmul_rn(__fsub_rn(sigmoidf_ref(x), y), norm);
    if (kind == DCLL_LOSS_SOFT_MARGIN) return __fmul_rn(__fmul_rn(-y, sigmoidf_ref(-y * x)), norm);
    if (kind == DCLL_LOSS_KL_DIV) return __fmul_rn(-y, norm);
    if (kind == DCLL_LOSS_POISSON_NLL) return __fmul_rn(__fsub_rn(expf(x), y), norm);
    // DCLL_LOSS_HINGE, torch's form for any target: where(y != 1, clamp_min(1 - x, 0), 0) + where(y != -1, x, 0); the
    // clamp passes its gradient at 1 - x == 0, so for y = 0 the slope at x = 1 is -1 + 1 = 0
    return ((y != -1.f) ? norm : 0.f) - ((y != 1.f && x <= 1.f) ? norm : 0.f);
}
// loss of one element before the 1/numel of the mean
__device__ __forceinline__ float loss_value_elem(float x, float y, int kind) {
    const float d = x - y;
    if (kind == DCLL_LOSS_SMOOTHL1) return fabsf(d) < 1.f ? 0.5f * d * d : fabsf(d) - 0.5f;
    if (kind == DCLL_LOSS_MSE) return d * d;
    if (kind == DCLL_LOSS_L1) return fabsf(d);
    if (kind == DCLL_LOSS_BCE_LOGITS) return fmaxf(x, 0.f) - y * x + log1pf(expf(-fabsf(x)));      // softplus(x) - y x
    if (kind == DCLL_LOSS_SOFT_MARGIN) {                                                            // softplus(-y x)
        const float z = -y * x;
        return fmaxf(z, 0.f) + log1pf(expf(-fabsf(z)));
    }
    if (kind == DCLL_LOSS_KL_DIV) return (y == 0.f ? 0.f : y * logf(y)) - y * x;                  // xlogy(y, y) - y x
    if (kind == DCLL_LOSS_POISSON_NLL) return expf(x) - y * x;
    return ((y != 1.f) ? fmaxf(1.f - x, 0.f) : 0.f) + ((y != -1.f) ? x : 0.f);                     // DCLL_LOSS_HINGE
}

// torch.nn.CrossEntropyLoss() with probability targets, mean over the B rows, for element k of one row x[0..K) with target
// row y: returns g_k = (softmax(x)_k * sum(y) - y_k) / B (torch's gradient also for rows that do not sum to 1) and adds
// -y_k log_softmax(x)_k / B to `val`.  The row maximum is subtracted before expf, so every finite row stays finite.
// Every caller of a row walks it whole, in the same fixed order (maximum, then the sums over k = 0..K-1): one CTA per row
// in readout_finish_kernel, one thread per element in loss_grad_kernel and dense_loss_grad_kernel all get the same bits
// from the same row values.
__device__ __forceinline__ float ce_grad_elem(const float *x, const float *y, int K, int k, int B, float &val) {
    float m = x[0];
    for (int j = 1; j < K; ++j) m = fmaxf(m, x[j]);
    float s = 0.f, ysum = 0.f;
    for (int j = 0; j < K; ++j) {
        s = __fadd_rn(s, expf(__fsub_rn(x[j], m)));
        ysum = __fadd_rn(ysum, y[j]);
    }
    const float inv_b = (float)(1.0 / (double)B);
    const float xk = __fsub_rn(x[k], m), yk = y[k];
    val += __fmul_rn(__fmul_rn(-yk, __fsub_rn(xk, logf(s))), inv_b);
    const float p = __fdiv_rn(expf(xk), s);
    return __fmul_rn(__fsub_rn(__fmul_rn(p, ysum), yk), inv_b);
}

}  // namespace dcll
