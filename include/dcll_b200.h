/* dcll_b200.h -- C ABI of the B200-native DCLL hot path (libdcll_b200.so).
 *
 * Plain pointers and sizes only: no torch / C++ types cross this boundary.  Every
 * pointer marked "device" is a CUDA device pointer owned by the caller (the Python
 * host mirror allocates them as torch tensors and passes data_ptr()).  All entry
 * points enqueue work on `stream` (a cudaStream_t passed as void*) and never
 * synchronise the host.  They return 0 on success or a negative DCLL_E* code;
 * dcll_last_error() returns a static message for the calling thread.
 *
 * The reference (ohjay/snn-modulation-classification) has no FFI of its own: its
 * boundary is the Python class API.  Each entry point below therefore cites the
 * reference *method* whose arithmetic it replaces (paths relative to the reference
 * root); the Python classes that keep the reference's signatures and call these
 * functions live in snn_modulation_classification_b200/dcll/pytorch_libdcll.py.
 */
#ifndef DCLL_B200_H
#define DCLL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DCLL_ABI_VERSION 12

enum { DCLL_OK = 0, DCLL_EINVAL = -1, DCLL_ECUDA = -2, DCLL_EUNSUPPORTED = -3 };

/* time-constant storage: the reference keeps alpha/alphas/tau_m__dt/tau_s__dt either as (1,)
 * tensors or, with random_tau, as (Cin,H,W) tensors holding one value per input channel
 * (dcll/pytorch_libdcll.py:349-356, :391-405). */
enum { DCLL_COEF_SCALAR = 0, DCLL_COEF_CHANNEL = 1, DCLL_COEF_ELEMENT = 2 };
/* layer input: dense float32 [B,Cin,H,W] spikes, or (layer 0 only, Cin == 1) the encoder's
 * int32 [B,2] (row, col) cell of the single spike of each sample. */
enum { DCLL_X_DENSE = 0, DCLL_X_CELLS = 1 };
/* loss classes train.py:173 can select (torch.nn.<class>() with default arguments); gradient of the mean-reduced loss.
 * CROSS_ENTROPY: probability targets, softmax over the K values of a row, mean over the B rows; every other kind is
 * element-wise, mean over the B*K elements.  BCE_LOGITS also serves MultiLabelSoftMarginLoss, SMOOTHL1 HuberLoss (delta 1);
 * KL_DIV takes log-probability inputs, POISSON_NLL log-rate inputs; HINGE is HingeEmbeddingLoss (margin 1). */
enum { DCLL_LOSS_SMOOTHL1 = 0, DCLL_LOSS_MSE = 1, DCLL_LOSS_L1 = 2,
       DCLL_LOSS_EXTERNAL = 3 /* any other loss class: the host supplies dL/dpvoutput (and dL/doutput) */,
       DCLL_LOSS_CROSS_ENTROPY = 4, DCLL_LOSS_BCE_LOGITS = 5, DCLL_LOSS_SOFT_MARGIN = 6, DCLL_LOSS_KL_DIV = 7,
       DCLL_LOSS_POISSON_NLL = 8, DCLL_LOSS_HINGE = 9 /* the last kind */ };
/* conv arithmetic: FP32 CUDA-core FMA (parity mode); split-bf16 x3 on tcgen05 tensor cores (both operands bf16 hi + lo, three
 * products); or F16X2: the same kernels with the TRACE operand as one fp16 value (eps1 lies in [0,1]: relative rounding 2^-12)
 * against split-fp16 weights / local gradients -- two products, no lo pass over the traces.  kind::f16 wants both operands in
 * one format, and fp16 has 5 exponent bits, so every operand image carries a power-of-two scale (exact): a_exp for the traces
 * (static bound from the time constants), g_exp for the local gradient (static bound from the frozen read-out and the batch
 * size), and a per-layer weight exponent the library tracks on the device (w_exp).  Needs w_exp and 32 input channels; layers
 * with one input channel keep the split-bf16 form (they are not bound by the tensor pipe). */
enum { DCLL_PREC_FP32 = 0, DCLL_PREC_BF16X3 = 1, DCLL_PREC_F16X2 = 2 };

/* torch.optim.Adam hyper-parameters + state of one parameter group
 * (dcll/pytorch_libdcll.py:634-638; train.py:164-168). */
typedef struct dcll_adam {
    double lr, beta1, beta2, eps, weight_decay;
    int64_t step;          /* number of updates already applied; incremented by the update call */
    float *m_w, *v_w;      /* device: exp_avg / exp_avg_sq of the weight */
    float *m_b, *v_b;      /* device: exp_avg / exp_avg_sq of the bias   */
} dcll_adam;

/* Update rule of one dcll_adam, for the _opt entry points (train.py --optim_type): the dcll_adam keeps lr, betas, eps,
 * weight_decay, step and the two float32 state tensors per parameter (exp_avg, and exp_avg_sq -- or exp_inf for Adamax,
 * in v_w / v_b).  Each rule follows torch's _single_tensor_<rule> operation order.
 *   ADAM   torch.optim.Adam (the entry points without _opt)
 *   ADAMW  torch.optim.AdamW, or Adam(decoupled_weight_decay=True); amsgrad=False
 *   ADAMAX torch.optim.Adamax
 *   NADAM  torch.optim.NAdam (decoupled_wd, momentum_decay; mu_product in/out)
 *   RADAM  torch.optim.RAdam (decoupled_wd)                                                                             */
enum { DCLL_OPT_ADAM = 0, DCLL_OPT_ADAMW = 1, DCLL_OPT_ADAMAX = 2, DCLL_OPT_NADAM = 3, DCLL_OPT_RADAM = 4 };
typedef struct dcll_optim {
    int32_t kind;          /* DCLL_OPT_*                                                                    */
    int32_t decoupled_wd;  /* NAdam / RAdam: decoupled_weight_decay (AdamW: always decoupled)              */
    double momentum_decay; /* NAdam                                                                         */
    float mu_product;      /* NAdam: torch's float32 state['mu_product'], before the call / after it        */
} dcll_optim;

/* One Conv2dDCLLlayer (dcll/pytorch_libdcll.py:512-612) with its i2h core
 * (ContinuousConv2D :296-429 or ContinuousRelativeRefractoryConv2D :432-509). */
typedef struct dcll_conv_layer {
    int32_t B, Cin, H, W;            /* input  [B,Cin,H,W]                                   */
    int32_t Cout, KH, KW, padH, padW; /* stride 1, dilation 1, groups 1 (every shipped spec)  */
    int32_t poolH, poolW;            /* 1 or 2 per axis (MaxPool2d k = stride, pad (k-1)//2) */
    int32_t K;                       /* target_size                                          */
    int32_t output_layer;            /* trainable output_ read-out present (:577-579)        */
    int32_t coef_mode;               /* DCLL_COEF_*                                          */
    int32_t x_mode;                  /* DCLL_X_*                                             */
    int32_t precision;               /* DCLL_PREC_*                                          */
    int32_t cur;                     /* which half of eps0/eps1 holds the current state;
                                        flipped by every forward step                        */
    int32_t write_pvmem;             /* materialise the membrane tensor (API path) or skip   */
    int32_t quantized;               /* 1: the convolution uses the int8 quantise->dequantise image of `weight`
                                        (per-output-channel symmetric, oracle/quant.py); `weight` stays the
                                        float32 master that Adam updates (straight-through)                */
    float alpharp, wrp;              /* wrp > 0: refractory variant                          */
    const float *alpha, *alphas, *tau_m, *tau_s; /* device                                   */
    float *weight;                   /* device [Cout,Cin,KH,KW]  (the nn.Parameter)          */
    float *weight_t;                 /* device [Cin,KH*KW,CoutPad] kernel-side copy,
                                        CoutPad = 32*ceil(Cout/32); dcll_conv_sync_weights.
                                        With quantized && weight_mma the allocation must hold
                                        Cout*Cin*KH*KW more floats (dense dequantised copy)   */
    void *weight_mma;                /* device bf16 [KH*KW][Cin/8][2][Cout][8]: {hi,lo} split weights in the
                                        tcgen05 B-operand layout (Cin = 1: [(KH+1)/2][2][2][Cout][8], the 8 slots
                                        being kernel columns; at least 4096 elements); required when precision is
                                        DCLL_PREC_BF16X3, refreshed together with weight_t       */
    float *bias;                     /* device [Cout]                                        */
    const float *wo, *bo;            /* device [K,F], [K]   frozen local read-out i2o        */
    float *wout, *bout;              /* device [K,F], [K]   output_ or NULL                  */
    float *eps0[2], *eps1[2];        /* device [B,Cin,H,W]  ping-pong state                  */
    void *eps1_mma;                  /* device bf16 [B][2][Cin/8][H][W][8]: {hi,lo} split image of the eps1 the last
                                        forward step produced, in the tcgen05 operand layout (16 bytes per position
                                        and channel group; with Cin = 1 the 8 slots hold eps1[y][x-3..x+4], i.e.
                                        2*B*8*H*W elements).  Required (2*B*max(Cin,8)*H*W bf16) when
                                        precision is DCLL_PREC_BF16X3 and weight_mma is set; written by
                                        dcll_conv_step_fwd / dcll_conv_core_fwd, read by the convolution and by
                                        dcll_conv_step_bwd_update of the same timestep          */
    float *arp;                      /* device [B,Cout,Hc,Wc] or NULL                        */
    /* per-step outputs (device) */
    float *spikes;                   /* [B,Cout,Hp,Wp] pooled spikes                         */
    float *pv;                       /* [B,Cout,Hp,Wp] pooled sigmoid                        */
    float *pvmem;                    /* [B,Cout,Hc,Wc] or NULL                               */
    uint8_t *pool_idx;               /* [B,Cout,Hp,Wp] argmax inside the pool window, or NULL
                                        when poolH == poolW == 1                             */
    float *pvoutput;                 /* [B,K]                                                */
    float *output;                   /* [B,K] logits of output_, or NULL                     */
    float *g_u;                      /* [B,Cout,Hp,Wp] training scratch: dL/d(membrane) at the
                                        pool argmax                                          */
    void *workspace;                 /* device scratch, dcll_conv_workspace_bytes()          */
    size_t workspace_bytes;
    /* DCLL_PREC_F16X2 only (ignored otherwise) */
    int32_t a_exp;                   /* eps1_mma holds fp16(eps1 * 2^a_exp): 2^a_exp * max eps1 <= 2^15, where
                                        max eps1 = tau_s/(1-alphas) * tau_m/(1-alpha) for spike input     */
    int32_t g_exp;                   /* g_u image holds fp16 {hi,lo} of g_u * 2^g_exp (saturating)         */
    int32_t *w_exp;                  /* device int32[4], zero-initialised by the caller, owned by the library afterwards:
                                        {exponent of the current weight_mma image, exponent of the next one,
                                         block ticket, running max |w| bits}; weight_mma holds fp16 {hi,lo} of w * 2^w_exp[0] */
} dcll_conv_layer;

typedef struct dcll_train_args {
    const float *target;             /* device [B,K] one-hot                                 */
    const float *g_o_ext, *g_o2_ext; /* device [B,K]: DCLL_LOSS_EXTERNAL only                */
    int32_t loss_kind;               /* DCLL_LOSS_*                                          */
    int32_t apply_update;            /* 1: fused Adam; 0: only write gradients (DP: allreduce
                                        then dcll_conv_apply_update)                         */
    dcll_adam adam_i2h;              /* optimizer  over i2h.{weight,bias}                    */
    dcll_adam adam_out;              /* optimizer2 over output_.{weight,bias}                */
    float *grad_w, *grad_b;          /* device, optional (NULL) unless apply_update == 0     */
    float *grad_wout, *grad_bout;    /* device, optional                                     */
    float *loss_out;                 /* device [1] or NULL: value of the local loss          */
} dcll_train_args;

/* -- library ------------------------------------------------------------------------------ */
int dcll_abi_version(void);
const char *dcll_last_error(void);
size_t dcll_sizeof_conv_layer(void);
size_t dcll_sizeof_train_args(void);

/* -- measurement hooks (bench.py) --------------------------------------------------------------- *
 * dcll_launch_count: kernels launched by this library since load (or since the last reset).
 * dcll_profile_enable(every_n): bracket the kernels of every n-th layer-step with CUDA events on the
 * launching stream (0 disables).  dcll_profile_read synchronises those events and returns, per kernel
 * class c (0 encode, 1 conv_fwd, 2 readout_fwd, 3 readout_bwd, 4 wgrad, 5 adam, 6 misc, 7 trace -- the trace/image
 * kernel of a tensor-core conv step, also contained in its conv_fwd bracket) and layer l (< 8), the summed milliseconds ms[c*8+l] and the number of sampled brackets n[c*8+l]; then clears. */
int64_t dcll_launch_count(int reset);
int dcll_profile_enable(int every_n);
int dcll_profile_read(double *ms, int64_t *n);
/* dcll_debug_timeline: in-kernel stopwatch of the persistent tensor-core kernels (DCLL_TIMELINE=1 in the environment before the
 * first launch, otherwise an error): copies [4 kernel kinds][148 CTAs][16 slots] SM-cycle counters of the last launch of each
 * kind (csrc/common.cuh TL_*; tools/timeline.py prints them).  Synchronises the device.  Returns the number of values. */
int dcll_debug_timeline(uint64_t *out, int n_u64);

/* -- encoder: data/utils.py:43-87 (iq2spiketrain) ------------------------------------------ *
 * x: device float32 [B,2,N]; cells: device int32 [T,B,2] = (cell_Q, cell_I) for samples
 * t_start .. t_start+T-1.  Bit-exact with the reference's torch-CPU arithmetic.              */
int dcll_iq_encode(const float *x, int B, int N, double min_I, double max_I, double min_Q, double max_Q,
                   int out_w, int out_h, int t_start, int T, int do_gamma, int32_t *cells, void *stream);
/* dense one-hot frames [T,B,1,H,W] float32 (what data/utils.py:57,81-82 materialises) */
int dcll_cells_to_frames(const int32_t *cells, int T, int B, int H, int W, float *frames, void *stream);

/* image2spiketrain (data/utils.py:15-40): frozen Poisson spike train of an image, out float32 [Tmax,B,Nin]:
 *   spike[t,b,n] = t < t_len[b] && !(u[b,t,n] < p[b,n]),  p = (1000 - gain*x[b,n]) / 1000 in float32.
 * u: device float64 [B,Tmax,Nin] = the uniforms of the reference's numpy stream (bit-exact parity for the same draws), or NULL:
 * a seeded counter-based generator on the device (same distribution, not the numpy stream). */
int dcll_image_encode(const float *x, const double *u, const int32_t *t_len, int B, int Nin, int Tmax, double gain,
                      uint64_t seed, float *out, void *stream);

/* -- conv layer step ------------------------------------------------------------------------ */
size_t dcll_conv_workspace_bytes(const dcll_conv_layer *L);
/* refresh weight_t from weight (after load_state_dict / external assignment) */
int dcll_conv_sync_weights(const dcll_conv_layer *L, void *stream);
/* Conv2dDCLLlayer.forward (:599-608) incl. i2h.forward (:407-426 / :485-509): trace update,
 * conv, refractory, sigmoid, threshold, pool, read-outs.  x: dense [B,Cin,H,W] or cells [B,2].
 * clout (device int32 [B], optional): argmax of pvoutput (or of output on the output layer),
 * DCLLClassification.forward :724-728.  Flips L->cur.                                        */
int dcll_conv_step_fwd(dcll_conv_layer *L, const void *x, int32_t *clout, void *stream);
/* The same step for a caller that walks the layers itself (data-parallel training: an allreduce sits between a
 * layer's backward and its next forward) but still wants what dcll_net_window does between two tensor-core layers of equal
 * geometry: with next != NULL, L's convolution epilogue also applies NEXT's trace recurrences (:415-416 of the next layer,
 * its input being L's spikes) and writes its operand image; the following call for that layer then passes trace_done = 1
 * and skips its own trace pass.  dcll_conv_chain_fusable(L, next) says whether a pair qualifies (1) or not (0). */
int dcll_conv_chain_fusable(const dcll_conv_layer *L, const dcll_conv_layer *next);
int dcll_conv_step_fwd_chain(dcll_conv_layer *L, const dcll_conv_layer *next, int trace_done, const void *x, int32_t *clout,
                             void *stream);
/* i2h.forward alone (ContinuousConv2D.forward :407-426): like the above without pooling-independent
 * read-outs; L->poolH/poolW must be 1 so that spikes/pv are the un-pooled tensors.  Flips L->cur. */
int dcll_conv_core_fwd(dcll_conv_layer *L, const void *x, void *stream);
/* DCLLBase.train_dcll :692-714 after the forward: local loss gradient, weight gradient and the
 * Adam step(s).  Increments a->adam_*.step when apply_update.                                */
int dcll_conv_step_bwd_update(dcll_conv_layer *L, dcll_train_args *a, void *stream);
/* Adam on gradients already in a->grad_* (data-parallel path, after the allreduce) */
int dcll_conv_apply_update(dcll_conv_layer *L, dcll_train_args *a, void *stream);
/* The same two calls with the update rules opt[0] (adam_i2h) and opt[1] (adam_out).  opt == NULL, or kind DCLL_OPT_ADAM,
 * is Adam exactly as above.  Writes back step (in dcll_adam) and mu_product (in opt) of every rule it applied. */
int dcll_conv_step_bwd_update_opt(dcll_conv_layer *L, dcll_train_args *a, dcll_optim *opt, void *stream);
int dcll_conv_apply_update_opt(dcll_conv_layer *L, dcll_train_args *a, dcll_optim *opt, void *stream);

/* -- dense layer: DenseDCLLlayer (dcll/pytorch_libdcll.py:198-266) over CLLDenseModule (:72-148) or
 *    CLLDenseRRPModule (:151-195).  Not instantiated by any entry point of the reference; FP32 tiled GEMMs. */
typedef struct dcll_dense_layer {
    int32_t B, In, Out, K;
    int32_t coef_mode;               /* DCLL_COEF_SCALAR or DCLL_COEF_CHANNEL ([In] vectors, random_tau)  */
    float alpharp, wrp;
    const float *alpha, *alphas, *tau_m, *tau_s;
    float *weight, *bias;            /* device [Out,In], [Out]                                            */
    const float *wo, *bo;            /* device [K,Out], [K]  frozen i2o                                   */
    float *eps0, *eps1;              /* device [B,In], updated in place (element-wise, no halo)           */
    float *arp;                      /* device [B,Out] or NULL                                            */
    float *spikes, *pv, *vmem;       /* device [B,Out] outputs                                            */
    float *pvoutput;                 /* device [B,K]                                                      */
    float *g_o, *g_u;                /* device scratch [B,K], [B,Out]                                     */
    float *grad_w, *grad_b;          /* device [Out,In], [Out]                                            */
} dcll_dense_layer;
size_t dcll_sizeof_dense_layer(void);
/* DenseDCLLlayer.forward :250-255 (x: device [B,In]) */
int dcll_dense_step_fwd(dcll_dense_layer *L, const float *x, int32_t *clout, void *stream);
/* local gradient (SURVEY appendix C: gW = ((g_o Wo) * s(1-s))^T eps1) + Adam on weight/bias when apply_update;
 * gradients are always left in grad_w / grad_b. */
int dcll_dense_step_bwd_update(dcll_dense_layer *L, dcll_train_args *a, void *stream);
/* the same with the update rule opt[0] of adam_i2h (NULL: Adam) */
int dcll_dense_step_bwd_update_opt(dcll_dense_layer *L, dcll_train_args *a, dcll_optim *opt, void *stream);

/* -- whole window: the T-loop of train.py:249-251 / test_radio_ml.py:144-145 ----------------- *
 * Runs `T` timesteps of ConvNetwork.learn (train != 0) or .test over `n_layers` chained
 * layers.  x0: layer-0 input for all timesteps, dense [T,B,Cin,H,W] or cells [T,B,2].
 * target: [B,K] (t_stride 0) or [T,B,K] (t_stride B*K).  iter0[l]: DCLLBase.iter of slice l
 * before the window (reset() sets 0).  clout: device int32 [T,n_layers,B] (rows before
 * burn-in are written too; the host keeps the reference's counting rule).                    */
int dcll_net_window(dcll_conv_layer *layers, dcll_train_args *train, int n_layers, const void *x0,
                    const float *target, int64_t target_t_stride, int T, int train_mode, int burnin,
                    const int32_t *iter0, int32_t *clout, void *stream);
/* Same, plus the activity statistics of DCLLBase.forward :658-661: every `hist_every`-th iteration of slice l
 * (iter % hist_every == 0) the 19-bin histogram of pv over [0,1] (np.histogram(pv, np.linspace(0,1,20))) is written to
 * hist[l][n][19] (device int32, n counts the sampled iterations of the window, at most hist_cap per layer).
 * hist == NULL or hist_every <= 0 disables it. */
int dcll_net_window_stats(dcll_conv_layer *layers, dcll_train_args *train, int n_layers, const void *x0,
                          const float *target, int64_t target_t_stride, int T, int train_mode, int burnin,
                          const int32_t *iter0, int32_t *clout, int32_t *hist, int hist_every, int hist_cap, void *stream);
/* the same with update rules opt[2*l] (train[l].adam_i2h) and opt[2*l+1] (train[l].adam_out); NULL: Adam everywhere.  A NAdam
 * mu_product is carried across the timesteps of the window and written back at the end. */
int dcll_net_window_stats_opt(dcll_conv_layer *layers, dcll_train_args *train, dcll_optim *opt, int n_layers, const void *x0,
                              const float *target, int64_t target_t_stride, int T, int train_mode, int burnin,
                              const int32_t *iter0, int32_t *clout, int32_t *hist, int hist_every, int hist_cap, void *stream);

/* -- data-parallel window (SURVEY.md section 8e; the reference has no multi-GPU code: train.py:249-251 over a batch shard) -- *
 * One process per GPU, identical weights, each rank its own B/world samples.  dcll_net_window_dp is dcll_net_window in
 * training mode with one raw ncclAllReduce (average) per layer and timestep of the layer's gradient bucket
 * [gW | gb | gWout | gbout] on a side stream, waited for right before the layer's next forward, where the identical Adam
 * step is applied on every rank.  NCCL is dlopen'ed from `nccl_lib` (the libnccl.so.2 torch has loaded; NULL = default
 * search path) -- the library itself links cudart only.  Rendezvous: rank 0 calls dcll_dp_unique_id, the host broadcasts the
 * 128 bytes (torch.distributed), every rank calls dcll_dp_create (collective).  max_ctas > 0 caps the CTAs NCCL may use, so
 * that the collectives do not evict the one-CTA-per-SM persistent kernels they overlap with.
 * train[l]: apply_update = 0 and grad_w, grad_b[, grad_wout, grad_bout] back to back in bucket[l] (bucket_floats[l] floats). */
typedef struct dcll_dp dcll_dp;
int dcll_dp_unique_id(const char *nccl_lib, void *id128);
int dcll_dp_create(const char *nccl_lib, const void *id128, int rank, int world, int max_ctas, dcll_dp **out);
int dcll_dp_destroy(dcll_dp *dp);
int dcll_net_window_dp(dcll_dp *dp, dcll_conv_layer *layers, dcll_train_args *train, int n_layers, const void *x0,
                       const float *target, int64_t target_t_stride, int T, int burnin, const int32_t *iter0, int32_t *clout,
                       float *const *bucket, const size_t *bucket_floats, void *stream);
/* the same with update rules opt[2*l], opt[2*l+1] as in dcll_net_window_stats_opt */
int dcll_net_window_dp_opt(dcll_dp *dp, dcll_conv_layer *layers, dcll_train_args *train, dcll_optim *opt, int n_layers,
                           const void *x0, const float *target, int64_t target_t_stride, int T, int burnin, const int32_t *iter0,
                           int32_t *clout, float *const *bucket, const size_t *bucket_floats, void *stream);

/* -- multi-timestep inference of the radio_ml_conv stack on a 16x16 plane (test_radio_ml.py:144-145, script geometry) -- *
 * One launch runs Tc timesteps of the three conv cores (1->32, 32->32, 32->32; 7x7, padding 3, no pooling) with one CTA
 * per sample: synaptic traces stay in registers, inter-layer spikes in shared memory, membranes in TMEM (tcgen05, split-bf16).
 * cells: device int32 [Tc][B][2]; pv_out[l]: device float32 [Tc][B][32*256] (sigmoid outputs of layer l, the read-out
 * input).  State (eps0/eps1 of the current half, arp) is read at the start and written back at the end; `cur` is not
 * flipped.  The read-outs then run batched over Tc*B rows with dcll_conv_readout_rows (descriptor with B = Tc*B).
 * Operand form of layers 1 and 2, from their descriptors: precision DCLL_PREC_F16X2 runs the f16x2 form of the
 * per-timestep forward (fp16 traces scaled by 2^a_exp against the fp16 {hi,lo} weight image of w_exp), any other
 * precision the split-bf16 form; layer 0 runs on the FMA pipe from weight_t in either case.  Quantised layers use the
 * images dcll_conv_sync_weights left in weight_t / weight_mma.  Layers 1 and 2 of different forms: DCLL_EUNSUPPORTED;
 * an f16x2 layer without w_exp or with a_exp outside [-100, 100]: DCLL_EINVAL.                                          */
int dcll_infer_stack16(const dcll_conv_layer *layers, int n_layers, const int32_t *cells, int Tc, float *const *pv_out,
                       void *stream);
int dcll_conv_readout_rows(const dcll_conv_layer *L, int32_t *clout, void *stream);

/* -- vote: dcll/pytorch_libdcll.py:44-61 ------------------------------------------------------ *
 * pred[b] = most frequent class of clout[t0..T,b] (first-seen wins ties, as Counter does).    */
int dcll_vote(const int32_t *clout, int T, int t_stride, int B, int K, int32_t *pred, void *stream);

/* -- quantised weights (defined by this repo, no reference counterpart; oracle/quant.py) ------ *
 * per-output-channel symmetric int8: s = max|w|/127 (1 if 0), q = clamp(rint(w/s),-127,127).  */
int dcll_quantize(const float *w, int rows, int cols, int8_t *codes, float *scales, void *stream);
int dcll_dequantize(const int8_t *codes, const float *scales, int rows, int cols, float *w, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* DCLL_B200_H */
