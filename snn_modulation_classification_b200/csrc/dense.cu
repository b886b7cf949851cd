// DenseDCLLlayer step (dcll/pytorch_libdcll.py:72-266), FP32.
//
// The dense layers are exported by the reference's library but instantiated by none of its entry points
// (SURVEY.md section 2, row 4), so this path favours simplicity: an element-wise trace kernel (HBM bound) and
// one strided, shared-memory tiled SGEMM with fused epilogues for the four contractions of a step
//   vmem = eps1 W^T + b            (:141)      pvoutput = pv Wo^T + bo        (:253)
//   g_u  = (g_o Wo) * pv (1 - pv)  (autograd)  gW = g_u^T eps1, gb = sum g_u  (autograd)
#include "common.cuh"

namespace dcll {

// eps0 = x*tau_s + alphas*eps0 ; eps1 = alpha*eps1 + eps0*tau_m   (:139-140), in place, one rounding per op
__global__ void dense_trace_kernel(const float *__restrict__ x, float *__restrict__ e0, float *__restrict__ e1,
                                   const float *__restrict__ alpha, const float *__restrict__ alphas,
                                   const float *__restrict__ tau_m, const float *__restrict__ tau_s, int per_feature,
                                   int In, size_t n) {
    pdl_entry();
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    int k = per_feature ? (int)(i % In) : 0;
    float n0 = __fadd_rn(__fmul_rn(x[i], tau_s[k]), __fmul_rn(alphas[k], e0[i]));
    float n1 = __fadd_rn(__fmul_rn(alpha[k], e1[i]), __fmul_rn(n0, tau_m[k]));
    e0[i] = n0;
    e1[i] = n1;
}

enum { EPI_BIAS = 0, EPI_NEURON = 1, EPI_SIGMOID_GRAD = 2 };
struct GemmP {
    const float *A, *Bm;       // C[m,n] = sum_k A[m*sam + k*sak] * Bm[n*sbn + k*sbk]
    long sam, sak, sbn, sbk;
    int M, N, Kd;
    float *C;                  // [M,N] row-major
    const float *bias;         // [N] or null
    // EPI_NEURON
    float *arp, *spikes, *pv;
    float alpharp, wrp;
    // EPI_SIGMOID_GRAD
    const float *pv_in;
};

template <int EPI>
__global__ void __launch_bounds__(256) sgemm_kernel(const GemmP p) {
    pdl_entry();
    constexpr int BT = 32, BKK = 16;
    __shared__ float As[BKK][BT + 1], Bs[BKK][BT + 1];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;   // 16 x 16 threads, 2 x 2 outputs each
    const int m0 = blockIdx.y * BT, n0 = blockIdx.x * BT;
    float acc[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
    for (int k0 = 0; k0 < p.Kd; k0 += BKK) {
        for (int i = threadIdx.x; i < BT * BKK; i += 256) {
            int kk = i % BKK, r = i / BKK;
            int m = m0 + r, n = n0 + r, k = k0 + kk;
            As[kk][r] = (m < p.M && k < p.Kd) ? p.A[m * p.sam + k * p.sak] : 0.f;
            Bs[kk][r] = (n < p.N && k < p.Kd) ? p.Bm[n * p.sbn + k * p.sbk] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < BKK; ++kk) {
            float a0 = As[kk][ty], a1 = As[kk][ty + 16], b0 = Bs[kk][tx], b1 = Bs[kk][tx + 16];
            acc[0][0] = fmaf(a0, b0, acc[0][0]), acc[0][1] = fmaf(a0, b1, acc[0][1]);
            acc[1][0] = fmaf(a1, b0, acc[1][0]), acc[1][1] = fmaf(a1, b1, acc[1][1]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            int m = m0 + ty + 16 * i, n = n0 + tx + 16 * j;
            if (m >= p.M || n >= p.N) continue;
            size_t o = (size_t)m * p.N + n;
            float v = acc[i][j] + (p.bias ? p.bias[n] : 0.f);
            if (EPI == EPI_NEURON) {
                float a = 0.f;
                if (p.arp) {                                       // :182-183
                    a = __fmul_rn(p.alpharp, p.arp[o]);
                    v = __fadd_rn(v, a);
                }
                float s = v > 0.f ? 1.f : 0.f;
                p.spikes[o] = s;
                p.pv[o] = sigmoidf_ref(v);
                if (p.arp) p.arp[o] = __fsub_rn(a, __fmul_rn(s, p.wrp));   // :189
            } else if (EPI == EPI_SIGMOID_GRAD) {
                float q = p.pv_in[o];
                v = v * (1.f - q) * q;
            }
            p.C[o] = v;
        }
}

template <int EPI>
static int gemm(const GemmP &p, cudaStream_t st) {
    dim3 grid(ceil_div(p.N, 32), ceil_div(p.M, 32));
    launch_k(sgemm_kernel<EPI>, grid, 256, 0, st, p);
    DCLL_LAUNCH_OK("sgemm_kernel");
    return DCLL_OK;
}

__global__ void dense_finish_kernel(const float *__restrict__ pvoutput, int B, int K, int32_t *__restrict__ clout) {
    pdl_entry();
    int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    int best = 0;
    float bv = pvoutput[(size_t)b * K];
    for (int k = 1; k < K; ++k) {
        float v = pvoutput[(size_t)b * K + k];
        if (v > bv) bv = v, best = k;
    }
    clout[b] = best;
}

__global__ void dense_loss_grad_kernel(const float *__restrict__ pvoutput, const float *__restrict__ target, int B, int K,
                                       int loss_kind, float *__restrict__ g_o) {
    pdl_entry();
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * K) return;
    if (loss_kind == DCLL_LOSS_CROSS_ENTROPY) {
        const int b = i / K;
        float unused = 0.f;   // the host computes the dense loss value itself
        g_o[i] = ce_grad_elem(pvoutput + (size_t)b * K, target + (size_t)b * K, K, i - b * K, B, unused);
    } else {
        g_o[i] = loss_grad_elem(pvoutput[i], target[i], loss_kind, B * K);
    }
}

__global__ void colsum_kernel(const float *__restrict__ g, int B, int N, float *__restrict__ out) {
    pdl_entry();
    int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    float s = 0.f;
    for (int b = 0; b < B; ++b) s += g[(size_t)b * N + n];
    out[n] = s;
}

}  // namespace dcll

using namespace dcll;

static int check_dense(const dcll_dense_layer *L, const char *who) {
    DCLL_REQUIRE(L && L->B > 0 && L->In > 0 && L->Out > 0 && L->K > 0, DCLL_EINVAL, "%s: bad dimensions", who);
    DCLL_REQUIRE(L->alpha && L->alphas && L->tau_m && L->tau_s && L->weight && L->bias && L->wo && L->bo && L->eps0 &&
                     L->eps1 && L->spikes && L->pv && L->vmem && L->pvoutput,
                 DCLL_EINVAL, "%s: null pointer", who);
    DCLL_REQUIRE(L->coef_mode == DCLL_COEF_SCALAR || L->coef_mode == DCLL_COEF_CHANNEL, DCLL_EINVAL,
                 "%s: time constants must be scalar or per input feature", who);
    DCLL_REQUIRE(!(L->wrp > 0.f) || L->arp, DCLL_EINVAL, "%s: refractory layer without arp state", who);
    return DCLL_OK;
}

extern "C" __attribute__((visibility("default"))) size_t dcll_sizeof_dense_layer(void) { return sizeof(dcll_dense_layer); }

extern "C" __attribute__((visibility("default"))) int dcll_dense_step_fwd(dcll_dense_layer *L, const float *x,
                                                                           int32_t *clout, void *stream) {
    int rc = check_dense(L, "dcll_dense_step_fwd");
    if (rc != DCLL_OK) return rc;
    DCLL_REQUIRE(x, DCLL_EINVAL, "dcll_dense_step_fwd: null input");
    cudaStream_t st = (cudaStream_t)stream;
    size_t n = (size_t)L->B * L->In;
    launch_k(dense_trace_kernel, (unsigned)((n + 255) / 256), 256, 0, st, x, L->eps0, L->eps1, L->alpha, L->alphas, L->tau_m,
                                                                    L->tau_s, L->coef_mode == DCLL_COEF_CHANNEL, L->In, n);
    DCLL_LAUNCH_OK("dense_trace_kernel");
    GemmP p = {};
    p.A = L->eps1, p.sam = L->In, p.sak = 1;          // eps1 [B,In]
    p.Bm = L->weight, p.sbn = L->In, p.sbk = 1;       // W [Out,In]
    p.M = L->B, p.N = L->Out, p.Kd = L->In, p.C = L->vmem, p.bias = L->bias;
    p.arp = L->wrp > 0.f ? L->arp : nullptr, p.spikes = L->spikes, p.pv = L->pv, p.alpharp = L->alpharp, p.wrp = L->wrp;
    rc = gemm<EPI_NEURON>(p, st);
    if (rc != DCLL_OK) return rc;
    GemmP q = {};
    q.A = L->pv, q.sam = L->Out, q.sak = 1;           // pv [B,Out]
    q.Bm = L->wo, q.sbn = L->Out, q.sbk = 1;          // Wo [K,Out]
    q.M = L->B, q.N = L->K, q.Kd = L->Out, q.C = L->pvoutput, q.bias = L->bo;
    rc = gemm<EPI_BIAS>(q, st);
    if (rc != DCLL_OK) return rc;
    if (clout) {
        launch_k(dense_finish_kernel, ceil_div(L->B, 128), 128, 0, st, L->pvoutput, L->B, L->K, clout);
        DCLL_LAUNCH_OK("dense_finish_kernel");
    }
    return DCLL_OK;
}

extern "C" __attribute__((visibility("default"))) int dcll_dense_step_bwd_update(dcll_dense_layer *L, dcll_train_args *a,
                                                                                  void *stream) {
    return dcll_dense_step_bwd_update_opt(L, a, nullptr, stream);
}

// opt: the update rule of adam_i2h, or null (Adam)
extern "C" __attribute__((visibility("default"))) int dcll_dense_step_bwd_update_opt(dcll_dense_layer *L, dcll_train_args *a,
                                                                                      dcll_optim *opt, void *stream) {
    int rc = check_dense(L, "dcll_dense_step_bwd_update");
    if (rc != DCLL_OK) return rc;
    DCLL_REQUIRE(!opt || (opt->kind >= DCLL_OPT_ADAM && opt->kind <= DCLL_OPT_RADAM), DCLL_EINVAL,
                 "dcll_dense_step_bwd_update_opt: unknown update rule");
    DCLL_REQUIRE(a && L->g_o && L->g_u && L->grad_w && L->grad_b, DCLL_EINVAL, "dcll_dense_step_bwd_update: null scratch");
    cudaStream_t st = (cudaStream_t)stream;
    const int nk = L->B * L->K;
    DCLL_REQUIRE(a->loss_kind >= DCLL_LOSS_SMOOTHL1 && a->loss_kind <= DCLL_LOSS_HINGE, DCLL_EINVAL,
                 "dcll_dense_step_bwd_update: unknown loss");
    if (a->loss_kind == DCLL_LOSS_EXTERNAL) {
        DCLL_REQUIRE(a->g_o_ext, DCLL_EINVAL, "dcll_dense_step_bwd_update: external loss gradient missing");
        DCLL_CUDA_OK(cudaMemcpyAsync(L->g_o, a->g_o_ext, sizeof(float) * nk, cudaMemcpyDeviceToDevice, st));
    } else {
        DCLL_REQUIRE(a->target, DCLL_EINVAL, "dcll_dense_step_bwd_update: null target");
        launch_k(dense_loss_grad_kernel, ceil_div(nk, 256), 256, 0, st, L->pvoutput, a->target, L->B, L->K, a->loss_kind, L->g_o);
        DCLL_LAUNCH_OK("dense_loss_grad_kernel");
    }
    GemmP p = {};                                      // g_u[b,o] = (sum_k g_o[b,k] Wo[k,o]) * pv (1-pv)
    p.A = L->g_o, p.sam = L->K, p.sak = 1;
    p.Bm = L->wo, p.sbn = 1, p.sbk = L->Out;
    p.M = L->B, p.N = L->Out, p.Kd = L->K, p.C = L->g_u, p.pv_in = L->pv;
    rc = gemm<EPI_SIGMOID_GRAD>(p, st);
    if (rc != DCLL_OK) return rc;
    GemmP q = {};                                      // gW[o,i] = sum_b g_u[b,o] eps1[b,i]
    q.A = L->g_u, q.sam = 1, q.sak = L->Out;
    q.Bm = L->eps1, q.sbn = 1, q.sbk = L->In;
    q.M = L->Out, q.N = L->In, q.Kd = L->B, q.C = L->grad_w;
    rc = gemm<EPI_BIAS>(q, st);
    if (rc != DCLL_OK) return rc;
    launch_k(colsum_kernel, ceil_div(L->Out, 128), 128, 0, st, L->g_u, L->B, L->Out, L->grad_b);
    DCLL_LAUNCH_OK("colsum_kernel");
    if (a->apply_update) {
        DCLL_REQUIRE(a->adam_i2h.m_w && a->adam_i2h.v_w && a->adam_i2h.m_b && a->adam_i2h.v_b, DCLL_EINVAL,
                     "dcll_dense_step_bwd_update: null Adam state");
        rc = dense_flat_update(a->adam_i2h, opt, L->weight, L->grad_w, (size_t)L->Out * L->In, L->bias, L->grad_b, (size_t)L->Out, st);
        if (rc != DCLL_OK) return rc;
    }
    return DCLL_OK;
}
