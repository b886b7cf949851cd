// Local weight gradient of one Conv2dDCLLlayer and the per-timestep Adam step, FP32 parity mode.
//
// Replaces (reference): loss.backward() + optimizer.step() of DCLLBase.train_dcll
// (dcll/pytorch_libdcll.py:704,711-712) for i2h.{weight,bias}.  There is no BPTT and no gradient
// w.r.t. the layer input (states and inter-layer spikes are detached, :424-425,:254,:606), so the
// backward pass is exactly one contraction:
//     gW[co,ci,kh,kw] = sum_{b,h,w} g_u[b,co,h,w] * eps1[b,ci,h+kh-padH,w+kw-padW],   gb[co] = sum g_u
// with g_u = dL/d(membrane) produced by readout_bwd_kernel (non-zero only at the pool argmax).
//
// Decomposition: the reduction runs over B*Hc*Wc positions (1M at 128x128, B=64) while the result has
// only Cout*Cin*KH*KW entries, so the position axis is split over CTAs (split-K) and every CTA keeps its
// slice of gW in registers: thread = (4 output channels, 1 input channel, 1 kernel row) x KW taps.
// Partials are summed in a fixed order by reduce_adam_kernel, which also applies Adam and refreshes the
// [Cin,KH*KW,CoutPad] weight copy the forward kernel consumes -- deterministic, no float atomics.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace dcll {

struct WgP {
    const float *g_u;        // [B,Cout,Hp,Wp]
    const uint8_t *pool_idx; // [B,Cout,Hp,Wp] or null
    const float *eps1;       // [B,Cin,H,W]  (state AFTER the forward step)
    float *partial;          // [S][nW + Cout]
    int B, Cin, H, W, Cout, padH, padW, Hc, Wc, Hp, Wp;
    int tiles_h, tiles_w, n_units, S, n_tot, nW;
};

__host__ __device__ constexpr int wg_ci_t(int kh) { return kh >= 7 ? 4 : (kh >= 5 ? 6 : (kh >= 3 ? 10 : 32)); }
__host__ __device__ constexpr int wg_plane(int halo_h, int pitch) {
    int s = halo_h * pitch;      // multiple of 4
    if (((s / 4) & 1) == 0) s += 4;  // (stride/4) odd: input-channel planes start in different 16-byte bank groups
    return s;
}

template <int KH, int KW, int PH, int PW>
__global__ void __launch_bounds__(8 * wg_ci_t(KH) * KH) wgrad_kernel(const WgP p) {
    pdl_entry();
    constexpr int TH = 16, SEGS = 2, TW = 16;
    constexpr int CI_T = wg_ci_t(KH);
    constexpr int NT = 8 * CI_T * KH;
    constexpr int HALO_H = TH + KH - 1, HALO_W = TW + KW - 1;
    constexpr int PITCH = ((TW + 8 > HALO_W ? TW + 8 : HALO_W) + 3) / 4 * 4;
    constexpr int PLANE = wg_plane(HALO_H, PITCH);
    constexpr int NX4 = (8 + KW - 1 + 3) / 4;

    extern __shared__ __align__(16) float wg_smem[];
    float *gs = wg_smem;                 // [pos][32 co], 16-byte chunks XOR-swizzled by pos&7
    float *xs = wg_smem + TH * TW * 32;  // [ci][halo row][pitch]

    const int tid = threadIdx.x;
    const int coq = tid & 7;
    const int ci_l = (tid >> 3) % CI_T;
    const int kh = tid / (8 * CI_T);
    const int ci0 = blockIdx.x * CI_T;
    const int s = blockIdx.y;
    const int z = blockIdx.z;
    const bool bias_thread = (blockIdx.x == 0) && ci_l == 0 && kh == 0;

    float acc[4][KW];
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int k = 0; k < KW; ++k) acc[c][k] = 0.f;
    float gb[4] = {0.f, 0.f, 0.f, 0.f};

    const int tiles = p.tiles_h * p.tiles_w;
    for (int u = s; u < p.n_units; u += p.S) {
        const int b = u / tiles;
        const int tile = u - b * tiles;
        const int th_i = tile / p.tiles_w, tw_i = tile - th_i * p.tiles_w;
        const int h0 = th_i * TH, w0 = tw_i * TW;
        __syncthreads();
        // ---- g_u tile -> shared, transposed to channel-last
        if (PH * PW == 1) {
            for (int i = tid; i < TH * TW * 8; i += NT) {
                int pos = i % (TH * TW), q = i / (TH * TW);
                int r = pos / TW, c = pos - r * TW;
                int oh = h0 + r, ow = w0 + c;
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (oh < p.Hc && ow < p.Wc) {
                    int co = z * 32 + q * 4;
                    size_t o = ((size_t)(b * p.Cout + co) * p.Hc + oh) * p.Wc + ow;
                    size_t cs = (size_t)p.Hc * p.Wc;
                    if (co < p.Cout) v.x = __ldg(p.g_u + o);
                    if (co + 1 < p.Cout) v.y = __ldg(p.g_u + o + cs);
                    if (co + 2 < p.Cout) v.z = __ldg(p.g_u + o + 2 * cs);
                    if (co + 3 < p.Cout) v.w = __ldg(p.g_u + o + 3 * cs);
                }
                *reinterpret_cast<float4 *>(gs + pos * 32 + ((q ^ (pos & 7)) << 2)) = v;
            }
        } else {
            // pooled grid: every pooled cell scatters its gradient to the argmax position of its window
            // and zeros to the rest; rows/columns not covered by any window are zero-filled first.
            for (int i = tid; i < TH * TW * 8; i += NT)
                *reinterpret_cast<float4 *>(gs + i * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
            __syncthreads();
            constexpr int PTH = TH / PH, PTW = TW / PW;
            for (int i = tid; i < PTH * PTW * 8; i += NT) {
                int pc = i % (PTH * PTW), q = i / (PTH * PTW);
                int pr = pc / PTW, pcx = pc - pr * PTW;
                int ohp = h0 / PH + pr, owp = w0 / PW + pcx;
                if (ohp < p.Hp && owp < p.Wp) {
                    int co = z * 32 + q * 4;
                    size_t o = ((size_t)(b * p.Cout + co) * p.Hp + ohp) * p.Wp + owp;
                    size_t cs = (size_t)p.Hp * p.Wp;
                    float gv[4] = {0.f, 0.f, 0.f, 0.f};
                    int iv[4] = {0, 0, 0, 0};
#pragma unroll
                    for (int c = 0; c < 4; ++c)
                        if (co + c < p.Cout) gv[c] = __ldg(p.g_u + o + c * cs), iv[c] = p.pool_idx[o + c * cs];
#pragma unroll
                    for (int wi = 0; wi < PH * PW; ++wi) {
                        int widx = (PW == 2) ? wi : wi * 2;  // stored index = dy*2 + dx
                        int dy = wi / PW, dx = wi % PW;
                        int pos = (pr * PH + dy) * TW + pcx * PW + dx;
                        float4 v = make_float4(iv[0] == widx ? gv[0] : 0.f, iv[1] == widx ? gv[1] : 0.f,
                                               iv[2] == widx ? gv[2] : 0.f, iv[3] == widx ? gv[3] : 0.f);
                        *reinterpret_cast<float4 *>(gs + pos * 32 + ((q ^ (pos & 7)) << 2)) = v;
                    }
                }
            }
        }
        // ---- eps1 halo tile -> shared
        for (int i = tid; i < CI_T * HALO_H * HALO_W; i += NT) {
            int cl = i / (HALO_H * HALO_W);
            int rem = i - cl * (HALO_H * HALO_W);
            int r = rem / HALO_W, c = rem - r * HALO_W;
            int gh = h0 - p.padH + r, gw = w0 - p.padW + c, ci = ci0 + cl;
            float v = 0.f;
            if (ci < p.Cin && gh >= 0 && gh < p.H && gw >= 0 && gw < p.W)
                v = __ldg(p.eps1 + ((size_t)(b * p.Cin + ci) * p.H + gh) * p.W + gw);
            xs[cl * PLANE + r * PITCH + c] = v;
        }
        __syncthreads();
        // ---- accumulate
#pragma unroll 1
        for (int row = 0; row < TH; ++row) {
#pragma unroll
            for (int seg = 0; seg < SEGS; ++seg) {
                const float *xrow = xs + ci_l * PLANE + (row + kh) * PITCH + seg * 8;
                float xr[NX4 * 4];
#pragma unroll
                for (int q = 0; q < NX4; ++q) {
                    float4 v = *reinterpret_cast<const float4 *>(xrow + 4 * q);
                    xr[4 * q] = v.x, xr[4 * q + 1] = v.y, xr[4 * q + 2] = v.z, xr[4 * q + 3] = v.w;
                }
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int pos = row * TW + seg * 8 + j;
                    float4 gv = *reinterpret_cast<const float4 *>(gs + pos * 32 + ((coq ^ (pos & 7)) << 2));
#pragma unroll
                    for (int k = 0; k < KW; ++k) {
                        acc[0][k] = fmaf(gv.x, xr[j + k], acc[0][k]);
                        acc[1][k] = fmaf(gv.y, xr[j + k], acc[1][k]);
                        acc[2][k] = fmaf(gv.z, xr[j + k], acc[2][k]);
                        acc[3][k] = fmaf(gv.w, xr[j + k], acc[3][k]);
                    }
                    if (bias_thread) gb[0] += gv.x, gb[1] += gv.y, gb[2] += gv.z, gb[3] += gv.w;
                }
            }
        }
    }
    // ---- partials, in the layout of the weight tensor [Cout,Cin,KH,KW] (+ bias at the end)
    float *out = p.partial + (size_t)s * p.n_tot;
    const int ci = ci0 + ci_l;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        int co = z * 32 + coq * 4 + c;
        if (co < p.Cout) {
            if (ci < p.Cin) {
#pragma unroll
                for (int k = 0; k < KW; ++k) out[((size_t)(co * p.Cin + ci) * KH + kh) * KW + k] = acc[c][k];
            }
            if (bias_thread) out[p.nW + co] = gb[c];
        }
    }
}

// Tail shared by the two reducers: thread (sl == 0, element i) holds the combined gradient in red[.][e]; Adam on the element,
// kernel-side weight copies, and -- F16X2 (w_exp != null) -- the fp16 image with the device-tracked exponent:
//   * the image written here is fp16 {hi,lo} of w * 2^k, k = w_exp[1], read by every block at its start;
//   * every block folds max |w_new| into w_exp[3] (bit pattern of a non-negative float orders like the float; the maximum does
//     not depend on the order, so this stays deterministic);
//   * the LAST block to finish (ticket in w_exp[2]) publishes slot 0 = the exponent this launch wrote the image with -- what the
//     next convolution must undo -- and slot 1 = the exponent for the next image from this step's maximum, and resets 2 and 3.
//     It is the only writer of the slots, and by then every other block has read slot 1.
constexpr int RED_U = 10;   // partial-block loads in flight per thread in the reducers below
template <class Sc>
__device__ __forceinline__ void reduce_adam_tail(float (&red)[4][64], int n_tot, int nW, int Cout, int CoutPad, int CinKK,
                                                 float *__restrict__ w, float *__restrict__ wt, float *__restrict__ bias,
                                                 float *__restrict__ m_w, float *__restrict__ v_w, float *__restrict__ m_b,
                                                 float *__restrict__ v_b, float *__restrict__ grad_w, float *__restrict__ grad_b, int apply,
                                                 const Sc &sc, __nv_bfloat16 *__restrict__ w_mma, int Cin, int KHKW, int KW,
                                                 int *__restrict__ w_exp, int kexp, float w_pre, float m_pre, float v_pre) {
    const int e = threadIdx.x & 63, sl = threadIdx.x >> 6;
    const int i = blockIdx.x * 64 + e;
    float wabs = 0.f;
    if (sl == 0 && i < n_tot) {
        const float g = ((red[0][e] + red[1][e]) + red[2][e]) + red[3][e];
        if (i < nW) {
            if (grad_w) grad_w[i] = g;
            if (apply) {
                float wv = w_pre, m = m_pre, v = v_pre;                   // loaded by the caller BEFORE the reduction (one round trip less)
                elem_update(wv, g, m, v, sc);
                w[i] = wv, m_w[i] = m, v_w[i] = v;
                wabs = fabsf(wv);
                int co = i / CinKK, r = i - co * CinKK;
                wt[(size_t)r * CoutPad + co] = wv;
                if (w_mma) {   // {hi,lo} copy in the tcgen05 B-operand layout [tap][ci/8][{hi,lo}][co][8] (conv_fwd_tc.cu)
                    const int ci = r / KHKW, tap = r - ci * KHKW;
                    size_t o = (size_t)tap * (2 * Cin * Cout) + ((size_t)(ci >> 3) * 2 * Cout + co) * 8 + (ci & 7);
                    if (Cin == 1) o = ((size_t)(tap / KW) * 2 * Cout + co) * 8 + tap % KW;   // [kh][part][co][8 column shifts]
                    if (w_exp) {
                        // (the exponent is one step old: 2^8 of headroom; a weight that outgrows it within ONE step saturates)
                        const float vs = fminf(fmaxf(__fmul_rn(wv, pow2i(kexp)), -65504.f), 65504.f);
                        const __half hi = __float2half_rn(vs);
                        reinterpret_cast<__half *>(w_mma)[o] = hi;
                        reinterpret_cast<__half *>(w_mma)[o + (size_t)Cout * 8] = __float2half_rn(vs - __half2float(hi));
                    } else {
                        __nv_bfloat16 hi = __float2bfloat16_rn(wv);
                        __nv_bfloat16 lo = __float2bfloat16_rn(wv - __bfloat162float(hi));
                        w_mma[o] = hi;
                        w_mma[o + (size_t)Cout * 8] = lo;
                    }
                }
            }
        } else {
            int co = i - nW;
            if (grad_b) grad_b[co] = g;
            if (apply) {
                float wv = bias[co], m = m_b[co], v = v_b[co];
                elem_update(wv, g, m, v, sc);
                bias[co] = wv, m_b[co] = m, v_b[co] = v;
            }
        }
    }
    if (w_exp && apply) {
        if (sl == 0) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) wabs = fmaxf(wabs, __shfl_xor_sync(0xffffffffu, wabs, o));
            if ((threadIdx.x & 31) == 0 && wabs > 0.f) atomicMax(reinterpret_cast<unsigned *>(w_exp + 3), __float_as_uint(wabs));
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();
            const int ticket = atomicAdd(w_exp + 2, 1);
            if (ticket == (int)gridDim.x - 1) {
                __threadfence();
                const unsigned mb = atomicExch(reinterpret_cast<unsigned *>(w_exp + 3), 0u);
                w_exp[0] = kexp;
                w_exp[1] = weight_exp_for(__uint_as_float(mb));
                w_exp[2] = 0;
            }
        }
    }
}

// parameters of the reducers' update tail (w, moments, gradients, kernel-side copies)
#define RED_TAIL_PARAMS                                                                                                          \
    float *__restrict__ w, float *__restrict__ wt, float *__restrict__ bias, float *__restrict__ m_w, float *__restrict__ v_w,   \
        float *__restrict__ m_b, float *__restrict__ v_b, float *__restrict__ grad_w, float *__restrict__ grad_b, int apply
#define RED_TAIL_PARAMS2 __nv_bfloat16 *__restrict__ w_mma, int Cin, int KHKW, int KW, int *__restrict__ w_exp
#define RED_TAIL_ARGS w, wt, bias, m_w, v_w, m_b, v_b, grad_w, grad_b, apply, sc, w_mma, Cin, KHKW, KW, w_exp

// grad = sum_s partial[s] (fixed order) ; Adam ; W, W^T, moments
template <class Sc>
__device__ __forceinline__ void reduce_body(const float *__restrict__ partial, int S, int n_tot, int nW, int Cout, int CoutPad,
                                            int CinKK, RED_TAIL_PARAMS, const Sc &sc, RED_TAIL_PARAMS2) {
    // CTA = 64 elements x 4 slices of the partial blocks (a single serial walk over ~150 blocks was pure load latency);
    // the slices are combined in a fixed order, so the result stays bit-reproducible
    __shared__ float red[4][64];
    const int e = threadIdx.x & 63, sl = threadIdx.x >> 6;
    const int i = blockIdx.x * 64 + e;
    const int kexp = w_exp ? *reinterpret_cast<volatile int *>(w_exp + 1) : 0;
    float g = 0.f, w_pre = 0.f, m_pre = 0.f, v_pre = 0.f;
    if (sl == 0 && i < nW && apply) w_pre = w[i], m_pre = m_w[i], v_pre = v_w[i];
    if (i < n_tot) {
        // RED_U loads in flight per thread, added in the same fixed order as a serial walk (a rolled loop waited one L2 round trip
        // per block: this kernel is pure latency, 10-12 us for 5 MB)
        // (the loads are UNCONDITIONAL, past the end the slice's last block is read again: predicated loads were scheduled
        //  load - add - load - add, one round trip each)
        const int s_hi = sl + 4 * ((S - 1 - sl) >> 2);                       // last block of this slice (S > sl inside the loop)
        for (int s0 = sl; s0 < S; s0 += 4 * RED_U) {
            float t[RED_U];
#pragma unroll
            for (int u = 0; u < RED_U; ++u) t[u] = __ldg(partial + (size_t)min(s0 + 4 * u, s_hi) * n_tot + i);
#pragma unroll
            for (int u = 0; u < RED_U; ++u)
                if (s0 + 4 * u < S) g += t[u];
        }
    }
    red[sl][e] = g;
    __syncthreads();
    reduce_adam_tail(red, n_tot, nW, Cout, CoutPad, CinKK, w, wt, bias, m_w, v_w, m_b, v_b, grad_w, grad_b, apply, sc, w_mma, Cin, KHKW,
                     KW, w_exp, kexp, w_pre, m_pre, v_pre);
}
__global__ void __launch_bounds__(256) reduce_adam_kernel(const float *__restrict__ partial, int S, int n_tot, int nW, int Cout,
                                                          int CoutPad, int CinKK, RED_TAIL_PARAMS, AdamScalars sc,
                                                          RED_TAIL_PARAMS2) {
    pdl_entry();
    reduce_body(partial, S, n_tot, nW, Cout, CoutPad, CinKK, RED_TAIL_ARGS);
}
__global__ void __launch_bounds__(256) reduce_opt_kernel(const float *__restrict__ partial, int S, int n_tot, int nW, int Cout,
                                                         int CoutPad, int CinKK, RED_TAIL_PARAMS, OptScalars sc, RED_TAIL_PARAMS2) {
    pdl_entry();
    reduce_body(partial, S, n_tot, nW, Cout, CoutPad, CinKK, RED_TAIL_ARGS);
}

// Same reduction + Adam tail for the partial blocks of wgrad_tc2_kernel (wgrad_tc2.cu): one compact block per CTA,
//   block[(co*32 + ci)*20 + a*5 + slot],  a = kernel column within the role (A: kw 0..3, B: kw 4..6), slot <-> kh = 4g - 1 + slot,
//   + 32 bias sums (role B blocks).  CTA c: pair c >> 1 (pairs [0, nA) = role A), kernel-row group g = c & 1.
// Element (kh, kw) lives in the role's CTAs with g = 0 when kh <= 3 (slot kh + 1) and with g = 1 when kh >= 3 (slot kh - 3);
// kh = 3 is the sum of both.  Blocks are walked in a fixed order by 4 slices that are combined in a fixed order.
template <class Sc>
__device__ __forceinline__ void reduce_rp_body(const float *__restrict__ partial, int nA, int nB, int blk, int nw_blk, int n_tot,
                                               int nW, int Cout, int CoutPad, int CinKK, RED_TAIL_PARAMS, const Sc &sc,
                                               RED_TAIL_PARAMS2) {
    __shared__ float red[4][64];
    const int e = threadIdx.x & 63, sl = threadIdx.x >> 6;
    const int i = blockIdx.x * 64 + e;
    // F16X2: the image written below is fp16 {hi,lo} of w * 2^k, k = w_exp[1] -- read by every block before any block can have
    // finished (the last block to finish is the only writer of the slots, see the end of the kernel)
    const int kexp = w_exp ? *reinterpret_cast<volatile int *>(w_exp + 1) : 0;
    float g = 0.f, w_pre = 0.f, m_pre = 0.f, v_pre = 0.f;
    if (sl == 0 && i < nW && apply) w_pre = w[i], m_pre = m_w[i], v_pre = v_w[i];
    if (i < nW) {
        const int cc = i / KHKW, tap = i - cc * KHKW;            // cc = co * Cin + ci
        const int kh = tap / KW, kw = tap - kh * KW;
        const bool roleA = kw < 4;
        const int a = roleA ? kw : kw - 4;
        const int c_first = roleA ? 0 : 2 * nA, c_last = roleA ? 2 * nA : 2 * (nA + nB);
        const size_t base = (size_t)cc * 20 + a * 5;
        // slice sl walks the blocks c = c_first + sl + 4 j, whose group (c & 1) is the parity of sl: either all or none of them
        // hold this element, and the slot is the same for all (RED_U loads in flight, fixed order as before)
        const int grp = (c_first + sl) & 1;
        if (grp == 0 ? kh <= 3 : kh >= 3) {
            const float *src = partial + base + (grp == 0 ? kh + 1 : kh - 3);
            const int c_hi = c_first + sl + 4 * ((c_last - 1 - c_first - sl) >> 2);   // last block of this slice (unconditional loads, see above)
            for (int c0 = c_first + sl; c0 < c_last; c0 += 4 * RED_U) {
                float t[RED_U];
#pragma unroll
                for (int u = 0; u < RED_U; ++u) t[u] = __ldg(src + (size_t)min(c0 + 4 * u, c_hi) * blk);
#pragma unroll
                for (int u = 0; u < RED_U; ++u)
                    if (c0 + 4 * u < c_last) g += t[u];
            }
        }
    } else if (i < n_tot) {
        const int c_last = 2 * (nA + nB);
        const float *src = partial + nw_blk + (i - nW);
        const int c_hi = 2 * nA + sl + 4 * ((c_last - 1 - 2 * nA - sl) >> 2);
        for (int c0 = 2 * nA + sl; c0 < c_last; c0 += 4 * RED_U) {
            float t[RED_U];
#pragma unroll
            for (int u = 0; u < RED_U; ++u) t[u] = __ldg(src + (size_t)min(c0 + 4 * u, c_hi) * blk);
#pragma unroll
            for (int u = 0; u < RED_U; ++u)
                if (c0 + 4 * u < c_last) g += t[u];
        }
    }
    red[sl][e] = g;
    __syncthreads();
    reduce_adam_tail(red, n_tot, nW, Cout, CoutPad, CinKK, w, wt, bias, m_w, v_w, m_b, v_b, grad_w, grad_b, apply, sc, w_mma, Cin, KHKW,
                     KW, w_exp, kexp, w_pre, m_pre, v_pre);
}
__global__ void __launch_bounds__(256) reduce_adam_rp_kernel(const float *__restrict__ partial, int nA, int nB, int blk, int nw_blk,
                                                             int n_tot, int nW, int Cout, int CoutPad, int CinKK, RED_TAIL_PARAMS,
                                                             AdamScalars sc, RED_TAIL_PARAMS2) {
    pdl_entry();
    reduce_rp_body(partial, nA, nB, blk, nw_blk, n_tot, nW, Cout, CoutPad, CinKK, RED_TAIL_ARGS);
}
__global__ void __launch_bounds__(256) reduce_opt_rp_kernel(const float *__restrict__ partial, int nA, int nB, int blk, int nw_blk,
                                                            int n_tot, int nW, int Cout, int CoutPad, int CinKK, RED_TAIL_PARAMS,
                                                            OptScalars sc, RED_TAIL_PARAMS2) {
    pdl_entry();
    reduce_rp_body(partial, nA, nB, blk, nw_blk, n_tot, nW, Cout, CoutPad, CinKK, RED_TAIL_ARGS);
}
#undef RED_TAIL_PARAMS
#undef RED_TAIL_PARAMS2
#undef RED_TAIL_ARGS

static int wg_n_ci_chunks(const dcll_conv_layer *L) {
    int ci_t = L->KH >= 7 ? 4 : (L->KH >= 5 ? 6 : (L->KH >= 3 ? 10 : 32));
    return ceil_div(L->Cin, ci_t);
}

int wgrad_units(const dcll_conv_layer *L) {
    Geo g = geo_of(L);
    return L->B * ceil_div(g.Hc, 16) * ceil_div(g.Wc, 16);
}

int wgrad_splits(const dcll_conv_layer *L) {
    int n_units = wgrad_units(L);
    int per_split_ctas = wg_n_ci_chunks(L) * ceil_div(L->Cout, 32);
    int S = max(1, min(n_units, (2 * 148) / per_split_ctas));
    int per = ceil_div(n_units, S);
    return ceil_div(n_units, per);
}

template <int KH, int KW>
constexpr size_t wg_smem_bytes() {
    constexpr int HALO_H = 16 + KH - 1, HALO_W = 16 + KW - 1;
    constexpr int PITCH = ((16 + 8 > HALO_W ? 16 + 8 : HALO_W) + 3) / 4 * 4;
    return sizeof(float) * (16 * 16 * 32 + wg_ci_t(KH) * wg_plane(HALO_H, PITCH));
}

template <int KH, int KW, int PH, int PW>
static int launch_wg_inst(const WgP &p, dim3 grid, cudaStream_t st) {
    constexpr int NT = 8 * wg_ci_t(KH) * KH;
    constexpr size_t smem = wg_smem_bytes<KH, KW>();
    DCLL_SMEM_ATTR((wgrad_kernel<KH, KW, PH, PW>), smem);
    launch_k(wgrad_kernel<KH, KW, PH, PW>, grid, NT, smem, st, p);
    DCLL_LAUNCH_OK("wgrad_kernel");
    return DCLL_OK;
}

template <int KH, int KW>
static int launch_wg(const WgP &p, const dcll_conv_layer *L, cudaStream_t st) {
    dim3 grid(wg_n_ci_chunks(L), p.S, ceil_div(L->Cout, 32));
    if (L->poolH == 1 && L->poolW == 1) return launch_wg_inst<KH, KW, 1, 1>(p, grid, st);
    if constexpr (KH > 1) {
        if (L->poolH == 2 && L->poolW == 2) return launch_wg_inst<KH, KW, 2, 2>(p, grid, st);
    } else {
        if (L->poolH == 1 && L->poolW == 2) return launch_wg_inst<KH, KW, 1, 2>(p, grid, st);
    }
    set_error("pooling (%d,%d) with kernel (%d,%d) has no sm_100a instantiation", L->poolH, L->poolW, KH, KW);
    return DCLL_EUNSUPPORTED;
}

// Adam on an already averaged gradient bucket [gW | gb | gWout | gbout] (data-parallel driver, dp.cu): the conv parameters go
// through reduce_adam_kernel with the bucket as its single partial block, so weight_t and the tensor-core weight image are
// refreshed by the same launch, as on the single-GPU path; output_ takes the flat kernel.  opt: the rules of adam_i2h, adam_out
// (null: Adam).
int launch_bucket_adam(const dcll_conv_layer *L, dcll_train_args *a, const float *bucket, cudaStream_t st, dcll_optim *opt) {
    Geo g = geo_of(L);
    const int n_tot = g.nW + L->Cout;
    {
        OptScalars buf;
        const OptScalars *so = next_opt_scalars(a->adam_i2h, opt, &buf);
        AdamScalars sc = adam_scalars(a->adam_i2h, a->adam_i2h.step + 1);
        dcll_adam &o = a->adam_i2h;
        ProfScope ps(KC_ADAM, 0, st);
#define RED_BUCKET(KERN, SC)                                                                                                          \
    launch_k(KERN, ceil_div(n_tot, 64), 256, 0, st, bucket, 1, n_tot, g.nW, L->Cout, g.CoutPad, L->Cin * L->KH * L->KW, L->weight,  \
             L->weight_t, L->bias, o.m_w, o.v_w, o.m_b, o.v_b, (float *)nullptr, (float *)nullptr, 1, SC,                            \
             L->quantized ? nullptr : reinterpret_cast<__nv_bfloat16 *>(L->weight_mma), L->Cin, L->KH * L->KW, L->KW,                \
             (prec_f16(L) && !L->quantized) ? L->w_exp : (int *)nullptr)   // F16X2: same image / exponent protocol as the single-GPU step
        if (so) {
            RED_BUCKET(reduce_opt_kernel, *so);
            DCLL_LAUNCH_OK("reduce_opt_kernel");
        } else {
            RED_BUCKET(reduce_adam_kernel, sc);
            DCLL_LAUNCH_OK("reduce_adam_kernel");
        }
#undef RED_BUCKET
        a->adam_i2h.step += 1;
        if (L->quantized) {
            int rc = sync_kernel_weights(L, st);
            if (rc != DCLL_OK) return rc;
        }
    }
    if (L->output_layer) {
        OptScalars buf;
        const OptScalars *sr = next_opt_scalars(a->adam_out, opt ? opt + 1 : nullptr, &buf);
        AdamScalars so = adam_scalars(a->adam_out, a->adam_out.step + 1);
        const float *gwout = bucket + n_tot, *gbout = gwout + (size_t)L->K * g.F;
        ProfScope ps(KC_ADAM, 1, st);
        const dcll_adam &o = a->adam_out;
        int rc = sr ? launch_opt_flat(L->wout, gwout, o.m_w, o.v_w, (size_t)L->K * g.F, *sr, st)
                    : launch_adam_flat(L->wout, gwout, o.m_w, o.v_w, (size_t)L->K * g.F, so, st);
        if (rc != DCLL_OK) return rc;
        rc = sr ? launch_opt_flat(L->bout, gbout, o.m_b, o.v_b, (size_t)L->K, *sr, st)
                : launch_adam_flat(L->bout, gbout, o.m_b, o.v_b, (size_t)L->K, so, st);
        if (rc != DCLL_OK) return rc;
        a->adam_out.step += 1;
    }
    return DCLL_OK;
}

int launch_wgrad(const dcll_conv_layer *L, dcll_train_args *a, cudaStream_t st, const OptScalars *so) {
    Geo g = geo_of(L);
    WsLayout ws = ws_layout(L);
    WgP p;
    p.g_u = L->g_u, p.pool_idx = L->pool_idx, p.eps1 = L->eps1[L->cur & 1];
    p.partial = (float *)((char *)L->workspace + ws.off_wg_part);
    p.B = L->B, p.Cin = L->Cin, p.H = L->H, p.W = L->W, p.Cout = L->Cout, p.padH = L->padH, p.padW = L->padW;
    p.Hc = g.Hc, p.Wc = g.Wc, p.Hp = g.Hp, p.Wp = g.Wp;
    p.tiles_h = ceil_div(g.Hc, 16), p.tiles_w = ceil_div(g.Wc, 16);
    p.n_units = wgrad_units(L), p.nW = g.nW, p.n_tot = g.nW + L->Cout;
    int rc;
    if (wgrad_tc2_supported(L)) {
        // row-pair N-concatenation kernel: g_u arrives as bf16 planes (readout_bwd2_kernel<.., IMG>), compact per-CTA partials
        int nA = 0, nB = 0;
        rc = launch_wgrad_tc2(L, p.partial, &nA, &nB, st);
        if (rc != DCLL_OK) return rc;
        AdamScalars sc = adam_scalars(a->adam_i2h, a->adam_i2h.step + 1);
        dcll_adam &o = a->adam_i2h;
        ProfScope ps(KC_ADAM, 0, st);
        const int blk = (int)(wgrad_tc2_partial_floats() / 148);
#define RED_RP(KERN, SC)                                                                                                              \
    launch_k(KERN, ceil_div(p.n_tot, 64), 256, 0, st, p.partial, nA, nB, blk, blk - L->Cout, p.n_tot, p.nW, L->Cout, g.CoutPad,         \
             L->Cin * L->KH * L->KW, L->weight, L->weight_t, L->bias, o.m_w, o.v_w, o.m_b, o.v_b, a->grad_w, a->grad_b, a->apply_update, \
             SC, L->quantized ? nullptr : reinterpret_cast<__nv_bfloat16 *>(L->weight_mma), L->Cin, L->KH * L->KW, L->KW,              \
             (prec_f16(L) && !L->quantized) ? L->w_exp : nullptr)
        if (so) {
            RED_RP(reduce_opt_rp_kernel, *so);
            DCLL_LAUNCH_OK("reduce_opt_rp_kernel");
        } else {
            RED_RP(reduce_adam_rp_kernel, sc);
            DCLL_LAUNCH_OK("reduce_adam_rp_kernel");
        }
#undef RED_RP
        if (a->apply_update && L->quantized) return sync_kernel_weights(L, st);
        return DCLL_OK;
    }
    DCLL_REQUIRE(!prec_f16(L), DCLL_EUNSUPPORTED,
                 "f16x2: the layer needs the row-pair weight-gradient kernel (even conv height, conv width a multiple of 8, K <= 32)");
    if (wgrad_tc_supported(L)) {
        p.S = wgrad_tc_splits(L);
        rc = launch_wgrad_tc(L, p.partial, p.S, st);
    } else {
        p.S = wgrad_splits(L);
        if (L->KH == 7 && L->KW == 7) rc = launch_wg<7, 7>(p, L, st);
        else if (L->KH == 5 && L->KW == 5) rc = launch_wg<5, 5>(p, L, st);
        else if (L->KH == 3 && L->KW == 3) rc = launch_wg<3, 3>(p, L, st);
        else if (L->KH == 1 && L->KW == 3) rc = launch_wg<1, 3>(p, L, st);
        else { set_error("kernel_size (%d,%d) has no sm_100a instantiation", L->KH, L->KW); return DCLL_EUNSUPPORTED; }
    }
    if (rc != DCLL_OK) return rc;
    AdamScalars sc = adam_scalars(a->adam_i2h, a->adam_i2h.step + 1);
    dcll_adam &o = a->adam_i2h;
    ProfScope ps(KC_ADAM, 0, st);
#define RED(KERN, SC)                                                                                                           \
    launch_k(KERN, ceil_div(p.n_tot, 64), 256, 0, st, p.partial, p.S, p.n_tot, p.nW, L->Cout, g.CoutPad, L->Cin * L->KH * L->KW,  \
             L->weight, L->weight_t, L->bias, o.m_w, o.v_w, o.m_b, o.v_b, a->grad_w, a->grad_b, a->apply_update, SC,                \
             L->quantized ? nullptr : reinterpret_cast<__nv_bfloat16 *>(L->weight_mma), L->Cin, L->KH * L->KW, L->KW, (int *)nullptr)
    if (so) {
        RED(reduce_opt_kernel, *so);
        DCLL_LAUNCH_OK("reduce_opt_kernel");
    } else {
        RED(reduce_adam_kernel, sc);
        DCLL_LAUNCH_OK("reduce_adam_kernel");
    }
#undef RED
    // reduce_adam_kernel refreshed weight_t and the tensor-core split itself; only the quantised image needs a pass
    if (a->apply_update && L->quantized) return sync_kernel_weights(L, st);
    return DCLL_OK;
}

}  // namespace dcll
