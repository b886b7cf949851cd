// Multi-timestep inference kernel for the radio_ml_conv stack on a 16x16 I/Q plane (scripts/train_radio_ml.sh geometry):
// layer 0 (1 -> 32 channels) and two 32 -> 32 layers, 7x7 kernels, padding 3, no pooling.
//
// Replaces, for Tc consecutive timesteps in ONE launch, the inner loop of test_radio_ml.py:144-145 /
// networks/__init__.py:182-185 over ContinuousConv2D.forward (dcll/pytorch_libdcll.py:407-426, :485-509).
//
//   * one CTA = one sample; the whole network state of that sample stays ON CHIP for the Tc timesteps:
//     the synaptic traces eps0/eps1 of every layer live in REGISTERS (each thread owns fixed (position, 8-channel
//     group) items across timesteps: 2 layers x 2 items x 8 channels x {eps0,eps1} = 64 registers), the spikes passed
//     from layer to layer live in shared memory as bytes, the membrane accumulators in TMEM;
//   * layers 1 and 2 run on tcgen05 exactly like conv_fwd_tc.cu (split-bf16, implicit im2col by descriptor shifts,
//     [W_hi|W_lo] concatenated along N, 12-stage cp.async.bulk weight ring); layer 0 (K = 49) runs on the FMA pipe;
//   * F16 (DCLL_PREC_F16X2 hidden layers): the operand form of the per-timestep f16x2 forward -- the trace tile is ONE fp16
//     plane set, fp16(eps1 * 2^a_exp), against the fp16 {hi,lo} image of w * 2^w_exp[0]: one kind::f16 MMA with N = 2C per
//     K chunk instead of the two bf16 MMAs, the power-of-two scales undone in the epilogue (conv_mma2_kernel's order);
//   * per timestep only the 8 bytes of the spike cell come in and pv (for the read-outs) goes out.
//
// The local read-outs are NOT inside this kernel on purpose: the frozen read-out matrices are 4*K*F bytes per layer
// (3.1 MB for the three layers + output_ at 16x16) and every element is used once per sample, so a per-sample CTA would
// re-stream them every timestep (18 TB/s of L2 traffic across 148 SMs).  Instead pv of the Tc timesteps is written out
// and readout_fwd_kernel sweeps each read-out matrix ONCE over Tc*B rows (dcll_conv_readout_rows).
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace dcll {

struct StackP {
    const int2 *cells;                 // [Tc][B] (row, col) of the single input spike
    int B, Tc;
    // per layer (0: 1->32, 1/2: 32->32)
    float *e0[3], *e1[3], *arp[3];     // state [B,Cin,16,16] / [B,32,16,16] (arp null when wrp == 0)
    const float *alpha[3], *alphas[3], *tau_m[3], *tau_s[3];
    int coef_mode[3];
    const float *w0t;                  // layer 0 weights [49][32] (weight_t of layer 0)
    const __nv_bfloat16 *w_mma[3];     // layers 1,2: tcgen05 B-operand copies
    const float *bias[3];
    float alpharp[3], wrp[3];
    float *pv[3];                      // [Tc][B][32*256]
    int a_exp[3];                      // F16 form, layers 1,2: the trace image holds fp16(eps1 * 2^a_exp)
    const int *w_exp[3];               // F16 form, layers 1,2: device exponent of the fp16 weight image
};

namespace st16 {
constexpr int NT = 512, HW = 16, NPOS = 256, C = 32, KH = 7, KW = 7, NTAPS = 49;
constexpr int ROWP = HW + KW - 1;                 // 22
constexpr int PLANE = ROWP * ROWP * 16;           // bytes per channel group of the halo tile
constexpr int PART = 4 * PLANE;
constexpr int TAP_BYTES = 2 * 4 * C * 16, NSTAGE = 12;
constexpr int ACC_COLS = 2 * C, TMEM_COLS = 128;  // 2 M-tiles x [hi*hi+lo*hi | hi*lo]  (F16: [A*W_hi | A*W_lo])
template <bool F16>
struct Smem {
    static constexpr int A_BYTES = F16 ? PART : 2 * PART;                      // F16: the fp16 part only
    static constexpr int OFF_RING = A_BYTES;
    static constexpr int OFF_SPK = OFF_RING + NSTAGE * TAP_BYTES;        // 2 x [256 pos][32 ch] bytes
    static constexpr int OFF_L0 = OFF_SPK + 2 * NPOS * C;                // float [22][24] padded eps1 tile of layer 0
    static constexpr int OFF_W0 = OFF_L0 + ROWP * 24 * 4;                // float [49][32]
    static constexpr int OFF_COEF = OFF_W0 + NTAPS * C * 4;              // float [2 hidden layers][4][32]
    static constexpr int OFF_BIAS = OFF_COEF + 2 * 4 * C * 4;            // float [3][32]
    static constexpr int OFF_BAR = OFF_BIAS + 3 * C * 4;
    static constexpr int SMEM = OFF_BAR + 256;
};
}  // namespace st16

template <bool F16>
__global__ void __launch_bounds__(st16::NT, 1) infer_stack16_kernel(const StackP p) {
    pdl_entry();
    using namespace st16;
    using namespace tc;
    using S = Smem<F16>;
    constexpr int A_BYTES = S::A_BYTES, OFF_RING = S::OFF_RING, OFF_SPK = S::OFF_SPK, OFF_L0 = S::OFF_L0, OFF_W0 = S::OFF_W0,
                  OFF_COEF = S::OFF_COEF, OFF_BIAS = S::OFF_BIAS, OFF_BAR = S::OFF_BAR;
    extern __shared__ __align__(128) unsigned char smem[];
    unsigned char *sA = smem, *sW = smem + OFF_RING;
    unsigned char *spk[2] = {smem + OFF_SPK, smem + OFF_SPK + NPOS * C};
    float *l0t = reinterpret_cast<float *>(smem + OFF_L0);
    float *w0s = reinterpret_cast<float *>(smem + OFF_W0);
    float *coef = reinterpret_cast<float *>(smem + OFF_COEF);
    float *bias_s = reinterpret_cast<float *>(smem + OFF_BIAS);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + OFF_BAR);
    uint64_t *full = bars, *empty = bars + NSTAGE, *acc_full = bars + 2 * NSTAGE;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * NSTAGE + 2);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int b = blockIdx.x;
    const int pos = tid & 255, r = pos >> 4, c = pos & 15;
    const int half = tid >> 8;                       // 0/1: which channel groups / channel half this thread owns

    // ---- one-time setup
    for (int i = tid; i < A_BYTES / 16; i += NT) reinterpret_cast<uint4 *>(sA)[i] = make_uint4(0u, 0u, 0u, 0u);   // zero halo border
    for (int i = tid; i < ROWP * 24; i += NT) l0t[i] = 0.f;
    for (int i = tid; i < NTAPS * C; i += NT) w0s[i] = p.w0t[i];
    for (int i = tid; i < 2 * 4 * C; i += NT) {
        const int l = 1 + i / (4 * C), which = (i / C) & 3, ch = i & 31;
        const float *src = which == 0 ? p.tau_s[l] : (which == 1 ? p.alphas[l] : (which == 2 ? p.alpha[l] : p.tau_m[l]));
        coef[i] = src[p.coef_mode[l] == DCLL_COEF_SCALAR ? 0 : ch];
    }
    for (int i = tid; i < 3 * C; i += NT) bias_s[i] = p.bias[i / C][i % C];
    if (tid == 0) {
        for (int s = 0; s < NSTAGE; ++s) mbar_init(full + s, 1), mbar_init(empty + s, 2);   // two MMA issuers commit
        mbar_init(acc_full, 2);
        mbar_fence_init();
    }
    if (warp == 2) tmem_alloc(tmem_slot, TMEM_COLS);
    fence_before();
    __syncthreads();
    fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // ---- thread-owned state: layer 0 (threads 0..255: one position), hidden layers (2 items x 8 channels each)
    const float c0_ts = p.tau_s[0][0], c0_as = p.alphas[0][0], c0_al = p.alpha[0][0], c0_tm = p.tau_m[0][0];
    float s0_e0 = 0.f, s0_e1 = 0.f;
    if (half == 1) s0_e0 = p.e0[0][(size_t)b * NPOS + pos], s0_e1 = p.e1[0][(size_t)b * NPOS + pos];   // owners: warps 8..15
    float he0[2][2][8], he1[2][2][8];
#pragma unroll
    for (int l = 0; l < 2; ++l)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int cg = half + 2 * h;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const size_t o = ((size_t)b * C + cg * 8 + k) * NPOS + pos;
                he0[l][h][k] = p.e0[l + 1][o];
                he1[l][h][k] = p.e1[l + 1][o];
            }
        }

    constexpr uint32_t IDESC_N2 = idesc_bf16(128, 2 * C, false, false), IDESC_N1 = idesc_bf16(128, C, false, false);
    constexpr uint32_t IDESC_F16 = idesc_f16a(128, 2 * C, false, false);
    float unscale[2] = {1.f, 1.f};
    if constexpr (F16) {
#pragma unroll
        for (int l = 0; l < 2; ++l) unscale[l] = pow2i(-(p.a_exp[l + 1] + __ldg(p.w_exp[l + 1])));
    }
    constexpr uint32_t A_HI = desc_hi(ROWP * 16), B_HI = desc_hi(128);
    const uint32_t a_lo_base = desc_lo(smem_u32(sA), PLANE), b_lo_base = desc_lo(smem_u32(sW), 2 * C * 16);
    const uint32_t elected = elect_one();
    uint32_t gtap = 0;      // taps consumed so far (MMA warp / producer lane keep identical copies)
    uint32_t acc_uses = 0;  // completed accumulator hand-overs

    // ---- layer 0 (single input channel, K = 49, FMA pipe), split so that timestep t+1 can run in the shadow of timestep t's MMAs
    auto layer0_trace = [&](int tt) {                 // state owners (warps 8..15, one position each)
        const int2 cell = __ldg(p.cells + (size_t)tt * p.B + b);
        const float xin = (r == cell.x && c == cell.y) ? 1.f : 0.f;
        s0_e0 = __fadd_rn(__fmul_rn(xin, c0_ts), __fmul_rn(c0_as, s0_e0));
        s0_e1 = __fadd_rn(__fmul_rn(c0_al, s0_e1), __fmul_rn(s0_e0, c0_tm));
        l0t[(r + 3) * 24 + c + 3] = s0_e1;
    };
    auto layer0_conv = [&](int tt, int hf) {          // this thread's position x output channels 16*hf .. 16*hf+15
        float acc[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) acc[k] = 0.f;
#pragma unroll 1
        for (int kh = 0; kh < KH; ++kh) {
#pragma unroll
            for (int kw = 0; kw < KW; ++kw) {
                const float xv = l0t[(r + kh) * 24 + c + kw];
                const float4 *w4 = reinterpret_cast<const float4 *>(w0s + (kh * KW + kw) * C + hf * 16);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float4 w = w4[q];
                    acc[4 * q] = fmaf(xv, w.x, acc[4 * q]), acc[4 * q + 1] = fmaf(xv, w.y, acc[4 * q + 1]);
                    acc[4 * q + 2] = fmaf(xv, w.z, acc[4 * q + 2]), acc[4 * q + 3] = fmaf(xv, w.w, acc[4 * q + 3]);
                }
            }
        }
        float *__restrict__ pvout = p.pv[0] + ((size_t)tt * p.B + b) * (C * NPOS);
        float *__restrict__ arp0 = p.arp[0] ? p.arp[0] + ((size_t)b * C + hf * 16) * NPOS + pos : nullptr;
        float av[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) av[k] = arp0 ? arp0[k * NPOS] : 0.f;      // all refractory loads before any store
        __align__(16) unsigned char sb[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            const int co = hf * 16 + k;
            float u = __fadd_rn(acc[k], bias_s[co]);
            float a = 0.f;
            if (arp0) {
                a = __fmul_rn(p.alpharp[0], av[k]);
                u = __fadd_rn(u, a);
            }
            const float sp = u > 0.f ? 1.f : 0.f;
            av[k] = __fsub_rn(a, __fmul_rn(sp, p.wrp[0]));
            sb[k] = (unsigned char)sp;
            pvout[co * NPOS + pos] = sigmoidf_ref(u);
        }
        if (arp0) {
#pragma unroll
            for (int k = 0; k < 16; ++k) arp0[k * NPOS] = av[k];
        }
        *reinterpret_cast<uint4 *>(spk[0] + pos * C + hf * 16) = *reinterpret_cast<const uint4 *>(sb);
    };
    // timestep 0: everybody helps (512 threads = 256 positions x 2 channel halves)
    if (p.Tc > 0) {
        if (half == 1) layer0_trace(0);
        __syncthreads();
        layer0_conv(0, half);
    }

    for (int t = 0; t < p.Tc; ++t) {
        // ================= layers 1, 2: tcgen05 =================
#pragma unroll
        for (int l = 0; l < 2; ++l) {
            const unsigned char *w_src = reinterpret_cast<const unsigned char *>(p.w_mma[l + 1]);
            // weight producer: first stages of this layer-step in flight during the prologue
            if (warp == 1 && lane == 0) {
                for (int i = 0; i < NSTAGE; ++i) {
                    const uint32_t g = gtap + i, s = g % NSTAGE;
                    if (g >= NSTAGE) mbar_wait(empty + s, ((g / NSTAGE) - 1) & 1);
                    mbar_expect_tx(full + s, TAP_BYTES);
                    bulk_g2s(sW + s * TAP_BYTES, w_src + (size_t)i * TAP_BYTES, TAP_BYTES, full + s);
                }
            }
            __syncthreads();   // spikes of the previous layer are complete (and layer 0's tile reads are done)
            // ---- prologue: trace update in registers, bf16 hi/lo split (F16: the scaled fp16 value) into the A tile interior
            const float *cf = coef + l * 4 * C;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int cg = half + 2 * h;
                const uint2 xb = *reinterpret_cast<const uint2 *>(spk[l] + pos * C + cg * 8);
                __align__(16) __nv_bfloat16 hi[8], lo[8];
                __align__(16) __half hf[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const int ch = cg * 8 + k;
                    const float xin = (float)(((k < 4 ? xb.x : xb.y) >> (8 * (k & 3))) & 0xffu);
                    const float n0 = __fadd_rn(__fmul_rn(xin, cf[ch]), __fmul_rn(cf[C + ch], he0[l][h][k]));
                    const float n1 = __fadd_rn(__fmul_rn(cf[2 * C + ch], he1[l][h][k]), __fmul_rn(n0, cf[3 * C + ch]));
                    he0[l][h][k] = n0, he1[l][h][k] = n1;
                    if constexpr (F16) {
                        hf[k] = __float2half_rn(__fmul_rn(n1, pow2i(p.a_exp[l + 1])));
                    } else {
                        hi[k] = __float2bfloat16_rn(n1);
                        lo[k] = __float2bfloat16_rn(n1 - __bfloat162float(hi[k]));
                    }
                }
                unsigned char *dst = sA + cg * PLANE + ((r + 3) * ROWP + c + 3) * 16;
                if constexpr (F16) {
                    *reinterpret_cast<uint4 *>(dst) = *reinterpret_cast<const uint4 *>(hf);
                } else {
                    *reinterpret_cast<uint4 *>(dst) = *reinterpret_cast<const uint4 *>(hi);
                    *reinterpret_cast<uint4 *>(dst + PART) = *reinterpret_cast<const uint4 *>(lo);
                }
            }
            fence_async_smem();
            __syncthreads();
            // ---- MMA issue (warps 0 and 2, one M-tile each: a single issuing thread tops out at ~53 cycles per MMA, the
            //      tensor pipe at ~44) / weight refill (one lane of warp 1)
            if (warp == 0 || warp == 2) {
                const int mt = warp >> 1;
                int kh = 0, kw = 0;
                for (int i = 0; i < NTAPS; ++i) {
                    const uint32_t g = gtap + i, s = g % NSTAGE;
                    mbar_wait(full + s, (g / NSTAGE) & 1);
                    fence_after();
                    if (elected) {
                        const uint32_t b_tap = b_lo_base + ((s * TAP_BYTES) >> 4);
                        {
                            const uint32_t a_tap = a_lo_base + (kh * ROWP + 8 * mt + kw);
                            const uint32_t d = tmem_base + mt * ACC_COLS;
#pragma unroll
                            for (int j = 0; j < 2; ++j) {
                                const uint64_t bd = desc(B_HI, b_tap + ((2 * j * 2 * C * 16) >> 4));
                                if constexpr (F16) {
                                    mma_bf16(d, desc(A_HI, a_tap + ((2 * j * PLANE) >> 4)), bd, IDESC_F16, (i | j) != 0);
                                } else {
                                    mma_bf16(d, desc(A_HI, a_tap + ((2 * j * PLANE) >> 4)), bd, IDESC_N2, (i | j) != 0);
                                    mma_bf16(d, desc(A_HI, a_tap + ((PART + 2 * j * PLANE) >> 4)), bd, IDESC_N1, 1);
                                }
                            }
                        }
                        commit(empty + s);
                        if (i == NTAPS - 1) commit(acc_full);
                    }
                    __syncwarp();
                    if (++kw == KW) kw = 0, ++kh;
                }
            } else if (warp == 1 && lane == 0) {
                for (int i = NSTAGE; i < NTAPS; ++i) {
                    const uint32_t g = gtap + i, s = g % NSTAGE;
                    mbar_wait(empty + s, ((g / NSTAGE) - 1) & 1);
                    mbar_expect_tx(full + s, TAP_BYTES);
                    bulk_g2s(sW + s * TAP_BYTES, w_src + (size_t)i * TAP_BYTES, TAP_BYTES, full + s);
                }
            } else if (l == 1 && half == 1 && t + 1 < p.Tc) {
                // warps 8..15 are idle while layer 2 is multiplied: they run layer 0 of the NEXT timestep now (its spike
                // buffer spk[0] was consumed by layer 1's prologue of this timestep; the __syncthreads at the top of
                // the next layer-1 step publishes it)
                layer0_trace(t + 1);
                asm volatile("bar.sync 1, 256;" ::: "memory");
                layer0_conv(t + 1, 0);
                layer0_conv(t + 1, 1);
            }
            gtap += NTAPS;
            __syncwarp();
            // ---- epilogue: all 16 warps (TMEM lane quarter = warp % 4), thread = one position x 16 channels
            mbar_wait(acc_full, acc_uses & 1);
            ++acc_uses;
            fence_after();
            {
                const int q = warp & 3, mt = (warp >> 2) & 1;
                const int m = q * 32 + lane, er = m >> 3, ec = 8 * mt + (m & 7), epos = er * HW + ec;
                float *__restrict__ pvout = p.pv[l + 1] + ((size_t)t * p.B + b) * (C * NPOS);
                float *__restrict__ arp = p.arp[l + 1] ? p.arp[l + 1] + (size_t)b * C * NPOS + epos : nullptr;
                {
                    const int n0 = 16 * (warp >> 3);
                    float av[16];
#pragma unroll
                    for (int k = 0; k < 16; ++k) av[k] = arp ? arp[(n0 + k) * NPOS] : 0.f;   // loads first, stores last
                    uint32_t v[16], v2[16];
                    ld16(tmem_base + ((uint32_t)(q * 32) << 16) + mt * ACC_COLS + n0, v);
                    ld16(tmem_base + ((uint32_t)(q * 32) << 16) + mt * ACC_COLS + C + n0, v2);
                    __align__(16) unsigned char sb[16];
#pragma unroll
                    for (int k = 0; k < 16; ++k) {
                        const int co = n0 + k;
                        float u = __fadd_rn(__uint_as_float(v[k]), __uint_as_float(v2[k]));
                        if constexpr (F16) u = __fmul_rn(u, unscale[l]);      // undo the power-of-two operand scales (exact)
                        u = __fadd_rn(u, bias_s[(l + 1) * C + co]);
                        float a = 0.f;
                        if (arp) {
                            a = __fmul_rn(p.alpharp[l + 1], av[k]);
                            u = __fadd_rn(u, a);
                        }
                        const float sp = u > 0.f ? 1.f : 0.f;
                        av[k] = __fsub_rn(a, __fmul_rn(sp, p.wrp[l + 1]));
                        sb[k] = (unsigned char)sp;
                        pvout[co * NPOS + epos] = sigmoidf_ref(u);
                    }
                    if (arp) {
#pragma unroll
                        for (int k = 0; k < 16; ++k) arp[(n0 + k) * NPOS] = av[k];
                    }
                    if (l == 0) *reinterpret_cast<uint4 *>(spk[1] + epos * C + n0) = *reinterpret_cast<const uint4 *>(sb);
                }
            }
            fence_before();
        }
        __syncthreads();   // accumulators drained, A tile and spike buffers free for the next timestep
        fence_after();
    }
    // ---- state back to global
    if (half == 1) p.e0[0][(size_t)b * NPOS + pos] = s0_e0, p.e1[0][(size_t)b * NPOS + pos] = s0_e1;
#pragma unroll
    for (int l = 0; l < 2; ++l)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int cg = half + 2 * h;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const size_t o = ((size_t)b * C + cg * 8 + k) * NPOS + pos;
                p.e0[l + 1][o] = he0[l][h][k];
                p.e1[l + 1][o] = he1[l][h][k];
            }
        }
    fence_before();
    __syncthreads();
    if (warp == 2) tmem_dealloc(tmem_base, TMEM_COLS);
}

static int stack16_check(const dcll_conv_layer *Ls, int n_layers, bool *f16) {
    DCLL_REQUIRE(Ls && n_layers == 3, DCLL_EUNSUPPORTED, "dcll_infer_stack16: needs exactly 3 layers");
    for (int l = 0; l < 3; ++l) {
        const dcll_conv_layer &L = Ls[l];
        DCLL_REQUIRE(L.H == 16 && L.W == 16 && L.KH == 7 && L.KW == 7 && L.padH == 3 && L.padW == 3 && L.poolH == 1 && L.poolW == 1 &&
                         L.Cout == 32 && L.Cin == (l == 0 ? 1 : 32) && L.B == Ls[0].B,
                     DCLL_EUNSUPPORTED, "dcll_infer_stack16: layer %d is not a 16x16, 7x7/pad 3, %d->32 channel layer", l, l ? 32 : 1);
        DCLL_REQUIRE(L.coef_mode != DCLL_COEF_ELEMENT, DCLL_EUNSUPPORTED, "dcll_infer_stack16: per-element time constants unsupported");
        DCLL_REQUIRE(L.weight_t && L.bias && L.eps0[L.cur & 1] && L.eps1[L.cur & 1] && (l == 0 || L.weight_mma) && (!(L.wrp > 0.f) || L.arp),
                     DCLL_EINVAL, "dcll_infer_stack16: null tensor in layer %d", l);
    }
    // operand form of the tensor-core layers 1 and 2: fp16 traces (f16x2) or split-bf16; one kernel instantiation runs both
    *f16 = Ls[1].precision == DCLL_PREC_F16X2;
    DCLL_REQUIRE((Ls[2].precision == DCLL_PREC_F16X2) == *f16, DCLL_EUNSUPPORTED,
                 "dcll_infer_stack16: layers 1 and 2 differ in operand form (one f16x2, one split-bf16)");
    for (int l = 1; l < 3 && *f16; ++l) {
        DCLL_REQUIRE(Ls[l].w_exp, DCLL_EINVAL, "dcll_infer_stack16: f16x2 layer %d has no w_exp", l);
        DCLL_REQUIRE(Ls[l].a_exp >= -100 && Ls[l].a_exp <= 100, DCLL_EINVAL, "dcll_infer_stack16: f16x2 layer %d: a_exp out of range", l);
    }
    return DCLL_OK;
}

template <bool F16>
static int launch_stack16(const StackP &p, cudaStream_t st) {
    DCLL_SMEM_ATTR(infer_stack16_kernel<F16>, st16::Smem<F16>::SMEM);
    launch_k(infer_stack16_kernel<F16>, p.B, st16::NT, st16::Smem<F16>::SMEM, st, p);
    DCLL_LAUNCH_OK("infer_stack16_kernel");
    return DCLL_OK;
}

}  // namespace dcll

using namespace dcll;

extern "C" __attribute__((visibility("default"))) int dcll_infer_stack16(const dcll_conv_layer *layers, int n_layers, const int32_t *cells,
                                                                         int Tc, float *const *pv_out, void *stream) {
    bool f16 = false;
    int rc = stack16_check(layers, n_layers, &f16);
    if (rc != DCLL_OK) return rc;
    DCLL_REQUIRE(cells && pv_out && pv_out[0] && pv_out[1] && pv_out[2] && Tc > 0, DCLL_EINVAL, "dcll_infer_stack16: bad arguments");
    StackP p;
    p.cells = reinterpret_cast<const int2 *>(cells);
    p.B = layers[0].B, p.Tc = Tc;
    for (int l = 0; l < 3; ++l) {
        const dcll_conv_layer &L = layers[l];
        const int cur = L.cur & 1;
        p.e0[l] = L.eps0[cur], p.e1[l] = L.eps1[cur], p.arp[l] = L.wrp > 0.f ? L.arp : nullptr;
        p.alpha[l] = L.alpha, p.alphas[l] = L.alphas, p.tau_m[l] = L.tau_m, p.tau_s[l] = L.tau_s, p.coef_mode[l] = L.coef_mode;
        p.w_mma[l] = reinterpret_cast<const __nv_bfloat16 *>(L.weight_mma);
        p.bias[l] = L.bias, p.alpharp[l] = L.alpharp, p.wrp[l] = L.wrp, p.pv[l] = pv_out[l];
        p.a_exp[l] = f16 ? L.a_exp : 0, p.w_exp[l] = f16 ? L.w_exp : nullptr;
    }
    p.w0t = layers[0].weight_t;   // [49][32] since CoutPad == 32
    return f16 ? launch_stack16<true>(p, (cudaStream_t)stream) : launch_stack16<false>(p, (cudaStream_t)stream);
}

// Read-outs of `rows` rows of pv (rows = Tc*B after dcll_infer_stack16): L->B must be set to `rows`, L->pv / pvoutput / output /
// workspace sized accordingly.  clout: int32 [rows].
extern "C" __attribute__((visibility("default"))) int dcll_conv_readout_rows(const dcll_conv_layer *L, int32_t *clout, void *stream) {
    DCLL_REQUIRE(L && L->pv && L->pvoutput && L->wo && L->bo && L->workspace, DCLL_EINVAL, "dcll_conv_readout_rows: null pointer");
    DCLL_REQUIRE(!L->output_layer || (L->wout && L->bout && L->output), DCLL_EINVAL, "dcll_conv_readout_rows: output layer without output_");
    DCLL_REQUIRE(L->workspace_bytes >= ws_layout(L).total, DCLL_EINVAL, "dcll_conv_readout_rows: workspace too small");
    return launch_readout_fwd(L, nullptr, 0, clout, nullptr, (cudaStream_t)stream);
}
