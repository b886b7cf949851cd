// Local read-outs of a Conv2dDCLLlayer and the local-loss gradient.
//
// Replaces (reference, dcll/pytorch_libdcll.py):
//   :602-603  pvoutput = i2o(flatten(pool(pv)))                     -> readout_fwd_kernel (+ finish)
//   :605-606  output   = output_(flatten.detach())  (last layer)    -> same kernel, extra K rows
//   :694-697  SmoothL1Loss(pvoutput, target) [+ (output, target)]   -> readout_finish_kernel (gradient only)
//   :724-728  clout.append(argmax)                                  -> readout_finish_kernel (device side)
//   :704      autograd: d loss / d membrane through i2o, pool, sigmoid -> readout_bwd_kernel
//             d loss / d output_.{weight,bias} + optimizer2.step()  -> readout_bwd_kernel<.,true> (fused)
//
// The read-out is a skinny GEMM [B,F] x [F,Ktot] whose frozen matrix (4*K*F bytes, 50 MB per layer at
// 128x128) must be amortised over the batch, so it is a separate HBM-bound pass over pv rather than an
// epilogue of the convolution: every CTA keeps a 32-wide slice of Wo in shared memory and sweeps it
// over all samples.  Partials are reduced in a fixed order (no float atomics): results are
// deterministic run to run.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace dcll {

constexpr int RO_BM = 64;   // samples per tile
constexpr int RO_BK = 64;   // features per pipeline stage
constexpr int RO_PITCH = RO_BK + 4;   // floats; (pitch/4) odd -> conflict-free float4 reads across rows

__device__ __forceinline__ void ro_cp16(void *smem_dst, const void *gmem_src) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem_src));
}
__device__ __forceinline__ void ro_zero16(void *smem_dst) { *reinterpret_cast<float4 *>(smem_dst) = make_float4(0.f, 0.f, 0.f, 0.f); }

// partial[blk][b][kt] = sum over this CTA's feature tiles of pv[b,f] * Wcat[kt,f],  Wcat = [wo ; wout]
// Two-stage cp.async pipeline: the (64 x 64) pv tile and the (Ktot x 64) read-out tile of stage s+1 stream into shared
// memory while stage s is multiplied; thread = 4 samples x KJ outputs, float4 along the feature axis.
// Requires F % 4 == 0 and 16-byte aligned rows (checked by the launcher; otherwise the scalar-load variant runs).
template <int KJ, bool VEC>
__global__ void __launch_bounds__(256, 3) readout_fwd_kernel(const float *__restrict__ pv, const float *__restrict__ wo,
                                                             const float *__restrict__ wout, int B, int F, int K, int Ktot,
                                                             float *__restrict__ partial) {
    pdl_entry();
    extern __shared__ __align__(16) float ro_smem[];
    constexpr int ROWS = RO_BM + 16 * KJ;                 // pv rows followed by read-out rows
    constexpr int STAGE = ROWS * RO_PITCH;
    const int tid = threadIdx.x;
    const int tb = tid & 15, tk = tid >> 4;
    const int n_ft = (F + RO_BK - 1) / RO_BK;

    auto issue = [&](int stage, int ft, int b0) {
        float *dst = ro_smem + stage * STAGE;
        const int f0 = ft * RO_BK;
        // ROWS x 16 chunks of 16 bytes
        for (int i = tid; i < ROWS * (RO_BK / 4); i += 256) {
            const int row = i / (RO_BK / 4), c4 = i - row * (RO_BK / 4);
            const int f = f0 + c4 * 4;
            float *d = dst + row * RO_PITCH + c4 * 4;
            const float *src = nullptr;
            if (row < RO_BM) {
                const int b = b0 + row;
                if (b < B) src = pv + (size_t)b * F + f;
            } else {
                const int k = row - RO_BM;
                if (k < Ktot) src = (k < K ? wo + (size_t)k * F : wout + (size_t)(k - K) * F) + f;
            }
            if (VEC) {
                if (src && f + 4 <= F) ro_cp16(d, src);
                else {
                    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (src) {
                        if (f < F) v.x = src[0];
                        if (f + 1 < F) v.y = src[1];
                        if (f + 2 < F) v.z = src[2];
                    }
                    *reinterpret_cast<float4 *>(d) = v;
                }
            } else {
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (src) {
                    if (f < F) v.x = __ldg(src);
                    if (f + 1 < F) v.y = __ldg(src + 1);
                    if (f + 2 < F) v.z = __ldg(src + 2);
                    if (f + 3 < F) v.w = __ldg(src + 3);
                }
                *reinterpret_cast<float4 *>(d) = v;
            }
        }
        asm volatile("cp.async.commit_group;\n" ::: "memory");
    };

    // grid.y strides over 64-sample tiles (small F / large B: not enough feature tiles to fill the machine)
    for (int b0 = blockIdx.y * RO_BM; b0 < B; b0 += gridDim.y * RO_BM) {
        float acc[4][KJ];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < KJ; ++j) acc[i][j] = 0.f;
        int ft = blockIdx.x, stage = 0;
        if (ft < n_ft) issue(0, ft, b0);
        for (; ft < n_ft; ft += gridDim.x, stage ^= 1) {
            const int nxt = ft + gridDim.x;
            if (nxt < n_ft) {
                issue(stage ^ 1, nxt, b0);
                asm volatile("cp.async.wait_group 1;\n" ::: "memory");
            } else {
                asm volatile("cp.async.wait_group 0;\n" ::: "memory");
            }
            __syncthreads();
            const float *pvs = ro_smem + stage * STAGE;
            const float *wos = pvs + RO_BM * RO_PITCH;
#pragma unroll 4
            for (int f4 = 0; f4 < RO_BK; f4 += 4) {
                float4 a[4], w[KJ];
#pragma unroll
                for (int i = 0; i < 4; ++i) a[i] = *reinterpret_cast<const float4 *>(pvs + (tb + 16 * i) * RO_PITCH + f4);
#pragma unroll
                for (int j = 0; j < KJ; ++j) w[j] = *reinterpret_cast<const float4 *>(wos + (tk + 16 * j) * RO_PITCH + f4);
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < KJ; ++j) {
                        acc[i][j] = fmaf(a[i].x, w[j].x, acc[i][j]);
                        acc[i][j] = fmaf(a[i].y, w[j].y, acc[i][j]);
                        acc[i][j] = fmaf(a[i].z, w[j].z, acc[i][j]);
                        acc[i][j] = fmaf(a[i].w, w[j].w, acc[i][j]);
                    }
            }
            __syncthreads();   // everyone is done with this stage before it is refilled two iterations later
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            int b = b0 + tb + 16 * i;
#pragma unroll
            for (int j = 0; j < KJ; ++j) {
                int k = tk + 16 * j;
                if (b < B && k < Ktot) partial[((size_t)blockIdx.x * B + b) * Ktot + k] = acc[i][j];
            }
        }
    }
}

// One CTA per sample: fixed-order reduction of the partials, + bias, loss gradient, argmax.
// blockDim.x / 64 slices walk the partial blocks (4 after the FP32 kernel, 16 after the tcgen05 kernel's many blocks).
__global__ void __launch_bounds__(1024) readout_finish_kernel(const float *__restrict__ partial, int n_part, int B, int K,
                                                             int Ktot, const float *__restrict__ bo,
                                                             const float *__restrict__ bout, const float *__restrict__ target,
                                                             int loss_kind, float *__restrict__ pvoutput,
                                                             float *__restrict__ output, float *__restrict__ g_o,
                                                             float *__restrict__ g_o2, int32_t *__restrict__ clout,
                                                             float *__restrict__ loss_out) {
    pdl_entry();
    __shared__ float red[16][64];
    __shared__ float vals[64];
    const int b = blockIdx.x, tid = threadIdx.x;
    const int kk = tid & 63, sl = tid >> 6, n_sl = blockDim.x >> 6;
    float s = 0.f;
    if (kk < Ktot) {
        // FIN_U loads in flight per thread, added in the same fixed order as a serial walk (a rolled loop paid one L2 round trip
        // per partial block: ~8 us per launch, three launches per timestep on the critical path)
        constexpr int FIN_U = 10;
        const float *src = partial + (size_t)b * Ktot + kk;
        const size_t pitch = (size_t)B * Ktot;
        // (unconditional loads -- past the end the slice's last block is read again -- so that they are issued back to back)
        const int c_hi = sl + n_sl * ((n_part - 1 - sl) / n_sl);
        for (int c0 = sl; c0 < n_part; c0 += n_sl * FIN_U) {
            float t[FIN_U];
#pragma unroll
            for (int u = 0; u < FIN_U; ++u) t[u] = src[(size_t)min(c0 + u * n_sl, c_hi) * pitch];
#pragma unroll
            for (int u = 0; u < FIN_U; ++u)
                if (c0 + u * n_sl < n_part) s += t[u];
        }
    }
    red[sl][kk] = s;
    __syncthreads();
    float lsum = 0.f;
    if (tid < Ktot) {
        const bool second = tid >= K;
        const int k = second ? tid - K : tid;
        float v = ((red[0][tid] + red[1][tid]) + red[2][tid]) + red[3][tid];
        for (int q = 4; q < n_sl; ++q) v += red[q][tid];
        v += second ? bout[k] : bo[k];
        vals[tid] = v;
        (second ? output : pvoutput)[(size_t)b * K + k] = v;
        if (target && loss_kind != DCLL_LOSS_CROSS_ENTROPY) {
            const float y = target[(size_t)b * K + k];
            float g = loss_grad_elem(v, y, loss_kind, B * K);
            (second ? g_o2 : g_o)[(size_t)b * K + k] = g;
            lsum = loss_value_elem(v, y, loss_kind) / (float)(B * K);
        }
    }
    __syncthreads();
    if (target && loss_kind == DCLL_LOSS_CROSS_ENTROPY && tid < Ktot) {
        // row-coupled: each head (pvoutput, output) gets its own softmax over the K values now in `vals`
        const bool second = tid >= K;
        const int k = second ? tid - K : tid;
        (second ? g_o2 : g_o)[(size_t)b * K + k] = ce_grad_elem(vals + (second ? K : 0), target + (size_t)b * K, K, k, B, lsum);
    }
    if (tid == 0) {
        // DCLLClassification.forward :725-728 -- argmax of output on the output layer, else of pvoutput;
        // first maximum wins, as torch.argmax does.
        if (clout) {
            const int base = (Ktot > K) ? K : 0;
            int best = 0;
            float bv = vals[base];
            for (int k = 1; k < K; ++k)
                if (vals[base + k] > bv) bv = vals[base + k], best = k;
            clout[b] = best;
        }
    }
    if (loss_out && target) {
        // diagnostic only (train_dcll returns it, ConvNetwork.learn drops it): order-dependent atomics are fine
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) lsum += __shfl_xor_sync(0xffffffffu, lsum, o);
        if ((tid & 31) == 0 && tid < 64 && lsum != 0.f) atomicAdd(loss_out, lsum);
    }
}

// Packed variant of the non-fused sweep above (g_u only): thread = TWO adjacent feature columns, every multiply-add is one
// FFMA2 (fma.rn.f32x2: two independent IEEE FMAs, so each lane-half is bit-identical to the scalar kernel).  The scalar
// kernel is instruction-issue bound (64 instructions per sample-feature, issue slots 67 % busy at 3.4 TB/s); here a
// sample costs 6 broadcast LDS.128 + 24 FFMA2 for two features.  Needs an even F and 8-byte aligned rows.  On the output
// layer it is paired with wout_grad_adam2_kernel (a fused packed sweep needs 179 registers -- one CTA per SM).
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
    unsigned long long ra = *reinterpret_cast<unsigned long long *>(&a), rb = *reinterpret_cast<unsigned long long *>(&b),
                       rc = *reinterpret_cast<unsigned long long *>(&c), rd;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
    return *reinterpret_cast<float2 *>(&rd);
}

__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
    unsigned long long ra = *reinterpret_cast<unsigned long long *>(&a), rb = *reinterpret_cast<unsigned long long *>(&b), rd;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
    return *reinterpret_cast<float2 *>(&rd);
}

// IMG: g_u leaves the kernel as a bf16 {hi,lo} operand image in the same buffer -- sample b occupies the same F*4 bytes,
//     [part 2][co/8][position/8][co % 8][8 positions] bf16,
// i.e. 128-byte core matrices (8 channels x 8 consecutive positions) of the K-major B operand of wgrad_tc2_kernel, which moves
// them with one tensor-map box per unit (full 128-byte lines; the first, plain-NCHW form of the image made every 16-byte piece
// its own half-used L2 sector).  The block -> feature map follows the image: a CTA = 8 channels x 64 consecutive positions.
// q32 = 32-bit address of the bf16 pair in the hi part of the sample; the lo part starts F/2 words later.
// F16X2 (g_scale != 0): fp16 {hi,lo} of g_u * g_scale, saturated to the fp16 range (the scale comes from a bound on |g_u|)
// (packed conversions: one F2FP per pair on the ALU pipe instead of two half-rate F2F and a byte permute)
__device__ __forceinline__ void store_gu_img_f16(uint32_t *q32, int half_f, float2 v, float g_scale) {
    const float x = fminf(fmaxf(__fmul_rn(v.x, g_scale), -65504.f), 65504.f), y = fminf(fmaxf(__fmul_rn(v.y, g_scale), -65504.f), 65504.f);
    const __half2 h = __floats2half2_rn(x, y);                              // low half = x
    const float2 hf = __half22float2(h);
    const __half2 l = __floats2half2_rn(x - hf.x, y - hf.y);
    q32[0] = *reinterpret_cast<const uint32_t *>(&h);
    q32[half_f] = *reinterpret_cast<const uint32_t *>(&l);
}
__device__ __forceinline__ void store_gu_img(uint32_t *q32, int half_f, float2 v) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(v.x, v.y);
    const uint32_t hb = *reinterpret_cast<const uint32_t *>(&h);
    const __nv_bfloat162 l = __floats2bfloat162_rn(v.x - __uint_as_float(hb << 16), v.y - __uint_as_float(hb & 0xffff0000u));
    q32[0] = hb;
    q32[half_f] = *reinterpret_cast<const uint32_t *>(&l);
}

// pv rows reach the thread through a ring of thread-PRIVATE shared-memory slots filled by 8-byte cp.async (LDGSTS): NG groups of
// UB rows, requested NG - 1 groups ahead -- no registers held while the loads fly and no barrier (a thread only ever reads what it
// copied itself).  With the register double buffer of the first packed version a CTA had 16 KB in flight (32 KB per SM): latency-
// bound at ~3.3 TB/s of reads; at B = 64 the whole 32-row slice of a CTA is now requested before the first multiply (64 KB per
// CTA).  The CTAs that share a block of Wo columns (the batch slices) are adjacent in the 1-D grid, so the second read of those
// columns hits L2 instead of DRAM.
constexpr int RB2_NG = 4;
__device__ __forceinline__ void cp_async8(uint32_t dst, const void *src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(src) : "memory");
}
template <int KMAX, int UB, int MINB, bool IMG>
__global__ void __launch_bounds__(256, MINB) readout_bwd2_kernel(const float *__restrict__ pv, const float *__restrict__ wo,
                                                              const float *__restrict__ g_o, int B, int F, int K, int b_per_blk,
                                                              float *__restrict__ g_u, int hw, int slices, float g_scale) {
    extern __shared__ __align__(16) float2 rb2_ring[];                 // [RB2_NG][UB][256]
    const int fblk = blockIdx.x / slices, slice = blockIdx.x - fblk * slices;
    pdl_entry();
    // g rows are read back as broadcast LDS.128 (4 k per load) and enter the FFMA2 as a scalar-broadcast operand: ptxas folds
    // the {g,g} pair into `FFMA2 Rd, Rg.F32, Rw.F32x2, Rs.F32x2`.  (Storing the rows duplicated {g,g} doubled the LDS traffic
    // and made the sweep L1TEX-bound: ncu l1tex throughput 74 %, short-scoreboard stalls above the DRAM ones.)
    __shared__ __align__(16) float gd[64][KMAX];
    static_assert(KMAX % 4 == 0, "float4 rows");
    const int tid = threadIdx.x;
    int f = 2 * (fblk * 256 + tid);
    bool fok = f < F;
    int img_word = 0;                                      // IMG: 32-bit word of this thread's bf16 pair inside one part of the sample
    if (IMG) {
        const int chunks = hw >> 3, blk_per_cog = (chunks + 7) >> 3;          // 8-position chunks per plane, 64-position blocks
        const int cog = fblk / blk_per_cog, pb = fblk - cog * blk_per_cog;
        // warp = one channel of the group, lanes = 64 consecutive positions: the pv / Wo loads stay 256-byte contiguous per warp
        // (with lanes = 8 channels x 8 positions they were 8 scattered sectors: +0.02 ms per launch, measured); the 4-byte image
        // stores of a warp land as 16-byte runs in 8 lines, whose other runs come from the 7 sibling warps of this CTA
        // (round 2: a warp covers TWO adjacent channels x 32 positions instead of one x 64, so that the 4-byte image stores of a
        //  warp fill whole 32-byte sectors -- the 16-byte runs of two adjacent channels are neighbours in the image; measured with
        //  the stores removed they cost 0.023 ms per launch as half sectors, the conversions 0.012)
        const int wq = tid >> 5, ln = tid & 31;
        const int co8 = (wq & 3) * 2 + (ln >> 4), c8 = pb * 8 + (wq >> 2) * 4 + ((ln >> 2) & 3), pr = ln & 3;
        f = (cog * 8 + co8) * hw + c8 * 8 + 2 * pr;
        fok = c8 < chunks && f < F;
        img_word = ((cog * chunks + c8) * 8 + co8) * 4 + pr;
    }
    const int b_begin = slice * b_per_blk, b_end = min(B, b_begin + b_per_blk);
    const uint32_t ring0 = (uint32_t)__cvta_generic_to_shared(rb2_ring) + tid * 8;
    // group g of the rows b0.. : UB rows of this thread's feature pair -> ring stage g % NG
    auto request = [&](int b0, int g) {
        const float *src = pv + (size_t)(b0 + g * UB) * F + f;
        const uint32_t dst = ring0 + (g % RB2_NG) * (UB * 256 * 8);
#pragma unroll
        for (int u = 0; u < UB; ++u, src += F) cp_async8(dst + u * (256 * 8), src);
    };
    // the first groups are requested before anything else, so they fly together with the Wo columns and the g_o rows
    if (fok && b_begin < b_end) {
        const int ng0 = min(64, b_end - b_begin) / UB;
#pragma unroll
        for (int g = 0; g < RB2_NG - 1; ++g) {
            if (g < ng0) request(b_begin, g);
            asm volatile("cp.async.commit_group;" ::: "memory");
        }
    }
    float2 w[KMAX];
#pragma unroll
    for (int k = 0; k < KMAX; ++k) w[k] = (k < K && fok) ? __ldg(reinterpret_cast<const float2 *>(wo + (size_t)k * F + f)) : make_float2(0.f, 0.f);
    for (int b0 = b_begin; b0 < b_end; b0 += 64) {
        const int nb = min(64, b_end - b0);
        __syncthreads();
        for (int i = tid; i < 64 * KMAX; i += 256) {
            int bb = i / KMAX, k = i - bb * KMAX;
            gd[bb][k] = (bb < nb && k < K) ? g_o[(size_t)(b0 + bb) * K + k] : 0.f;
        }
        __syncthreads();
        if (fok) {
            const size_t rowF = (size_t)F;
            const float *pvp = pv + (size_t)b0 * F + f;
            float *gup = g_u + (size_t)b0 * F + f;
            const float2 one2 = make_float2(1.f, 1.f), neg2 = make_float2(-1.f, -1.f);
            auto sample = [&](int bb, float2 p) {
                float2 s = make_float2(0.f, 0.f);
                const float4 *g4 = reinterpret_cast<const float4 *>(gd[bb]);
#pragma unroll
                for (int k = 0; k < KMAX; k += 4) {
                    const float4 g = g4[k >> 2];
                    s = ffma2(make_float2(g.x, g.x), w[k], s);
                    s = ffma2(make_float2(g.y, g.y), w[k + 1], s);
                    s = ffma2(make_float2(g.z, g.z), w[k + 2], s);
                    s = ffma2(make_float2(g.w, g.w), w[k + 3], s);
                }
                // s * (1 - pv) * pv, each lane-half rounded exactly like the scalar expression (1 - pv == fma(pv, -1, 1))
                return fmul2(fmul2(s, ffma2(p, neg2, one2)), p);
            };
            int bb = 0;
            // full groups of UB rows through the cp.async ring (requested RB2_NG - 1 groups ahead; the first ones at kernel entry)
            {
                const int ng = nb / UB;
                if (b0 != b_begin) {
#pragma unroll
                    for (int g = 0; g < RB2_NG - 1; ++g) {
                        if (g < ng) request(b0, g);
                        asm volatile("cp.async.commit_group;" ::: "memory");
                    }
                }
                for (int g = 0; g < ng; ++g, bb += UB) {
                    if (g + RB2_NG - 1 < ng) request(b0, g + RB2_NG - 1);   // its stage was read by this thread one iteration ago
                    asm volatile("cp.async.commit_group;" ::: "memory");
                    asm volatile("cp.async.wait_group %0;" ::"n"(RB2_NG - 1) : "memory");
                    const float2 *stage = rb2_ring + (g % RB2_NG) * (UB * 256) + tid;
                    float2 cur[UB];
#pragma unroll
                    for (int u = 0; u < UB; ++u) cur[u] = stage[u * 256];
                    float *q = gup;
#pragma unroll
                    for (int u = 0; u < UB; ++u, q += rowF) {
                        const float2 v = sample(bb + u, cur[u]);
                        if (IMG && g_scale != 0.f) store_gu_img_f16(reinterpret_cast<uint32_t *>(q - f) + img_word, F >> 1, v, g_scale);
                        else if (IMG) store_gu_img(reinterpret_cast<uint32_t *>(q - f) + img_word, F >> 1, v);
                        else *reinterpret_cast<float2 *>(q) = v;
                    }
                    gup = q;
                }
                asm volatile("cp.async.wait_group 0;" ::: "memory");
                pvp += (size_t)ng * UB * rowF;
            }
            for (; bb < nb; ++bb, pvp += rowF, gup += rowF) {
                const float2 v = sample(bb, __ldg(reinterpret_cast<const float2 *>(pvp)));
                if (IMG && g_scale != 0.f) store_gu_img_f16(reinterpret_cast<uint32_t *>(gup - f) + img_word, F >> 1, v, g_scale);
                else if (IMG) store_gu_img(reinterpret_cast<uint32_t *>(gup - f) + img_word, F >> 1, v);
                else *reinterpret_cast<float2 *>(gup) = v;
            }
        }
    }
}

// The three kernels that reduce the output_ gradient and apply its update (readout_update.cuh) exist twice: with Adam
// (readout_bwd_kernel, wout_grad_adam_kernel, wout_grad_adam2_kernel) and, for the rules of dcll_optim, with OptScalars
// (readout_bwd_opt_kernel, wout_grad_opt_kernel, wout_grad_opt2_kernel).  The file is included once per rule, so the Adam kernels
// are compiled from exactly their own text (a shared __device__ body loses what __launch_bounds__ tells the compiler about
// threadIdx and changes the Adam kernels' machine code).
#define UPD_SCALARS AdamScalars
#define UPD_NAME(adam, opt) adam
#include "readout_update.cuh"
#undef UPD_SCALARS
#undef UPD_NAME
#define UPD_SCALARS OptScalars
#define UPD_NAME(adam, opt) opt
#include "readout_update.cuh"
#undef UPD_SCALARS
#undef UPD_NAME

// g_o / g_o2 from stored read-outs (layer-level API: the target is only known after forward returned).  One thread per
// element; with cross-entropy each thread walks its row (K <= 32, rows stay in L1) exactly as readout_finish_kernel does.
__global__ void loss_grad_kernel(const float *__restrict__ pvoutput, const float *__restrict__ output,
                                 const float *__restrict__ target, int B, int K, int loss_kind, float *__restrict__ g_o,
                                 float *__restrict__ g_o2, float *__restrict__ loss_out) {
    pdl_entry();
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    float lsum = 0.f;
    if (i < B * K && loss_kind == DCLL_LOSS_CROSS_ENTROPY) {
        const int b = i / K, k = i - b * K;
        const float *y = target + (size_t)b * K;
        g_o[i] = ce_grad_elem(pvoutput + (size_t)b * K, y, K, k, B, lsum);
        if (output) g_o2[i] = ce_grad_elem(output + (size_t)b * K, y, K, k, B, lsum);
    } else if (i < B * K) {
        float t = target[i];
        g_o[i] = loss_grad_elem(pvoutput[i], t, loss_kind, B * K);
        lsum = loss_value_elem(pvoutput[i], t, loss_kind) / (float)(B * K);
        if (output) {
            g_o2[i] = loss_grad_elem(output[i], t, loss_kind, B * K);
            lsum += loss_value_elem(output[i], t, loss_kind) / (float)(B * K);
        }
    }
    if (loss_out) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) lsum += __shfl_xor_sync(0xffffffffu, lsum, o);
        if ((threadIdx.x & 31) == 0 && lsum != 0.f) atomicAdd(loss_out, lsum);
    }
}

// generic Adam (or a dcll_optim rule) over a flat parameter (data-parallel path: gradients arrive from the allreduce)
template <class Sc>
__device__ __forceinline__ void flat_body(float *__restrict__ w, const float *__restrict__ g, float *__restrict__ m,
                                          float *__restrict__ v, size_t n, const Sc &sc) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    float wv = w[i], mv = m[i], vv = v[i];
    elem_update(wv, g[i], mv, vv, sc);
    w[i] = wv, m[i] = mv, v[i] = vv;
}
__global__ void adam_flat_kernel(float *__restrict__ w, const float *__restrict__ g, float *__restrict__ m,
                                 float *__restrict__ v, size_t n, AdamScalars sc) {
    pdl_entry();
    flat_body(w, g, m, v, n, sc);
}
__global__ void opt_flat_kernel(float *__restrict__ w, const float *__restrict__ g, float *__restrict__ m,
                                float *__restrict__ v, size_t n, OptScalars sc) {
    pdl_entry();
    flat_body(w, g, m, v, n, sc);
}

int launch_readout_fwd(const dcll_conv_layer *L, const float *target, int loss_kind, int32_t *clout, float *loss_out,
                       cudaStream_t st) {
    Geo g = geo_of(L);
    WsLayout ws = ws_layout(L);
    char *base = (char *)L->workspace;
    float *partial = (float *)(base + ws.off_ro_part);
    float *g_o = (float *)(base + ws.off_go), *g_o2 = (float *)(base + ws.off_go2);
    if (readout_tc_supported(L)) {
        int rc = launch_readout_tc(L, partial, st);
        if (rc != DCLL_OK) return rc;
        launch_k(readout_finish_kernel, L->B, ws.n_ro_tc > 16 ? 1024 : 256, 0, st, partial, ws.n_ro_tc, L->B, L->K, g.Ktot, L->bo, L->bout, target, loss_kind,
                                                      L->pvoutput, L->output, g_o, g_o2, clout, loss_out);
        DCLL_LAUNCH_OK("readout_finish_kernel");
        return DCLL_OK;
    }
    const int kj = ceil_div(g.Ktot, 16);
    DCLL_REQUIRE(kj >= 1 && kj <= 4, DCLL_EUNSUPPORTED, "read-out width %d > 64 unsupported", g.Ktot);
    const bool vec = (g.F % 4 == 0) && (((uintptr_t)L->pv | (uintptr_t)L->wo | (uintptr_t)L->wout) % 16 == 0);
#define RO_CFG(J)                                                                                            \
    DCLL_SMEM_ATTR((readout_fwd_kernel<J, true>), 2 * (RO_BM + 16 * J) * RO_PITCH * sizeof(float));          \
    DCLL_SMEM_ATTR((readout_fwd_kernel<J, false>), 2 * (RO_BM + 16 * J) * RO_PITCH * sizeof(float));
    RO_CFG(1) RO_CFG(2) RO_CFG(3) RO_CFG(4)
#undef RO_CFG
    // batch tiles in grid.y until the grid holds ~4 CTAs per SM
    const int b_tiles = ceil_div(L->B, RO_BM);
    dim3 grid(ws.n_ro, max(1, min(b_tiles, ceil_div(4 * 148, ws.n_ro))));
#define RO_CASE(J)                                                                                                        \
    case J: {                                                                                                             \
        size_t sm = 2 * (RO_BM + 16 * J) * RO_PITCH * sizeof(float);                                                      \
        if (vec) launch_k(readout_fwd_kernel<J, true>, grid, 256, sm, st, L->pv, L->wo, L->wout, L->B, g.F, L->K, g.Ktot, partial); \
        else launch_k(readout_fwd_kernel<J, false>, grid, 256, sm, st, L->pv, L->wo, L->wout, L->B, g.F, L->K, g.Ktot, partial);    \
        break;                                                                                                            \
    }
    switch (kj) { RO_CASE(1) RO_CASE(2) RO_CASE(3) RO_CASE(4) }
#undef RO_CASE
    DCLL_LAUNCH_OK("readout_fwd_kernel");
    launch_k(readout_finish_kernel, L->B, 256, 0, st, partial, ws.n_ro, L->B, L->K, g.Ktot, L->bo, L->bout, target, loss_kind,
                                                 L->pvoutput, L->output, g_o, g_o2, clout, loss_out);
    DCLL_LAUNCH_OK("readout_finish_kernel");
    return DCLL_OK;
}

int launch_loss_grad(const dcll_conv_layer *L, const float *target, int loss_kind, float *loss_out, cudaStream_t st) {
    WsLayout ws = ws_layout(L);
    char *base = (char *)L->workspace;
    float *g_o = (float *)(base + ws.off_go), *g_o2 = (float *)(base + ws.off_go2);
    int n = L->B * L->K;
    launch_k(loss_grad_kernel, ceil_div(n, 256), 256, 0, st, L->pvoutput, L->output_layer ? L->output : nullptr, target, L->B, L->K,
                                                        loss_kind, g_o, g_o2, loss_out);
    DCLL_LAUNCH_OK("loss_grad_kernel");
    return DCLL_OK;
}

int launch_readout_bwd(const dcll_conv_layer *L, dcll_train_args *a, cudaStream_t st, const OptScalars *so) {
    Geo g = geo_of(L);
    WsLayout ws = ws_layout(L);
    char *base = (char *)L->workspace;
    const float *g_o = (const float *)(base + ws.off_go), *g_o2 = (const float *)(base + ws.off_go2);
    DCLL_REQUIRE(L->K <= 32, DCLL_EUNSUPPORTED, "target_size %d > 32 unsupported in the backward read-out", L->K);
    // g_u alone: packed kernel (two features per thread, FFMA2) when rows are 8-byte aligned, else the scalar kernel.
    // Output layer with a large F: ONE scalar sweep over pv serves g_u and gWout (+ Adam); with a small F the output_
    // gradient gets its own kernel below.
    const bool packed = (g.F % 2 == 0) && (((uintptr_t)L->pv | (uintptr_t)L->wo | (uintptr_t)L->g_u) % 8 == 0);
    AdamScalars sc = {};
    const bool big_out = L->output_layer && ceil_div(g.F, 256) >= 2 * 148;
    const bool packed_out = big_out && packed && (!a->apply_update || (a->adam_out.m_w && a->adam_out.v_w)) &&
                            (((uintptr_t)L->wout | (uintptr_t)a->adam_out.m_w | (uintptr_t)a->adam_out.v_w | (uintptr_t)a->grad_wout) % 8 == 0);
    // odd F / unaligned rows: the scalar fused sweep -- never when the weight-gradient kernel expects g_u in image form (then the
    // packed g_u sweep below runs and the output_ gradient takes the generic kernel)
    const bool fused_out = big_out && !packed_out && !wgrad_tc2_supported(L);
    int fblk = ceil_div(g.F, (packed && !fused_out) ? 512 : 256);
    const int hw = g.Hp * g.Wp;
    if (wgrad_tc2_supported(L)) fblk = (L->Cout / 8) * ceil_div(hw / 8, 8);   // image-ordered blocks: 8 channels x 64 positions
    if (packed_out) {
        // large F: packed g_u sweep below + packed output_ gradient/Adam kernel (pv read twice, both at >= 4 waves)
        sc = adam_scalars(a->adam_out, a->adam_out.step + 1);
        dcll_adam &o = a->adam_out;
        const int grid = ceil_div(g.F, 256);
        constexpr int ring_bytes = RB2_NG * 8 * 256 * 8;
#define WG2(KERN, KM, SC)                                                                                                 \
    DCLL_SMEM_ATTR(KERN<KM>, ring_bytes);                                                                                 \
    launch_k(KERN<KM>, grid, 256, ring_bytes, st, L->pv, g_o2, L->B, g.F, L->K, L->wout, L->bout, o.m_w, o.v_w, o.m_b,    \
                                                     o.v_b, a->grad_wout, a->grad_bout, a->apply_update, SC)
        if (so) {
            if (L->K <= 16) { WG2(wout_grad_opt2_kernel, 16, *so); }
            else if (L->K <= 24) { WG2(wout_grad_opt2_kernel, 24, *so); }
            else { WG2(wout_grad_opt2_kernel, 32, *so); }
            DCLL_LAUNCH_OK("wout_grad_opt2_kernel");
        } else {
            if (L->K <= 16) { WG2(wout_grad_adam2_kernel, 16, sc); }
            else if (L->K <= 24) { WG2(wout_grad_adam2_kernel, 24, sc); }
            else { WG2(wout_grad_adam2_kernel, 32, sc); }
            DCLL_LAUNCH_OK("wout_grad_adam2_kernel");
        }
#undef WG2
    } else if (L->output_layer && !fused_out) {
        // small F: the output_ gradient gets its own kernel (batch split over warps inside the CTA)
        sc = adam_scalars(a->adam_out, a->adam_out.step + 1);
        dcll_adam &o = a->adam_out;
        dim3 grid(ceil_div(g.F, 32), ceil_div(L->K, 8));
        if (so) {
            launch_k(wout_grad_opt_kernel<8>, grid, 256, 0, st, L->pv, g_o2, L->B, g.F, L->K, L->wout, L->bout, o.m_w, o.v_w, o.m_b,
                     o.v_b, a->grad_wout, a->grad_bout, a->apply_update, *so);
            DCLL_LAUNCH_OK("wout_grad_opt_kernel");
        } else {
            launch_k(wout_grad_adam_kernel<8>, grid, 256, 0, st, L->pv, g_o2, L->B, g.F, L->K, L->wout, L->bout, o.m_w, o.v_w, o.m_b, o.v_b,
                                                          a->grad_wout, a->grad_bout, a->apply_update, sc);
            DCLL_LAUNCH_OK("wout_grad_adam_kernel");
        }
    }
#define RB_LAUNCH(KM, WO, GRID, BPER, ...) \
    launch_k(readout_bwd_kernel<KM, WO>, GRID, 256, 0, st, L->pv, L->wo, g_o, WO ? g_o2 : nullptr, L->B, g.F, L->K, BPER, L->g_u, __VA_ARGS__)
    if (fused_out) {
        // the output_ gradient reduces over the whole batch inside one thread: no batch slicing
        sc = adam_scalars(a->adam_out, a->adam_out.step + 1);
        dcll_adam &o = a->adam_out;
        dim3 grid(fblk, 1);
#define RB_OPT(KM)                                                                                                               \
    launch_k(readout_bwd_opt_kernel<KM, true>, grid, 256, 0, st, L->pv, L->wo, g_o, g_o2, L->B, g.F, L->K, L->B, L->g_u, L->wout, L->bout, \
             o.m_w, o.v_w, o.m_b, o.v_b, a->grad_wout, a->grad_bout, a->apply_update, *so)
        if (so) {
            if (L->K <= 16) RB_OPT(16);
            else if (L->K <= 24) RB_OPT(24);
            else RB_OPT(32);
        } else if (L->K <= 16)
            RB_LAUNCH(16, true, grid, L->B, L->wout, L->bout, o.m_w, o.v_w, o.m_b, o.v_b, a->grad_wout, a->grad_bout, a->apply_update, sc);
        else if (L->K <= 24)
            RB_LAUNCH(24, true, grid, L->B, L->wout, L->bout, o.m_w, o.v_w, o.m_b, o.v_b, a->grad_wout, a->grad_bout, a->apply_update, sc);
        else
            RB_LAUNCH(32, true, grid, L->B, L->wout, L->bout, o.m_w, o.v_w, o.m_b, o.v_b, a->grad_wout, a->grad_bout, a->apply_update, sc);
#undef RB_OPT
    } else {
        // enough CTAs for >= 4 waves of 3 CTAs per SM (a 2.3-wave grid loses 23 % to the partial last wave): slice the batch
        // (packed kernel, round 2: with the pv rows in the cp.async ring a CTA's fixed cost -- its Wo columns and g_o rows, one DRAM
        //  round trip before the first multiply -- is what more slices multiply; two waves of 2 CTAs per SM are enough.  Measured at
        //  128x128, B = 64: one slice 0.066 / 0.083 ms against 0.074 / 0.089 with two.)
        int slices = max(1, min(ceil_div(L->B, 32), ceil_div((packed ? 2 * 2 : 4 * 3) * 148, fblk)));
        {
            static int sl_env = -1;                                       // DCLL_RB2_SLICES=n: force the number of batch slices (A/B)
            if (sl_env < 0) {
                const char *e = getenv("DCLL_RB2_SLICES");
                sl_env = e ? atoi(e) : 0;
            }
            if (sl_env > 0) slices = sl_env;
        }
        int b_per = ceil_div(ceil_div(L->B, slices), 32) * 32;
        slices = ceil_div(L->B, b_per);
        dim3 grid(fblk, slices);
        float *nf = nullptr;
        if (packed) {
            const unsigned grid1 = (unsigned)fblk * slices;                   // 1-D: the slices of a feature block are adjacent
            constexpr int ring_bytes = RB2_NG * 8 * 256 * 8;
            const float g_scale = prec_f16(L) ? pow2i(L->g_exp) : 0.f;   // F16X2: the image is fp16 {hi,lo} of g_u * 2^g_exp
            // DCLL_RB_TC=1: the K-sum as a skinny tcgen05 GEMM per 128 features (readout_bwd_tc.cu), F16X2 image form only
            if (g_scale != 0.f && wgrad_tc2_supported(L) && readout_bwd_tc_supported(L, hw, g.F))
                return launch_readout_bwd_tc(L, g_o, hw, g.F, g_scale, st);
            // 8 rows in flight per thread, next group prefetched: 128 registers, 2 CTAs per SM (4 rows at 3 CTAs per SM was slower)
            // image form of g_u (bf16 {hi,lo} planes in the same buffer) when the row-pair weight-gradient kernel consumes it
#define RB2_M(KM, MB)                                                                                                              \
    do {                                                                                                                           \
        if (wgrad_tc2_supported(L)) {                                                                                              \
            DCLL_SMEM_ATTR((readout_bwd2_kernel<KM, 8, MB, true>), ring_bytes);                                                    \
            launch_k(readout_bwd2_kernel<KM, 8, MB, true>, grid1, 256, ring_bytes, st, L->pv, L->wo, g_o, L->B, g.F, L->K, b_per, L->g_u, hw, slices, g_scale); \
        } else {                                                                                                                   \
            DCLL_SMEM_ATTR((readout_bwd2_kernel<KM, 8, MB, false>), ring_bytes);                                                   \
            launch_k(readout_bwd2_kernel<KM, 8, MB, false>, grid1, 256, ring_bytes, st, L->pv, L->wo, g_o, L->B, g.F, L->K, b_per, L->g_u, hw, slices, 0.f); \
        }                                                                                                                          \
    } while (0)
            // CTAs per SM: two.  With the rows in the cp.async ring instead of registers three fit for K <= 24 (80 registers, a few
            // bytes of spill) but run SLOWER (measured, 128x128 B = 64: 0.084 / 0.121 ms against 0.075 / 0.102); DCLL_RB2_MINB=3 selects it
            static int minb = -1;
            if (minb < 0) {
                const char *e = getenv("DCLL_RB2_MINB");
                minb = (e && atoi(e) == 3) ? 3 : 2;
            }
#define RB2(KM)                  \
    do {                         \
        if (minb == 3 && KM <= 24) RB2_M(KM, 3); \
        else RB2_M(KM, 2);       \
    } while (0)
            if (L->K <= 16) { RB2(16); }
            else if (L->K <= 24) { RB2(24); }
            else { RB2(32); }
#undef RB2
#undef RB2_M
        } else if (L->K <= 16)
            RB_LAUNCH(16, false, grid, b_per, nf, nf, nf, nf, nf, nf, nf, nf, 0, sc);
        else if (L->K <= 24)
            RB_LAUNCH(24, false, grid, b_per, nf, nf, nf, nf, nf, nf, nf, nf, 0, sc);
        else
            RB_LAUNCH(32, false, grid, b_per, nf, nf, nf, nf, nf, nf, nf, nf, 0, sc);
    }
#undef RB_LAUNCH
    DCLL_LAUNCH_OK("readout_bwd_kernel");
    return DCLL_OK;
}

int launch_adam_flat(float *w, const float *g, float *m, float *v, size_t n, const AdamScalars &sc, cudaStream_t st) {
    launch_k(adam_flat_kernel, (unsigned)((n + 255) / 256), 256, 0, st, w, g, m, v, n, sc);
    DCLL_LAUNCH_OK("adam_flat_kernel");
    return DCLL_OK;
}

int launch_opt_flat(float *w, const float *g, float *m, float *v, size_t n, const OptScalars &sc, cudaStream_t st) {
    launch_k(opt_flat_kernel, (unsigned)((n + 255) / 256), 256, 0, st, w, g, m, v, n, sc);
    DCLL_LAUNCH_OK("opt_flat_kernel");
    return DCLL_OK;
}

}  // namespace dcll
