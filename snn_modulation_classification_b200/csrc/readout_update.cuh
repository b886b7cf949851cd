// Included twice by readout.cu, with UPD_SCALARS = AdamScalars / UPD_NAME(adam, opt) = adam and with OptScalars / opt: the
// kernels that reduce the output_ gradient and apply the update of optimizer2 to it (no include guard, on purpose).

// g_u[b,f] = (sum_k g_o[b,k] Wo[k,f]) * (1 - pv) * pv      (gradient w.r.t. the membrane at the pool argmax)
// Thread = one feature column of Wo held in registers, swept over a slice of the batch (4 samples in flight).
// WOUT variant (output layer, whole batch per CTA): the same sweep also accumulates
//   gWout[k,f] = sum_b g_o2[b,k] pv[b,f]   and applies optimizer2.step() (Adam, lr 1e-4, torch defaults;
//   dcll/pytorch_libdcll.py:636-638,713-714) thread-locally, so pv is read once for both purposes.
template <int KMAX, bool WOUT>
__global__ void __launch_bounds__(256) UPD_NAME(readout_bwd_kernel, readout_bwd_opt_kernel)(const float *__restrict__ pv, const float *__restrict__ wo,
                                                          const float *__restrict__ g_o, const float *__restrict__ g_o2, int B,
                                                          int F, int K, int b_per_blk, float *__restrict__ g_u,
                                                          float *__restrict__ wout, float *__restrict__ bout,
                                                          float *__restrict__ m_w, float *__restrict__ v_w,
                                                          float *__restrict__ m_b, float *__restrict__ v_b,
                                                          float *__restrict__ grad_w, float *__restrict__ grad_b, int apply,
                                                          UPD_SCALARS sc) {
    pdl_entry();
    // rows are read back as float4 (one broadcast LDS.128 per 4 FMAs; scalar LDS made the sweep LDS-issue bound)
    __shared__ __align__(16) float gs[64][KMAX];
    __shared__ __align__(16) float gs2[WOUT ? 64 : 1][KMAX];
    static_assert(KMAX % 4 == 0, "float4 rows");
    const int tid = threadIdx.x;
    const int f = blockIdx.x * 256 + tid;
    const bool fok = f < F;
    float w[KMAX], acc[WOUT ? KMAX : 1];
#pragma unroll
    for (int k = 0; k < KMAX; ++k) w[k] = (k < K && fok) ? __ldg(wo + (size_t)k * F + f) : 0.f;
    if (WOUT) {
#pragma unroll
        for (int k = 0; k < KMAX; ++k) acc[k] = 0.f;
    }
    float bsum = 0.f;
    const int b_begin = blockIdx.y * b_per_blk, b_end = min(B, b_begin + b_per_blk);
    for (int b0 = b_begin; b0 < b_end; b0 += 64) {
        const int nb = min(64, b_end - b0);
        __syncthreads();
        for (int i = tid; i < 64 * KMAX; i += 256) {
            int bb = i / KMAX, k = i - bb * KMAX;
            const bool ok = bb < nb && k < K;
            gs[bb][k] = ok ? g_o[(size_t)(b0 + bb) * K + k] : 0.f;
            if (WOUT) gs2[bb][k] = ok ? g_o2[(size_t)(b0 + bb) * K + k] : 0.f;
        }
        __syncthreads();
        if (fok) {
            constexpr int UB = 8;   // samples in flight per thread (16 was slower: fewer resident CTAs)
            for (int bb = 0; bb < nb; bb += UB) {
                float pvv[UB];
#pragma unroll
                for (int u = 0; u < UB; ++u) pvv[u] = (bb + u < nb) ? __ldg(pv + (size_t)(b0 + bb + u) * F + f) : 0.f;
#pragma unroll
                for (int u = 0; u < UB; ++u) {
                    if (bb + u >= nb) break;
                    float s = 0.f;
                    const float4 *g4 = reinterpret_cast<const float4 *>(gs[bb + u]);
#pragma unroll
                    for (int k = 0; k < KMAX; k += 4) {
                        const float4 g = g4[k >> 2];
                        s = fmaf(g.x, w[k], s), s = fmaf(g.y, w[k + 1], s), s = fmaf(g.z, w[k + 2], s), s = fmaf(g.w, w[k + 3], s);
                    }
                    g_u[(size_t)(b0 + bb + u) * F + f] = s * (1.f - pvv[u]) * pvv[u];
                    if (WOUT) {
                        const float4 *h4 = reinterpret_cast<const float4 *>(gs2[bb + u]);
#pragma unroll
                        for (int k = 0; k < KMAX; k += 4) {
                            const float4 g = h4[k >> 2];
                            acc[k] = fmaf(g.x, pvv[u], acc[k]), acc[k + 1] = fmaf(g.y, pvv[u], acc[k + 1]);
                            acc[k + 2] = fmaf(g.z, pvv[u], acc[k + 2]), acc[k + 3] = fmaf(g.w, pvv[u], acc[k + 3]);
                        }
                    }
                }
            }
        }
        if (WOUT && blockIdx.x == 0 && tid < K)
            for (int bb = 0; bb < nb; ++bb) bsum += gs2[bb][tid];
    }
    if (WOUT) {
        if (fok) {
#pragma unroll
            for (int k = 0; k < KMAX; ++k) {
                if (k < K) {
                    size_t o = (size_t)k * F + f;
                    if (grad_w) grad_w[o] = acc[k];
                    if (apply) {
                        float wv = wout[o], m = m_w[o], v = v_w[o];
                        elem_update(wv, acc[k], m, v, sc);
                        wout[o] = wv, m_w[o] = m, v_w[o] = v;
                    }
                }
            }
        }
        if (blockIdx.x == 0 && tid < K) {
            if (grad_b) grad_b[tid] = bsum;
            if (apply) {
                float wv = bout[tid], m = m_b[tid], v = v_b[tid];
                elem_update(wv, bsum, m, v, sc);
                bout[tid] = wv, m_b[tid] = m, v_b[tid] = v;
            }
        }
    }
}

// output_ gradient + Adam alone, for small feature counts (16x16 planes: F = 8192), where the fused sweep above would
// leave each thread with a serial loop over the whole batch.  CTA = 32 features x 8 batch slices (one warp each, so the
// pv loads are 128-byte coalesced and g_o2 is a warp-broadcast load) x KG outputs (grid.y); fixed-order reduction of the
// 8 slices through shared memory, then Adam.
template <int KG>
__global__ void __launch_bounds__(256) UPD_NAME(wout_grad_adam_kernel, wout_grad_opt_kernel)(const float *__restrict__ pv, const float *__restrict__ g_o2, int B,
                                                             int F, int K, float *__restrict__ wout, float *__restrict__ bout,
                                                             float *__restrict__ m_w, float *__restrict__ v_w,
                                                             float *__restrict__ m_b, float *__restrict__ v_b,
                                                             float *__restrict__ grad_w, float *__restrict__ grad_b, int apply,
                                                             UPD_SCALARS sc) {
    pdl_entry();
    __shared__ float red[8][KG][33];
    __shared__ float bred[8][KG];
    const int fx = threadIdx.x & 31, bs = threadIdx.x >> 5;
    const int f = blockIdx.x * 32 + fx;
    const int k0 = blockIdx.y * KG;
    const bool fok = f < F;
    float acc[KG], bsum[KG];
#pragma unroll
    for (int k = 0; k < KG; ++k) acc[k] = 0.f, bsum[k] = 0.f;
    for (int b = bs; b < B; b += 8 * 4) {
        float pvv[4], g[4][KG];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int bb = b + 8 * u;
            pvv[u] = (bb < B && fok) ? __ldg(pv + (size_t)bb * F + f) : 0.f;
#pragma unroll
            for (int k = 0; k < KG; ++k) g[u][k] = (bb < B && k0 + k < K) ? __ldg(g_o2 + (size_t)bb * K + k0 + k) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int k = 0; k < KG; ++k) acc[k] = fmaf(g[u][k], pvv[u], acc[k]), bsum[k] += g[u][k];
    }
#pragma unroll
    for (int k = 0; k < KG; ++k) red[bs][k][fx] = acc[k];
    if (fx == 0) {
#pragma unroll
        for (int k = 0; k < KG; ++k) bred[bs][k] = bsum[k];
    }
    __syncthreads();
    if (bs == 0 && fok) {
#pragma unroll
        for (int k = 0; k < KG; ++k) {
            if (k0 + k < K) {
                float gsum = 0.f;
#pragma unroll
                for (int s = 0; s < 8; ++s) gsum += red[s][k][fx];
                size_t o = (size_t)(k0 + k) * F + f;
                if (grad_w) grad_w[o] = gsum;
                if (apply) {
                    float wv = wout[o], m = m_w[o], v = v_w[o];
                    elem_update(wv, gsum, m, v, sc);
                    wout[o] = wv, m_w[o] = m, v_w[o] = v;
                }
            }
        }
    }
    if (blockIdx.x == 0 && threadIdx.x < KG && k0 + threadIdx.x < K) {
        const int k = k0 + threadIdx.x;
        float gsum = 0.f;
        for (int s = 0; s < 8; ++s) gsum += bred[s][threadIdx.x];
        if (grad_b) grad_b[k] = gsum;
        if (apply) {
            float wv = bout[k], m = m_b[k], v = v_b[k];
            elem_update(wv, gsum, m, v, sc);
            bout[k] = wv, m_b[k] = m, v_b[k] = v;
        }
    }
}

// output_ gradient + Adam for LARGE feature counts (128x128 planes: F = 524 288), the companion of readout_bwd2_kernel on
// the output layer.  The fused scalar sweep (readout_bwd_kernel<., true>) keeps the whole batch serial in one thread with
// 48 scalar FMAs per sample-feature and a 2.3-wave grid (0.27 ms against a 0.09 ms HBM floor); splitting it into the packed
// g_u sweep plus this kernel re-reads pv once (134 MB, 0.02 ms) but both halves run packed and with >= 4 waves.
// CTA = 128 feature PAIRS x 2 halves of the OUTPUT index k: a thread accumulates gWout[k][f, f+1] for its KMAX/2 outputs over
// the whole batch in order (FFMA2 with the g_o2 value as broadcast operand, rows prefetched one group ahead) and then applies
// Adam to exactly those elements -- no cross-thread reduction.  The two halves read the same pv rows (second read: L1/L2).
// (First version: halves of the BATCH, all KMAX outputs per thread -- 128 registers, 2 CTAs per SM, 0.104 ms.)
template <int KMAX>
__global__ void __launch_bounds__(256, 3) UPD_NAME(wout_grad_adam2_kernel, wout_grad_opt2_kernel)(const float *__restrict__ pv, const float *__restrict__ g_o2, int B,
                                                                 int F, int K, float *__restrict__ wout, float *__restrict__ bout,
                                                                 float *__restrict__ m_w, float *__restrict__ v_w,
                                                                 float *__restrict__ m_b, float *__restrict__ v_b,
                                                                 float *__restrict__ grad_w, float *__restrict__ grad_b, int apply,
                                                                 UPD_SCALARS sc) {
    pdl_entry();
    constexpr int KH = KMAX / 2, UB = 8;
    static_assert(KH % 4 == 0, "float4 rows per half");
    __shared__ __align__(16) float gd[64][KMAX];                  // broadcast LDS.128 rows, see readout_bwd2_kernel
    extern __shared__ __align__(16) float2 rb2_ring[];            // [RB2_NG][UB][256]: thread-private cp.async slots (readout_bwd2_kernel)
    const int tid = threadIdx.x, pair = tid & 127, half = tid >> 7;
    const int f = 2 * (blockIdx.x * 128 + pair);
    const bool fok = f < F;
    const int kbase = half * KH;
    const size_t rowF = (size_t)F;
    const uint32_t ring0 = (uint32_t)__cvta_generic_to_shared(rb2_ring) + tid * 8;
    auto request = [&](int b0, int g) {
        const float *src = pv + (size_t)(b0 + g * UB) * F + f;
        const uint32_t dst = ring0 + (g % RB2_NG) * (UB * 256 * 8);
#pragma unroll
        for (int u = 0; u < UB; ++u, src += F) cp_async8(dst + u * (256 * 8), src);
    };
    if (fok) {
        const int ng0 = min(64, B) / UB;
#pragma unroll
        for (int g = 0; g < RB2_NG - 1; ++g) {
            if (g < ng0) request(0, g);
            asm volatile("cp.async.commit_group;" ::: "memory");
        }
    }
    // the Adam tail reads w, m, v of this thread's outputs in dependent rounds: pull their lines into L2 now, while the batch streams
    // (no measurable effect at 128x128, B = 64 -- 0.102 ms either way -- kept because it is free)
    if (fok && apply) {
#pragma unroll
        for (int k = 0; k < KH; ++k) {
            if (kbase + k < K) {
                const size_t o = (size_t)(kbase + k) * F + f;
                asm volatile("prefetch.global.L2 [%0];" ::"l"(wout + o));
                asm volatile("prefetch.global.L2 [%0];" ::"l"(m_w + o));
                asm volatile("prefetch.global.L2 [%0];" ::"l"(v_w + o));
            }
        }
    }
    // The Adam tail's w, m, v rows travel through the SAME ring as extra groups behind the last pv rows (TG = KH / 2 groups of
    // 2 outputs x {w, m, v}), requested RB2_NG - 1 groups ahead like everything else: their DRAM latency is covered by the last
    // multiplies and by the Adam arithmetic of the groups before them.  (Loading them in dependent rounds after the sweep left
    // every CTA waiting four times: 18 % of the samples on the first use of each round.)
    constexpr int TG = KH / 2;
    static_assert(KH % 2 == 0 && 6 <= UB, "tail groups of two outputs fit a ring group");
    const bool chain_ok = apply && K == KMAX;
    bool chained = false;
    int ng_last = 0;
    auto request_tail = [&](int tg) {
        const uint32_t dst = ring0 + ((ng_last + tg) % RB2_NG) * (UB * 256 * 8);
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const size_t o = (size_t)(kbase + 2 * tg + j) * F + f;
            cp_async8(dst + (3 * j + 0) * (256 * 8), wout + o);
            cp_async8(dst + (3 * j + 1) * (256 * 8), m_w + o);
            cp_async8(dst + (3 * j + 2) * (256 * 8), v_w + o);
        }
    };
    float2 acc[KH];
#pragma unroll
    for (int k = 0; k < KH; ++k) acc[k] = make_float2(0.f, 0.f);
    for (int b0 = 0; b0 < B; b0 += 64) {
        const int nb = min(64, B - b0);
        __syncthreads();
        for (int i = tid; i < 64 * KMAX; i += 256) {
            int bb = i / KMAX, k = i - bb * KMAX;
            gd[bb][k] = (bb < nb && k < K) ? g_o2[(size_t)(b0 + bb) * K + k] : 0.f;
        }
        __syncthreads();
        if (fok) {
            const float *pvp = pv + (size_t)b0 * F + f;
            auto sample = [&](int bb, float2 p) {
                const float4 *g4 = reinterpret_cast<const float4 *>(&gd[bb][kbase]);
#pragma unroll
                for (int k = 0; k < KH; k += 4) {
                    const float4 g = g4[k >> 2];
                    acc[k] = ffma2(make_float2(g.x, g.x), p, acc[k]);
                    acc[k + 1] = ffma2(make_float2(g.y, g.y), p, acc[k + 1]);
                    acc[k + 2] = ffma2(make_float2(g.z, g.z), p, acc[k + 2]);
                    acc[k + 3] = ffma2(make_float2(g.w, g.w), p, acc[k + 3]);
                }
            };
            int bb = 0;
            {
                const int ng = nb / UB;
                const bool chain = chain_ok && b0 + 64 >= B && ng >= RB2_NG - 1;   // last batch block: the tail follows in the ring
                if (chain) chained = true, ng_last = ng;
                if (b0 != 0) {
#pragma unroll
                    for (int g = 0; g < RB2_NG - 1; ++g) {
                        if (g < ng) request(b0, g);
                        asm volatile("cp.async.commit_group;" ::: "memory");
                    }
                }
                for (int g = 0; g < ng; ++g, bb += UB) {
                    if (g + RB2_NG - 1 < ng) request(b0, g + RB2_NG - 1);
                    else if (chain && g + RB2_NG - 1 - ng < TG) request_tail(g + RB2_NG - 1 - ng);
                    asm volatile("cp.async.commit_group;" ::: "memory");
                    asm volatile("cp.async.wait_group %0;" ::"n"(RB2_NG - 1) : "memory");
                    const float2 *stage = rb2_ring + (g % RB2_NG) * (UB * 256) + tid;
                    float2 cur[UB];
#pragma unroll
                    for (int u = 0; u < UB; ++u) cur[u] = stage[u * 256];
#pragma unroll
                    for (int u = 0; u < UB; ++u) sample(bb + u, cur[u]);
                }
                if (!chain) asm volatile("cp.async.wait_group 0;" ::: "memory");
                pvp += (size_t)ng * UB * rowF;
            }
            for (; bb < nb; ++bb, pvp += rowF) sample(bb, __ldg(reinterpret_cast<const float2 *>(pvp)));
        }
    }
    if (fok && chained) {
#pragma unroll
        for (int tg = 0; tg < TG; ++tg) {
            if (tg + RB2_NG - 1 < TG) request_tail(tg + RB2_NG - 1);
            asm volatile("cp.async.commit_group;" ::: "memory");
            asm volatile("cp.async.wait_group %0;" ::"n"(RB2_NG - 1) : "memory");
            const float2 *stage = rb2_ring + ((ng_last + tg) % RB2_NG) * (UB * 256) + tid;
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const size_t o = (size_t)(kbase + 2 * tg + j) * F + f;
                float2 w = stage[(3 * j + 0) * 256], m = stage[(3 * j + 1) * 256], v = stage[(3 * j + 2) * 256];
                const float2 g = acc[2 * tg + j];
                if (grad_w) *reinterpret_cast<float2 *>(grad_w + o) = g;
                elem_update(w.x, g.x, m.x, v.x, sc);
                elem_update(w.y, g.y, m.y, v.y, sc);
                *reinterpret_cast<float2 *>(wout + o) = w;
                *reinterpret_cast<float2 *>(m_w + o) = m;
                *reinterpret_cast<float2 *>(v_w + o) = v;
            }
        }
    } else if (fok) {
        // Adam tail on this thread's own outputs, TB rows at a time with every load issued before the first store
        constexpr int TB = (KH % 3 == 0) ? 3 : 4;
        static_assert(KH % TB == 0, "tail groups");
#pragma unroll
        for (int kk = 0; kk < KH; kk += TB) {
            float2 w[TB], m[TB], v[TB];
#pragma unroll
            for (int j = 0; j < TB; ++j) {
                const size_t o = (size_t)(kbase + kk + j) * F + f;
                if (apply && kbase + kk + j < K) {
                    w[j] = *reinterpret_cast<const float2 *>(wout + o);
                    m[j] = *reinterpret_cast<const float2 *>(m_w + o);
                    v[j] = *reinterpret_cast<const float2 *>(v_w + o);
                }
            }
#pragma unroll
            for (int j = 0; j < TB; ++j) {
                if (kbase + kk + j < K) {
                    const size_t o = (size_t)(kbase + kk + j) * F + f;
                    const float2 g = acc[kk + j];
                    if (grad_w) *reinterpret_cast<float2 *>(grad_w + o) = g;
                    if (apply) {
                        elem_update(w[j].x, g.x, m[j].x, v[j].x, sc);
                        elem_update(w[j].y, g.y, m[j].y, v[j].y, sc);
                        *reinterpret_cast<float2 *>(wout + o) = w[j];
                        *reinterpret_cast<float2 *>(m_w + o) = m[j];
                        *reinterpret_cast<float2 *>(v_w + o) = v[j];
                    }
                }
            }
        }
    }
    if (blockIdx.x == 0 && tid < K) {
        float bsum = 0.f;
        for (int b = 0; b < B; ++b) bsum += g_o2[(size_t)b * K + tid];
        if (grad_b) grad_b[tid] = bsum;
        if (apply) {
            float wv = bout[tid], m = m_b[tid], v = v_b[tid];
            elem_update(wv, bsum, m, v, sc);
            bout[tid] = wv, m_b[tid] = m, v_b[tid] = v;
        }
    }
}
