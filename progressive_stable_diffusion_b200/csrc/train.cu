// Training-step kernels (SURVEY.md 8f row f1; reference: src/models/diffusion_module_ip.py:392-462 training_step, :500-536
// configure_optimizers; Lightning "16-mixed" + gradient_clip_val, src/pipelines/training/training_pipeline_ip.py:103-123).
//   dadd_layernorm_bwd     backward of the 48 LayerNorms (dx, dgamma, dbeta)
//   dadd_geglu_bwd         backward of the GEGLU gate (value * gelu(gate), exact erf form)
//   dadd_groupnorm_bwd     backward of GroupNorm (+ per-(sample, channel) additive term) (+ SiLU), NHWC
//   dadd_minsnr_mse        Min-SNR-weighted MSE loss and its gradient in one pass
//   dadd_sumsq / dadd_clip_coef / dadd_adamw_step   gradient-norm clipping and AdamW over the flat fp32 buckets of the
//                          data-parallel trainer (one launch per bucket, no host synchronisation)
//   dadd_ema_update        EMA weight averaging over the same buckets (the reference's EMAWeightAveraging callback)
// All reductions are two-stage and atomics-free: results are bit-reproducible run to run.  HBM-bound elementwise / row-wise
// work: 16-byte accesses, fp32 arithmetic, grids sized in multiples of the SM count.
#include "common.cuh"

namespace daddk {

// ------------------------------------------------------------------------------------------------ LayerNorm backward
// A warp owns a row at a time (grid-stride over rows); lane l holds vectors l, l + 32, ... of the row (NV of them).  Per row:
//   xhat = (x - mean) * rstd,  g = dy * gamma,  dx = rstd * (g - mean(g) - xhat * mean(g * xhat))
// and dgamma += dy * xhat, dbeta += dy accumulate in registers across the warp's rows; the warps of a CTA are combined in
// shared memory, CTAs through part[cta][2][C] and a second tiny kernel.
template <typename T, int NV>
__global__ void __launch_bounds__(256) ln_bwd_kernel(const T* __restrict__ x, const T* __restrict__ dy, const float* __restrict__ gamma,
                                                     T* __restrict__ dx, float* __restrict__ part, int64_t rows, int C, float eps) {
    extern __shared__ float ln_sm[];                             // [warps][2][C]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int nvec = C >> 3;
    const float inv_c = 1.0f / (float)C;
    float gm[NV][8], dg[NV][8], db[NV][8];
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        const int iv = lane + j * 32;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            gm[j][i] = iv < nvec ? gamma[(iv << 3) + i] : 0.0f;
            dg[j][i] = 0.0f;
            db[j][i] = 0.0f;
        }
    }
    for (int64_t row = (int64_t)blockIdx.x * nw + warp; row < rows; row += (int64_t)gridDim.x * nw) {
        float fx[NV][8], fy[NV][8];
        float s = 0.0f;
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            const int iv = lane + j * 32;
#pragma unroll
            for (int i = 0; i < 8; ++i) fx[j][i] = fy[j][i] = 0.0f;
            if (iv < nvec) {
                Vec8<T> a, b;
                a.load(x + row * C + (iv << 3));
                b.load(dy + row * C + (iv << 3));
                a.unpack(fx[j]);
                b.unpack(fy[j]);
#pragma unroll
                for (int i = 0; i < 8; ++i) s += fx[j][i];
            }
        }
        const float mean = warp_sum(s) * inv_c;
        float q = 0.0f;
#pragma unroll
        for (int j = 0; j < NV; ++j)
            if (lane + j * 32 < nvec) {
#pragma unroll
                for (int i = 0; i < 8; ++i) { const float d = fx[j][i] - mean; q = fmaf(d, d, q); }
            }
        const float rstd = rsqrtf(warp_sum(q) * inv_c + eps);
        float c1 = 0.0f, c2 = 0.0f;
#pragma unroll
        for (int j = 0; j < NV; ++j)
            if (lane + j * 32 < nvec) {
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float xh = (fx[j][i] - mean) * rstd, g = fy[j][i] * gm[j][i];
                    fx[j][i] = xh;
                    c1 += g;
                    c2 = fmaf(g, xh, c2);
                    dg[j][i] = fmaf(fy[j][i], xh, dg[j][i]);
                    db[j][i] += fy[j][i];
                }
            }
        c1 = warp_sum(c1) * inv_c;
        c2 = warp_sum(c2) * inv_c;
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            const int iv = lane + j * 32;
            if (iv < nvec) {
                float o[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) o[i] = rstd * (fy[j][i] * gm[j][i] - c1 - fx[j][i] * c2);
                Vec8<T> t;
                t.pack(o);
                t.store(dx + row * C + (iv << 3));
            }
        }
    }
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        const int iv = lane + j * 32;
        if (iv < nvec) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                ln_sm[(warp * 2 + 0) * C + (iv << 3) + i] = dg[j][i];
                ln_sm[(warp * 2 + 1) * C + (iv << 3) + i] = db[j][i];
            }
        }
    }
    __syncthreads();
    for (int c = threadIdx.x; c < 2 * C; c += blockDim.x) {
        float a = 0.0f;
        for (int w = 0; w < nw; ++w) a += ln_sm[(w * 2 + c / C) * C + c % C];
        part[(size_t)blockIdx.x * 2 * C + c] = a;
    }
}

// out[c] = sum_i part[i][c]  (c < n), one thread per column, fixed order
__global__ void column_sum_kernel(const float* __restrict__ part, float* __restrict__ out, int nparts, int n) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
    float a = 0.0f;
    for (int i = 0; i < nparts; ++i) a += part[(size_t)i * n + c];
    out[c] = a;
}

// ------------------------------------------------------------------------------------------------ GEGLU backward
// proj = [value | gate] (M, 2I); y = value * gelu(gate);  dvalue = dy * gelu(gate),  dgate = dy * value * gelu'(gate)
template <typename T>
__global__ void __launch_bounds__(256) geglu_bwd_kernel(const T* __restrict__ proj, const T* __restrict__ dy, T* __restrict__ dproj,
                                                        int64_t M, int I) {
    const int nv = I >> 3;
    const int64_t total = M * nv;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t row = idx / nv;
        const int col = (int)(idx % nv) << 3;
        Vec8<T> a, g, d;
        a.load(proj + row * 2 * I + col);
        g.load(proj + row * 2 * I + I + col);
        d.load(dy + row * I + col);
        float fa[8], fg[8], fd[8], oa[8], og[8];
        a.unpack(fa);
        g.unpack(fg);
        d.unpack(fd);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float z = fg[i];
            const float cdf = 0.5f * (1.0f + erff(z * 0.70710678118654752f));
            const float pdf = 0.39894228040143268f * __expf(-0.5f * z * z);
            oa[i] = fd[i] * z * cdf;
            og[i] = fd[i] * fa[i] * (cdf + z * pdf);
        }
        a.pack(oa);
        g.pack(og);
        a.store(dproj + row * 2 * I + col);
        g.store(dproj + row * 2 * I + I + col);
    }
}

// ------------------------------------------------------------------------------------------------ GroupNorm backward (NHWC)
// x (B, HW, C) 16-bit, a = chan_add (B, C) fp32 or null: z = ((x + a - mean_g) * rstd_g) * gamma + beta, y = silu(z) or z.
// Three flat passes over grid (chunks, B), thread = fixed 8-channel column x pixel phase, each followed by a tiny finalise:
//   pass 0: per-channel (n, mean, M2) of x + a over the chunk          -> per (b, g) mean, rstd (Chan combination)
//   pass 1: per-channel P1 = sum dz, P2 = sum dz * xhat (dz = dy * act') -> per (b, g) s1 = sum gamma P1, s2 = sum gamma P2;
//                                                                          dgamma[c] = sum_b P2, dbeta[c] = sum_b P1
//   pass 2: dx = rstd * (dz * gamma - (s1 + xhat * s2) / n), and sum_p dx per (b, c) = gradient of the additive term.
constexpr int GNB_THREADS = 256;      // target block size; a block is V x PH threads (V = C / 8 columns, up to 512)

struct GnbPlan {
    int V, PH, npx, chunks;
};
static GnbPlan gnb_plan(int B, int C, int HW) {
    GnbPlan p;
    p.V = C >> 3;
    p.PH = GNB_THREADS / p.V;
    if (p.PH < 1) p.PH = 1;
    p.npx = p.PH * 8;
    if (p.npx > HW) p.npx = HW;
    p.chunks = (HW + p.npx - 1) / p.npx;
    while ((int64_t)p.chunks * B < 2 * num_sms() && p.npx > p.PH) {
        p.npx = p.npx / 2 < p.PH ? p.PH : p.npx / 2;
        p.chunks = (HW + p.npx - 1) / p.npx;
    }
    return p;
}

template <typename T, int MODE>
__global__ void __launch_bounds__(512) gnb_pass_kernel(const T* __restrict__ x, const float* __restrict__ chan_add,
                                                               const T* __restrict__ dy, const float* __restrict__ gamma,
                                                               const float* __restrict__ beta, const float2* __restrict__ stats,
                                                               const float2* __restrict__ gsum, T* __restrict__ dx,
                                                               float* __restrict__ part, int HW, int C, int G, int npx,
                                                               int apply_silu) {
    extern __shared__ float gnb_sm[];                            // [PH][C][2]
    const int V = C >> 3, PH = blockDim.x / V;
    const int tid = threadIdx.x, v = tid % V, ph = tid / V, c0 = v << 3, cpg = C / G;
    const int b = blockIdx.y, chunk = blockIdx.x, chunks = gridDim.x;
    const bool active = tid < V * PH;
    const int p0 = chunk * npx, p1 = min(HW, p0 + npx);
    const T* xb = x + (size_t)b * HW * C + c0;
    float add[8], acc0[8], acc1[8], K[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        add[i] = (chan_add && active) ? chan_add[(size_t)b * C + c0 + i] : 0.0f;
        acc0[i] = acc1[i] = 0.0f;
    }
    float mu[8], rs[8], gm[8], bt[8], s1[8], s2[8];
    if (active) {
        if constexpr (MODE == 0) {
            Vec8<T> t;
            t.load(xb);                                          // shift: the channel's value at pixel 0 of the sample
            t.unpack(K);
#pragma unroll
            for (int i = 0; i < 8; ++i) K[i] += add[i];
        } else {
            const float inv_n = 1.0f / ((float)cpg * (float)HW);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int g = (c0 + i) / cpg;
                const float2 st = stats[(size_t)b * G + g];
                mu[i] = st.x;
                rs[i] = st.y;
                gm[i] = gamma[c0 + i];
                bt[i] = beta[c0 + i];
                if constexpr (MODE == 2) {
                    const float2 gs = gsum[(size_t)b * G + g];
                    s1[i] = gs.x * inv_n;
                    s2[i] = gs.y * inv_n;
                }
            }
        }
        for (int p = p0 + ph; p < p1; p += PH) {
            Vec8<T> tx;
            tx.load(xb + (size_t)p * C);
            float fx[8];
            tx.unpack(fx);
            if constexpr (MODE == 0) {
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float d = fx[i] + add[i] - K[i];
                    acc0[i] += d;
                    acc1[i] = fmaf(d, d, acc1[i]);
                }
            } else {
                Vec8<T> td;
                td.load(dy + ((size_t)b * HW + p) * C + c0);
                float fd[8], o[8];
                td.unpack(fd);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float xh = (fx[i] + add[i] - mu[i]) * rs[i];
                    float dz = fd[i];
                    if (apply_silu) {
                        const float z = fmaf(xh, gm[i], bt[i]);
                        const float sg = __fdividef(1.0f, 1.0f + __expf(-z));
                        dz *= sg * (1.0f + z * (1.0f - sg));
                    }
                    if constexpr (MODE == 1) {
                        acc0[i] += dz;
                        acc1[i] = fmaf(dz, xh, acc1[i]);
                    } else {
                        o[i] = rs[i] * (dz * gm[i] - s1[i] - xh * s2[i]);
                        acc0[i] += o[i];
                    }
                }
                if constexpr (MODE == 2) {
                    Vec8<T> to;
                    to.pack(o);
                    to.store(dx + ((size_t)b * HW + p) * C + c0);
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            gnb_sm[((size_t)ph * C + c0 + i) * 2 + 0] = acc0[i];
            gnb_sm[((size_t)ph * C + c0 + i) * 2 + 1] = acc1[i];
        }
    }
    __syncthreads();
    // combine the pixel phases (fixed order) -> part[b][chunk][c][2] (MODE 0 also needs the count: chunk sizes are implied)
    for (int c = tid; c < C; c += blockDim.x) {
        float a0 = 0.0f, a1 = 0.0f;
        for (int q = 0; q < PH; ++q) {
            a0 += gnb_sm[((size_t)q * C + c) * 2 + 0];
            a1 += gnb_sm[((size_t)q * C + c) * 2 + 1];
        }
        float* o = part + (((size_t)b * chunks + chunk) * C + c) * 2;
        o[0] = a0;
        o[1] = a1;
    }
}

// pass-0 finalise: one warp per (b, g).  Channel c of the group has shifted sums S1 = sum d, S2 = sum d^2 over all chunks with
// d = x + a - K_c: mean_c = K_c + S1 / HW, M2_c = S2 - S1^2 / HW; channels combine with Chan's formula.
template <typename T>
__global__ void gnb_final0_kernel(const float* __restrict__ part, const T* __restrict__ x, const float* __restrict__ chan_add,
                                  float2* __restrict__ stats, int HW, int C, int G, int chunks, float eps) {
    const int b = blockIdx.x / G, g = blockIdx.x % G, cpg = C / G, lane = threadIdx.x;
    float n = 0.0f, mean = 0.0f, m2 = 0.0f;
    for (int j = lane; j < cpg; j += 32) {
        const int c = g * cpg + j;
        float S1 = 0.0f, S2 = 0.0f;
        for (int k = 0; k < chunks; ++k) {
            const float* p = part + (((size_t)b * chunks + k) * C + c) * 2;
            S1 += p[0];
            S2 += p[1];
        }
        const float K = to_f(x[(size_t)b * HW * C + c]) + (chan_add ? chan_add[(size_t)b * C + c] : 0.0f);
        const float nc = (float)HW, mc = K + S1 / nc, qc = fmaxf(S2 - S1 * S1 / nc, 0.0f);
        if (n == 0.0f) { n = nc; mean = mc; m2 = qc; }
        else {
            const float nn = n + nc, d = mc - mean;
            mean += d * (nc / nn);
            m2 += qc + d * d * (n * nc / nn);
            n = nn;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float n2 = __shfl_xor_sync(0xffffffffu, n, o), mean2 = __shfl_xor_sync(0xffffffffu, mean, o),
                    q2 = __shfl_xor_sync(0xffffffffu, m2, o);
        if (n2 > 0.0f) {
            if (n == 0.0f) { n = n2; mean = mean2; m2 = q2; }
            else {
                const float nn = n + n2, d = mean2 - mean;
                mean += d * (n2 / nn);
                m2 += q2 + d * d * (n * n2 / nn);
                n = nn;
            }
        }
    }
    if (lane == 0) stats[(size_t)b * G + g] = make_float2(mean, rsqrtf(m2 / n + eps));
}

// pass-1 finalise: P[b][c] = sum over chunks (kept for the dgamma / dbeta column sums); gsum[b][g] = (sum gamma P1, sum gamma P2)
__global__ void gnb_final1_kernel(const float* __restrict__ part, const float* __restrict__ gamma, float* __restrict__ pbc,
                                  float2* __restrict__ gsum, int C, int G, int chunks) {
    const int b = blockIdx.x / G, g = blockIdx.x % G, cpg = C / G, lane = threadIdx.x;
    float s1 = 0.0f, s2 = 0.0f;
    for (int j = lane; j < cpg; j += 32) {
        const int c = g * cpg + j;
        float P1 = 0.0f, P2 = 0.0f;
        for (int k = 0; k < chunks; ++k) {
            const float* p = part + (((size_t)b * chunks + k) * C + c) * 2;
            P1 += p[0];
            P2 += p[1];
        }
        pbc[((size_t)b * C + c) * 2 + 0] = P1;
        pbc[((size_t)b * C + c) * 2 + 1] = P2;
        s1 = fmaf(gamma[c], P1, s1);
        s2 = fmaf(gamma[c], P2, s2);
    }
    s1 = warp_sum(s1);
    s2 = warp_sum(s2);
    if (lane == 0) gsum[(size_t)b * G + g] = make_float2(s1, s2);
}

// dgamma[c] = sum_b P2[b][c], dbeta[c] = sum_b P1[b][c]
__global__ void gnb_param_kernel(const float* __restrict__ pbc, float* __restrict__ dgamma, float* __restrict__ dbeta, int B, int C) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    float a = 0.0f, d = 0.0f;
    for (int b = 0; b < B; ++b) {
        d += pbc[((size_t)b * C + c) * 2 + 0];
        a += pbc[((size_t)b * C + c) * 2 + 1];
    }
    dgamma[c] = a;
    dbeta[c] = d;
}

// dadd[b][c] = sum over chunks of pass 2's first accumulator
__global__ void gnb_final2_kernel(const float* __restrict__ part, float* __restrict__ dadd, int C, int chunks, int total) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;           // i = b * C + c
    if (i >= total) return;
    const int b = i / C, c = i % C;
    float a = 0.0f;
    for (int k = 0; k < chunks; ++k) a += part[(((size_t)b * chunks + k) * C + c) * 2];
    dadd[i] = a;
}

// ------------------------------------------------------------------------------------------------ Min-SNR MSE loss
// loss = mean_b w_b * mean_e (pred - target)^2 ;  grad = 2 w_b (pred - target) / (B E).  One CTA per (sample, slice).
__global__ void __launch_bounds__(256) minsnr_mse_kernel(const float* __restrict__ pred, const float* __restrict__ target,
                                                         const float* __restrict__ w, float* __restrict__ grad,
                                                         float* __restrict__ part, int E, int B, float upstream) {
    __shared__ float red[8];
    const int b = blockIdx.y;
    const float wb = w[b], gs = 2.0f * wb * upstream / ((float)B * (float)E);
    float a = 0.0f;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < E; e += gridDim.x * blockDim.x) {
        const float d = pred[(size_t)b * E + e] - target[(size_t)b * E + e];
        a = fmaf(d, d, a);
        if (grad) grad[(size_t)b * E + e] = gs * d;
    }
    a = warp_sum(a);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = a;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.0f;
        for (int i = 0; i < 8; ++i) t += red[i];
        part[b * gridDim.x + blockIdx.x] = t * wb / ((float)B * (float)E);
    }
}
__global__ void sum_small_kernel(const float* __restrict__ part, float* __restrict__ out, int n) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        float t = 0.0f;
        for (int i = 0; i < n; ++i) t += part[i];
        out[0] = t;
    }
}

// ------------------------------------------------------------------------------------------------ clipping + AdamW
__global__ void __launch_bounds__(256) sumsq_kernel(const float* __restrict__ g, int64_t n, float* __restrict__ part) {
    __shared__ float red[8];
    // a thread's fp32 chain is folded into a double every 256 float4s: thousands of terms in one fp32 accumulator (few partials
    // for a large buffer) drift low by a few 1e-6; shorter chains (every trainer bucket) give the plain fp32 sum, bit for bit
    float a = 0.0f;
    double folded = 0.0;
    int chain = 0;
    const int64_t n4 = n >> 2;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        const float4 v = reinterpret_cast<const float4*>(g)[i];
        a = fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, fmaf(v.w, v.w, a))));
        if (++chain == 256) {
            folded += (double)a;
            a = 0.0f;
            chain = 0;
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (int64_t i = n4 << 2; i < n; ++i) a = fmaf(g[i], g[i], a);
    a = (float)(folded + (double)a);
    a = warp_sum(a);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = a;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.0f;
        for (int i = 0; i < 8; ++i) t += red[i];
        part[blockIdx.x] = t;
    }
}
// coef = grad_scale * min(1, max_norm / (grad_scale * sqrt(sum part) + 1e-6));  norm_out = grad_scale * sqrt(sum part)
__global__ void clip_coef_kernel(const float* __restrict__ part, int n, float max_norm, float grad_scale, float* __restrict__ out) {
    __shared__ double red[32];
    double a = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) a += (double)part[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = a;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += red[i];
        const float norm = grad_scale * (float)sqrt(t);
        // a non-finite norm (fp16 overflow under a loss scale) poisons the coefficient: dadd_adamw_step then skips the update
        out[0] = !isfinite(norm) ? __int_as_float(0x7fc00000) : (max_norm > 0.0f ? grad_scale * fminf(1.0f, max_norm / (norm + 1e-6f)) : grad_scale);
        out[1] = norm;
    }
}
// torch.optim.AdamW semantics (decoupled decay first, then the moment update); g is scaled by *coef on the fly
// dev_state != nullptr: {learning-rate scale, step number} live on the device (bc1 / bc2 ignored): a captured CUDA graph of the
// whole training step replays with the right bias corrections and schedule without any host-side argument changing
__global__ void __launch_bounds__(256) adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                    float* __restrict__ v, int64_t n, float lr, float b1, float b2, float eps,
                                                    float wd, float bc1, float bc2, const float* __restrict__ coef,
                                                    const float* __restrict__ dev_state) {
    const float c = coef ? coef[0] : 1.0f;
    if (!isfinite(c)) return;                                    // overflowed step: leave parameters and moments untouched
    if (dev_state) {
        lr *= dev_state[0];
        const float t = dev_state[1];
        bc1 = 1.0f - powf(b1, t);
        bc2 = 1.0f - powf(b2, t);
    }
    const float step = lr / bc1, rbc2 = rsqrtf(bc2);
    const int64_t n4 = n >> 2;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        float4 pp = reinterpret_cast<float4*>(p)[i], mm = reinterpret_cast<float4*>(m)[i], vv = reinterpret_cast<float4*>(v)[i];
        const float4 gg = reinterpret_cast<const float4*>(g)[i];
        float* P = &pp.x; float* M = &mm.x; float* V = &vv.x; const float* Gp = &gg.x;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float gk = Gp[k] * c;
            P[k] *= 1.0f - lr * wd;
            M[k] = fmaf(b1, M[k], (1.0f - b1) * gk);
            V[k] = fmaf(b2, V[k], (1.0f - b2) * gk * gk);
            P[k] -= step * M[k] / (sqrtf(V[k]) * rbc2 + eps);
        }
        reinterpret_cast<float4*>(p)[i] = pp;
        reinterpret_cast<float4*>(m)[i] = mm;
        reinterpret_cast<float4*>(v)[i] = vv;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (int64_t i = n4 << 2; i < n; ++i) {
            const float gk = g[i] * c;
            p[i] *= 1.0f - lr * wd;
            m[i] = fmaf(b1, m[i], (1.0f - b1) * gk);
            v[i] = fmaf(b2, v[i], (1.0f - b2) * gk * gk);
            p[i] -= step * m[i] / (sqrtf(v[i]) * rbc2 + eps);
        }
}

}  // namespace daddk

using namespace daddk;

extern "C" int64_t dadd_layernorm_bwd_workspace_bytes(int C) { return (int64_t)2 * num_sms() * 2 * C * sizeof(float); }

extern "C" int dadd_layernorm_bwd(const void* x, const void* dy, const float* gamma, void* dx, float* dgamma, float* dbeta,
                                  float* workspace, int64_t rows, int C, float eps, int dtype, void* stream) {
    DADD_REQUIRE(x && dy && gamma && dx && dgamma && dbeta && workspace, "dadd_layernorm_bwd");
    DADD_REQUIRE(dtype16_ok(dtype) && C % 8 == 0 && C >= 8 && C <= 2048 && rows >= 0, "dadd_layernorm_bwd");
    DADD_REQUIRE(dbeta == dgamma + C, "dadd_layernorm_bwd");         // one (2, C) buffer: the column sums are written as a single row
    cudaStream_t s = (cudaStream_t)stream;
    if (rows == 0) {
        cudaMemsetAsync(dgamma, 0, C * sizeof(float), s);
        cudaMemsetAsync(dbeta, 0, C * sizeof(float), s);
        return 0;
    }
    const int warps = 4;                                             // 4 warps x 2 x C floats of shared memory <= 64 KB
    int64_t want = (rows + warps - 1) / warps;
    const int grid = (int)(want < 2 * num_sms() ? want : 2 * num_sms());
    const size_t smem = (size_t)warps * 2 * C * sizeof(float);
    const int nv = ((C >> 3) + 31) / 32;
#define DADD_LNB(NVV)                                                                                                      \
    DADD_DISPATCH_16(dtype, T, {                                                                                           \
        auto kern = ln_bwd_kernel<T, NVV>;                                                                                 \
        if (smem > 48 * 1024 && cuda_ok(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), \
                                        "dadd_layernorm_bwd smem")) return 2;                                              \
        kern<<<grid, warps * 32, smem, s>>>((const T*)x, (const T*)dy, gamma, (T*)dx, workspace, rows, C, eps);           \
    })
    if (nv <= 2) DADD_LNB(2);
    else if (nv <= 3) DADD_LNB(3);
    else if (nv <= 5) DADD_LNB(5);
    else DADD_LNB(8);
#undef DADD_LNB
    if (int rc = launched("dadd_layernorm_bwd")) return rc;
    column_sum_kernel<<<(2 * C + 255) / 256, 256, 0, s>>>(workspace, dgamma, grid, 2 * C);      // dgamma | dbeta must be adjacent
    return launched("dadd_layernorm_bwd(column sums)");
}

extern "C" int dadd_geglu_bwd(const void* proj, const void* dy, void* dproj, int64_t M, int inner, int dtype, void* stream) {
    DADD_REQUIRE(proj && dy && dproj, "dadd_geglu_bwd");
    DADD_REQUIRE(dtype16_ok(dtype) && inner % 8 == 0 && inner > 0 && M >= 0, "dadd_geglu_bwd");
    if (M == 0) return 0;
    const int64_t total = M * (inner >> 3);
    int64_t blocks = (total + 255) / 256;
    const int grid = (int)(blocks < 8 * (int64_t)num_sms() ? blocks : 8 * (int64_t)num_sms());
    DADD_DISPATCH_16(dtype, T, (geglu_bwd_kernel<T><<<grid, 256, 0, (cudaStream_t)stream>>>((const T*)proj, (const T*)dy, (T*)dproj, M, inner)));
    return launched("dadd_geglu_bwd");
}

extern "C" int64_t dadd_groupnorm_bwd_workspace_bytes(int B, int C, int HW, int G) {
    const GnbPlan p = gnb_plan(B, C, HW);
    return ((int64_t)B * p.chunks * C * 2 + (int64_t)B * C * 2 + (int64_t)B * G * 4) * sizeof(float);
}

extern "C" int dadd_groupnorm_bwd(const void* x, const float* chan_add, const void* dy, const float* gamma, const float* beta,
                                  void* dx, float* dgamma, float* dbeta, float* dchan_add, float* workspace, int B, int HW, int C,
                                  int G, float eps, int apply_silu, int dtype, void* stream) {
    DADD_REQUIRE(x && dy && gamma && beta && dx && dgamma && dbeta && workspace, "dadd_groupnorm_bwd");
    DADD_REQUIRE(dtype16_ok(dtype) && C % 8 == 0 && G > 0 && C % G == 0 && C / 8 <= 512 && B >= 0 && HW > 0, "dadd_groupnorm_bwd");
    DADD_REQUIRE(!dchan_add || chan_add, "dadd_groupnorm_bwd");
    if (B == 0) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    const GnbPlan p = gnb_plan(B, C, HW);
    float* part = workspace;
    float* pbc = part + (size_t)B * p.chunks * C * 2;
    float2* stats = reinterpret_cast<float2*>(pbc + (size_t)B * C * 2);
    float2* gsum = stats + (size_t)B * G;
    const dim3 grid(p.chunks, B);
    const size_t smem = (size_t)p.PH * C * 2 * sizeof(float);
    DADD_DISPATCH_16(dtype, T, {
        auto k0 = gnb_pass_kernel<T, 0>;
        auto k1 = gnb_pass_kernel<T, 1>;
        auto k2 = gnb_pass_kernel<T, 2>;
        if (smem > 48 * 1024) {
            if (cuda_ok(cudaFuncSetAttribute(k0, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "dadd_groupnorm_bwd smem")) return 2;
            if (cuda_ok(cudaFuncSetAttribute(k1, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "dadd_groupnorm_bwd smem")) return 2;
            if (cuda_ok(cudaFuncSetAttribute(k2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "dadd_groupnorm_bwd smem")) return 2;
        }
        k0<<<grid, p.V * p.PH, smem, s>>>((const T*)x, chan_add, nullptr, gamma, beta, nullptr, nullptr, nullptr, part, HW, C, G, p.npx, apply_silu);
        if (int rc = launched("dadd_groupnorm_bwd(stats)")) return rc;
        gnb_final0_kernel<T><<<B * G, 32, 0, s>>>(part, (const T*)x, chan_add, stats, HW, C, G, p.chunks, eps);
        if (int rc = launched("dadd_groupnorm_bwd(stats finalise)")) return rc;
        k1<<<grid, p.V * p.PH, smem, s>>>((const T*)x, chan_add, (const T*)dy, gamma, beta, stats, nullptr, nullptr, part, HW, C, G, p.npx, apply_silu);
        if (int rc = launched("dadd_groupnorm_bwd(sums)")) return rc;
        gnb_final1_kernel<<<B * G, 32, 0, s>>>(part, gamma, pbc, gsum, C, G, p.chunks);
        if (int rc = launched("dadd_groupnorm_bwd(sums finalise)")) return rc;
        gnb_param_kernel<<<(C + 255) / 256, 256, 0, s>>>(pbc, dgamma, dbeta, B, C);
        if (int rc = launched("dadd_groupnorm_bwd(dgamma)")) return rc;
        k2<<<grid, p.V * p.PH, smem, s>>>((const T*)x, chan_add, (const T*)dy, gamma, beta, stats, gsum, (T*)dx, part, HW, C, G, p.npx, apply_silu);
        if (int rc = launched("dadd_groupnorm_bwd(dx)")) return rc;
    });
    if (dchan_add) {
        gnb_final2_kernel<<<(B * C + 255) / 256, 256, 0, s>>>(part, dchan_add, C, p.chunks, B * C);
        return launched("dadd_groupnorm_bwd(dchan_add)");
    }
    return 0;
}

extern "C" int dadd_minsnr_mse(const float* pred, const float* target, const float* weight, float* loss, float* grad,
                               float* workspace, int B, int64_t E, float upstream, void* stream) {
    DADD_REQUIRE(pred && target && weight && loss && workspace && B > 0 && E > 0 && E < (1ll << 31), "dadd_minsnr_mse");
    cudaStream_t s = (cudaStream_t)stream;
    int slices = (int)((E + 256 * 16 - 1) / (256 * 16));
    if (slices > 64) slices = 64;
    minsnr_mse_kernel<<<dim3(slices, B), 256, 0, s>>>(pred, target, weight, grad, workspace, (int)E, B, upstream);
    if (int rc = launched("dadd_minsnr_mse")) return rc;
    sum_small_kernel<<<1, 32, 0, s>>>(workspace, loss, slices * B);
    return launched("dadd_minsnr_mse(sum)");
}
extern "C" int64_t dadd_minsnr_mse_workspace_bytes(int B) { return (int64_t)B * 64 * sizeof(float); }

extern "C" int dadd_sumsq(const float* g, int64_t n, float* partials, int n_partials, void* stream) {
    // (an empty buffer may come without an address: torch hands out NULL for zero elements; its partial sums are zeros)
    DADD_REQUIRE((g || n == 0) && partials && n >= 0 && n_partials > 0 && ((uintptr_t)g % 16) == 0, "dadd_sumsq");
    sumsq_kernel<<<n_partials, 256, 0, (cudaStream_t)stream>>>(g, n, partials);
    return launched("dadd_sumsq");
}

extern "C" int dadd_clip_coef(const float* partials, int n, float max_norm, float grad_scale, float* coef_and_norm, void* stream) {
    DADD_REQUIRE(partials && coef_and_norm && n > 0, "dadd_clip_coef");
    clip_coef_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(partials, n, max_norm, grad_scale, coef_and_norm);
    return launched("dadd_clip_coef");
}

// EMA weight averaging over a flat bucket: avg += (p - avg) * (1 - decay)  (torch.optim.swa_utils.get_ema_avg_fn, the avg_fn of the
// reference's EMAWeightAveraging callback, src/callbacks/ema_callback.py:414-436); first = 1: avg = p (AveragedModel's first update).
// An overflowed step (coef[0] not finite: the parameters were left untouched) still averages, like the callback does.
__global__ void __launch_bounds__(256) ema_kernel(float* __restrict__ avg, const float* __restrict__ p, int64_t n, float omd, int first) {
    const int64_t n4 = n >> 2;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        const float4 pp = reinterpret_cast<const float4*>(p)[i];
        float4 aa = reinterpret_cast<float4*>(avg)[i];
        if (first) {
            aa = pp;
        } else {
            aa.x = fmaf(pp.x - aa.x, omd, aa.x);
            aa.y = fmaf(pp.y - aa.y, omd, aa.y);
            aa.z = fmaf(pp.z - aa.z, omd, aa.z);
            aa.w = fmaf(pp.w - aa.w, omd, aa.w);
        }
        reinterpret_cast<float4*>(avg)[i] = aa;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (int64_t i = n4 << 2; i < n; ++i) avg[i] = first ? p[i] : fmaf(p[i] - avg[i], omd, avg[i]);
}

extern "C" int dadd_ema_update(float* avg, const float* p, int64_t n, float decay, int first, void* stream) {
    DADD_REQUIRE(avg && p && n >= 0, "dadd_ema_update");
    DADD_REQUIRE(decay >= 0.0f && decay <= 1.0f, "dadd_ema_update");
    DADD_REQUIRE((((uintptr_t)avg | (uintptr_t)p) % 16) == 0, "dadd_ema_update");
    if (n == 0) return 0;
    int64_t blocks = ((n >> 2) + 255) / 256;
    if (blocks < 1) blocks = 1;
    const int grid = (int)(blocks < 8 * (int64_t)num_sms() ? blocks : 8 * (int64_t)num_sms());
    ema_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(avg, p, n, (float)(1.0 - (double)decay), first);
    return launched("dadd_ema_update");
}

extern "C" int dadd_adamw_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2, float eps,
                               float weight_decay, float bias_corr1, float bias_corr2, const float* coef, void* stream) {
    DADD_REQUIRE(p && g && m && v && n >= 0, "dadd_adamw_step");
    DADD_REQUIRE((((uintptr_t)p | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v) % 16) == 0, "dadd_adamw_step");
    if (n == 0) return 0;
    int64_t blocks = ((n >> 2) + 255) / 256;
    if (blocks < 1) blocks = 1;
    const int grid = (int)(blocks < 8 * (int64_t)num_sms() ? blocks : 8 * (int64_t)num_sms());
    adamw_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(p, g, m, v, n, lr, beta1, beta2, eps, weight_decay, bias_corr1, bias_corr2, coef, nullptr);
    return launched("dadd_adamw_step");
}

extern "C" int dadd_adamw_step_dev(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2, float eps,
                                   float weight_decay, const float* dev_state, const float* coef, void* stream) {
    DADD_REQUIRE(p && g && m && v && dev_state && n >= 0, "dadd_adamw_step_dev");
    DADD_REQUIRE((((uintptr_t)p | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v) % 16) == 0, "dadd_adamw_step_dev");
    if (n == 0) return 0;
    int64_t blocks = ((n >> 2) + 255) / 256;
    if (blocks < 1) blocks = 1;
    const int grid = (int)(blocks < 8 * (int64_t)num_sms() ? blocks : 8 * (int64_t)num_sms());
    adamw_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(p, g, m, v, n, lr, beta1, beta2, eps, weight_decay, 1.0f, 1.0f, coef, dev_state);
    return launched("dadd_adamw_step_dev");
}

// ------------------------------------------------------------------------------------------------ cross-attention backward
// Backward of the triple-pathway core (dadd_cross_attn_fwd; attention_processor_routing_gates.py:148-178): per (sample, head)
//   o_i = sum_s g_s sum_{j in seg s} p_ij v_j,   p = per-segment softmax(q_i . k_j * scale)
//   dp_ij = g_s (do_i . v_j),  ds_ij = p_ij (dp_ij - sum_{j' in seg} p_ij' dp_ij'),
//   dq_i = scale sum_j ds_ij k_j,  dk_j = scale sum_i ds_ij q_i,  dv_j = sum_i g_s p_ij do_i.
// L <= 48 condition tokens: 480 d flop per query row - 0.3 % of the training step - so this runs on the CUDA cores in fp32.
// CTA = one (sample, head) x one slice of query rows, walking 32-row tiles: K, V and the tile of Q / dO sit in shared memory
// (pitch d + 1), dK / dV accumulate in registers across the tiles (fixed order), the slices' partials are summed by a second
// kernel: no atomics, bit-reproducible.
namespace daddk {
constexpr int XB_ROWS = 32, XB_THREADS = 256, XB_MAXOUT = 30;      // 48 * 160 / 256 outputs per thread at most

template <typename T>
__global__ void __launch_bounds__(XB_THREADS) cross_attn_bwd_kernel(const T* __restrict__ q, int64_t q_stride, const T* __restrict__ kc,
                                                                    const T* __restrict__ vc, const float* __restrict__ gates,
                                                                    const T* __restrict__ dout, int64_t do_stride, T* __restrict__ dq,
                                                                    int64_t dq_stride, float* __restrict__ dk_part, float* __restrict__ dv_part,
                                                                    int H, int N, int d, int L, int seg_len, float scale, int rows_per_split) {
    extern __shared__ float xb_sm[];
    const int dp = d + 1, lp = L + 1;
    float* sK = xb_sm;                      // [L][dp]
    float* sV = sK + L * dp;                // [L][dp]
    float* sQ = sV + L * dp;                // [32][dp]
    float* sD = sQ + XB_ROWS * dp;          // [32][dp]   dO tile
    float* sS = sD + XB_ROWS * dp;          // [32][lp]   scores -> scale * dS
    float* sP = sS + XB_ROWS * lp;          // [32][lp]   dP -> gate * P
    const int tid = threadIdx.x, bh = blockIdx.x, b = bh / H, h = bh % H, split = blockIdx.y, splits = gridDim.y;
    const int nseg = L / seg_len;
    const int row0 = split * rows_per_split, row1 = min(N, row0 + rows_per_split);
    const T* kb = kc + (size_t)bh * L * d;
    const T* vb = vc + (size_t)bh * L * d;
    for (int i = tid; i < L * d; i += XB_THREADS) {
        sK[(i / d) * dp + i % d] = to_f(kb[i]);
        sV[(i / d) * dp + i % d] = to_f(vb[i]);
    }
    float dka[XB_MAXOUT], dva[XB_MAXOUT];
#pragma unroll
    for (int i = 0; i < XB_MAXOUT; ++i) dka[i] = dva[i] = 0.0f;
    for (int r0 = row0; r0 < row1; r0 += XB_ROWS) {
        __syncthreads();                                            // previous tile fully consumed (and K / V loaded)
        for (int i = tid; i < XB_ROWS * d; i += XB_THREADS) {
            const int r = i / d, c = i % d, row = r0 + r;
            const bool live = row < row1;
            sQ[r * dp + c] = live ? to_f(q[((size_t)b * N + row) * q_stride + h * d + c]) : 0.0f;
            sD[r * dp + c] = live ? to_f(dout[((size_t)b * N + row) * do_stride + h * d + c]) : 0.0f;
        }
        __syncthreads();
        for (int i = tid; i < XB_ROWS * L; i += XB_THREADS) {
            const int r = i / L, j = i % L;
            float s = 0.0f, g = 0.0f;
            for (int c = 0; c < d; ++c) {
                s = fmaf(sQ[r * dp + c], sK[j * dp + c], s);
                g = fmaf(sD[r * dp + c], sV[j * dp + c], g);
            }
            sS[r * lp + j] = s * scale;
            sP[r * lp + j] = g * gates[j / seg_len];
        }
        __syncthreads();
        for (int i = tid; i < XB_ROWS * nseg; i += XB_THREADS) {
            const int r = i / nseg, sg = i % nseg;
            float* s = sS + r * lp + sg * seg_len;
            float* p = sP + r * lp + sg * seg_len;
            const float gate = gates[sg];
            float m = -INFINITY;
            for (int j = 0; j < seg_len; ++j) m = fmaxf(m, s[j]);
            float sum = 0.0f;
            for (int j = 0; j < seg_len; ++j) { s[j] = __expf(s[j] - m); sum += s[j]; }
            const float inv = 1.0f / sum;
            float dot = 0.0f;
            for (int j = 0; j < seg_len; ++j) { s[j] *= inv; dot = fmaf(s[j], p[j], dot); }
            for (int j = 0; j < seg_len; ++j) {
                const float pj = s[j];
                s[j] = scale * pj * (p[j] - dot);                  // scale * dS
                p[j] = gate * pj;                                   // gate * P
            }
        }
        __syncthreads();
        for (int i = tid; i < XB_ROWS * d; i += XB_THREADS) {
            const int r = i / d, c = i % d, row = r0 + r;
            if (row < row1) {
                float a = 0.0f;
                for (int j = 0; j < L; ++j) a = fmaf(sS[r * lp + j], sK[j * dp + c], a);
                if constexpr (std::is_same_v<T, __nv_bfloat16>) dq[((size_t)b * N + row) * dq_stride + h * d + c] = __float2bfloat16(a);
                else dq[((size_t)b * N + row) * dq_stride + h * d + c] = __float2half(a);
            }
        }
#pragma unroll
        for (int i = 0; i < XB_MAXOUT; ++i) {
            const int o = tid + i * XB_THREADS;
            if (o < L * d) {
                const int j = o / d, c = o % d;
                float a = dka[i], v = dva[i];
#pragma unroll 8
                for (int r = 0; r < XB_ROWS; ++r) {
                    a = fmaf(sS[r * lp + j], sQ[r * dp + c], a);
                    v = fmaf(sP[r * lp + j], sD[r * dp + c], v);
                }
                dka[i] = a;
                dva[i] = v;
            }
        }
    }
#pragma unroll
    for (int i = 0; i < XB_MAXOUT; ++i) {
        const int o = tid + i * XB_THREADS;
        if (o < L * d) {
            dk_part[((size_t)bh * splits + split) * L * d + o] = dka[i];
            dv_part[((size_t)bh * splits + split) * L * d + o] = dva[i];
        }
    }
}

// out[bh][o] = sum_split part[bh][split][o], both tensors in one launch (blockIdx.y selects dK / dV)
__global__ void cross_attn_bwd_reduce_kernel(const float* __restrict__ dk_part, const float* __restrict__ dv_part, float* __restrict__ dk,
                                             float* __restrict__ dv, int64_t total, int per, int splits) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const float* part = blockIdx.y ? dv_part : dk_part;
    const int64_t bh = i / per, o = i % per;
    float a = 0.0f;
    for (int s = 0; s < splits; ++s) a += part[(bh * splits + s) * per + o];
    (blockIdx.y ? dv : dk)[i] = a;
}
}  // namespace daddk

static int xb_splits(int BH, int N) {
    int s = (2 * num_sms() + BH - 1) / BH;
    const int max_s = (N + 2 * XB_ROWS - 1) / (2 * XB_ROWS);
    if (s > max_s) s = max_s;
    return s < 1 ? 1 : s;
}

extern "C" int64_t dadd_cross_attn_bwd_workspace_bytes(int B, int H, int N, int d, int L) {
    return (int64_t)2 * B * H * xb_splits(B * H, N) * L * d * sizeof(float);
}

extern "C" int dadd_cross_attn_bwd(const void* q, int64_t q_stride, const void* k_cat, const void* v_cat, const float* gates,
                                   const void* dout, int64_t do_stride, void* dq, int64_t dq_stride, float* dk, float* dv,
                                   float* workspace, int B, int H, int N, int d, int L, int seg_len, float scale, int dtype, void* stream) {
    DADD_REQUIRE(q && k_cat && v_cat && gates && dout && dq && dk && dv && workspace, "dadd_cross_attn_bwd");
    DADD_REQUIRE(dtype16_ok(dtype) && B >= 0 && H > 0 && N >= 0 && d > 0 && d <= 160, "dadd_cross_attn_bwd");
    DADD_REQUIRE(seg_len > 0 && L % seg_len == 0 && L > 0 && L <= 48, "dadd_cross_attn_bwd");
    DADD_REQUIRE(q_stride >= (int64_t)H * d && do_stride >= (int64_t)H * d && dq_stride >= (int64_t)H * d, "dadd_cross_attn_bwd");
    if (B == 0 || N == 0) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    const int BH = B * H, splits = xb_splits(BH, N);
    int rows = (N + splits - 1) / splits;
    rows = (rows + XB_ROWS - 1) / XB_ROWS * XB_ROWS;
    const size_t smem = ((size_t)2 * L * (d + 1) + 2 * XB_ROWS * (d + 1) + 2 * XB_ROWS * (L + 1)) * sizeof(float);
    float* dk_part = workspace;
    float* dv_part = workspace + (size_t)BH * splits * L * d;
    DADD_DISPATCH_16(dtype, T, {
        auto kern = cross_attn_bwd_kernel<T>;
        if (smem > 48 * 1024 && cuda_ok(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "dadd_cross_attn_bwd smem")) return 2;
        kern<<<dim3(BH, splits), XB_THREADS, smem, s>>>((const T*)q, q_stride, (const T*)k_cat, (const T*)v_cat, gates, (const T*)dout, do_stride,
                                                        (T*)dq, dq_stride, dk_part, dv_part, H, N, d, L, seg_len, scale, rows);
    });
    if (int rc = launched("dadd_cross_attn_bwd")) return rc;
    const int64_t total = (int64_t)BH * L * d;
    cross_attn_bwd_reduce_kernel<<<dim3((unsigned)((total + 255) / 256), 2), 256, 0, s>>>(dk_part, dv_part, dk, dv, total, L * d, splits);
    return launched("dadd_cross_attn_bwd(reduce)");
}
