// Pairwise squared-distance statistics of two fp32 feature sets without the distance matrix: the CMMD, improved precision /
// recall, density / coverage and realism metrics of the evaluation sweep (reference: src/pipelines/evaluation/
// evaluation_pipeline.py:577-839, 978-1179, which materialise cdist matrices in torch).
//   d2[i][j] = max(|x_i|^2 + |y_j|^2 - 2 x_i . y_j, 0)       X: [M][D], Y: [N][D], row-major fp32
// One persistent tcgen05 GEMM computes 128 x 256 tiles of X Y^T into TMEM; the epilogue turns each tile into d2 and folds
// it into per-(row, column slice) state, so no distance ever reaches global memory:
//   RBF_SUM  sum_ij exp(-gamma d2)         per-row sums in double, one partial per (row block, slice), summed in fixed order
//   KNN      k-th smallest d2 of each row  per-slice sorted top-k lists, merged by a second pass (same_set: j == i excluded)
//   COUNT    #{j : d2[i][j] <= r[j]}       per-slice int32 counts, summed; COVER is the same count, finished as count > 0
//   RATIO_MAX max_j r[j] / (d2[i][j] + eps) per-slice maxima (IEEE division, running max from 0), max-merged
// COVER, COUNT and RATIO_MAX share one kernel instance (the radius instance): Args::mode picks the reduction once per tile.
// Precision: fp32-faithful via error-compensated TF32.  A pre-pass splits every row into hi = tf32(x) (round to nearest) and
// lo = x - hi (exact in fp32) and computes |x|^2 in double; the MMA accumulates lo_x.hi_y + hi_x.lo_y + hi_x.hi_y (kind::tf32,
// fp32 in TMEM).  What is dropped is lo_x.lo_y (<= 2^-22 |x||y|) and the tf32 truncation of lo (<= 2^-21 |x||y| per term).
// Layout: warps 0-3 epilogue (TMEM lane == row), warp 4 TMA producer, warp 5 MMA issuer.  A stage holds one 32-column
// K-block of {X_hi, X_lo} (128 rows) and {Y_hi, Y_lo} (256 rows), 128-byte swizzle, zero-filled edges; two accumulators of
// 256 TMEM columns let tile t + 1 be multiplied while tile t drains.  Every item (row block, column slice) is computed by one
// CTA in a fixed order, so results are bit-reproducible and independent of the grid.
#include "tc_util.cuh"

namespace daddk {
namespace pw {

using namespace daddk::tc;

constexpr int NTHREADS = 192;
constexpr int TBM = 128, TBN = 256, BK = 32, STAGES = 2, KMAX = 16;
constexpr uint32_t A_BYTES = TBM * BK * 4, B_BYTES = TBN * BK * 4;
constexpr uint32_t STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;
constexpr int ITEM_TARGET = 4 * 148;          // slices are chosen from the shape alone (not the device) so results do not depend on it

struct Bars {
    uint64_t full[STAGES], empty[STAGES];
    uint64_t acc_full[2], acc_empty[2];
    uint32_t tmem_base;
};

struct Plan {
    int64_t nrb, nct, tps, S, items;
    int64_t off_xhi, off_xlo, off_yhi, off_ylo, off_nx, off_ny, off_part, total;
};

static int64_t up256(int64_t b) { return (b + 255) & ~int64_t(255); }

static Plan make_plan(int64_t M, int64_t N, int D, int mode, int k, int same_set) {
    Plan p{};
    p.nrb = (M + TBM - 1) / TBM;
    p.nct = (N + TBN - 1) / TBN;
    int64_t S = (ITEM_TARGET + p.nrb - 1) / p.nrb;
    if (S > p.nct) S = p.nct;
    if (S < 1) S = 1;
    p.tps = (p.nct + S - 1) / S;
    p.S = (p.nct + p.tps - 1) / p.tps;          // no empty slice
    p.items = p.nrb * p.S;
    const int64_t xb = up256(M * D * 4), yb = same_set ? 0 : up256(N * D * 4);
    int64_t o = 0;
    p.off_xhi = o; o += xb;
    p.off_xlo = o; o += xb;
    p.off_yhi = same_set ? p.off_xhi : o; o += yb;
    p.off_ylo = same_set ? p.off_xlo : o; o += yb;
    p.off_nx = o; o += up256(M * 4);
    p.off_ny = same_set ? p.off_nx : o; o += same_set ? 0 : up256(N * 4);
    p.off_part = o;
    if (mode == DADD_PAIRWISE_RBF_SUM) o += up256(p.items * 8);
    else if (mode == DADD_PAIRWISE_KNN) o += up256(M * p.S * k * 4);
    else o += up256(M * p.S * 4);                 // radius modes: one int32 count or float max per (row, slice)
    p.total = o;
    return p;
}

__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ uint64_t desc_add(uint64_t desc, uint32_t bytes) { return desc + (uint64_t)(bytes >> 4); }
__device__ __forceinline__ void named_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
                 : "memory");
}

// Sorted (ascending) top-k insert over a register array; k <= KMAX is a runtime bound, so every index stays static.
__device__ __forceinline__ void topk_insert(float (&best)[KMAX], float v, int k) {
#pragma unroll
    for (int q = 0; q < KMAX; ++q) {
        if (q < k) {
            const float lo = fminf(best[q], v);
            v = fmaxf(best[q], v);
            best[q] = lo;
        }
    }
}
__device__ __forceinline__ float topk_last(const float (&best)[KMAX], int k) {
    float r = best[0];
#pragma unroll
    for (int q = 1; q < KMAX; ++q)
        if (q == k - 1) r = best[q];
    return r;
}

// hi = tf32(x) (round to nearest), lo = x - hi, sq = |x|^2 (double sum, rounded once).  One warp per row.
__global__ void __launch_bounds__(256) split_kernel(const float* __restrict__ x, float* __restrict__ hi, float* __restrict__ lo,
                                                     float* __restrict__ sq, int64_t rows, int D) {
    const int64_t r = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (r >= rows) return;
    const float4* src = reinterpret_cast<const float4*>(x + r * D);
    float4* h4 = reinterpret_cast<float4*>(hi + r * D);
    float4* l4 = reinterpret_cast<float4*>(lo + r * D);
    double s = 0.0;
    for (int c = lane; c < D / 4; c += 32) {
        const float4 v = src[c];
        float e[4] = {v.x, v.y, v.z, v.w}, h[4], l[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            uint32_t t;
            asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t) : "f"(e[q]));
            h[q] = __uint_as_float(t);
            l[q] = e[q] - h[q];
            s += (double)e[q] * (double)e[q];
        }
        h4[c] = make_float4(h[0], h[1], h[2], h[3]);
        l4[c] = make_float4(l[0], l[1], l[2], l[3]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) sq[r] = (float)s;
}

struct Args {
    const float *nx, *ny, *radii;
    void* part;
    int M, N, D, k, same_set, mode;
    float gamma;                                  // RBF_SUM: gamma; RATIO_MAX: eps
    int S, tps, nct, items;
};

// The radius instance's reduction of one 128 x 256 TMEM tile into this thread's row: a count of d2 <= r (COUNT, COVER) or a
// running max of r / (d2 + eps) (RATIO_MAX).  Padded columns have r = -1: they neither count nor raise the max (which starts at 0).
template <bool RATIO>
__device__ __forceinline__ void radius_tile(uint32_t taddr, const float* ny, const float* rr, float nxi, float eps, int& cnt,
                                            float& rmax) {
#pragma unroll 1
    for (int ch = 0; ch < TBN / 32; ++ch) {
        uint32_t v[32];
        tmem_ld32(taddr + ch * 32, v);
        tmem_wait_ld();
#pragma unroll
        for (int e = 0; e < 32; ++e) {
            const int j = ch * 32 + e;
            const float d2 = fmaxf(fmaf(-2.0f, __uint_as_float(v[e]), nxi + ny[j]), 0.0f);
            if (RATIO) rmax = fmaxf(rmax, __fdiv_rn(rr[j], d2 + eps));
            else cnt += d2 <= rr[j] ? 1 : 0;
        }
    }
}

template <int MODE>
__global__ void __launch_bounds__(NTHREADS, 1)
pairwise_kernel(const __grid_constant__ CUtensorMap txh, const __grid_constant__ CUtensorMap txl,
                const __grid_constant__ CUtensorMap tyh, const __grid_constant__ CUtensorMap tyl, const Args p) {
    constexpr uint32_t TMEM_COLS = 512;
    constexpr uint32_t IDESC = instr_desc_tf32(TBN);

    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    unsigned char* sStage = smem;
    float* sNy = reinterpret_cast<float*>(sStage + STAGES * STAGE_BYTES);     // [2 accumulators][TBN]
    float* sR = sNy + 2 * TBN;                                                  // [2][TBN] (radius modes)
    double* sRed = reinterpret_cast<double*>(sR + 2 * TBN);                     // [4] (RBF_SUM)
    Bars* bars = reinterpret_cast<Bars*>(sRed + 4);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int kblocks = (p.D + BK - 1) / BK;

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&bars->full[s], 1);
            mbar_init(&bars->empty[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&bars->acc_full[a], 1);
            mbar_init(&bars->acc_empty[a], 4);                                  // one arrival per epilogue warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 5) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&bars->tmem_base)), "n"(TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    fence_before();
    __syncthreads();
    fence_after();
    const uint32_t tmem = bars->tmem_base;

    if (warp == 4) {
        if (lane == 0) {
            // ---------------------------------------------------------------------------------------- TMA producer
            uint32_t it = 0;
            for (int item = blockIdx.x; item < p.items; item += gridDim.x) {
                const int m0 = (item / p.S) * TBM, s = item % p.S;
                const int ct_end = min(p.nct, (s + 1) * p.tps);
                for (int ct = s * p.tps; ct < ct_end; ++ct) {
                    for (int kb = 0; kb < kblocks; ++kb, ++it) {
                        const uint32_t st = it % STAGES;
                        mbar_wait(&bars->empty[st], ((it / STAGES) & 1) ^ 1);
                        const uint32_t base = smem_u32(sStage + st * STAGE_BYTES);
                        mbar_expect_tx(&bars->full[st], STAGE_BYTES);
                        tma_load_2d(base, &txh, &bars->full[st], kb * BK, m0);
                        tma_load_2d(base + A_BYTES, &txl, &bars->full[st], kb * BK, m0);
                        tma_load_2d(base + 2 * A_BYTES, &tyh, &bars->full[st], kb * BK, ct * TBN);
                        tma_load_2d(base + 2 * A_BYTES + B_BYTES, &tyl, &bars->full[st], kb * BK, ct * TBN);
                    }
                }
            }
        }
    } else if (warp == 5) {
        // -------------------------------------------------------------------------------------------- MMA issuer
        const bool leader = elect_one();
        uint32_t it = 0, t = 0;
        for (int item = blockIdx.x; item < p.items; item += gridDim.x) {
            const int s = item % p.S;
            const int ct_end = min(p.nct, (s + 1) * p.tps);
            for (int ct = s * p.tps; ct < ct_end; ++ct, ++t) {
                const uint32_t a = t & 1;
                if (t >= 2) mbar_wait(&bars->acc_empty[a], ((t >> 1) - 1) & 1);
                fence_after();
                for (int kb = 0; kb < kblocks; ++kb, ++it) {
                    const uint32_t st = it % STAGES;
                    mbar_wait(&bars->full[st], (it / STAGES) & 1);
                    fence_after();
                    if (leader) {
                        const uint32_t base = smem_u32(sStage + st * STAGE_BYTES);
                        const uint64_t dxh = smem_desc(base, 16, 1024), dxl = smem_desc(base + A_BYTES, 16, 1024);
                        const uint64_t dyh = smem_desc(base + 2 * A_BYTES, 16, 1024), dyl = smem_desc(base + 2 * A_BYTES + B_BYTES, 16, 1024);
                        const uint32_t d = tmem + a * TBN;
#pragma unroll
                        for (int k = 0; k < BK / 8; ++k) {          // the two small correction terms first, then hi . hi
                            mma_ss_tf32(d, desc_add(dxl, k * 32), desc_add(dyh, k * 32), IDESC, (kb > 0 || k > 0) ? 1u : 0u);
                            mma_ss_tf32(d, desc_add(dxh, k * 32), desc_add(dyl, k * 32), IDESC, 1u);
                            mma_ss_tf32(d, desc_add(dxh, k * 32), desc_add(dyh, k * 32), IDESC, 1u);
                        }
                        mma_commit(&bars->empty[st]);
                        if (kb + 1 == kblocks) mma_commit(&bars->acc_full[a]);
                    }
                    __syncwarp();
                }
            }
        }
    } else {
        // ---------------------------------------------------------------------------------------- epilogue (warps 0-3)
        const int row = warp * 32 + lane;
        const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
        uint32_t t = 0;
        for (int item = blockIdx.x; item < p.items; item += gridDim.x) {
            const int rb = item / p.S, s = item % p.S;
            const int gi = rb * TBM + row;
            const bool row_ok = gi < p.M;
            const float nxi = row_ok ? p.nx[gi] : 0.0f;
            double rsum = 0.0;
            float best[KMAX];
#pragma unroll
            for (int q = 0; q < KMAX; ++q) best[q] = __int_as_float(0x7f800000);
            float kth = __int_as_float(0x7f800000);
            int cnt = 0;
            float rmax = 0.0f;
            const int ct_end = min(p.nct, (s + 1) * p.tps);
            for (int ct = s * p.tps; ct < ct_end; ++ct, ++t) {
                const uint32_t a = t & 1;
                const int c0 = ct * TBN;
                float* ny = sNy + a * TBN;
                float* rr = sR + a * TBN;
                for (int j = row; j < TBN; j += 128) {                // (slot a was last read two tiles ago)
                    const int col = c0 + j;
                    ny[j] = col < p.N ? p.ny[col] : 0.0f;
                    if (MODE == DADD_PAIRWISE_COUNT) rr[j] = col < p.N ? p.radii[col] : -1.0f;
                }
                mbar_wait(&bars->acc_full[a], (t >> 1) & 1);
                fence_after();
                named_sync(1, 128);
                if (MODE == DADD_PAIRWISE_COUNT) {
                    if (p.mode == DADD_PAIRWISE_RATIO_MAX) radius_tile<true>(tmem + a * TBN + lane_base, ny, rr, nxi, p.gamma, cnt, rmax);
                    else radius_tile<false>(tmem + a * TBN + lane_base, ny, rr, nxi, p.gamma, cnt, rmax);
                } else {
#pragma unroll 1
                    for (int ch = 0; ch < TBN / 32; ++ch) {
                        uint32_t v[32];
                        tmem_ld32(tmem + a * TBN + ch * 32 + lane_base, v);
                        tmem_wait_ld();
#pragma unroll
                        for (int e = 0; e < 32; ++e) {
                            const int j = ch * 32 + e, col = c0 + j;
                            const float d2 = fmaxf(fmaf(-2.0f, __uint_as_float(v[e]), nxi + ny[j]), 0.0f);
                            if (MODE == DADD_PAIRWISE_RBF_SUM) {
                                if (col < p.N) rsum += (double)expf(-p.gamma * d2);
                            } else if (col < p.N && d2 < kth && !(p.same_set && col == gi)) {
                                topk_insert(best, d2, p.k);
                                kth = topk_last(best, p.k);
                            }
                        }
                    }
                }
                fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->acc_empty[a]);
            }
            if (MODE == DADD_PAIRWISE_RBF_SUM) {
                double r = row_ok ? rsum : 0.0;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
                if (lane == 0) sRed[warp] = r;
                named_sync(1, 128);
                if (row == 0) reinterpret_cast<double*>(p.part)[item] = ((sRed[0] + sRed[1]) + sRed[2]) + sRed[3];
            } else if (row_ok) {
                if (MODE == DADD_PAIRWISE_KNN) {
                    float* dst = reinterpret_cast<float*>(p.part) + ((int64_t)gi * p.S + s) * p.k;
#pragma unroll
                    for (int q = 0; q < KMAX; ++q)
                        if (q < p.k) dst[q] = best[q];
                } else if (p.mode == DADD_PAIRWISE_RATIO_MAX) {
                    reinterpret_cast<float*>(p.part)[(int64_t)gi * p.S + s] = rmax;
                } else {
                    reinterpret_cast<int*>(p.part)[(int64_t)gi * p.S + s] = cnt;
                }
            }
        }
    }
    fence_before();
    __syncthreads();
    if (warp == 5) {
        fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(TMEM_COLS));
    }
}

// One block: the per-item partial sums in a fixed order (thread t takes items t, t + 1024, ...; then a fixed tree).
__global__ void __launch_bounds__(1024) rbf_finish_kernel(const double* __restrict__ part, int items, double* __restrict__ out) {
    __shared__ double sh[1024];
    double s = 0.0;
    for (int i = threadIdx.x; i < items; i += 1024) s += part[i];
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int w = 512; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) sh[threadIdx.x] += sh[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[0] = sh[0];
}

__global__ void knn_finish_kernel(const float* __restrict__ part, int M, int S, int k, float* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    float best[KMAX];
#pragma unroll
    for (int q = 0; q < KMAX; ++q) best[q] = __int_as_float(0x7f800000);
    const float* src = part + (int64_t)i * S * k;
    for (int e = 0; e < S * k; ++e) topk_insert(best, src[e], k);
    out[i] = topk_last(best, k);
}

// Radius modes, slices in order: COUNT sums the counts (int32 out), COVER writes count > 0 (uint8 out), RATIO_MAX takes the max.
__global__ void radius_finish_kernel(const void* __restrict__ part, int M, int S, int mode, void* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    if (mode == DADD_PAIRWISE_RATIO_MAX) {
        const float* src = reinterpret_cast<const float*>(part) + (int64_t)i * S;
        float r = 0.0f;
        for (int s = 0; s < S; ++s) r = fmaxf(r, src[s]);
        reinterpret_cast<float*>(out)[i] = r;
        return;
    }
    const int* src = reinterpret_cast<const int*>(part) + (int64_t)i * S;
    int c = 0;
    for (int s = 0; s < S; ++s) c += src[s];
    if (mode == DADD_PAIRWISE_COUNT) reinterpret_cast<int*>(out)[i] = c;
    else reinterpret_cast<uint8_t*>(out)[i] = c > 0 ? 1 : 0;
}

// 2-D row-major fp32 (rows, cols), box = 32 columns (128 bytes) x box_rows, 128-byte swizzle, zero fill beyond the edges
static int make_map_f32(CUtensorMap* map, const void* base, int64_t rows, int64_t cols, int box_rows) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return fail("%s: cuTensorMapEncodeTiled is unavailable", "dadd_pairwise");
    const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)cols * 4};
    const cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail("%s: cuTensorMapEncodeTiled failed (CUresult %lld)", "dadd_pairwise", (long long)r);
    return 0;
}

template <int MODE>
static int launch_main(const CUtensorMap (&maps)[4], const Args& a, cudaStream_t s) {
    const size_t smem = (size_t)STAGES * STAGE_BYTES + 4 * TBN * sizeof(float) + 4 * sizeof(double) + sizeof(Bars) + 1024;
    auto kern = pairwise_kernel<MODE>;
    if (cuda_ok(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "dadd_pairwise smem")) return 2;
    const int grid = a.items < num_sms() ? a.items : num_sms();
    kern<<<grid, NTHREADS, smem, s>>>(maps[0], maps[1], maps[2], maps[3], a);
    return launched("dadd_pairwise");
}

}  // namespace pw
}  // namespace daddk

using namespace daddk;

static bool radius_mode(int mode) {
    return mode == DADD_PAIRWISE_COVER || mode == DADD_PAIRWISE_COUNT || mode == DADD_PAIRWISE_RATIO_MAX;
}

static int pairwise_check(int64_t M, int64_t N, int D, int mode, int k, int same_set) {
    if (mode != DADD_PAIRWISE_RBF_SUM && mode != DADD_PAIRWISE_KNN && !radius_mode(mode))
        return fail("%s: unknown mode %lld", "dadd_pairwise", (long long)mode);
    if (M < 1 || N < 1 || M > (1ll << 30) || N > (1ll << 30))
        return fail("%s: needs 1 <= M, N <= 2^30 (M = %lld, N = %lld)", "dadd_pairwise", (long long)M, (long long)N);
    if (D < 8 || D % 8 != 0 || D > (1 << 20)) return fail("%s: needs D %% 8 == 0 and 8 <= D <= 2^20 (D = %lld)", "dadd_pairwise", (long long)D);
    if (same_set && (N != M || radius_mode(mode)))
        return fail("%s: same_set needs N == M and mode RBF_SUM or KNN (N = %lld, M = %lld)", "dadd_pairwise", (long long)N, (long long)M);
    if (mode == DADD_PAIRWISE_KNN) {
        if (k < 1 || k > pw::KMAX) return fail("%s: KNN needs 1 <= k <= 16 (k = %lld)", "dadd_pairwise", (long long)k);
        if (N <= k + (same_set ? 1 : 0))
            return fail("%s: KNN needs more than k columns, more than k + 1 with same_set (N = %lld, k = %lld)", "dadd_pairwise",
                        (long long)N, (long long)k);
    }
    return 0;
}

extern "C" int64_t dadd_pairwise_workspace_bytes(int64_t M, int64_t N, int D, int mode, int k, int same_set) {
    if (pairwise_check(M, N, D, mode, k, same_set)) return -1;
    return pw::make_plan(M, N, D, mode, k, same_set).total;
}

extern "C" int dadd_pairwise(const float* x, const float* y, int64_t M, int64_t N, int D, int mode, int k, int same_set, float gamma,
                             const float* radii, void* out, void* workspace, int64_t workspace_bytes, void* stream) {
    if (pairwise_check(M, N, D, mode, k, same_set)) return 1;
    DADD_REQUIRE(x && out && workspace, "dadd_pairwise");
    DADD_REQUIRE(same_set ? (y == nullptr || y == x) : y != nullptr, "dadd_pairwise");
    if (radius_mode(mode) && !radii) return fail("%s: COVER, COUNT and RATIO_MAX need radii (got NULL)", "dadd_pairwise");
    if (mode == DADD_PAIRWISE_RATIO_MAX && !(gamma > 0.0f && gamma < INFINITY))
        return fail("%s: RATIO_MAX needs a finite eps > 0, passed as gamma (eps = %g)", "dadd_pairwise", (double)gamma);
    DADD_REQUIRE(((uintptr_t)x | (uintptr_t)y | (uintptr_t)workspace) % 16 == 0, "dadd_pairwise");
    const pw::Plan pl = pw::make_plan(M, N, D, mode, k, same_set);
    if (workspace_bytes < pl.total)
        return fail("%s: workspace of %lld bytes is smaller than dadd_pairwise_workspace_bytes() = %lld", "dadd_pairwise",
                    (long long)workspace_bytes, (long long)pl.total);
    cudaStream_t s = (cudaStream_t)stream;
    char* ws = (char*)workspace;
    float *xhi = (float*)(ws + pl.off_xhi), *xlo = (float*)(ws + pl.off_xlo), *yhi = (float*)(ws + pl.off_yhi),
          *ylo = (float*)(ws + pl.off_ylo), *nx = (float*)(ws + pl.off_nx), *ny = (float*)(ws + pl.off_ny);
    CUtensorMap maps[4];
    if (pw::make_map_f32(&maps[0], xhi, M, D, pw::TBM) || pw::make_map_f32(&maps[1], xlo, M, D, pw::TBM) ||
        pw::make_map_f32(&maps[2], yhi, N, D, pw::TBN) || pw::make_map_f32(&maps[3], ylo, N, D, pw::TBN))
        return 1;
    pw::split_kernel<<<(unsigned)((M + 7) / 8), 256, 0, s>>>(x, xhi, xlo, nx, M, D);
    if (int rc = launched("dadd_pairwise split")) return rc;
    if (!same_set) {
        pw::split_kernel<<<(unsigned)((N + 7) / 8), 256, 0, s>>>(y, yhi, ylo, ny, N, D);
        if (int rc = launched("dadd_pairwise split")) return rc;
    }
    pw::Args a{nx, ny, radii, ws + pl.off_part, (int)M, (int)N, D, k, same_set, mode, gamma, (int)pl.S, (int)pl.tps, (int)pl.nct,
               (int)pl.items};
    int rc;
    if (mode == DADD_PAIRWISE_RBF_SUM) rc = pw::launch_main<DADD_PAIRWISE_RBF_SUM>(maps, a, s);
    else if (mode == DADD_PAIRWISE_KNN) rc = pw::launch_main<DADD_PAIRWISE_KNN>(maps, a, s);
    else rc = pw::launch_main<DADD_PAIRWISE_COUNT>(maps, a, s);     // the radius instance: COVER, COUNT, RATIO_MAX
    if (rc) return rc;
    const unsigned fb = (unsigned)((M + 255) / 256);
    if (mode == DADD_PAIRWISE_RBF_SUM) pw::rbf_finish_kernel<<<1, 1024, 0, s>>>((const double*)a.part, a.items, (double*)out);
    else if (mode == DADD_PAIRWISE_KNN) pw::knn_finish_kernel<<<fb, 256, 0, s>>>((const float*)a.part, a.M, a.S, k, (float*)out);
    else pw::radius_finish_kernel<<<fb, 256, 0, s>>>(a.part, a.M, a.S, mode, out);
    return launched("dadd_pairwise finish");
}
