// fgr.cu -- registration::FastGlobalRegistration (fast_global_registration.cu:103-431) and knn::BruteForceNN
// (bruteforce_nn.inl:33-135).
//   feature_nn_kernel : exact nearest neighbour in feature space, both directions from ONE distance evaluation, with
//                       O(n + m) memory (the reference writes the n_ref x n_query distance matrix, once per direction).
//   fgr_normalize     : means of both clouds and the global scale (NormalizePointCloud, :197-265).
//   fgr_mutual / fgr_tuple / fgr_pairs : cross check + tuple test + truncation (AdvancedMatching, :103-194).
//   fgr_gnc_kernel    : the whole Geman-McClure / graduated non-convexity loop in one block
//                       (OptimizePairwiseRegistration, :309-372) and GetInvTransformationOriginalScale (:376-389).
// Arithmetic contract (DESIGN.md section 4, "FastGlobalRegistration"): feature d2 = one FMA chain over the features in
// order from 0; means = float64 sums in a fixed order (256 strided partials, then the partials in order), rounded once,
// divided by (float)n; norms sqrtf(dot3); the per-pair JTJ / JTr are float32 in the reference's operation order and
// are summed over pairs in float64, in pair order, rounded once.
#include <float.h>
#include <math.h>
#include <string.h>

#include <algorithm>

#include "cphb_internal.cuh"
// ldlt6_solve / se3_exp / matmul4 / identity4 of the ICP epilogue; internal linkage here, so that their host-side
// stubs do not collide with icp.cu's at link time
namespace {
#include "icp_types.cuh"
#include "icp_solve.cuh"
}  // namespace

#define FNN_TILE 128
#define FNN_THREADS 256
#define FGR_THREADS 256

__device__ __forceinline__ unsigned long long fnn_key(float d2, unsigned idx) {
    return ((unsigned long long)__float_as_uint(d2) << 32) | idx;
}
__device__ __forceinline__ unsigned long long umin64(unsigned long long a, unsigned long long b) { return a < b ? a : b; }

// One block = a 128 x 128 tile of (A row, B row) pairs; each thread holds an 8 x 8 register tile.  Features are staged
// in shared memory KC at a time (KC divides Dim: 33 | 33, 44 | 352), so no padding work is done.  The distance of a
// pair is fma(d_k, d_k, .) over k in order, d_k = a_k - b_k; (a - b)^2 == (b - a)^2 bit for bit, so the same value
// serves both directions.  Keys (d2 bits << 32 | index) are non-negative floats first, so the 64-bit minimum is the
// smallest distance and, among equal distances, the smallest index -- the reference's strict-< ascending scan.
// TWO_WAY = false drops the column direction (knn::BruteForceNN).  A non-finite feature sets *bad.
template <int Dim, bool TWO_WAY>
__global__ void __launch_bounds__(FNN_THREADS) feature_nn_kernel(const float *__restrict__ A, int na, const float *__restrict__ B,
                                                                 int nb, unsigned long long *keyA, unsigned long long *keyB,
                                                                 int *bad) {
    constexpr int KC = (Dim % 33 == 0) ? 33 : 44;
    static_assert(Dim % KC == 0, "feature chunk must divide Dim");
    __shared__ __align__(16) float sA[KC][FNN_TILE];
    __shared__ __align__(16) float sB[KC][FNN_TILE];
    __shared__ unsigned long long rowmin[FNN_TILE], colmin[FNN_TILE];
    const int a0 = blockIdx.y * FNN_TILE, b0 = blockIdx.x * FNN_TILE;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    if (threadIdx.x < FNN_TILE) colmin[threadIdx.x] = ~0ull;
    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    bool nonfinite = false;
    for (int k0 = 0; k0 < Dim; k0 += KC) {
        for (int e = threadIdx.x; e < FNN_TILE * KC; e += FNN_THREADS) {
            const int r = e % FNN_TILE, k = e / FNN_TILE;
            const float va = (a0 + r < na) ? A[(size_t)(a0 + r) * Dim + k0 + k] : 0.f;
            const float vb = (b0 + r < nb) ? B[(size_t)(b0 + r) * Dim + k0 + k] : 0.f;
            nonfinite |= !isfinite(va) || !isfinite(vb);
            sA[k][r] = va;
            sB[k][r] = vb;
        }
        __syncthreads();
#pragma unroll 11
        for (int k = 0; k < KC; ++k) {
            const float4 x0 = *reinterpret_cast<const float4 *>(&sA[k][ty * 8]);
            const float4 x1 = *reinterpret_cast<const float4 *>(&sA[k][ty * 8 + 4]);
            const float4 y0 = *reinterpret_cast<const float4 *>(&sB[k][tx * 8]);
            const float4 y1 = *reinterpret_cast<const float4 *>(&sB[k][tx * 8 + 4]);
            const float a[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
            const float b[8] = {y0.x, y0.y, y0.z, y0.w, y1.x, y1.y, y1.z, y1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float d = __fsub_rn(a[i], b[j]);
                    acc[i][j] = __fmaf_rn(d, d, acc[i][j]);
                }
        }
        __syncthreads();
    }
    if (nonfinite) atomicExch(bad, 1);
    // row minima: the 16 threads of a row group are one half warp
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        unsigned long long key = ~0ull;
#pragma unroll
        for (int j = 0; j < 8; ++j)
            if (b0 + tx * 8 + j < nb) key = umin64(key, fnn_key(acc[i][j], (unsigned)(b0 + tx * 8 + j)));
#pragma unroll
        for (int o = 8; o >= 1; o >>= 1) key = umin64(key, __shfl_xor_sync(CPHB_FULL, key, o));
        if (tx == 0) rowmin[ty * 8 + i] = key;
    }
    if (TWO_WAY) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            unsigned long long key = ~0ull;
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (a0 + ty * 8 + i < na) key = umin64(key, fnn_key(acc[i][j], (unsigned)(a0 + ty * 8 + i)));
            key = umin64(key, __shfl_xor_sync(CPHB_FULL, key, 16));
            if ((ty & 1) == 0) atomicMin(&colmin[tx * 8 + j], key);
        }
    }
    __syncthreads();
    if (threadIdx.x < FNN_TILE) {
        const int t = threadIdx.x;
        if (a0 + t < na) atomicMin(&keyA[a0 + t], rowmin[t]);
        if (TWO_WAY && b0 + t < nb) atomicMin(&keyB[b0 + t], colmin[t]);
    }
}

__global__ void fnn_decode_kernel(const unsigned long long *key, size_t n, int32_t *idx, float *d2) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned long long k = key[i];
    idx[i] = (int32_t)(unsigned)(k & 0xffffffffu);
    if (d2) d2[i] = __uint_as_float((unsigned)(k >> 32));
}

// keys must hold ~0 on entry.  Rows of A find their nearest row of B (keyA); with keyB also the reverse.
static int launch_feature_nn(const float *A, size_t na, const float *B, size_t nb, int dim, unsigned long long *keyA,
                             unsigned long long *keyB, int *bad, cudaStream_t s) {
    const dim3 grid((unsigned)((nb + FNN_TILE - 1) / FNN_TILE), (unsigned)((na + FNN_TILE - 1) / FNN_TILE));
    if (dim == 33) {
        if (keyB) CPHB_LAUNCH((feature_nn_kernel<33, true>), grid, FNN_THREADS, 0, s, A, (int)na, B, (int)nb, keyA, keyB, bad);
        else CPHB_LAUNCH((feature_nn_kernel<33, false>), grid, FNN_THREADS, 0, s, A, (int)na, B, (int)nb, keyA, keyB, bad);
    } else {
        if (keyB) CPHB_LAUNCH((feature_nn_kernel<352, true>), grid, FNN_THREADS, 0, s, A, (int)na, B, (int)nb, keyA, keyB, bad);
        else CPHB_LAUNCH((feature_nn_kernel<352, false>), grid, FNN_THREADS, 0, s, A, (int)na, B, (int)nb, keyA, keyB, bad);
    }
    CPHB_CHECK_LAUNCH();
    return CPHB_OK;
}

static int check_feature_args(const char *fn, size_t n_points, size_t n_features, int dim) {
    if (dim != 33 && dim != 352) {
        cphb_set_error("%s: feature dimension %d (only 33 and 352 are supported)", fn, dim);
        return CPHB_ERR_INVALID;
    }
    if (n_points != n_features) {
        cphb_set_error("%s: %zu points but %zu features", fn, n_points, n_features);
        return CPHB_ERR_INVALID;
    }
    // grid.y of the matcher and int32 indices
    if (n_points > (size_t)65535 * FNN_TILE) {
        cphb_set_error("%s: %zu feature rows exceed the matcher's limit of %d", fn, n_points, 65535 * FNN_TILE);
        return CPHB_ERR_INVALID;
    }
    return CPHB_OK;
}

extern "C" int cphb_feature_nn(const float *ref, size_t n_ref, const float *query, size_t n_query, int dim, int32_t *idx_out,
                               float *d2_out, int32_t *ref_idx_out, float *ref_d2_out, void *stream) {
    cudaStream_t s = (cudaStream_t)stream;
    int rc = check_feature_args("cphb_feature_nn", n_ref, n_ref, dim);
    if (!rc) rc = check_feature_args("cphb_feature_nn", n_query, n_query, dim);
    if (rc) return rc;
    const bool two_way = ref_idx_out != nullptr;
    if (n_query == 0 && !(two_way && n_ref)) return CPHB_OK;
    if (n_ref == 0 || n_query == 0 || !ref || !query || !idx_out) {
        cphb_set_error("cphb_feature_nn: empty set on one side or null argument");
        return CPHB_ERR_INVALID;
    }
    const size_t n_keys = n_query + (two_way ? n_ref : 0);
    unsigned long long *key = nullptr;
    int *bad = nullptr;
    rc = cphb_alloc_async((void **)&key, sizeof(unsigned long long) * n_keys, s);
    if (!rc) rc = cphb_alloc_async((void **)&bad, sizeof(int), s);
    if (!rc) {
        cudaMemsetAsync(key, 0xff, sizeof(unsigned long long) * n_keys, s);
        cudaMemsetAsync(bad, 0, sizeof(int), s);
        rc = launch_feature_nn(query, n_query, ref, n_ref, dim, key, two_way ? key + n_query : nullptr, bad, s);
    }
    int h_bad = 0;
    if (!rc) {
        CPHB_LAUNCH(fnn_decode_kernel, (unsigned)((n_query + 255) / 256), 256, 0, s, key, n_query, idx_out, d2_out);
        if (two_way)
            CPHB_LAUNCH(fnn_decode_kernel, (unsigned)((n_ref + 255) / 256), 256, 0, s, key + n_query, n_ref, ref_idx_out, ref_d2_out);
        cudaMemcpyAsync(&h_bad, bad, sizeof(int), cudaMemcpyDeviceToHost, s);
        if (cudaStreamSynchronize(s) != cudaSuccess) {
            cphb_set_error("cphb_feature_nn: %s", cudaGetErrorString(cudaGetLastError()));
            rc = CPHB_ERR_CUDA;
        }
    }
    cphb_free_async(key, s);
    cphb_free_async(bad, s);
    if (!rc && h_bad) {
        cphb_set_error("cphb_feature_nn: non-finite feature value");
        rc = CPHB_ERR_INVALID;
    }
    return rc;
}

// ---------------------------------------------------------------------------------------------------------------------
// FastGlobalRegistration
// ---------------------------------------------------------------------------------------------------------------------
struct FgrNorm {
    float mean[2][3];  // source, target
    float scale;       // largest centred point norm over both clouds
    float scale_global;
};

// NormalizePointCloud (:197-265), one block: thread t sums points t, t + 256, ... in float64, thread 0 adds the 256
// partials in order; mean = (float)sum / (float)n; scale = max sqrtf(dot3(p - mean)) over both clouds.
__global__ void __launch_bounds__(FGR_THREADS) fgr_normalize_kernel(const float *src, size_t ns, const float *tgt, size_t nt,
                                                                    int use_absolute_scale, FgrNorm *out) {
    __shared__ double part[FGR_THREADS][3];
    __shared__ float mean[3];
    __shared__ unsigned smax;
    if (threadIdx.x == 0) smax = 0u;
    for (int c = 0; c < 2; ++c) {
        const float *p = c ? tgt : src;
        const size_t n = c ? nt : ns;
        double a0 = 0.0, a1 = 0.0, a2 = 0.0;
        for (size_t i = threadIdx.x; i < n; i += FGR_THREADS) {
            a0 = __dadd_rn(a0, (double)p[3 * i]);
            a1 = __dadd_rn(a1, (double)p[3 * i + 1]);
            a2 = __dadd_rn(a2, (double)p[3 * i + 2]);
        }
        part[threadIdx.x][0] = a0; part[threadIdx.x][1] = a1; part[threadIdx.x][2] = a2;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t0 = 0.0, t1 = 0.0, t2 = 0.0;
            for (int t = 0; t < FGR_THREADS; ++t) {
                t0 = __dadd_rn(t0, part[t][0]); t1 = __dadd_rn(t1, part[t][1]); t2 = __dadd_rn(t2, part[t][2]);
            }
            mean[0] = __fdiv_rn((float)t0, (float)n);
            mean[1] = __fdiv_rn((float)t1, (float)n);
            mean[2] = __fdiv_rn((float)t2, (float)n);
            for (int k = 0; k < 3; ++k) out->mean[c][k] = mean[k];
        }
        __syncthreads();
        float m = 0.f;
        for (size_t i = threadIdx.x; i < n; i += FGR_THREADS) {
            const float x = __fsub_rn(p[3 * i], mean[0]), y = __fsub_rn(p[3 * i + 1], mean[1]), z = __fsub_rn(p[3 * i + 2], mean[2]);
            m = fmaxf(m, sqrtf(dot3(x, y, z, x, y, z)));
        }
        atomicMax(&smax, __float_as_uint(m));  // non-negative floats order as their bits
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        out->scale = __uint_as_float(smax);
        out->scale_global = use_absolute_scale ? 1.f : out->scale;
    }
}

__device__ __forceinline__ void fgr_point(const float *p, size_t i, const float *mean, float scale_global, float *o) {
#pragma unroll
    for (int k = 0; k < 3; ++k) o[k] = __fdiv_rn(__fsub_rn(p[3 * i + k], mean[k]), scale_global);
}

// cross check: fi point i is kept when its nearest fj point j has i as its own nearest fi point
__global__ void fgr_mutual_kernel(const unsigned long long *key_i, size_t ni, const unsigned long long *key_j, uint8_t *keep) {
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (i >= ni) return;
    const unsigned j = (unsigned)(key_i[i] & 0xffffffffu);
    keep[i] = (unsigned)(key_j[j] & 0xffffffffu) == (unsigned)i;
}

// thrust::minstd_rand (a = 48271, m = 2^31 - 1, seed 1): discard(idx) is a modular power.
__device__ __host__ __forceinline__ unsigned long long minstd_pow(unsigned long long e) {
    unsigned long long r = 1, b = 48271;
    while (e) {
        if (e & 1) r = r * b % 2147483647ull;
        b = b * b % 2147483647ull;
        e >>= 1;
    }
    return r;
}
// uniform_int_distribution(0, ncorr - 1) through thrust's float64 uniform_real_distribution
__device__ __forceinline__ int minstd_draw(unsigned long long x, size_t ncorr) {
    return (int)(__dmul_rn(__ddiv_rn((double)(x - 1), 2147483646.0), (double)ncorr));
}
__device__ __forceinline__ void fgr_trial_draws(size_t idx, size_t ncorr, int r[3]) {
    unsigned long long x = minstd_pow(idx);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        x = x * 48271ull % 2147483647ull;
        r[k] = minstd_draw(x, ncorr);
    }
}

struct FgrMatch {
    const float *pi, *pj;          // fi / fj clouds (raw)
    const int32_t *mutual;         // ascending fi indices that passed the cross check
    const unsigned long long *key_i;  // fi point -> nearest fj point
    const FgrNorm *norm;
    int ci, cj;                    // which cloud (0 source, 1 target) fi / fj are
    size_t ncorr;
    float tuple_scale;
};

__device__ __forceinline__ void fgr_pair(const FgrMatch &m, int r, int &i, int &j) {
    i = m.mutual[r];
    j = (int)(unsigned)(m.key_i[i] & 0xffffffffu);
}

// compute_tuple_constraint_functor (:17-101): one thread per trial, pass flag per trial
__global__ void fgr_tuple_kernel(FgrMatch m, size_t n_trial, uint8_t *pass) {
    size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (idx >= n_trial) return;
    int r[3];
    fgr_trial_draws(idx, m.ncorr, r);
    const float sg = m.norm->scale_global;
    float pi[3][3], pj[3][3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        int i, j;
        fgr_pair(m, r[k], i, j);
        fgr_point(m.pi, i, m.norm->mean[m.ci], sg, pi[k]);
        fgr_point(m.pj, j, m.norm->mean[m.cj], sg, pj[k]);
    }
    bool cond = true;
    const float s = m.tuple_scale;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const int l = (k + 1) % 3;
        const float dx = __fsub_rn(pi[k][0], pi[l][0]), dy = __fsub_rn(pi[k][1], pi[l][1]), dz = __fsub_rn(pi[k][2], pi[l][2]);
        const float ex = __fsub_rn(pj[k][0], pj[l][0]), ey = __fsub_rn(pj[k][1], pj[l][1]), ez = __fsub_rn(pj[k][2], pj[l][2]);
        const float li = sqrtf(dot3(dx, dy, dz, dx, dy, dz)), lj = sqrtf(dot3(ex, ey, ez, ex, ey, ez));
        cond = cond && (__fmul_rn(li, s) < lj) && (lj < __fdiv_rn(li, s));
    }
    pass[idx] = cond;
}

// the first n_pairs pairs of the passing trials, in trial order, as (source index, target index)
__global__ void fgr_pairs_kernel(FgrMatch m, const int32_t *passed, size_t n_pairs, int swapped, int32_t *out) {
    size_t p = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (p >= n_pairs) return;
    int r[3];
    fgr_trial_draws((size_t)passed[p / 3], m.ncorr, r);
    int i, j;
    fgr_pair(m, r[p % 3], i, j);
    out[2 * p] = swapped ? j : i;
    out[2 * p + 1] = swapped ? i : j;
}

// OptimizePairwiseRegistration (:309-372) + GetInvTransformationOriginalScale (:376-389), one block.
// P / Q: scratch [n][3] for the gathered source points and the target working copy.
__global__ void __launch_bounds__(FGR_THREADS) fgr_gnc_kernel(const float *src, const float *tgt, const int32_t *pairs, int n,
                                                              const FgrNorm *norm, int iteration_number, int decrease_mu,
                                                              float division_factor, float max_corr, float *P, float *Q,
                                                              float *trace_T, float *T_out) {
    __shared__ float vals[27][FGR_THREADS];
    __shared__ double S[27];
    __shared__ float trans[16], delta[16];
    const float sg = norm->scale_global;
    for (int k = threadIdx.x; k < n; k += FGR_THREADS) {
        fgr_point(src, (size_t)pairs[2 * k], norm->mean[0], sg, P + 3 * k);
        fgr_point(tgt, (size_t)pairs[2 * k + 1], norm->mean[1], sg, Q + 3 * k);
    }
    if (threadIdx.x == 0) identity4(trans);
    __syncthreads();
    float par = sg;  // the reference starts from scale_global, not scale_start (:423-424)
    if (n >= 10) {
        for (int itr = 0; itr < iteration_number; ++itr) {
            if (threadIdx.x < 27) S[threadIdx.x] = 0.0;
            for (int c0 = 0; c0 < n; c0 += FGR_THREADS) {
                const int k = c0 + threadIdx.x;
                if (k < n) {
                    // compute_jacobian_functor (:267-307)
                    const float q0 = Q[3 * k], q1 = Q[3 * k + 1], q2 = Q[3 * k + 2];
                    const float r0 = __fsub_rn(P[3 * k], q0), r1 = __fsub_rn(P[3 * k + 1], q1), r2 = __fsub_rn(P[3 * k + 2], q2);
                    const float temp = __fdiv_rn(par, __fadd_rn(dot3(r0, r1, r2, r0, r1, r2), par));
                    const float s = __fmul_rn(temp, temp);
                    const float J[3][6] = {{0.f, -q2, q1, -1.f, 0.f, 0.f}, {q2, 0.f, -q0, 0.f, -1.f, 0.f}, {-q1, q0, 0.f, 0.f, 0.f, -1.f}};
                    const float rr[3] = {r0, r1, r2};
                    int e = 0;
#pragma unroll
                    for (int a = 0; a < 6; ++a)
#pragma unroll
                        for (int b = a; b < 6; ++b) {
                            float v = 0.f;
#pragma unroll
                            for (int w = 0; w < 3; ++w) v = __fadd_rn(v, __fmul_rn(__fmul_rn(J[w][a], J[w][b]), s));
                            vals[e++][threadIdx.x] = v;
                        }
#pragma unroll
                    for (int a = 0; a < 6; ++a) {
                        float v = 0.f;
#pragma unroll
                        for (int w = 0; w < 3; ++w) v = __fadd_rn(v, __fmul_rn(__fmul_rn(J[w][a], rr[w]), s));
                        vals[21 + a][threadIdx.x] = v;
                    }
                }
                __syncthreads();
                if (threadIdx.x < 27) {
                    const int m = min(FGR_THREADS, n - c0);
                    double acc = S[threadIdx.x];
                    for (int t = 0; t < m; ++t) acc = __dadd_rn(acc, (double)vals[threadIdx.x][t]);
                    S[threadIdx.x] = acc;
                }
                __syncthreads();
            }
            if (threadIdx.x == 0) {
                // SolveLinearSystemPSD<6>(-JTJ, JTr) (:347-348): no symmetry or determinant check
                float A[36], b[6], x[6];
                int p = 0;
                for (int a = 0; a < 6; ++a)
                    for (int c = a; c < 6; ++c) {
                        const float v = -(float)S[p++];
                        A[6 * a + c] = v;
                        A[6 * c + a] = v;
                    }
                for (int a = 0; a < 6; ++a) b[a] = (float)S[21 + a];
                ldlt6_solve(A, b, x);
                se3_exp(x, delta);
                matmul4(delta, trans, trans);
                if (trace_T)
                    for (int e = 0; e < 16; ++e) trace_T[16 * itr + e] = trans[e];
            }
            __syncthreads();
            for (int k = threadIdx.x; k < n; k += FGR_THREADS) {
                const float x = Q[3 * k], y = Q[3 * k + 1], z = Q[3 * k + 2];
                Q[3 * k] = __fadd_rn(dot3(delta[0], delta[1], delta[2], x, y, z), delta[3]);
                Q[3 * k + 1] = __fadd_rn(dot3(delta[4], delta[5], delta[6], x, y, z), delta[7]);
                Q[3 * k + 2] = __fadd_rn(dot3(delta[8], delta[9], delta[10], x, y, z), delta[11]);
            }
            if (decrease_mu && itr % 4 == 0 && par > max_corr) par = __fdiv_rn(par, division_factor);
            __syncthreads();
        }
    } else if (trace_T) {
        for (int e = threadIdx.x; e < 16 * iteration_number; e += FGR_THREADS) trace_T[e] = (e % 16 % 5 == 0) ? 1.f : 0.f;
    }
    if (threadIdx.x == 0) {
        // [R^T | -R^T (-R mean_t + t scale_global + mean_s)]
        const float *ms = norm->mean[0], *mt = norm->mean[1];
        float v[3];
        for (int k = 0; k < 3; ++k) {
            const float rm = dot3(trans[4 * k], trans[4 * k + 1], trans[4 * k + 2], mt[0], mt[1], mt[2]);
            v[k] = __fadd_rn(__fadd_rn(-rm, __fmul_rn(trans[4 * k + 3], sg)), ms[k]);
        }
        for (int r = 0; r < 3; ++r) {
            for (int c = 0; c < 3; ++c) T_out[4 * r + c] = trans[4 * c + r];
            T_out[4 * r + 3] = -dot3(trans[r], trans[4 + r], trans[8 + r], v[0], v[1], v[2]);
        }
        T_out[12] = T_out[13] = T_out[14] = 0.f;
        T_out[15] = 1.f;
    }
}

extern "C" void cphb_fgr_default_option(cphb_fgr_option *o) {
    o->division_factor = 1.4f;
    o->use_absolute_scale = 0;
    o->decrease_mu = 1;
    o->maximum_correspondence_distance = 0.025f;
    o->iteration_number = 64;
    o->tuple_scale = 0.95f;
    o->maximum_tuple_count = 1000;
}

struct FgrWork {
    FgrNorm *norm = nullptr;
    unsigned long long *key = nullptr;  // [n_fi + n_fj]
    int *bad = nullptr;
    uint8_t *flags = nullptr;
    int32_t *mutual = nullptr, *passed = nullptr;
    void release(cudaStream_t s) {
        cphb_free_async(norm, s);
        cphb_free_async(key, s);
        cphb_free_async(bad, s);
        cphb_free_async(flags, s);
        cphb_free_async(mutual, s);
        cphb_free_async(passed, s);
    }
};

// NormalizePointCloud + AdvancedMatching.  pairs_out: device, 2 * max(maximum_tuple_count, 0) int32.
// h_counts: pairs written, mutual matches, trials, passing pairs.  Leaves w.norm for the pose solve.
static int fgr_match(const float *src, size_t ns, const float *tgt, size_t nt, const float *fs, const float *ft, int dim,
                     const cphb_fgr_option &opt, int32_t *pairs_out, int64_t h_counts[4], FgrWork &w, cudaStream_t s) {
    const bool swapped = nt > ns;
    const float *pi = swapped ? tgt : src, *pj = swapped ? src : tgt, *fi = swapped ? ft : fs, *fj = swapped ? fs : ft;
    const size_t ni = swapped ? nt : ns, nj = swapped ? ns : nt;
    int rc = cphb_alloc_async((void **)&w.norm, sizeof(FgrNorm), s);
    if (!rc) rc = cphb_alloc_async((void **)&w.key, sizeof(unsigned long long) * (ni + nj), s);
    if (!rc) rc = cphb_alloc_async((void **)&w.bad, sizeof(int), s);
    if (!rc) rc = cphb_alloc_async((void **)&w.flags, ni, s);
    if (!rc) rc = cphb_alloc_async((void **)&w.mutual, sizeof(int32_t) * ni, s);
    if (rc) return rc;
    CPHB_CUDA(cudaMemsetAsync(w.key, 0xff, sizeof(unsigned long long) * (ni + nj), s));
    CPHB_CUDA(cudaMemsetAsync(w.bad, 0, sizeof(int), s));
    CPHB_LAUNCH(fgr_normalize_kernel, 1, FGR_THREADS, 0, s, src, ns, tgt, nt, opt.use_absolute_scale, w.norm);
    CPHB_CHECK_LAUNCH();
    rc = launch_feature_nn(fi, ni, fj, nj, dim, w.key, w.key + ni, w.bad, s);
    if (rc) return rc;
    int h_bad = 0;
    CPHB_CUDA(cudaMemcpyAsync(&h_bad, w.bad, sizeof(int), cudaMemcpyDeviceToHost, s));
    CPHB_CUDA(cudaStreamSynchronize(s));
    if (h_bad) {
        // deliberate deviation: the reference would match NaN / inf features silently
        cphb_set_error("FastGlobalRegistration: non-finite feature value");
        return CPHB_ERR_INVALID;
    }
    CPHB_LAUNCH(fgr_mutual_kernel, (unsigned)((ni + 255) / 256), 256, 0, s, w.key, ni, w.key + ni, w.flags);
    CPHB_CHECK_LAUNCH();
    size_t ncorr = 0;
    rc = cphb_compact_flags(w.flags, ni, w.mutual, &ncorr, s);
    if (rc) return rc;
    const size_t n_trial = ncorr * 100;
    size_t n_pass_trials = 0;
    FgrMatch m{pi, pj, w.mutual, w.key, w.norm, swapped ? 1 : 0, swapped ? 0 : 1, ncorr, opt.tuple_scale};
    if (n_trial) {
        cphb_free_async(w.flags, s);
        w.flags = nullptr;
        rc = cphb_alloc_async((void **)&w.flags, n_trial, s);
        if (!rc) rc = cphb_alloc_async((void **)&w.passed, sizeof(int32_t) * n_trial, s);
        if (rc) return rc;
        CPHB_LAUNCH(fgr_tuple_kernel, (unsigned)((n_trial + 255) / 256), 256, 0, s, m, n_trial, w.flags);
        CPHB_CHECK_LAUNCH();
        rc = cphb_compact_flags(w.flags, n_trial, w.passed, &n_pass_trials, s);
        if (rc) return rc;
    }
    const size_t n_res = 3 * n_pass_trials;
    const size_t n_pairs = std::min(n_res, (size_t)std::max(opt.maximum_tuple_count, 0));
    if (n_pairs) {
        CPHB_LAUNCH(fgr_pairs_kernel, (unsigned)((n_pairs + 255) / 256), 256, 0, s, m, w.passed, n_pairs, swapped ? 1 : 0,
                    pairs_out);
        CPHB_CHECK_LAUNCH();
    }
    h_counts[0] = (int64_t)n_pairs;
    h_counts[1] = (int64_t)ncorr;
    h_counts[2] = (int64_t)n_trial;
    h_counts[3] = (int64_t)n_res;
    return CPHB_OK;
}

static int fgr_check(const char *fn, const float *src, size_t ns, const float *tgt, size_t nt, const float *fs, size_t nfs,
                     const float *ft, size_t nft, int dim, const cphb_fgr_option *opt) {
    int rc = check_feature_args(fn, ns, nfs, dim);
    if (!rc) rc = check_feature_args(fn, nt, nft, dim);
    if (rc) return rc;
    if (!opt || (ns && (!src || !fs)) || (nt && (!tgt || !ft))) {
        cphb_set_error("%s: null argument", fn);
        return CPHB_ERR_INVALID;
    }
    return CPHB_OK;
}

extern "C" int cphb_fgr_advanced_matching(const float *source_points, size_t n_source, const float *target_points,
                                          size_t n_target, const float *source_features, size_t n_source_features,
                                          const float *target_features, size_t n_target_features, int dim,
                                          const cphb_fgr_option *option, int32_t *pairs_out, int64_t h_counts[4],
                                          void *stream) {
    cudaStream_t s = (cudaStream_t)stream;
    int rc = fgr_check("cphb_fgr_advanced_matching", source_points, n_source, target_points, n_target, source_features,
                       n_source_features, target_features, n_target_features, dim, option);
    if (rc) return rc;
    if (!h_counts) {
        cphb_set_error("cphb_fgr_advanced_matching: null h_counts");
        return CPHB_ERR_INVALID;
    }
    for (int k = 0; k < 4; ++k) h_counts[k] = 0;
    if (n_source == 0 || n_target == 0) return CPHB_OK;
    if (!pairs_out && option->maximum_tuple_count > 0) {
        cphb_set_error("cphb_fgr_advanced_matching: null pairs_out");
        return CPHB_ERR_INVALID;
    }
    FgrWork w;
    rc = fgr_match(source_points, n_source, target_points, n_target, source_features, target_features, dim, *option, pairs_out,
                   h_counts, w, s);
    w.release(s);
    if (cudaStreamSynchronize(s) != cudaSuccess && !rc) {
        cphb_set_error("cphb_fgr_advanced_matching: %s", cudaGetErrorString(cudaGetLastError()));
        rc = CPHB_ERR_CUDA;
    }
    return rc;
}

extern "C" int cphb_fast_global_registration(const cphb_cloud *source, const cphb_cloud *target, const float *source_features,
                                             size_t n_source_features, const float *target_features,
                                             size_t n_target_features, int dim, const cphb_fgr_option *option,
                                             cphb_icp_result *h_result, int32_t *corr_out, float *trace_T, void *stream) {
    cudaStream_t s = (cudaStream_t)stream;
    if (!source || !target || !h_result) {
        cphb_set_error("cphb_fast_global_registration: null argument");
        return CPHB_ERR_INVALID;
    }
    int rc = fgr_check("cphb_fast_global_registration", source->points, source->n, target->points, target->n,
                       source_features, n_source_features, target_features, n_target_features, dim, option);
    if (rc) return rc;
    memset(h_result, 0, sizeof(*h_result));
    for (int k = 0; k < 16; ++k) h_result->transformation[k] = (k % 5 == 0) ? 1.f : 0.f;
    if (source->n == 0 || target->n == 0) {
        // the reference logs "Invalid source or target pointcloud." and returns RegistrationResult() (:400-404)
        cphb_set_error("cphb_fast_global_registration: Invalid source or target pointcloud.");
        return CPHB_OK;
    }
    const int iters = std::max(option->iteration_number, 0);
    const size_t cap = (size_t)std::max(option->maximum_tuple_count, 0);
    FgrWork w;
    int32_t *pairs = nullptr;
    float *PQ = nullptr, *T_dev = nullptr;
    int64_t counts[4] = {0, 0, 0, 0};
    rc = cphb_alloc_async((void **)&pairs, sizeof(int32_t) * 2 * (cap + 1), s);
    if (!rc) rc = fgr_match(source->points, source->n, target->points, target->n, source_features, target_features, dim,
                            *option, pairs, counts, w, s);
    if (!rc) rc = cphb_alloc_async((void **)&PQ, sizeof(float) * 6 * ((size_t)counts[0] + 1), s);
    if (!rc) rc = cphb_alloc_async((void **)&T_dev, sizeof(float) * 16, s);
    float h_T[16];
    float gnc_ms = 0.f;
    cudaEvent_t ev[2] = {nullptr, nullptr};
    if (!rc) {
        const int n = (int)counts[0];
        cudaEventCreate(&ev[0]);
        cudaEventCreate(&ev[1]);
        cudaEventRecord(ev[0], s);
        CPHB_LAUNCH(fgr_gnc_kernel, 1, FGR_THREADS, 0, s, source->points, target->points, pairs, n, w.norm, iters,
                    option->decrease_mu, option->division_factor, option->maximum_correspondence_distance, PQ, PQ + 3 * n,
                    trace_T, T_dev);
        cudaError_t e = cudaGetLastError();
        cudaEventRecord(ev[1], s);
        if (e == cudaSuccess) e = cudaMemcpyAsync(h_T, T_dev, sizeof(h_T), cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        if (e == cudaSuccess) cudaEventElapsedTime(&gnc_ms, ev[0], ev[1]);
        if (e != cudaSuccess) {
            cphb_set_error("fgr_gnc_kernel: %s", cudaGetErrorString(e));
            rc = CPHB_ERR_CUDA;
        }
    }
    for (int k = 0; k < 2; ++k)
        if (ev[k]) cudaEventDestroy(ev[k]);
    w.release(s);
    cphb_free_async(pairs, s);
    cphb_free_async(PQ, s);
    cphb_free_async(T_dev, s);
    if (rc) {
        cudaStreamSynchronize(s);
        return rc;
    }
    // EvaluateRegistration on the original clouds (:428-431)
    rc = cphb_evaluate_registration(source, target, option->maximum_correspondence_distance, h_T, h_result, corr_out, stream);
    // loop_ms / loop_launches: the pose loop (one kernel), not the evaluation
    h_result->loop_ms = gnc_ms;
    h_result->loop_launches = 1;
    h_result->iterations = counts[0] >= 10 ? iters : 0;
    return rc;
}
