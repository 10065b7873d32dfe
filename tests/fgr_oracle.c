/* fgr_oracle.c -- CPU restatement of registration::FastGlobalRegistration (fast_global_registration.cu) and
 * knn::BruteForceNN (bruteforce_nn.inl) under the arithmetic contract of DESIGN.md section 4.
 *
 * Test infrastructure only.  It is compiled together with oracle/oracle.c (included below, unchanged) so that the
 * 6x6 LDLT, the se(3) exponential and the 4x4 composition are the oracle's own; tests/fgr_oracle.py builds it into a
 * temporary directory.  Every FMA is an explicit fmaf() (built with -ffp-contract=off). */
#include "oracle.c"

typedef struct {
    float division_factor;
    int use_absolute_scale;
    int decrease_mu;
    float maximum_correspondence_distance;
    int iteration_number;
    float tuple_scale;
    int maximum_tuple_count;
} orc_fgr_option; /* cphb_fgr_option */

/* bruteforce_nn.inl:33-98: d2 = fma(d_k, d_k, .) over k in order from 0, d_k = query_k - ref_k; the first ref index
 * with the smallest value (strict < while scanning ascending) */
static void feature_nn_one(const float *ref, int nr, const float *q, int dim, int32_t *idx, float *d2) {
    int best = 0;
    float bd = 0.f;
    for (int r = 0; r < nr; ++r) {
        const float *f = ref + (size_t)r * dim;
        float s = 0.f;
        for (int k = 0; k < dim; ++k) {
            const float d = q[k] - f[k];
            s = fmaf(d, d, s);
        }
        if (r == 0 || s < bd) { bd = s; best = r; }
    }
    *idx = best;
    *d2 = bd;
}

void orc_feature_nn(const float *ref, int nr, const float *query, int nq, int dim, int32_t *idx, float *d2) {
#pragma omp parallel for schedule(dynamic, 16)
    for (int i = 0; i < nq; ++i) feature_nn_one(ref, nr, query + (size_t)i * dim, dim, idx + i, d2 + i);
}

/* thrust::minstd_rand, seed 1, discard(idx), three draws of uniform_int_distribution(0, ncorr - 1)
 * (thrust/random/detail/uniform_{int,real}_distribution.inl: float64 (x - min) / (1 + max - min) * ncorr) */
void orc_minstd_draws(unsigned long long idx, long long ncorr, int out[3]) {
    unsigned long long r = 1, b = 48271, e = idx;
    while (e) {
        if (e & 1) r = r * b % 2147483647ull;
        b = b * b % 2147483647ull;
        e >>= 1;
    }
    for (int k = 0; k < 3; ++k) {
        r = r * 48271ull % 2147483647ull;
        out[k] = (int)(((double)(r - 1) / 2147483646.0) * (double)ncorr);
    }
}

/* NormalizePointCloud (:197-265): out = mean_source[3], mean_target[3], scale, scale_global.  Sums: 256 strided
 * float64 partials, then the partials in order (the device's fixed order), rounded once, / (float)n. */
void orc_fgr_normalize(const float *src, int ns, const float *tgt, int nt, int use_absolute_scale, float out[8]) {
    float scale = 0.f;
    for (int c = 0; c < 2; ++c) {
        const float *p = c ? tgt : src;
        const int n = c ? nt : ns;
        double tot[3] = {0, 0, 0};
        for (int t = 0; t < 256; ++t) {
            double a[3] = {0, 0, 0};
            for (int i = t; i < n; i += 256)
                for (int k = 0; k < 3; ++k) a[k] += (double)p[3 * i + k];
            for (int k = 0; k < 3; ++k) tot[k] += a[k];
        }
        float *m = out + 3 * c;
        for (int k = 0; k < 3; ++k) m[k] = (float)tot[k] / (float)n;
        for (int i = 0; i < n; ++i) {
            const float x = p[3 * i] - m[0], y = p[3 * i + 1] - m[1], z = p[3 * i + 2] - m[2];
            const float nn = sqrtf(dot3f(x, y, z, x, y, z));
            if (nn > scale) scale = nn;
        }
    }
    out[6] = scale;
    out[7] = use_absolute_scale ? 1.f : scale;
}

static void fgr_point(const float *p, int i, const float *mean, float sg, float o[3]) {
    for (int k = 0; k < 3; ++k) o[k] = (p[3 * i + k] - mean[k]) / sg;
}

/* AdvancedMatching (:103-194).  pairs_out: 2 * maximum_tuple_count int32 (source, target); counts = pairs written,
 * mutual matches, trials, pairs of passing trials; mutual_out (optional, 2 * max(ns, nt)): the cross-checked (fi, fj)
 * pairs in fi order.  Returns 1 when the clouds were swapped. */
int orc_fgr_advanced_matching(const float *src, int ns, const float *tgt, int nt, const float *fs, const float *ft, int dim,
                              const orc_fgr_option *opt, int32_t *pairs_out, long long counts[4], int32_t *mutual_out) {
    float norm[8];
    orc_fgr_normalize(src, ns, tgt, nt, opt->use_absolute_scale, norm);
    const int swapped = nt > ns;
    const float *pi = swapped ? tgt : src, *pj = swapped ? src : tgt, *fi = swapped ? ft : fs, *fj = swapped ? fs : ft;
    const int ni = swapped ? nt : ns, nj = swapped ? ns : nt;
    const float *mi = norm + (swapped ? 3 : 0), *mj = norm + (swapped ? 0 : 3), sg = norm[7];
    int32_t *nn_i = malloc(sizeof(int32_t) * ni), *nn_j = malloc(sizeof(int32_t) * nj);
    float *d_i = malloc(sizeof(float) * ni), *d_j = malloc(sizeof(float) * nj);
    orc_feature_nn(fj, nj, fi, ni, dim, nn_i, d_i);
    orc_feature_nn(fi, ni, fj, nj, dim, nn_j, d_j);
    int32_t *mut = malloc(sizeof(int32_t) * 2 * ni);
    long long ncorr = 0;
    for (int i = 0; i < ni; ++i)
        if (nn_j[nn_i[i]] == i) { mut[2 * ncorr] = i; mut[2 * ncorr + 1] = nn_i[i]; ++ncorr; }
    if (mutual_out) memcpy(mutual_out, mut, sizeof(int32_t) * 2 * ncorr);
    const long long n_trial = ncorr * 100, cap = opt->maximum_tuple_count > 0 ? opt->maximum_tuple_count : 0;
    long long n_res = 0, written = 0;
    const float s = opt->tuple_scale;
    for (long long idx = 0; idx < n_trial; ++idx) {
        int r[3];
        orc_minstd_draws((unsigned long long)idx, ncorr, r);
        float a[3][3], b[3][3];
        for (int k = 0; k < 3; ++k) {
            fgr_point(pi, mut[2 * r[k]], mi, sg, a[k]);
            fgr_point(pj, mut[2 * r[k] + 1], mj, sg, b[k]);
        }
        int cond = 1;
        for (int k = 0; k < 3; ++k) {
            const int l = (k + 1) % 3;
            const float dx = a[k][0] - a[l][0], dy = a[k][1] - a[l][1], dz = a[k][2] - a[l][2];
            const float ex = b[k][0] - b[l][0], ey = b[k][1] - b[l][1], ez = b[k][2] - b[l][2];
            const float li = sqrtf(dot3f(dx, dy, dz, dx, dy, dz)), lj = sqrtf(dot3f(ex, ey, ez, ex, ey, ez));
            cond = cond && (li * s < lj) && (lj < li / s);
        }
        if (!cond) continue;
        for (int k = 0; k < 3; ++k, ++n_res) {
            if (written >= cap) continue;
            const int i = mut[2 * r[k]], j = mut[2 * r[k] + 1];
            pairs_out[2 * written] = swapped ? j : i;
            pairs_out[2 * written + 1] = swapped ? i : j;
            ++written;
        }
    }
    counts[0] = written;
    counts[1] = ncorr;
    counts[2] = n_trial;
    counts[3] = n_res;
    free(nn_i); free(nn_j); free(d_i); free(d_j); free(mut);
    return swapped;
}

/* OptimizePairwiseRegistration (:309-372) + GetInvTransformationOriginalScale (:376-389); trace (optional):
 * iteration_number x 16, the normalised pose after every iteration */
void orc_fgr_optimize(const float *src, int ns, const float *tgt, int nt, const int32_t *pairs, int n,
                      const orc_fgr_option *opt, float T_out[16], float *trace) {
    float norm[8];
    orc_fgr_normalize(src, ns, tgt, nt, opt->use_absolute_scale, norm);
    const float sg = norm[7];
    float *P = malloc(sizeof(float) * 3 * (n + 1)), *Q = malloc(sizeof(float) * 3 * (n + 1));
    for (int k = 0; k < n; ++k) {
        fgr_point(src, pairs[2 * k], norm, sg, P + 3 * k);
        fgr_point(tgt, pairs[2 * k + 1], norm + 3, sg, Q + 3 * k);
    }
    float trans[16], delta[16];
    identity4(trans);
    float par = sg; /* scale_global, not scale_start (:423-424) */
    for (int itr = 0; itr < opt->iteration_number; ++itr) {
        if (n < 10) {
            if (trace) memcpy(trace + 16 * itr, trans, sizeof(trans));
            continue;
        }
        double S[27] = {0};
        for (int k = 0; k < n; ++k) { /* compute_jacobian_functor (:267-307) */
            const float q0 = Q[3 * k], q1 = Q[3 * k + 1], q2 = Q[3 * k + 2];
            const float r0 = P[3 * k] - q0, r1 = P[3 * k + 1] - q1, r2 = P[3 * k + 2] - q2;
            const float temp = par / (dot3f(r0, r1, r2, r0, r1, r2) + par);
            const float s = temp * temp;
            const float J[3][6] = {{0.f, -q2, q1, -1.f, 0.f, 0.f}, {q2, 0.f, -q0, 0.f, -1.f, 0.f}, {-q1, q0, 0.f, 0.f, 0.f, -1.f}};
            const float rr[3] = {r0, r1, r2};
            int e = 0;
            for (int a = 0; a < 6; ++a)
                for (int b = a; b < 6; ++b) {
                    float v = 0.f;
                    for (int w = 0; w < 3; ++w) v = v + (J[w][a] * J[w][b]) * s;
                    S[e++] += (double)v;
                }
            for (int a = 0; a < 6; ++a) {
                float v = 0.f;
                for (int w = 0; w < 3; ++w) v = v + (J[w][a] * rr[w]) * s;
                S[21 + a] += (double)v;
            }
        }
        float A[36], b[6], x[6];
        int p = 0;
        for (int a = 0; a < 6; ++a)
            for (int c = a; c < 6; ++c) {
                const float v = -(float)S[p++];
                A[6 * a + c] = v;
                A[6 * c + a] = v;
            }
        for (int a = 0; a < 6; ++a) b[a] = (float)S[21 + a];
        ldlt6_solve(A, b, x); /* SolveLinearSystemPSD<6>(-JTJ, JTr): no symmetry / determinant check */
        se3_exp(x, delta);
        orc_matmul4(delta, trans, trans);
        if (trace) memcpy(trace + 16 * itr, trans, sizeof(trans));
        orc_transform_points(Q, n, delta);
        if (opt->decrease_mu && itr % 4 == 0 && par > opt->maximum_correspondence_distance) par = par / opt->division_factor;
    }
    const float *ms = norm, *mt = norm + 3;
    float v[3];
    for (int k = 0; k < 3; ++k) {
        const float rm = dot3f(trans[4 * k], trans[4 * k + 1], trans[4 * k + 2], mt[0], mt[1], mt[2]);
        v[k] = (-rm + trans[4 * k + 3] * sg) + ms[k];
    }
    for (int r = 0; r < 3; ++r) {
        for (int c = 0; c < 3; ++c) T_out[4 * r + c] = trans[4 * c + r];
        T_out[4 * r + 3] = -dot3f(trans[r], trans[4 + r], trans[8 + r], v[0], v[1], v[2]);
    }
    T_out[12] = T_out[13] = T_out[14] = 0.f;
    T_out[15] = 1.f;
    free(P);
    free(Q);
}
