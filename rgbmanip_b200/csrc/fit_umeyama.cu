// Pose fit, branch B of ADA/interface_v5.py:322-338 (direct_regression = False, use_depth = True):
// RANSAC over 5-point Umeyama similarity hypotheses + refit on the best inlier set
// (ADA/lib/align.py:44-102 estimateSimilarityTransform, :10-41 estimateSimilarityUmeyama), followed by the same
// box construction as branch A (interface_v5.py:354-374).  One CTA per environment, everything in fp64 like numpy.
// The 128 x 5 sample indices come either from a caller-supplied table (exact replay of a numpy stream in the parity
// tests) or from a counter-based hash (same distribution as np.random.randint, different stream).
#include "stages.cuh"

namespace adp {

constexpr int UM_THREADS = 256;
constexpr int UM_MAXP = 1024;
constexpr int UM_ITERS = 128;

struct Sim3 {
    double s;
    double R[9];
    double t[3];
    bool ok;
};

__device__ inline void jacobi_eig3(double a[3][3], double v[3][3]) {
    // symmetric 3x3 eigen-decomposition by cyclic Jacobi rotations: a -> diagonal, v = eigenvectors (columns)
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) v[i][j] = (i == j) ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 30; ++sweep) {
        const double off = fabs(a[0][1]) + fabs(a[0][2]) + fabs(a[1][2]);
        const double diag = fabs(a[0][0]) + fabs(a[1][1]) + fabs(a[2][2]);
        if (off <= 1e-18 * diag || off == 0.0) break;
        for (int p = 0; p < 2; ++p)
            for (int q = p + 1; q < 3; ++q) {
                if (a[p][q] == 0.0) continue;
                const double theta = (a[q][q] - a[p][p]) / (2.0 * a[p][q]);
                const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
                for (int k = 0; k < 3; ++k) {
                    const double akp = a[k][p], akq = a[k][q];
                    a[k][p] = c * akp - s * akq; a[k][q] = s * akp + c * akq;
                }
                for (int k = 0; k < 3; ++k) {
                    const double apk = a[p][k], aqk = a[q][k];
                    a[p][k] = c * apk - s * aqk; a[q][k] = s * apk + c * aqk;
                }
                for (int k = 0; k < 3; ++k) {
                    const double vkp = v[k][p], vkq = v[k][q];
                    v[k][p] = c * vkp - s * vkq; v[k][q] = s * vkp + c * vkq;
                }
            }
    }
}

__device__ inline double det3(const double m[3][3]) {
    return m[0][0] * (m[1][1] * m[2][2] - m[1][2] * m[2][1]) - m[0][1] * (m[1][0] * m[2][2] - m[1][2] * m[2][0]) +
           m[0][2] * (m[1][0] * m[2][1] - m[1][1] * m[2][0]);
}

// Umeyama from sufficient statistics: centroids sc/tc, covariance cov = E[(t - tc)(s - sc)^T], varP = sum of source variances
__device__ inline Sim3 umeyama_from_stats(const double sc[3], const double tc[3], const double cov[3][3], double varP) {
    Sim3 r;
    r.ok = true;
    // SVD of cov via the eigen-decomposition of cov^T cov
    double b[3][3], V[3][3];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) b[i][j] = cov[0][i] * cov[0][j] + cov[1][i] * cov[1][j] + cov[2][i] * cov[2][j];
    jacobi_eig3(b, V);
    double lam[3] = {b[0][0], b[1][1], b[2][2]};
    int ord[3] = {0, 1, 2};
    for (int i = 0; i < 2; ++i)
        for (int j = i + 1; j < 3; ++j) if (lam[ord[j]] > lam[ord[i]]) { int t = ord[i]; ord[i] = ord[j]; ord[j] = t; }
    double Vs[3][3], sig[3], U[3][3];
    for (int c = 0; c < 3; ++c) {
        sig[c] = sqrt(fmax(lam[ord[c]], 0.0));
        for (int k = 0; k < 3; ++k) Vs[k][c] = V[k][ord[c]];
    }
    for (int c = 0; c < 2; ++c) {
        double n = 0;
        for (int k = 0; k < 3; ++k) { U[k][c] = cov[k][0] * Vs[0][c] + cov[k][1] * Vs[1][c] + cov[k][2] * Vs[2][c]; n += U[k][c] * U[k][c]; }
        n = sqrt(n);
        if (!(n > 0.0)) { r.ok = false; n = 1.0; }
        for (int k = 0; k < 3; ++k) U[k][c] /= n;
    }
    // third left vector: along cov * v2 when that is numerically meaningful, else the cross product (sign fixed below)
    double u2[3] = {U[1][0] * U[2][1] - U[2][0] * U[1][1], U[2][0] * U[0][1] - U[0][0] * U[2][1], U[0][0] * U[1][1] - U[1][0] * U[0][1]};
    double w2[3], dot = 0;
    for (int k = 0; k < 3; ++k) { w2[k] = cov[k][0] * Vs[0][2] + cov[k][1] * Vs[1][2] + cov[k][2] * Vs[2][2]; dot += w2[k] * u2[k]; }
    const double sgn = (dot < 0.0) ? -1.0 : 1.0;
    for (int k = 0; k < 3; ++k) U[k][2] = sgn * u2[k];
    double Vh[3][3];
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) Vh[i][j] = Vs[j][i];
    if (det3(U) * det3(Vh) < 0.0) {          // align.py:25-28
        sig[2] = -sig[2];
        for (int k = 0; k < 3; ++k) U[k][2] = -U[k][2];
    }
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) r.R[3 * i + j] = U[i][0] * Vh[0][j] + U[i][1] * Vh[1][j] + U[i][2] * Vh[2][j];
    r.s = (sig[0] + sig[1] + sig[2]) / varP;
    for (int i = 0; i < 3; ++i) r.t[i] = tc[i] - r.s * (r.R[3 * i] * sc[0] + r.R[3 * i + 1] * sc[1] + r.R[3 * i + 2] * sc[2]);
    if (!isfinite(r.s)) r.ok = false;
    return r;
}

__device__ inline Sim3 umeyama_small(const double* S, const double* T, const int* idx, int n) {
    double sc[3] = {0, 0, 0}, tc[3] = {0, 0, 0};
    for (int i = 0; i < n; ++i) for (int k = 0; k < 3; ++k) { sc[k] += S[3 * idx[i] + k]; tc[k] += T[3 * idx[i] + k]; }
    for (int k = 0; k < 3; ++k) { sc[k] /= n; tc[k] /= n; }
    double cov[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}}, varP = 0;
    for (int i = 0; i < n; ++i) {
        double ds[3], dt[3];
        for (int k = 0; k < 3; ++k) { ds[k] = S[3 * idx[i] + k] - sc[k]; dt[k] = T[3 * idx[i] + k] - tc[k]; varP += ds[k] * ds[k]; }
        for (int a = 0; a < 3; ++a) for (int b = 0; b < 3; ++b) cov[a][b] += dt[a] * ds[b];
    }
    for (int a = 0; a < 3; ++a) for (int b = 0; b < 3; ++b) cov[a][b] /= n;
    varP /= n;
    return umeyama_from_stats(sc, tc, cov, varP);
}

__device__ __forceinline__ uint32_t um_mix(uint32_t x) {
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    return x;
}

__device__ double block_sum_d(double v, double* red) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0;
    for (int i = 0; i < UM_THREADS / 32; ++i) s += red[i];
    __syncthreads();
    return s;
}

__global__ void __launch_bounds__(UM_THREADS)
fit_umeyama_kernel(const float* __restrict__ nocs, const float* __restrict__ depth, const int* __restrict__ choose,
                   const double* __restrict__ Kp, const double* __restrict__ E, const uint8_t* __restrict__ valid,
                   const int* __restrict__ rand_idx, uint32_t seed, double* __restrict__ bbox, double* __restrict__ scale_out,
                   double* __restrict__ rot_out, double* __restrict__ trans_out, int P, int S_img) {
    extern __shared__ double smd[];
    double* S = smd;                    // [P][3] source = NOCS
    double* T = smd + 3 * UM_MAXP;      // [P][3] target = camera points
    double* hyp = T + 3 * UM_MAXP;      // [128][13]  s*R (9), t (3), scale
    __shared__ double red[UM_THREADS / 32];
    __shared__ int s_int[4];
    __shared__ double s_best;
    const int b = blockIdx.x, tid = threadIdx.x;
    double* out = bbox + (size_t)b * 24;
    auto sentinel = [&]() {
        if (tid < 24) out[tid] = 10.0 + (double)(((tid / 3) >> (2 - tid % 3)) & 1);
        if (tid == 0 && scale_out) scale_out[b] = nan("");
    };
    if (valid && !valid[b]) { sentinel(); return; }
    const double* k = Kp + 9 * b;
    for (int i = tid; i < P; i += UM_THREADS) {
        const int pix = choose[(size_t)b * P + i];
        const double z = (double)depth[(size_t)b * P + i];
        const int y = pix / S_img, x = pix - y * S_img;
        T[3 * i] = ((double)x - k[2]) * z / k[0];
        T[3 * i + 1] = ((double)y - k[5]) * z / k[4];
        T[3 * i + 2] = z;
        for (int c = 0; c < 3; ++c) S[3 * i + c] = (double)nocs[((size_t)b * P + i) * 3 + c];
    }
    __syncthreads();
    // source centroid and diameter -> inlier threshold (align.py:53-58)
    double acc[3] = {0, 0, 0};
    for (int i = tid; i < P; i += UM_THREADS) for (int c = 0; c < 3; ++c) acc[c] += S[3 * i + c];
    double sc0[3];
    for (int c = 0; c < 3; ++c) sc0[c] = block_sum_d(acc[c], red) / P;
    double mx = 0;
    for (int i = tid; i < P; i += UM_THREADS) {
        const double dx = S[3 * i] - sc0[0], dy = S[3 * i + 1] - sc0[1], dz = S[3 * i + 2] - sc0[2];
        mx = fmax(mx, sqrt(dx * dx + dy * dy + dz * dz));
    }
    for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((tid & 31) == 0) red[tid >> 5] = mx;
    __syncthreads();
    mx = red[0];
    for (int i = 1; i < UM_THREADS / 32; ++i) mx = fmax(mx, red[i]);
    __syncthreads();
    const double inlier_t = 2.0 * mx / 10.0;

    // all 128 five-point hypotheses are independent of each other: one thread each
    if (tid < UM_ITERS) {
        int idx[5];
        for (int q = 0; q < 5; ++q)
            idx[q] = rand_idx ? rand_idx[((size_t)b * UM_ITERS + tid) * 5 + q]
                              : (int)(um_mix(seed ^ um_mix((uint32_t)(b * UM_ITERS + tid) * 5u + q + 0x9e3779b9u)) % (uint32_t)P);
        const Sim3 h = umeyama_small(S, T, idx, 5);
        double* o = hyp + 13 * tid;
        for (int q = 0; q < 9; ++q) o[q] = h.s * h.R[q];
        for (int q = 0; q < 3; ++q) o[9 + q] = h.t[q];
        o[12] = h.ok ? h.s : nan("");
    }
    if (tid == 0) { s_int[0] = 0; s_int[1] = -1; s_int[2] = 0; s_int[3] = 0; s_best = 0.0; }   // best inlier count, best hypothesis, scratch
    __syncthreads();

    // sequential scan of the hypotheses with the reference's early exit (align.py:68-87)
    for (int it = 0; it < UM_ITERS; ++it) {
        const double* h = hyp + 13 * it;
        const double thr = h[12] * inlier_t;       // NaN threshold -> no inliers, like a failed comparison in numpy
        int cnt = 0;
        for (int i = tid; i < P; i += UM_THREADS) {
            const double sx = S[3 * i], sy = S[3 * i + 1], sz = S[3 * i + 2];
            const double rx = T[3 * i] - (h[0] * sx + h[1] * sy + h[2] * sz + h[9]);
            const double ry = T[3 * i + 1] - (h[3] * sx + h[4] * sy + h[5] * sz + h[10]);
            const double rz = T[3 * i + 2] - (h[6] * sx + h[7] * sy + h[8] * sz + h[11]);
            cnt += sqrt(rx * rx + ry * ry + rz * rz) < thr;
        }
        for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        if ((tid & 31) == 0) atomicAdd(&s_int[2], cnt);
        __syncthreads();
        if (tid == 0) {
            const int n = s_int[2];
            s_int[2] = 0;
            if (n > s_int[0]) { s_int[0] = n; s_int[1] = it; s_best = (double)n / (double)P; }
            const double r5 = s_best * s_best * s_best * s_best * s_best;
            s_int[3] = (1.0 - pow(1.0 - r5, (double)it)) > 0.99 ? 1 : 0;
        }
        __syncthreads();
        if (s_int[3]) break;
    }
    __syncthreads();
    const int best_it = s_int[1];
    if (s_best < 0.1 || best_it < 0) { sentinel(); return; }     // align.py:89-91 -> interface_v5.py:351-352

    // refit on the inliers of the best hypothesis (align.py:93-95)
    const double* h = hyp + 13 * best_it;
    const double thr = h[12] * inlier_t;
    auto is_inlier = [&](int i) {
        const double sx = S[3 * i], sy = S[3 * i + 1], sz = S[3 * i + 2];
        const double rx = T[3 * i] - (h[0] * sx + h[1] * sy + h[2] * sz + h[9]);
        const double ry = T[3 * i + 1] - (h[3] * sx + h[4] * sy + h[5] * sz + h[10]);
        const double rz = T[3 * i + 2] - (h[6] * sx + h[7] * sy + h[8] * sz + h[11]);
        return sqrt(rx * rx + ry * ry + rz * rz) < thr;
    };
    double a6[6] = {0, 0, 0, 0, 0, 0};
    double cntd = 0;
    for (int i = tid; i < P; i += UM_THREADS)
        if (is_inlier(i)) { cntd += 1.0; for (int c = 0; c < 3; ++c) { a6[c] += S[3 * i + c]; a6[3 + c] += T[3 * i + c]; } }
    const double n_in = block_sum_d(cntd, red);
    double scn[3], tcn[3];
    for (int c = 0; c < 3; ++c) { scn[c] = block_sum_d(a6[c], red) / n_in; tcn[c] = block_sum_d(a6[3 + c], red) / n_in; }
    double cv[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}, vp = 0;
    for (int i = tid; i < P; i += UM_THREADS)
        if (is_inlier(i)) {
            double ds[3], dt[3];
            for (int c = 0; c < 3; ++c) { ds[c] = S[3 * i + c] - scn[c]; dt[c] = T[3 * i + c] - tcn[c]; vp += ds[c] * ds[c]; }
            for (int a = 0; a < 3; ++a) for (int c = 0; c < 3; ++c) cv[3 * a + c] += dt[a] * ds[c];
        }
    double cov[3][3];
    for (int q = 0; q < 9; ++q) cov[q / 3][q % 3] = block_sum_d(cv[q], red) / n_in;
    const double varP = block_sum_d(vp, red) / n_in;
    // half extents of the box: max |nocs| (interface_v5.py:355)
    double hmax[3] = {0, 0, 0};
    for (int i = tid; i < P; i += UM_THREADS) for (int c = 0; c < 3; ++c) hmax[c] = fmax(hmax[c], fabs(S[3 * i + c]));
    double half3[3];
    for (int c = 0; c < 3; ++c) {
        double m = hmax[c];
        for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
        if ((tid & 31) == 0) red[tid >> 5] = m;
        __syncthreads();
        m = red[0];
        for (int i = 1; i < UM_THREADS / 32; ++i) m = fmax(m, red[i]);
        __syncthreads();
        half3[c] = m;
    }
    if (tid == 0) {
        const Sim3 f = umeyama_from_stats(scn, tcn, cov, varP);
        if (scale_out) scale_out[b] = f.s;
        if (rot_out) for (int q = 0; q < 9; ++q) rot_out[9 * b + q] = f.R[q];
        if (trans_out) for (int q = 0; q < 3; ++q) trans_out[3 * b + q] = f.t[q];
        double inv[16];
        bool fin = f.ok && invert4x4(E + 16 * b, inv);
        for (int i = 0; i < 16 && fin; ++i) fin = isfinite(inv[i]);
        double cam[8][3];
        for (int c = 0; c < 8 && fin; ++c) {
            const double sx = (c & 2) ? -1.0 : 1.0, sy = (c & 4) ? -1.0 : 1.0, sz = (c & 1) ? -1.0 : 1.0;
            const double p[3] = {sx * half3[0] * f.s, sy * half3[1] * f.s, sz * half3[2] * f.s};
            for (int r = 0; r < 3; ++r) {
                // the reference stores R and t in a float32 4x4 (interface_v5.py:359-361)
                cam[c][r] = (double)(float)f.R[3 * r] * p[0] + (double)(float)f.R[3 * r + 1] * p[1] + (double)(float)f.R[3 * r + 2] * p[2] +
                            (double)(float)f.t[r];
                fin = fin && isfinite(cam[c][r]);
            }
        }
        if (fin) {
            for (int c = 0; c < 8; ++c)
                for (int r = 0; r < 3; ++r)
                    out[3 * c + r] = inv[4 * r] * cam[c][0] + inv[4 * r + 1] * cam[c][1] + inv[4 * r + 2] * cam[c][2] + inv[4 * r + 3];
        } else {
            for (int i = 0; i < 24; ++i) out[i] = 10.0 + (double)(((i / 3) >> (2 - i % 3)) & 1);
        }
    }
}

int fit_umeyama_run(const float* nocs, const float* depth, const int* choose, const double* Kp, const double* E, const uint8_t* valid,
                    const int* rand_idx, uint32_t seed, double* bbox, double* scale_out, double* rot_out, double* trans_out, int B,
                    int P, int S, cudaStream_t stream) {
    ADP_CHECK_ARG(P <= UM_MAXP, "at most 1024 points per env");
    if (B == 0) return ADP_OK;
    const size_t smem = (size_t)(6 * UM_MAXP + 13 * UM_ITERS) * sizeof(double);
    static int attr[kMaxDevices];
    ADP_TRY(ensure_dyn_smem(fit_umeyama_kernel, (int)smem, attr));
    fit_umeyama_kernel<<<B, UM_THREADS, smem, stream>>>(nocs, depth, choose, Kp, E, valid, rand_idx, seed, bbox, scale_out, rot_out,
                                                       trans_out, P, S);
    ADP_CUDA(cudaGetLastError());
    return ADP_OK;
}

}  // namespace adp
