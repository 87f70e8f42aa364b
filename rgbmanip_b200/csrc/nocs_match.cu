// Branch C of the pose fit, device part (ADA/lib/utils.py:121-195, depth_estimation_from_nocs_matches; taken when
// direct_regression = False and use_depth = False, ADA/interface_v5.py:339-349):
//   1. mutual nearest neighbours between the NOCS maps of the two views (1024 x 1024 distances, np.argmin = first minimum),
//   2. keep matches closer than 0.01 in NOCS space,
//   3. epipolar filter |x1^T F21 x2| < 1 px, F21 = K^-T [t]x R K^-1 from the UNCROPPED intrinsics and the relative pose
//      E1 E2^-1 ([t]x is stored as float32 in the reference),
//   4. linear triangulation of the surviving pixel pairs (the DLT of cv2.triangulatePoints: the right singular vector of the
//      smallest singular value of the 4 x 4 system, here the eigenvector of A^T A by cyclic Jacobi in fp64),
//   5. transform into the view-1 camera frame (left_pose @ X).
// One CTA of 1024 threads per environment, both NOCS maps in shared memory.  The median scale of the matched set is taken by
// the fit kernel in points mode (csrc/fit.cu); the PnP tail (cv2.solvePnPRansac) stays on the host.
#include "stages.cuh"

namespace adp {

constexpr int NM_P = 1024;

// np.linalg.norm(a - b) of float32 triples exactly as numpy evaluates it: sqrt of the sequential fp32 sum of squares
__device__ __forceinline__ float nocs_dist(const float3& a, const float3& b) {
    const float dx = __fsub_rn(a.x, b.x), dy = __fsub_rn(a.y, b.y), dz = __fsub_rn(a.z, b.z);
    return __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz)));
}

// image coordinates of sampled crop pixel `pix` (interface_v5.py:136-145): x / ratio + cmin, y / ratio + rmin.  `ratio` is a
// np.float64 scalar in the reference (numpy-integer window bounds), so under NumPy >= 2 the arithmetic is float64; the PnP gets
// the float32 rounding of it (interface_v5.py:348 astype)
__device__ __forceinline__ double2 crop_to_image(int pix, int S, int rmin, int rmax, int cmin) {
    const double ratio = (double)S / (double)(rmax - rmin);
    const int y = pix / S, x = pix - y * S;
    return make_double2(__dadd_rn(__ddiv_rn((double)x, ratio), (double)cmin), __dadd_rn(__ddiv_rn((double)y, ratio), (double)rmin));
}

// eigenvector of the smallest eigenvalue of the symmetric 4 x 4 matrix m (cyclic Jacobi, fp64)
__device__ void smallest_eigvec4(double m[4][4], double* out) {
    double v[4][4];
    for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) v[i][j] = (i == j) ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 30; ++sweep) {
        double off = 0.0;
        for (int p = 0; p < 4; ++p) for (int q = p + 1; q < 4; ++q) off += m[p][q] * m[p][q];
        double diag = 0.0;
        for (int p = 0; p < 4; ++p) diag += m[p][p] * m[p][p];
        if (off <= 1e-30 * diag) break;
        for (int p = 0; p < 4; ++p)
            for (int q = p + 1; q < 4; ++q) {
                if (m[p][q] == 0.0) continue;
                const double theta = (m[q][q] - m[p][p]) / (2.0 * m[p][q]);
                const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
                for (int k = 0; k < 4; ++k) {      // columns p, q of m
                    const double a = m[k][p], b = m[k][q];
                    m[k][p] = c * a - s * b; m[k][q] = s * a + c * b;
                }
                for (int k = 0; k < 4; ++k) {      // rows p, q of m
                    const double a = m[p][k], b = m[q][k];
                    m[p][k] = c * a - s * b; m[q][k] = s * a + c * b;
                }
                for (int k = 0; k < 4; ++k) {
                    const double a = v[k][p], b = v[k][q];
                    v[k][p] = c * a - s * b; v[k][q] = s * a + c * b;
                }
            }
    }
    int best = 0;
    for (int i = 1; i < 4; ++i) if (m[i][i] < m[best][best]) best = i;
    for (int k = 0; k < 4; ++k) out[k] = v[k][best];
}

__global__ void __launch_bounds__(NM_P)
nocs_match_kernel(const float* __restrict__ nocs1, const float* __restrict__ nocs2, const int* __restrict__ choose1,
                  const int* __restrict__ choose2, const int* __restrict__ win1, const int* __restrict__ win2,
                  const double* __restrict__ K, const double* __restrict__ E1, const double* __restrict__ E2,
                  const uint8_t* __restrict__ valid, int S, float* __restrict__ pts2d1, float* __restrict__ pts_cam,
                  float* __restrict__ nocs_m, int* __restrict__ count, int* __restrict__ match_ids, int P) {
    __shared__ float3 n1[NM_P], n2[NM_P];
    __shared__ int l2r[NM_P], r2l[NM_P];
    __shared__ int wsum[32];
    __shared__ double F21[9], Pm[2][12], Lp[16];
    const int b = blockIdx.x, i = threadIdx.x;
    const bool inr = i < P;
    if (inr) {
        const float* a = nocs1 + ((size_t)b * P + i) * 3;
        const float* c = nocs2 + ((size_t)b * P + i) * 3;
        n1[i] = make_float3(a[0], a[1], a[2]);
        n2[i] = make_float3(c[0], c[1], c[2]);
    }
    const int* w1 = win1 + 4 * b;
    const int* w2 = win2 + 4 * b;
    double2 px1 = make_double2(0.0, 0.0);
    if (inr) {
        px1 = crop_to_image(choose1[(size_t)b * P + i], S, w1[0], w1[1], w1[2]);
        pts2d1[((size_t)b * P + i) * 2] = (float)px1.x;
        pts2d1[((size_t)b * P + i) * 2 + 1] = (float)px1.y;
    }
    if (valid && !valid[b]) {
        if (i == 0) count[b] = 0;
        return;
    }
    if (i == 0) {
        // relative pose E1 E2^-1, F21 = K^-T [t]x R K^-1 (utils.py:146-158), projections P = K E[:3] (interface_v5.py:340-343)
        const double* k = K + 9 * b;
        const double* e1 = E1 + 16 * b;
        const double* e2 = E2 + 16 * b;
        double inv2[16], rel[16], Ki[9];
        invert4x4(e2, inv2);
        for (int r = 0; r < 4; ++r)
            for (int c = 0; c < 4; ++c) {
                double s = 0;
                for (int q = 0; q < 4; ++q) s += e1[4 * r + q] * inv2[4 * q + c];
                rel[4 * r + c] = s;
            }
        {   // inverse of the 3 x 3 intrinsics (general, by cofactors)
            const double a = k[0], bq = k[1], c = k[2], d = k[3], e = k[4], f = k[5], g = k[6], h = k[7], ii = k[8];
            const double det = a * (e * ii - f * h) - bq * (d * ii - f * g) + c * (d * h - e * g);
            Ki[0] = (e * ii - f * h) / det; Ki[1] = (c * h - bq * ii) / det; Ki[2] = (bq * f - c * e) / det;
            Ki[3] = (f * g - d * ii) / det; Ki[4] = (a * ii - c * g) / det; Ki[5] = (c * d - a * f) / det;
            Ki[6] = (d * h - e * g) / det; Ki[7] = (bq * g - a * h) / det; Ki[8] = (a * e - bq * d) / det;
        }
        const double t0 = rel[3], t1 = rel[7], t2 = rel[11];
        const double tx[9] = {0.0, (double)(float)(-t2), (double)(float)t1, (double)(float)t2, 0.0, (double)(float)(-t0),
                              (double)(float)(-t1), (double)(float)t0, 0.0};
        double A[9], Bm[9], Cm[9];
        for (int r = 0; r < 3; ++r)            // A = K^-T tx
            for (int c = 0; c < 3; ++c) { double s = 0; for (int q = 0; q < 3; ++q) s += Ki[3 * q + r] * tx[3 * q + c]; A[3 * r + c] = s; }
        for (int r = 0; r < 3; ++r)            // B = A R
            for (int c = 0; c < 3; ++c) { double s = 0; for (int q = 0; q < 3; ++q) s += A[3 * r + q] * rel[4 * q + c]; Bm[3 * r + c] = s; }
        for (int r = 0; r < 3; ++r)            // F = B K^-1
            for (int c = 0; c < 3; ++c) { double s = 0; for (int q = 0; q < 3; ++q) s += Bm[3 * r + q] * Ki[3 * q + c]; Cm[3 * r + c] = s; }
        for (int q = 0; q < 9; ++q) F21[q] = Cm[q];
        for (int v = 0; v < 2; ++v) {
            const double* e = v ? e2 : e1;
            for (int r = 0; r < 3; ++r)
                for (int c = 0; c < 4; ++c) Pm[v][4 * r + c] = k[3 * r] * e[c] + k[3 * r + 1] * e[4 + c] + k[3 * r + 2] * e[8 + c];
        }
        for (int q = 0; q < 16; ++q) Lp[q] = e1[q];
    }
    __syncthreads();
    // ---- 1. nearest neighbours both ways (first minimum, like np.argmin)
    if (inr) {
        float best = INFINITY, bestr = INFINITY;
        int bj = 0, bi = 0;
        const float3 a = n1[i], c = n2[i];
        for (int j = 0; j < P; ++j) {
            const float d = nocs_dist(a, n2[j]);        // dis[i, j]
            if (d < best) { best = d; bj = j; }
            const float e = nocs_dist(n1[j], c);        // dis[j, i]
            if (e < bestr) { bestr = e; bi = j; }
        }
        l2r[i] = bj;
        r2l[i] = bi;
    }
    __syncthreads();
    // ---- 2./3. mutual check, NOCS distance, epipolar distance
    bool keep = false;
    int j = 0;
    double2 px2 = make_double2(0.0, 0.0);
    if (inr) {
        j = l2r[i];
        keep = (r2l[j] == i) && (nocs_dist(n1[i], n2[j]) < 0.01f);
        if (keep) {
            px2 = crop_to_image(choose2[(size_t)b * P + j], S, w2[0], w2[1], w2[2]);
            // (x1^T F21) x2 in fp64 with x = (u, v, 1)
            const double u1 = px1.x, v1 = px1.y, u2 = px2.x, v2 = px2.y;
            const double r0 = u1 * F21[0] + v1 * F21[3] + F21[6], r1 = u1 * F21[1] + v1 * F21[4] + F21[7], r2 = u1 * F21[2] + v1 * F21[5] + F21[8];
            keep = fabs(r0 * u2 + r1 * v2 + r2) < 1.0;
        }
    }
    // ---- compaction in ascending view-1 index (the order of numpy's boolean masking)
    const unsigned int bal = __ballot_sync(0xffffffffu, keep);
    const int lane = i & 31, w = i >> 5;
    if (lane == 0) wsum[w] = __popc(bal);
    __syncthreads();
    if (w == 0) {
        int s = wsum[lane];
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += y;
        }
        wsum[lane] = s;                                  // inclusive
    }
    __syncthreads();
    const int pos = (w > 0 ? wsum[w - 1] : 0) + __popc(bal & ((1u << lane) - 1u));
    if (i == 0) count[b] = wsum[31];
    if (!keep) return;
    // ---- 4. DLT triangulation: rows x P[2] - P[0], y P[2] - P[1] for both views; 5. into the view-1 camera frame
    double A[4][4];
    {
        const double xs[2] = {px1.x, px2.x}, ys[2] = {px1.y, px2.y};
        for (int v = 0; v < 2; ++v)
            for (int c = 0; c < 4; ++c) {
                A[2 * v][c] = xs[v] * Pm[v][8 + c] - Pm[v][c];
                A[2 * v + 1][c] = ys[v] * Pm[v][8 + c] - Pm[v][4 + c];
            }
    }
    double M[4][4];
    for (int r = 0; r < 4; ++r)
        for (int c = 0; c < 4; ++c) { double s = 0; for (int q = 0; q < 4; ++q) s += A[q][r] * A[q][c]; M[r][c] = s; }
    double X[4];
    smallest_eigvec4(M, X);
    const double xw = X[0] / X[3], yw = X[1] / X[3], zw = X[2] / X[3];
    float* o = pts_cam + ((size_t)b * P + pos) * 3;
    for (int r = 0; r < 3; ++r) o[r] = (float)(Lp[4 * r] * xw + Lp[4 * r + 1] * yw + Lp[4 * r + 2] * zw + Lp[4 * r + 3]);
    float* nn = nocs_m + ((size_t)b * P + pos) * 3;
    nn[0] = n1[i].x; nn[1] = n1[i].y; nn[2] = n1[i].z;
    if (match_ids) { match_ids[((size_t)b * P + pos) * 2] = i; match_ids[((size_t)b * P + pos) * 2 + 1] = j; }
}

int nocs_match_run(const float* nocs1, const float* nocs2, const int* choose1, const int* choose2, const int* win1, const int* win2,
                   const double* K, const double* E1, const double* E2, const uint8_t* valid, int S, float* pts2d1, float* pts_cam,
                   float* nocs_m, int* count, int* match_ids, int B, int P, cudaStream_t stream) {
    ADP_CHECK_ARG(P == NM_P, "1024 sampled pixels per view");
    if (B == 0) return ADP_OK;
    nocs_match_kernel<<<B, NM_P, 0, stream>>>(nocs1, nocs2, choose1, choose2, win1, win2, K, E1, E2, valid, S, pts2d1, pts_cam,
                                             nocs_m, count, match_ids, P);
    ADP_CUDA(cudaGetLastError());
    return ADP_OK;
}

}  // namespace adp
