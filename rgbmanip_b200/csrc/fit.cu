// Per-environment pose fit, branch A of ADA/interface_v5.py:318-321 (the one every shipped config takes):
//   back-projection (ADA/lib/utils.py:99-112), scale = exact median over all point pairs of
//   |dc| / |dn| with |dn| > 0.01 and |dc| < 0.3 (utils.py:76-96), t = mean(c) - mean(s R n) (utils.py:114-119),
//   box corners + world transform + finite check (interface_v5.py:354-374, utils.py:40-74).
// One thread-block CLUSTER of 4 CTAs per environment: every CTA keeps the 1024 points in shared memory and owns a quarter
// of the pairs.  The median is an exact radix select over the pair ratios (11 + 11 + 10 bits of the positive-float bit
// pattern) of the SQUARED ratio q = |dc|^2 / |dn|^2 (monotone in the ratio, so the same pair is selected; the square root
// is taken once, in double, on the selected value).  q is RECOMPUTED in every pass from the points in shared memory
// (explicitly rounded intrinsics in a fixed order, so every pass sees the same bits): ~30 instructions per pair instead of a
// 2 MB-per-environment scratch row that is written once and re-read three times.  The per-CTA histograms are summed over distributed shared memory, so every CTA
// of the cluster derives the same digit without a broadcast.
#include "stages.cuh"

#include <cooperative_groups.h>

namespace adp {

namespace cg = cooperative_groups;

constexpr int FIT_THREADS = 512;
constexpr int FIT_G = 4;        // CTAs per environment (cluster size)
constexpr int FIT_MAXP = 1024;
constexpr int FIT_KB = 4;       // pair offsets evaluated per batch

__device__ __forceinline__ float block_reduce_sum(float v, float* red) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    float s = 0.f;
    for (int i = 0; i < FIT_THREADS / 32; ++i) s += red[i];
    __syncthreads();
    return s;
}
__device__ __forceinline__ float block_reduce_max(float v, float* red) {
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    float s = red[0];
    for (int i = 1; i < FIT_THREADS / 32; ++i) s = fmaxf(s, red[i]);
    __syncthreads();
    return s;
}

// squared ratio |dc|^2 / |dn|^2 of one pair, or a negative value when the pair is filtered out (utils.py:84-92:
// |dn| > 0.01 and |dc| < 0.3, tested on the squares).  Explicitly rounded intrinsics: no FMA contraction freedom, so
// re-evaluations are bit-identical.  Point layout: a = (cx, cy, cz, nx), a2 = (ny, nz).
__device__ __forceinline__ float pair_q(const float4& a, const float2& a2, const float4& b, const float2& b2) {
    const float dnx = __fsub_rn(a.w, b.w), dny = __fsub_rn(a2.x, b2.x), dnz = __fsub_rn(a2.y, b2.y);
    const float dn2 = __fmaf_rn(dnz, dnz, __fmaf_rn(dny, dny, __fmul_rn(dnx, dnx)));
    const float dcx = __fsub_rn(a.x, b.x), dcy = __fsub_rn(a.y, b.y), dcz = __fsub_rn(a.z, b.z);
    const float dc2 = __fmaf_rn(dcz, dcz, __fmaf_rn(dcy, dcy, __fmul_rn(dcx, dcx)));
    return (dn2 > 1e-4f && dc2 < 0.09f) ? __fdividef(dc2, dn2) : -1.f;
}

// warp-aggregated shared-memory histogram increment (the leading digit of most ratios falls into a handful of bins)
__device__ __forceinline__ void hist_add(unsigned int* hist, unsigned int bin, bool active) {
    const unsigned int act = __ballot_sync(0xffffffffu, active);
    if (!active) return;
    const unsigned int peers = __match_any_sync(act, bin);
    if ((threadIdx.x & 31) == (unsigned)(__ffs(peers) - 1)) atomicAdd(&hist[bin], (unsigned int)__popc(peers));
}

constexpr int FIT_BINS = 2048;   // 11 + 11 + 10 bit radix passes over the positive-float bit pattern

// Every unordered pair exactly once, perfectly balanced: point j is paired with (j + k) mod P for k = 1 .. P/2 (for even
// P the last offset k = P/2 only from j < P/2).  A thread keeps its own points j = tid, tid + 512 in registers and reads
// the partner from shared memory (consecutive lanes -> consecutive words); CTA `rank` of the cluster owns the offsets
// k = 1 + rank, 1 + rank + FIT_G, ...
template <typename F>
__device__ __forceinline__ void fit_for_each_ratio(int P, int rank, const float4* pa, const float2* pb, F&& body) {
    const int tid = threadIdx.x;
    float4 own[2];
    float2 own2[2];
    bool have[2];
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        const int j = tid + q * FIT_THREADS;
        have[q] = j < P;
        own[q] = pa[have[q] ? j : 0];
        own2[q] = pb[have[q] ? j : 0];
    }
    const int kmax = P / 2;
    // batches of FIT_KB offsets: all shared-memory loads and the arithmetic of a batch are issued before its histogram
    // atomics (which the compiler will not move loads across), so several pairs are in flight per thread
    for (int k0 = 1 + rank; k0 <= kmax; k0 += FIT_G * FIT_KB) {
        float r[FIT_KB][2];
#pragma unroll
        for (int u = 0; u < FIT_KB; ++u) {
            const int k = k0 + u * FIT_G;
            const bool kval = k <= kmax;
            const bool half_only = (2 * k == P);
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const int j = tid + q * FIT_THREADS;
                int o = j + k;
                if (o >= P) o -= P;
                const bool act = kval && have[q] && !(half_only && j >= k);
                const int oo = act ? o : 0;
                const float v = pair_q(own[q], own2[q], pa[oo], pb[oo]);
                r[u][q] = act ? v : -1.f;
            }
        }
#pragma unroll
        for (int u = 0; u < FIT_KB; ++u)
#pragma unroll
            for (int q = 0; q < 2; ++q) body(r[u][q]);      // called by every thread of the warp (negative = no pair / filtered out)
    }
}

__global__ void __cluster_dims__(FIT_G, 1, 1) __launch_bounds__(FIT_THREADS, 2)
fit_kernel(const float* __restrict__ nocs, const float* __restrict__ depth, const int* __restrict__ choose,
           const double* __restrict__ Kp, const float* __restrict__ R, const double* __restrict__ E, const uint8_t* __restrict__ valid,
           double* __restrict__ bbox, double* __restrict__ scale_out, double* __restrict__ trans_out,
           const float* __restrict__ pts_cam, const int* __restrict__ pts_count, int P, int S) {
    __shared__ float4 pa[FIT_MAXP];              // (cx, cy, cz, nx): camera-frame point + first NOCS coordinate
    __shared__ float2 pb[FIT_MAXP];              // (ny, nz)
    __shared__ unsigned int hist[FIT_BINS];      // this CTA's digit histogram (read by the whole cluster)
    __shared__ unsigned int htot[FIT_BINS];      // cluster-wide sum
    __shared__ float red[FIT_THREADS / 32];
    __shared__ unsigned int s_part[2];           // this CTA's partial counts: [0] valid ratios, [1] ratios below the median candidate
    __shared__ float s_pmax;                     // this CTA's largest ratio below the median candidate
    __shared__ unsigned int s_sel[3];
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const int b = blockIdx.x / FIT_G, tid = threadIdx.x;
    double* out = bbox + (size_t)b * 24;
    const bool ok_in = !valid || valid[b];
    if (!ok_in) {      // uniform over the cluster
        if (rank == 0) {
            if (tid < 24) out[tid] = 10.0 + (double)((tid / 3 >> (2 - tid % 3)) & 1);   // unit cube + 10 (interface_v5.py:232-241)
            if (tid == 0) { if (scale_out) scale_out[b] = nan(""); }
        }
        return;
    }
    const double* k = Kp + 9 * b;
    const double fx = k[0], fy = k[4], pcx = k[2], pcy = k[5];     // (unused in points mode)
    if (pts_cam) {
        // points mode (branch C, utils.py:189-193): camera-frame points come from the triangulation of the matched pixels,
        // `nocs` holds their NOCS coordinates in the same (compacted) order, the first pts_count[b] entries are valid.  The rest
        // is parked far apart: every pair with one of them fails the |dc| < 0.3 filter.
        const int cnt = pts_count[b];
        for (int i = tid; i < P; i += FIT_THREADS) {
            const float* pp = pts_cam + ((size_t)b * P + i) * 3;
            const float* nn = nocs + ((size_t)b * P + i) * 3;
            if (i < cnt) { pa[i] = make_float4(pp[0], pp[1], pp[2], nn[0]); pb[i] = make_float2(nn[1], nn[2]); }
            else { pa[i] = make_float4(1.0e6f * (float)(i + 1), 0.f, 0.f, 0.f); pb[i] = make_float2(0.f, 0.f); }
        }
    } else
    for (int i = tid; i < P; i += FIT_THREADS) {
        const int pix = choose[(size_t)b * P + i];
        const double z = (double)depth[(size_t)b * P + i];
        const int y = pix / S, x = pix - y * S;
        const float* nn = nocs + ((size_t)b * P + i) * 3;
        pa[i] = make_float4((float)(((double)x - pcx) * z / fx), (float)(((double)y - pcy) * z / fy), (float)z, nn[0]);
        pb[i] = make_float2(nn[1], nn[2]);
    }
    for (int i = tid; i < FIT_BINS; i += FIT_THREADS) hist[i] = 0;
    if (tid < 2) s_part[tid] = 0u;
    __syncthreads();

    // unordered pairs: the reference's ordered-pair list holds every ratio twice, which leaves the median unchanged.
    // pass A: histogram of the leading 11 bits + count of the valid ratios
    {
        unsigned int c = 0;
        fit_for_each_ratio(P, rank, pa, pb, [&](float r) {
            c += r >= 0.f;
            hist_add(hist, __float_as_uint(r) >> 21, r >= 0.f);
        });
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
        if ((tid & 31) == 0) atomicAdd(&s_part[0], c);
    }
    cluster.sync();
    long long m = 0;
    for (int r = 0; r < FIT_G; ++r) m += (long long)cluster.map_shared_rank(s_part, r)[0];
    double scale = nan("");
    if (m > 0) {       // uniform over the cluster
        // rank (0-based) of the upper middle element among the m sorted ratios; the lower one is rank (m-1)/2
        const long long k_hi = m / 2;
        const long long k_lo = (m - 1) / 2;
        unsigned int prefix = 0, pmask = 0;
        long long need = k_hi + 1;      // find the (k_hi+1)-th smallest
        const int shifts[3] = {21, 10, 0};
        const int widths[3] = {11, 11, 10};
        for (int pass = 0; pass < 3; ++pass) {
            const int shift = shifts[pass];
            const unsigned int bmask = (1u << widths[pass]) - 1u;
            if (pass > 0) {
                // digits below the leading one are spread evenly: plain shared-memory atomics, no warp aggregation
                fit_for_each_ratio(P, rank, pa, pb, [&](float r) {
                    const unsigned int key = __float_as_uint(r);
                    if (r >= 0.f && (key & pmask) == prefix) atomicAdd(&hist[(key >> shift) & bmask], 1u);
                });
                cluster.sync();
            }
            // cluster-wide histogram: every CTA sums the four per-CTA histograms over distributed shared memory
            for (int i = tid; i < FIT_BINS; i += FIT_THREADS) {
                unsigned int v = 0;
#pragma unroll
                for (int r = 0; r < FIT_G; ++r) v += cluster.map_shared_rank(hist, r)[i];
                htot[i] = v;
            }
            cluster.sync();                     // all remote reads of hist are done: it may be cleared for the next pass
            for (int i = tid; i < FIT_BINS; i += FIT_THREADS) hist[i] = 0;
            if (tid < 32) {
                // warp 0 scans the histogram: each lane sums a contiguous slice, then the slices are walked in order
                const int per = FIT_BINS / 32;
                long long part = 0;
                for (int q = 0; q < per; ++q) part += htot[tid * per + q];
                long long incl = part;
                for (int o = 1; o < 32; o <<= 1) {
                    const long long y = __shfl_up_sync(0xffffffffu, incl, o);
                    if (tid >= o) incl += y;
                }
                const long long excl = incl - part;
                const bool mine = (excl < need) && (need <= incl);
                if (mine) {
                    long long acc = excl;
                    int bsel = tid * per;
                    for (; bsel < tid * per + per; ++bsel) {
                        if (acc + (long long)htot[bsel] >= need) break;
                        acc += htot[bsel];
                    }
                    s_sel[0] = (unsigned int)bsel;
                    s_sel[1] = (unsigned int)(need - acc);
                    // lower middle (rank need-1 inside the current prefix group): same bin, or the largest occupied bin below it;
                    // 0xFFFFFFFF = it lies before this group (only meaningful after the last digit)
                    unsigned int lows = 0xFFFFFFFFu;
                    if (need - 1 > acc) lows = (unsigned int)bsel;
                    else if (need - 1 >= 1) {
                        int q = bsel - 1;
                        while (q > 0 && htot[q] == 0) --q;
                        lows = (unsigned int)q;
                    }
                    s_sel[2] = lows;
                }
            }
            __syncthreads();
            prefix |= s_sel[0] << shift;
            pmask |= bmask << shift;
            need = (long long)s_sel[1];
            __syncthreads();
        }
        const float v_hi = __uint_as_float(prefix);
        // lower middle (even m): inside the last prefix group it is read off the last histogram; otherwise it is the largest
        // element below v_hi, found by one more sweep (rare: v_hi is then the smallest value of its 22-bit prefix group)
        float v_lo = v_hi;
        if (k_lo < k_hi) {       // uniform over the cluster
            const unsigned int lows = s_sel[2];
            if (lows != 0xFFFFFFFFu) {
                v_lo = __uint_as_float((prefix & ~((1u << widths[2]) - 1u)) | lows);
            } else {
                float mx = -1.f;
                fit_for_each_ratio(P, rank, pa, pb, [&](float r) {
                    if (r >= 0.f && r < v_hi) mx = fmaxf(mx, r);
                });
                mx = block_reduce_max(mx, red);
                if (tid == 0) s_pmax = mx;
                cluster.sync();
                float mxall = -1.f;
                for (int r = 0; r < FIT_G; ++r) mxall = fmaxf(mxall, *cluster.map_shared_rank(&s_pmax, r));
                v_lo = mxall;
            }
        }
        // the select ran on q = ratio^2
        scale = 0.5 * (sqrt((double)v_lo) + sqrt((double)v_hi));
    }
    cluster.sync();       // no CTA leaves (or reuses shared memory) while a peer may still read its partial results
    if (rank != 0) return;

    // ---- translation: mean(cam) - mean(s R nocs);  half extents: max |nocs|
    const float smx = block_reduce_sum([&] { float s = 0.f; for (int i = tid; i < P; i += FIT_THREADS) s += pa[i].x; return s; }(), red);
    const float smy = block_reduce_sum([&] { float s = 0.f; for (int i = tid; i < P; i += FIT_THREADS) s += pa[i].y; return s; }(), red);
    const float smz = block_reduce_sum([&] { float s = 0.f; for (int i = tid; i < P; i += FIT_THREADS) s += pa[i].z; return s; }(), red);
    const float snx = block_reduce_sum([&] { float s = 0.f; for (int i = tid; i < P; i += FIT_THREADS) s += pa[i].w; return s; }(), red);
    const float sny = block_reduce_sum([&] { float s = 0.f; for (int i = tid; i < P; i += FIT_THREADS) s += pb[i].x; return s; }(), red);
    const float snz = block_reduce_sum([&] { float s = 0.f; for (int i = tid; i < P; i += FIT_THREADS) s += pb[i].y; return s; }(), red);
    const float hx = block_reduce_max([&] { float s = 0.f; for (int i = tid; i < P; i += FIT_THREADS) s = fmaxf(s, fabsf(pa[i].w)); return s; }(), red);
    const float hy = block_reduce_max([&] { float s = 0.f; for (int i = tid; i < P; i += FIT_THREADS) s = fmaxf(s, fabsf(pb[i].x)); return s; }(), red);
    const float hz = block_reduce_max([&] { float s = 0.f; for (int i = tid; i < P; i += FIT_THREADS) s = fmaxf(s, fabsf(pb[i].y)); return s; }(), red);

    if (tid == 0) {
        const float* Rb = R + 9 * b;
        const double mc[3] = {(double)smx / P, (double)smy / P, (double)smz / P};
        const double mn[3] = {(double)snx / P, (double)sny / P, (double)snz / P};
        double t[3];
        for (int r = 0; r < 3; ++r)
            t[r] = mc[r] - scale * ((double)Rb[3 * r] * mn[0] + (double)Rb[3 * r + 1] * mn[1] + (double)Rb[3 * r + 2] * mn[2]);
        if (scale_out) scale_out[b] = scale;
        if (trans_out) for (int r = 0; r < 3; ++r) trans_out[3 * b + r] = t[r];
        const double half[3] = {(double)hx * scale, (double)hy * scale, (double)hz * scale};   // size / 2
        double inv[16];
        bool fin = invert4x4(E + 16 * b, inv);
        for (int i = 0; i < 16 && fin; ++i) fin = isfinite(inv[i]);
        double cam[8][3];
        for (int c = 0; c < 8 && fin; ++c) {
            // corner order of get_3d_bbox (utils.py:40-58): (+++, ++-, -++, -+-, +-+, +--, --+, ---)
            const double sx = (c & 2) ? -1.0 : 1.0, sy = (c & 4) ? -1.0 : 1.0, sz = (c & 1) ? -1.0 : 1.0;
            const double p[3] = {sx * half[0], sy * half[1], sz * half[2]};
            for (int r = 0; r < 3; ++r) {
                // the reference stores R and t in a float32 4x4 (interface_v5.py:359-361)
                cam[c][r] = (double)Rb[3 * r] * p[0] + (double)Rb[3 * r + 1] * p[1] + (double)Rb[3 * r + 2] * p[2] + (double)(float)t[r];
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

int fit_run(const float* nocs, const float* depth, const int* choose, const double* Kp, const float* R, const double* E,
            const uint8_t* valid, double* bbox, double* scale_out, double* trans_out, const float* pts_cam, const int* pts_count,
            int B, int P, int S, cudaStream_t stream) {
    ADP_CHECK_ARG(P <= FIT_MAXP, "at most 1024 points per env");
    ADP_CHECK_ARG(!pts_cam || pts_count, "points mode needs the per-env point counts");
    if (B == 0) return ADP_OK;
    fit_kernel<<<B * FIT_G, FIT_THREADS, 0, stream>>>(nocs, depth, choose, Kp, R, E, valid, bbox, scale_out, trans_out, pts_cam, pts_count, P, S);
    ADP_CUDA(cudaGetLastError());
    return ADP_OK;
}

}  // namespace adp
