// fit_kernels.cu — pose fit (fdcm_fit_matches; rules in include/fdcm_b200.h): Gauss-Newton iterations of oriented
// point-to-line least squares of every match against the build scene's lines (sm_100a).
//
//   fit_grid_count_kernel + CUB scan + fit_grid_fill_kernel   per kFitCell-px cell of the map, the scene lines that can come
//                                                            within max_distance of a point of the cell.  A superset: rule 3
//                                                            takes the least (d2, j), so extra entries change no result and
//                                                            the fill may use atomic cursors
//   fit_eval_kernel<kScaled>                                one warp per match: per iteration the correspondences of every
//                                                            sample (lane i mod 32 takes sample i of a line), a butterfly
//                                                            reduction of the normal equations, the 3x3 (scaled: 4x4) solve and the update
//                                                            on every lane (the same values everywhere); then the stats pass
//                                                            and the evaluate<Dt3Cpu> score of the final pose
// Built with -fmad=false like every kernel of the library: the double arithmetic is the rules', operation by operation.
#include <climits>

#include <cub/device/device_scan.cuh>

#include "common.cuh"
#include "kernels.h"

namespace fdcm {

// A point p of cell (cx, cy) lies within kFitCell / sqrt(2) of the cell's centre, and a sample of a valid pose lies at most
// a rounding error outside the map (its cell index is clamped): a line within max_distance of p is within
// max_distance + 2 + 0.7072 kFitCell of the centre.
static inline double fit_reach(float max_distance) { return (double)max_distance + 2.0 + 0.7072 * kFitCell; }

// visit(cell) for every cell whose centre lies within reach of the (non-degenerate) line
template <class Visit>
__device__ __forceinline__ void fit_line_cells(const float4 l, double reach, int gx, int gy, Visit visit) {
    const double ax = l.x, ay = l.y, dx = (double)l.z - ax, dy = (double)l.w - ay;
    const double l2 = dx * dx + dy * dy;
    if (!(l2 > 0.0)) return;   // never a candidate (rule 3)
    const double S = kFitCell;
    const int cx0 = max(0, (int)floor((fmin(ax, (double)l.z) - reach) / S)), cx1 = min(gx - 1, (int)floor((fmax(ax, (double)l.z) + reach) / S));
    const int cy0 = max(0, (int)floor((fmin(ay, (double)l.w) - reach) / S)), cy1 = min(gy - 1, (int)floor((fmax(ay, (double)l.w) + reach) / S));
    const double r2 = reach * reach;
    for (int cy = cy0; cy <= cy1; ++cy)
        for (int cx = cx0; cx <= cx1; ++cx) {
            const double px = (cx + 0.5) * S, py = (cy + 0.5) * S;
            double u = ((px - ax) * dx + (py - ay) * dy) / l2;
            u = u < 0.0 ? 0.0 : (u > 1.0 ? 1.0 : u);
            const double ex = px - (ax + u * dx), ey = py - (ay + u * dy);
            if (ex * ex + ey * ey <= r2) visit(cy * gx + cx);
        }
}

__global__ void fit_grid_count_kernel(const float4* __restrict__ lines, int n, double reach, int gx, int gy,
                                      unsigned long long* __restrict__ cnt) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    fit_line_cells(lines[j], reach, gx, gy, [&](int c) { atomicAdd(cnt + c, 1ull); });
}

__global__ void fit_grid_fill_kernel(const float4* __restrict__ lines, int n, double reach, int gx, int gy,
                                     const unsigned long long* __restrict__ off, unsigned long long* __restrict__ cursor,
                                     int32_t* __restrict__ items) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    fit_line_cells(lines[j], reach, gx, gy, [&](int c) { items[off[c] + atomicAdd(cursor + c, 1ull)] = j; });
}

size_t fit_grid_scan_bytes(int n_cells) {
    size_t bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, bytes, (const unsigned long long*)nullptr, (unsigned long long*)nullptr, n_cells + 1);
    return bytes;
}

void launch_fit_grid_count(const float4* d_lines, int n_lines, float max_distance, int gx, int gy, unsigned long long* d_cnt,
                           unsigned long long* d_off, void* d_temp, size_t temp_bytes, cudaStream_t s) {
    if (n_lines > 0) fit_grid_count_kernel<<<(n_lines + 127) / 128, 128, 0, s>>>(d_lines, n_lines, fit_reach(max_distance), gx, gy, d_cnt);
    cub::DeviceScan::ExclusiveSum(d_temp, temp_bytes, d_cnt, d_off, gx * gy + 1, s);
}

void launch_fit_grid_fill(const float4* d_lines, int n_lines, float max_distance, int gx, int gy, const unsigned long long* d_off,
                          unsigned long long* d_cursor, int32_t* d_items, cudaStream_t s) {
    if (n_lines > 0)
        fit_grid_fill_kernel<<<(n_lines + 127) / 128, 128, 0, s>>>(d_lines, n_lines, fit_reach(max_distance), gx, gy, d_off, d_cursor,
                                                                   d_items);
}

// ---- the fit ---------------------------------------------------------------------------------------------------------
struct FitPose { double m0, m1, m3, m4, ex, ey; };

// rule 1: the float32 rounding F of a pose
__device__ __forceinline__ void fit_round(const FitPose& P, float shx, float shy, float* F) {
    F[0] = (float)P.m0; F[1] = (float)P.m1; F[2] = (float)(P.ex - (double)shx);
    F[3] = (float)P.m3; F[4] = (float)P.m4; F[5] = (float)(P.ey - (double)shy);
}

// refinement rule 4 for the float pose F, warp-wide: no NaN, every posed end point inside the map
__device__ bool fit_valid(const float4* __restrict__ tl, int L, const float* F, const MapView& map, const SlopeTableDev& table,
                          int lane) {
    const float offx = map.shift_x + F[2], offy = map.shift_y + F[5];
    const float Wm1 = (float)(map.dm.W - 1), Hm1 = (float)(map.dm.H - 1);
    bool bad = false;
    for (int q = lane; q < L && !bad; q += 32) {
        const PosedLine pl = pose_line(__ldg(tl + q), F, offx, offy, table);
        bad = !(0.f <= pl.x1 && pl.x1 <= Wm1 && 0.f <= pl.y1 && pl.y1 <= Hm1 && 0.f <= pl.x2 && pl.x2 <= Wm1 && 0.f <= pl.y2 &&
                pl.y2 <= Hm1);
    }
    return !__any_sync(0xffffffffu, bad);
}

// sums of rule 4: A00 A01 A02 A11 A12 A22 g0 g1 g2 rr; of rule 4' (scaled): A00 A01 A02 A03 A11 A12 A13 A22 A23 A33 g0 g1 g2
// g3 rr
template <bool kScaled>
constexpr int kFitSums = kScaled ? 15 : 10;

// rule 3 + 4 at pose P (float rounding F, centre c): every lane's sums, then the butterfly; also rho^2 (rule 2)
template <bool kScaled>
__device__ void fit_pass(const FitLaunch& p, const SlopeTableDev& table, const float4* __restrict__ tl, int L, const FitPose& P,
                         const float* F, double cx, double cy, double ax, double ay, int lane, double* acc, int& n_in, double& rho2) {
    const float offx = p.map.shift_x + F[2], offy = p.map.shift_y + F[5];
    const int D = p.map.dm.D, tol = p.prm.bin_tolerance;
    const double md2 = (double)p.prm.max_distance * (double)p.prm.max_distance;
#pragma unroll
    for (int k = 0; k < kFitSums<kScaled>; ++k) acc[k] = 0.0;
    n_in = 0;
    rho2 = 0.0;
    for (int q = 0; q < L; ++q) {
        const float4 v = __ldg(tl + q);
        const int n = fit_line_samples(v.x, v.y, v.z, v.w, p.prm.sample_step);
        if (n == 0) continue;
        const int b = pose_line(v, F, offx, offy, table).bin;
        for (int i = lane; i < n; i += 32) {
            double sx, sy;
            fit_sample(v.x, v.y, v.z, v.w, i, n, sx, sy);
            const double rx = sx - ax, ry = sy - ay, d2a = rx * rx + ry * ry;
            rho2 = d2a > rho2 ? d2a : rho2;
            const double px = (P.m0 * sx + P.m1 * sy) + P.ex, py = (P.m3 * sx + P.m4 * sy) + P.ey;
            int cxi = (int)floor(px / kFitCell), cyi = (int)floor(py / kFitCell);
            cxi = min(max(cxi, 0), p.gx - 1);
            cyi = min(max(cyi, 0), p.gy - 1);
            const int c = cyi * p.gx + cxi;
            double best = INFINITY;
            int bj = INT_MAX;
            for (unsigned long long k = __ldg(p.cell_off + c), k1 = __ldg(p.cell_off + c + 1); k < k1; ++k) {
                const int j = __ldg(p.cell_items + k);
                int db = abs(__ldg(p.scene_bins + j) - b);
                db = min(db, D - db);
                if (db > tol) continue;
                const float4 S = __ldg(p.scene + j);
                const double Ax = S.x, Ay = S.y, dx = (double)S.z - Ax, dy = (double)S.w - Ay;
                const double l2 = dx * dx + dy * dy;
                if (!(l2 > 0.0)) continue;
                double u = ((px - Ax) * dx + (py - Ay) * dy) / l2;
                u = u < 0.0 ? 0.0 : (u > 1.0 ? 1.0 : u);
                const double ex = px - (Ax + u * dx), ey = py - (Ay + u * dy);
                const double d2 = ex * ex + ey * ey;
                if (d2 <= md2 && (d2 < best || (d2 == best && j < bj))) {
                    best = d2;
                    bj = j;
                }
            }
            if (bj == INT_MAX) continue;
            const float4 S = __ldg(p.scene + bj);
            const double Ax = S.x, Ay = S.y, dx = (double)S.z - Ax, dy = (double)S.w - Ay;
            const double l = sqrt(dx * dx + dy * dy);
            const double nx = -dy / l, ny = dx / l;
            const double r = nx * (px - Ax) + ny * (py - Ay);
            const double jt = ny * (px - cx) - nx * (py - cy);
            if constexpr (kScaled) {
                const double js = nx * (px - cx) + ny * (py - cy);
                acc[0] = acc[0] + nx * nx;  acc[1] = acc[1] + nx * ny;  acc[2] = acc[2] + nx * jt;  acc[3] = acc[3] + nx * js;
                acc[4] = acc[4] + ny * ny;  acc[5] = acc[5] + ny * jt;  acc[6] = acc[6] + ny * js;
                acc[7] = acc[7] + jt * jt;  acc[8] = acc[8] + jt * js;  acc[9] = acc[9] + js * js;
                acc[10] = acc[10] + nx * r; acc[11] = acc[11] + ny * r; acc[12] = acc[12] + jt * r; acc[13] = acc[13] + js * r;
                acc[14] = acc[14] + r * r;
            } else {
                acc[0] = acc[0] + nx * nx; acc[1] = acc[1] + nx * ny; acc[2] = acc[2] + nx * jt;
                acc[3] = acc[3] + ny * ny; acc[4] = acc[4] + ny * jt; acc[5] = acc[5] + jt * jt;
                acc[6] = acc[6] + nx * r;  acc[7] = acc[7] + ny * r;  acc[8] = acc[8] + jt * r;
                acc[9] = acc[9] + r * r;
            }
            ++n_in;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int k = 0; k < kFitSums<kScaled>; ++k) acc[k] = acc[k] + __shfl_xor_sync(0xffffffffu, acc[k], o);
        n_in += __shfl_xor_sync(0xffffffffu, n_in, o);
        const double o2 = __shfl_xor_sync(0xffffffffu, rho2, o);
        rho2 = o2 > rho2 ? o2 : rho2;
    }
}

// rule 4: the damped Cholesky solve; false when a radicand is not > 0
__device__ __forceinline__ bool fit_solve(const double* a, double* d) {
    const double lam = 1e-9 * ((a[0] + a[3]) + a[5]);
    const double b00 = a[0] + lam, b11 = a[3] + lam, b22 = a[5] + lam;
    if (!(b00 > 0.0)) return false;
    const double l00 = sqrt(b00), l10 = a[1] / l00, l20 = a[2] / l00;
    const double r1 = b11 - l10 * l10;
    if (!(r1 > 0.0)) return false;
    const double l11 = sqrt(r1), l21 = (a[4] - l20 * l10) / l11;
    const double r2 = (b22 - l20 * l20) - l21 * l21;
    if (!(r2 > 0.0)) return false;
    const double l22 = sqrt(r2);
    const double y0 = -a[6] / l00, y1 = (-a[7] - l10 * y0) / l11, y2 = ((-a[8] - l20 * y0) - l21 * y1) / l22;
    d[2] = y2 / l22;
    d[1] = (y1 - l21 * d[2]) / l11;
    d[0] = ((y0 - l10 * d[1]) - l20 * d[2]) / l00;
    return true;
}

// rule 4': the damped 4x4 Cholesky solve in the header's order; false when a radicand is not > 0.  d = (dx, dy, dth, ds)
__device__ __forceinline__ bool fit_solve_scaled(const double* a, double* d) {
    const double lam = 1e-9 * (((a[0] + a[4]) + a[7]) + a[9]);
    const double b00 = a[0] + lam, b11 = a[4] + lam, b22 = a[7] + lam, b33 = a[9] + lam;
    if (!(b00 > 0.0)) return false;
    const double l00 = sqrt(b00), l10 = a[1] / l00, l20 = a[2] / l00, l30 = a[3] / l00;
    const double r1 = b11 - l10 * l10;
    if (!(r1 > 0.0)) return false;
    const double l11 = sqrt(r1), l21 = (a[5] - l20 * l10) / l11, l31 = (a[6] - l30 * l10) / l11;
    const double r2 = (b22 - l20 * l20) - l21 * l21;
    if (!(r2 > 0.0)) return false;
    const double l22 = sqrt(r2), l32 = ((a[8] - l30 * l20) - l31 * l21) / l22;
    const double r3 = ((b33 - l30 * l30) - l31 * l31) - l32 * l32;
    if (!(r3 > 0.0)) return false;
    const double l33 = sqrt(r3);
    const double y0 = -a[10] / l00, y1 = (-a[11] - l10 * y0) / l11, y2 = ((-a[12] - l20 * y0) - l21 * y1) / l22;
    const double y3 = (((-a[13] - l30 * y0) - l31 * y1) - l32 * y2) / l33;
    d[3] = y3 / l33;
    d[2] = (y2 - l32 * d[3]) / l22;
    d[1] = ((y1 - l21 * d[2]) - l31 * d[3]) / l11;
    d[0] = (((y0 - l10 * d[1]) - l20 * d[2]) - l30 * d[3]) / l00;
    return true;
}

constexpr int kFitThreads = 128;

template <bool kScaled>
__global__ void __launch_bounds__(kFitThreads) fit_eval_kernel(const __grid_constant__ FitLaunch p,
                                                               const __grid_constant__ SlopeTableDev table) {
    const long long h = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (h >= p.n) return;   // whole warp
    const fdcm_match m = p.in[h];
    const int t = m.tmpl_idx - p.tmpl_idx_base;   // (the host checks the indices)
    const int l0 = p.offsets[t], L = p.offsets[t + 1] - l0;
    const float4* tl = p.lines + l0;
    const float shx = p.map.shift_x, shy = p.map.shift_y;
    fdcm_match r = m;
    fdcm_fit_stats st{0, 0, 0, NAN};
    if (L == 0 || !fit_valid(tl, L, m.transform, p.map, table, lane)) {   // an invalid input (rule 6)
        if (lane == 0) {
            r.score = NAN;
            p.out[h] = r;
            if (p.stats) p.stats[h] = st;
        }
        return;
    }
    int n_samples = 0;
    for (int q = lane; q < L; q += 32) {
        const float4 v = __ldg(tl + q);
        n_samples += fit_line_samples(v.x, v.y, v.z, v.w, p.prm.sample_step);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) n_samples += __shfl_xor_sync(0xffffffffu, n_samples, o);
    const float2 af = p.anchors[t];
    const double ax = af.x, ay = af.y;
    FitPose P{(double)m.transform[0], (double)m.transform[1], (double)m.transform[3], (double)m.transform[4],
              (double)m.transform[2] + (double)shx, (double)m.transform[5] + (double)shy};
    float F[6];
    for (int k = 0; k < 6; ++k) F[k] = m.transform[k];
    double acc[kFitSums<kScaled>], rho2 = 0.0;
    int n_in = 0, iters = 0;
    bool at_pose = false;   // acc / n_in hold the correspondences of the current pose
    for (int it = 0; it < p.prm.iterations; ++it) {
        const double cx = (P.m0 * ax + P.m1 * ay) + P.ex, cy = (P.m3 * ax + P.m4 * ay) + P.ey;
        fit_pass<kScaled>(p, table, tl, L, P, F, cx, cy, ax, ay, lane, acc, n_in, rho2);
        at_pose = true;
        if (n_in < p.prm.min_inliers) break;
        double d[kScaled ? 4 : 3];
        if constexpr (kScaled) {
            if (!fit_solve_scaled(acc, d)) break;
        } else {
            if (!fit_solve(acc, d)) break;
        }
        // rule 5: the half-angle rotation about c, then the translation
        const double tau = d[2] * 0.5, k = 1.0 + tau * tau;
        double cr = (1.0 - tau * tau) / k, sr = (2.0 * tau) / k;
        if constexpr (kScaled) {   // rule 5': the scale step about c
            const double f = 1.0 + d[3];
            cr = f * cr;
            sr = f * sr;
        }
        const double ux = P.ex - cx, uy = P.ey - cy;
        const FitPose N{cr * P.m0 - sr * P.m3, cr * P.m1 - sr * P.m4, sr * P.m0 + cr * P.m3, sr * P.m1 + cr * P.m4,
                        ((cr * ux - sr * uy) + cx) + d[0], ((sr * ux + cr * uy) + cy) + d[1]};
        double sigma = 0.0;   // the scale of the pose before the update
        if constexpr (kScaled) {
            const double sig_n = sqrt(N.m0 * N.m4 - N.m1 * N.m3);
            if (!(sig_n >= (double)p.min_scale && sig_n <= (double)p.max_scale)) break;   // (NaN fails too)
            sigma = sqrt(P.m0 * P.m4 - P.m1 * P.m3);
        }
        float FN[6];
        fit_round(N, shx, shy, FN);
        if (!fit_valid(tl, L, FN, p.map, table, lane)) break;
        P = N;
        for (int q = 0; q < 6; ++q) F[q] = FN[q];
        ++iters;
        at_pose = false;
        if constexpr (kScaled) {
            const double rho = sqrt(rho2);
            const double ad0 = fabs(d[0]), ad1 = fabs(d[1]), adt = (fabs(d[2]) * sigma) * rho, ads = (fabs(d[3]) * sigma) * rho;
            const double s01 = ad0 > ad1 ? ad0 : ad1, sts = adt > ads ? adt : ads;
            const double step = s01 > sts ? s01 : sts;
            if (step <= (double)p.prm.tolerance) break;
        } else {
            const double ad0 = fabs(d[0]), ad1 = fabs(d[1]), adt = fabs(d[2]) * sqrt(rho2);
            const double step = ad0 > ad1 ? (ad0 > adt ? ad0 : adt) : (ad1 > adt ? ad1 : adt);
            if (step <= (double)p.prm.tolerance) break;
        }
    }
    if (!at_pose) {
        const double cx = (P.m0 * ax + P.m1 * ay) + P.ex, cy = (P.m3 * ax + P.m4 * ay) + P.ey;
        fit_pass<kScaled>(p, table, tl, L, P, F, cx, cy, ax, ay, lane, acc, n_in, rho2);
    }
    if (lane != 0) return;
    // rule 6: the score of F, evaluate<Dt3Cpu> in Eigen's order (refinement's scoring terms)
    const float offx = shx + F[2], offy = shy + F[5];
    const float raw = eigen_sum_lazy(L, [&](int q) {
        const PosedLine pl = pose_line(__ldg(tl + q), F, offx, offy, table);
        return line_cost(p.map.planes, (size_t)p.map.dm.pitch, p.map.dm.plane_elems, pl.bin, pl.x1, pl.y1, pl.x2, pl.y2);
    });
    r.score = p.denom ? raw / p.denom[t] : raw;
    for (int q = 0; q < 6; ++q) r.transform[q] = F[q];
    p.out[h] = r;
    if (p.stats) {
        st.n_samples = n_samples;
        st.n_inliers = n_in;
        st.iterations = iters;
        st.rms = n_in > 0 ? (float)sqrt(acc[kFitSums<kScaled> - 1] / (double)n_in) : NAN;
        p.stats[h] = st;
    }
}

void launch_fit_eval(const FitLaunch& p, const SlopeTableDev& table, cudaStream_t s) {
    if (p.n <= 0) return;
    const long long blocks = (p.n + kFitThreads / 32 - 1) / (kFitThreads / 32);
    if (p.scaled) fit_eval_kernel<true><<<(unsigned)blocks, kFitThreads, 0, s>>>(p, table);
    else fit_eval_kernel<false><<<(unsigned)blocks, kFitThreads, 0, s>>>(p, table);
}

}   // namespace fdcm
