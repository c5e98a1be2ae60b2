// coverage_kernels.cu — match verification (fdcm_match_coverage, fdcm_search_verify, fdcm_search_dense_verify; rules in
// include/fdcm_b200.h): oriented edge coverage of posed templates against the map's 1-bit edge masks (sm_100a).
//
//   coverage_planes_kernel  + coverage_window_kernel   the dilated mask of (radius, bin_tolerance): bit (b, y, x) is the OR of
//                                                      the edge bits of the planes within the tolerance of b over the
//                                                      (2r+1)^2 window around (x, y); afterwards every sample is one bit gather
//   coverage_eval_kernel                               one warp per match: validity, then the raster samples of every posed
//                                                      line, one gather per lane and sample, counted with ballot + popc
// Built with -fmad=false like every kernel of the library: the posed end points are the refinement's, operation by operation.
#include "common.cuh"
#include "kernels.h"

namespace fdcm {

// planes first: tmp[b][y][w] = OR of mask[q][y][w] over the planes q within the tolerance of b (circular)
__global__ void __launch_bounds__(256) coverage_planes_kernel(const uint32_t* __restrict__ mask, MapDims dm, int tol,
                                                              uint32_t* __restrict__ tmp) {
    const size_t plane_words = (size_t)dm.H * dm.wwords;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= plane_words * dm.D) return;
    const int b = (int)(i / plane_words);
    const size_t off = i - (size_t)b * plane_words;
    uint32_t v = 0;
    if (2 * tol + 1 >= dm.D) {
        for (int q = 0; q < dm.D; ++q) v |= __ldg(mask + (size_t)q * plane_words + off);
    } else {
        for (int d = -tol; d <= tol; ++d) {
            const int q = (b + d + dm.D) % dm.D;
            v |= __ldg(mask + (size_t)q * plane_words + off);
        }
    }
    tmp[i] = v;
}

// then the window: rows [y - r, y + r] of the map by OR, columns [x - r, x + r] by funnel shifts with the neighbouring
// words (r < 32); bits at x >= W stay clear
__global__ void __launch_bounds__(256) coverage_window_kernel(const uint32_t* __restrict__ tmp, MapDims dm, int r,
                                                              uint32_t* __restrict__ dil) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)dm.D * dm.H * dm.wwords) return;
    const int w = (int)(i % dm.wwords);
    const size_t row = i / dm.wwords;   // b * H + y
    const int y = (int)(row % dm.H);
    const size_t plane_row0 = row - y;
    const int y0 = max(0, y - r), y1 = min(dm.H - 1, y + r);
    uint32_t prev = 0, cur = 0, next = 0;
    for (int yy = y0; yy <= y1; ++yy) {
        const uint32_t* src = tmp + (plane_row0 + yy) * dm.wwords;
        cur |= __ldg(src + w);
        if (w > 0) prev |= __ldg(src + w - 1);
        if (w + 1 < dm.wwords) next |= __ldg(src + w + 1);
    }
    uint32_t v = cur;
    for (int s = 1; s <= r; ++s) v |= __funnelshift_l(prev, cur, s) | __funnelshift_r(cur, next, s);
    const int x0 = w * 32;
    if (x0 + 32 > dm.W) v &= x0 >= dm.W ? 0u : (1u << (dm.W - x0)) - 1u;
    dil[i] = v;
}

void launch_coverage_dilate(const uint32_t* d_mask, const MapDims& dm, int radius, int tol, uint32_t* d_tmp, uint32_t* d_dil,
                            cudaStream_t s) {
    const size_t words = (size_t)dm.D * dm.H * dm.wwords;
    if (words == 0) return;
    const unsigned blocks = (unsigned)((words + 255) / 256);
    coverage_planes_kernel<<<blocks, 256, 0, s>>>(d_mask, dm, tol, d_tmp);
    coverage_window_kernel<<<blocks, 256, 0, s>>>(d_tmp, dm, radius, d_dil);
}

constexpr int kCoverageThreads = 256;

__global__ void __launch_bounds__(kCoverageThreads) coverage_eval_kernel(const __grid_constant__ CoverageLaunch p,
                                                                         const __grid_constant__ SlopeTableDev table) {
    const long long h = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (h >= p.n) return;   // whole warp
    if (p.valid && !p.valid[h]) return;
    const fdcm_match m = p.rec[h];
    const int t = m.tmpl_idx - p.tmpl_idx_base;
    const MapDims dm = p.dm;
    // rule 2: validity of every posed end point, and n_total (rule 3)
    bool bad = t < 0 || t >= p.n_tmpl;   // (the host checks the indices; a record of the search is always in range)
    int l0 = 0, L = 0;
    if (!bad) {
        l0 = p.offsets[t];
        L = p.offsets[t + 1] - l0;
    }
    const float offx = p.shift_x + m.transform[2], offy = p.shift_y + m.transform[5];
    const float Wm1 = (float)(dm.W - 1), Hm1 = (float)(dm.H - 1);
    int total = 0;
    for (int q = lane; q < L && !bad; q += 32) {
        const PosedLine pl = pose_line(__ldg(p.lines + l0 + q), m.transform, offx, offy, table);
        // (a NaN in T or in an end point reaches every posed coordinate and fails these tests)
        if (!(0.f <= pl.x1 && pl.x1 <= Wm1 && 0.f <= pl.y1 && pl.y1 <= Hm1 && 0.f <= pl.x2 && pl.x2 <= Wm1 && 0.f <= pl.y2 &&
              pl.y2 <= Hm1)) {
            bad = true;
            break;
        }
        total += RasterLineDev(pl.x1, pl.y1, pl.x2, pl.y2).n;
    }
    bad = __any_sync(0xffffffffu, bad) || L == 0;
    if (bad) {
        if (p.coverage) p.coverage[h] = NAN;
        else if (lane == 0) p.valid[h] = 0;
        return;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) total += __shfl_xor_sync(0xffffffffu, total, o);
    // rule 4: one bit gather of the dilated mask per sample.  Filter mode stops once the threshold decision is certain:
    // the final count lies in [covered, covered + remaining] and (float)c / (float)total is non-decreasing in c.
    const float ftotal = (float)total;
    int covered = 0, done = 0;
    for (int q = 0; q < L; ++q) {
        const PosedLine pl = pose_line(__ldg(p.lines + l0 + q), m.transform, offx, offy, table);
        const RasterLineDev rl(pl.x1, pl.y1, pl.x2, pl.y2);
        const uint32_t* plane = p.dil + (size_t)pl.bin * dm.H * dm.wwords;
        for (int i0 = 0; i0 < rl.n; i0 += 32) {
            bool hit = false;
            const int i = i0 + lane;
            if (i < rl.n) {
                long long x, y;
                rl.at(i, x, y);
                // (the samples of end points inside the map lie inside the map; the test guards the gather)
                if (x >= 0 && y >= 0 && x < dm.W && y < dm.H)
                    hit = (__ldg(plane + (size_t)y * dm.wwords + (x >> 5)) >> (x & 31)) & 1u;
            }
            covered += __popc(__ballot_sync(0xffffffffu, hit));
        }
        done += rl.n;
        if (!p.coverage) {
            if ((float)covered / ftotal >= p.min_coverage) return;                   // kept whatever follows
            if ((float)(covered + (total - done)) / ftotal < p.min_coverage) break;  // removed whatever follows
        }
    }
    const float c = (float)covered / ftotal;
    if (p.coverage) {
        if (lane == 0) p.coverage[h] = c;
    } else if (lane == 0 && !(c >= p.min_coverage)) {
        p.valid[h] = 0;
    }
}

void launch_coverage_eval(const CoverageLaunch& p, const SlopeTableDev& table, cudaStream_t s) {
    if (p.n <= 0) return;
    const long long blocks = (p.n + kCoverageThreads / 32 - 1) / (kCoverageThreads / 32);
    coverage_eval_kernel<<<(unsigned)blocks, kCoverageThreads, 0, s>>>(p, table);
}

}   // namespace fdcm
