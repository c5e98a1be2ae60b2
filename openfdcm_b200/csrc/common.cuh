// common.cuh — shared device/host declarations of libfdcm_b200 (sm_100a only).
// Built with -fmad=false: every float op below is a separately rounded IEEE binary32 operation, as in
// the reference's SSE2 build (reference CMakeLists.txt:29-32: no -march, no FMA).
#pragma once
#include <cuda_runtime.h>
#include <cfloat>
#include <cstdint>

namespace fdcm {

constexpr int kMaxDepthDev = 64;
constexpr int kMaxPropSteps = 4 * kMaxDepthDev;
constexpr uint16_t kNoEdge16 = 0xFFFFu;

// geometry of the device feature map: [D][H][pitch] fp32 planes, pitch % 32 == 0 (128-byte rows)
struct MapDims {
    int D, H, W, pitch;
    int wwords;              // mask words per row = pitch / 32
    size_t plane_elems;      // H * pitch
};

struct PropParams {          // propagateOrientation schedule (dt3cpu.cpp:77-107)
    int n_steps;
    float w[kMaxPropSteps];
    uint8_t c1[kMaxPropSteps];
    uint8_t c2[kMaxPropSteps];
};

struct IntegralParams {      // lineIntegral direction per plane (core/imgproc.h:41-48)
    float rx[kMaxDepthDev], ry[kMaxDepthDev];
    int mode[kMaxDepthDev];  // 1: x-major, 2: y-major, 0: no-op
};

struct SlopeTableDev {       // see host_math.hpp SlopeTable
    int n_thr;
    int nan_bin;
    float thr[kMaxDepthDev + 8];
    uint8_t piece_bin[kMaxDepthDev + 9];
};

// ---- device float helpers --------------------------------------------------------------------
// (long)std::round(x): half away from zero, then truncating conversion
__device__ __forceinline__ long long round_to_ll(float x) { return (long long)roundf(x); }

// the reference's `x - 2.0*cond*x` (double) for rasterizeVector: +-x, zero always +0 (host_math.hpp)
__device__ __forceinline__ float signed_pick_dev(float x, bool negate) { return x == 0.f ? 0.f : (negate ? -x : x); }

// rasterizeVector (core/drawing.h:57-67)
__device__ __forceinline__ void rasterize_vector_dev(float vx, float vy, float& ox, float& oy) {
    const float t = vy / vx;
    if (t >= -1.0f && t < 1.0f) {
        const bool c = vx < 0;
        ox = c ? -1.f : 1.f;
        oy = signed_pick_dev(t, c);
        return;
    }
    const bool c = vy < 0;
    const float inv = 1.f / t;
    ox = signed_pick_dev(inv, c);
    oy = c ? -1.f : 1.f;
}

// relativelyEqual(x, 0.0f) (core/math.h:183-189): |x| <= eps_f + 1e-10*|x| evaluated in double
__device__ __forceinline__ bool rel_eq_zero(float x) {
    const double ax = (double)fabsf(x);
    return ax <= (double)FLT_EPSILON + 1e-10 * ax;
}

// Eigen 3.4.0 LinSpaced<float>(n, lo, hi)(i) (see oracle / SURVEY App. A.7)
struct LinSpacedDev {
    float lo, hi, step;
    int size1;
    bool flip;
    __device__ LinSpacedDev() : lo(0.f), hi(0.f), step(0.f), size1(1), flip(false) {}
    __device__ LinSpacedDev(int n, float lo_, float hi_)
        : lo(lo_), hi(hi_), step(n == 1 ? 0.f : (hi_ - lo_) / (float)(n - 1)), size1(n == 1 ? 1 : n - 1),
          flip(fabsf(hi_) < fabsf(lo_)) {}
    __device__ __forceinline__ float at(int i) const {
        if (flip) return (i == 0) ? lo : (hi - (float)(size1 - i) * step);
        return (i == size1) ? hi : (lo + (float)i * step);
    }
};

// rasterizeLine (core/drawing.h:74-102) of the line (p1x, p1y) - (p2x, p2y), without clipping: n pixels, pixel i at(i)
struct RasterLineDev {
    int n;
    int kind;                // 0: one pixel, 1: x fixed (steep), 2: y fixed (flat), 3: both vary
    long long fx, fy;        // the fixed coordinate of kinds 0..2
    LinSpacedDev lx, ly;
    __device__ RasterLineDev(float p1x, float p1y, float p2x, float p2y) {
        fx = round_to_ll(p1x);
        fy = round_to_ll(p1y);
        if (fabsf(p2x - p1x) <= 1e-5f && fabsf(p2y - p1y) <= 1e-5f) {
            n = 1;
            kind = 0;
            return;
        }
        const float lvx = p2x - p1x, lvy = p2y - p1y;
        float rx, ry;
        rasterize_vector_dev(lvx, lvy, rx, ry);
        if (rel_eq_zero(rx)) {
            n = (int)(lvy / ry) + 1;
            kind = 1;
            ly = LinSpacedDev(n, p1y, p2y);
            return;
        }
        if (rel_eq_zero(ry)) {
            n = (int)(lvx / rx) + 1;
            kind = 2;
            lx = LinSpacedDev(n, p1x, p2x);
            return;
        }
        const float a = lvx / rx, b = lvy / ry;
        n = (int)((a < b) ? b : a) + 1;   // std::max(a, b)
        kind = 3;
        lx = LinSpacedDev(n, p1x, p2x);
        ly = LinSpacedDev(n, p1y, p2y);
    }
    __device__ __forceinline__ void at(int i, long long& x, long long& y) const {
        x = (kind & 2) ? round_to_ll(lx.at(i)) : fx;
        y = (kind & 1) ? round_to_ll(ly.at(i)) : fy;
    }
};

// orientation bin of a slope through the host-built threshold table (dt3cpu.h:93-114 semantics)
__device__ __forceinline__ int bin_of_slope_dev(const SlopeTableDev& t, float slope) {
    if (slope != slope) return t.nan_bin;
    int lo = 0, hi = t.n_thr;   // count thresholds <= slope
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (t.thr[mid] <= slope) lo = mid + 1; else hi = mid;
    }
    return t.piece_bin[lo];
}

// Eigen 3.4.0 VectorXf::sum() order (Redux.h, SSE2 packet 4, 2x unrolled) over lazily produced terms
template <class CostFn>
__device__ __forceinline__ float eigen_sum_lazy(int n, CostFn c) {
    if (n < 4) {
        if (n == 0) return 0.f;
        float r = c(0);
        for (int i = 1; i < n; ++i) r = r + c(i);
        return r;
    }
    const int n4 = n & ~3, n8 = n & ~7;
    float A0 = c(0), A1 = c(1), A2 = c(2), A3 = c(3);
    if (n4 > 4) {
        float B0 = c(4), B1 = c(5), B2 = c(6), B3 = c(7);
        for (int i = 8; i < n8; i += 8) {
            const float c0 = c(i), c1 = c(i + 1), c2 = c(i + 2), c3 = c(i + 3);
            const float c4 = c(i + 4), c5 = c(i + 5), c6 = c(i + 6), c7 = c(i + 7);
            A0 = A0 + c0; A1 = A1 + c1; A2 = A2 + c2; A3 = A3 + c3;
            B0 = B0 + c4; B1 = B1 + c5; B2 = B2 + c6; B3 = B3 + c7;
        }
        A0 = A0 + B0; A1 = A1 + B1; A2 = A2 + B2; A3 = A3 + B3;
        if (n4 > n8) {
            const float c0 = c(n8), c1 = c(n8 + 1), c2 = c(n8 + 2), c3 = c(n8 + 3);
            A0 = A0 + c0; A1 = A1 + c1; A2 = A2 + c2; A3 = A3 + c3;
        }
    }
    float r = (A0 + A2) + (A1 + A3);
    for (int i = n4; i < n; ++i) r = r + c(i);
    return r;
}

// line q of the template posed by T (refinement rule 4): map-coordinate end points and the orientation bin
struct PosedLine { float x1, y1, x2, y2; int bin; };
__device__ __forceinline__ PosedLine pose_line(const float4 v, const float* T, float offx, float offy, const SlopeTableDev& table) {
    const float x1 = T[0] * v.x + T[1] * v.y, y1 = T[3] * v.x + T[4] * v.y;
    const float x2 = T[0] * v.z + T[1] * v.w, y2 = T[3] * v.z + T[4] * v.w;
    PosedLine p;
    p.bin = bin_of_slope_dev(table, (y2 - y1) / (x2 - x1));
    p.x1 = x1 + offx; p.y1 = y1 + offy;
    p.x2 = x2 + offx; p.y2 = y2 + offy;
    return p;
}

// the evaluate<Dt3Cpu> term of one posed line (dt3cpu.cpp:126-179): |plane(x1, y1) - plane(x2, y2)| of its plane at the
// truncated map-coordinate end points, which the caller has checked to lie inside the map
__device__ __forceinline__ float line_cost(const float* planes, size_t pitch, size_t plane_elems, int bin, float x1, float y1, float x2,
                                           float y2) {
    const int ix1 = (int)x1, iy1 = (int)y1, ix2 = (int)x2, iy2 = (int)y2;
    const float* P = planes + (size_t)bin * plane_elems;
    return fabsf(__ldg(P + (size_t)iy1 * pitch + ix1) - __ldg(P + (size_t)iy2 * pitch + ix2));
}

}   // namespace fdcm
