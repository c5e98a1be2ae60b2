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

}   // namespace fdcm
