// dt3_kernels.cu — hot path 1: DT3 feature-map build kernels (sm_100a).
//
// Pipeline (reference: buildCpuFeaturemap, matching/featuremaps/dt3cpu.h:174-234):
//   K1 raster_kernel            drawLines: clipLines + rasterizeLine per orientation plane  -> 1-bit edge mask
//   K2 dt_col_exact_kernel      first (vertical) pass of distanceTransform on the binary mask -> u16 distance
//      dt_pass_literal_kernel   Felzenszwalb lower-envelope pass, literal incl. the in-place aliasing
//      dt_row_l1_kernel         L1 second pass
//   K3 propagate_kernel         propagateOrientation: 4*D circular min-plus steps, D values in registers
//   K4 integral_tma.cu          lineIntegral: sequential fp32 running sums along each plane's discrete lines
// Layout: orientation-major [D][H][pitch] fp32, pitch % 32 == 0.
// All float arithmetic is non-fused (-fmad=false) and ordered exactly as the reference's expressions.
#include <cstdlib>

#include "common.cuh"
#include "kernels.h"

namespace fdcm {

// =============================================================================================
// K1: clip + rasterise scene lines into the per-plane edge bit mask
// =============================================================================================
__device__ __forceinline__ int outcode_dev(float x, float y, float xmax, float ymax) {
    int code = 0;   // core/src/drawing.cpp:37-50 (LEFT=1 RIGHT=2 BOTTOM=4 TOP=8), box [0,xmax]x[0,ymax]
    if (x < 0.f) code |= 1; else if (x > xmax) code |= 2;
    if (y < 0.f) code |= 4; else if (y > ymax) code |= 8;
    return code;
}

// Cohen-Sutherland (core/src/drawing.cpp:64-112); returns false when the line is purged
__device__ bool clip_line_dev(float& x1, float& y1, float& x2, float& y2, float xmax, float ymax) {
    int c1 = outcode_dev(x1, y1, xmax, ymax);
    int c2 = outcode_dev(x2, y2, xmax, ymax);
    for (int it = 0; it < 16; ++it) {   // the reference loop ends after <= 4 clips; bound guards NaN input
        if (c1 == 0 && c2 == 0) return true;
        if (c1 & c2) return false;
        if (c1 != 0) {
            if (c1 & 8)      { x1 = x1 + (x2 - x1) * (ymax - y1) / (y2 - y1); y1 = ymax; }
            else if (c1 & 4) { x1 = x1 + (x2 - x1) * (0.f - y1) / (y2 - y1); y1 = 0.f; }
            else if (c1 & 2) { y1 = y1 + (y2 - y1) * (xmax - x1) / (x2 - x1); x1 = xmax; }
            else if (c1 & 1) { y1 = y1 + (y2 - y1) * (0.f - x1) / (x2 - x1); x1 = 0.f; }
            c1 = outcode_dev(x1, y1, xmax, ymax);
            continue;
        }
        if (c2 & 8)      { x2 = x2 + (x1 - x2) * (ymax - y2) / (y1 - y2); y2 = ymax; }
        else if (c2 & 4) { x2 = x2 + (x1 - x2) * (0.f - y2) / (y1 - y2); y2 = 0.f; }
        else if (c2 & 2) { y2 = y2 + (y1 - y2) * (xmax - x2) / (x1 - x2); x2 = xmax; }
        else if (c2 & 1) { y2 = y2 + (y1 - y2) * (0.f - x2) / (x1 - x2); x2 = 0.f; }
        c2 = outcode_dev(x2, y2, xmax, ymax);
    }
    return false;
}

__device__ __forceinline__ void set_edge(uint32_t* mask, const MapDims& dm, int plane, long long x, long long y) {
    if (x < 0 || y < 0 || x >= dm.W || y >= dm.H) return;   // unreachable after clipping; guards NaN input
    atomicOr(mask + ((size_t)plane * dm.H + (size_t)y) * dm.wwords + (x >> 5), 1u << (x & 31));
}

// one warp per scene line (lines already shifted by the scene translation, dt3cpu.h:185)
__global__ void __launch_bounds__(256) raster_kernel(const float4* __restrict__ lines, const int32_t* __restrict__ bins,
                                                     int n_lines, MapDims dm, uint32_t* __restrict__ mask) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= n_lines) return;
    const float4 l = lines[warp];
    const int plane = bins[warp];
    float p1x = l.x, p1y = l.y, p2x = l.z, p2y = l.w;
    if (!clip_line_dev(p1x, p1y, p2x, p2y, (float)(dm.W - 1), (float)(dm.H - 1))) return;   // core/drawing.h:117-118
    // rasterizeLine (core/drawing.h:74-102)
    const RasterLineDev rl(p1x, p1y, p2x, p2y);
    for (int i = lane; i < rl.n; i += 32) {
        long long x, y;
        rl.at(i, x, y);
        set_edge(mask, dm, plane, x, y);
    }
}


// =============================================================================================
// K2b: the literal Felzenszwalb pass (core/imgproc.h:91-130) for maps beyond the integer-exact regime (side > 2897),
// where float(q^2) rounds and the reference's float arithmetic has to be replayed operation by operation.
// One thread per COLUMN walks down its column: plane, envelope stack (v, z) and output accesses of a warp are
// coalesced 128-byte rows.  The reference runs the same column pass twice with a transposition in between
// (imgproc.h:186-190); so does this path (transpose_square_kernel), instead of a row pass whose lanes would sit a
// whole pitch apart.  The second loop reproduces the reference's in-place read of img(v_k, i): when v_k < q the
// value has already been overwritten.
// kSrc: where the pass reads its input from
//   kSrcPlane: the plane itself (second call)
//   kSrcMask : the 1-bit edge mask, f = edge ? 0 : FLT_MAX (first call: the {0, FLT_MAX} image of imgproc.h:174-175 is
//              never materialised)
//   kSrcG16  : explicit u16 distances g, f = g * g, 0xFFFF -> FLT_MAX (fdcm_debug_dt_rows)
// =============================================================================================
struct EnvEntry { int v; float z; };
enum { kSrcPlane = 0, kSrcMask = 1, kSrcG16 = 2 };

template <int kSrc>
__global__ void __launch_bounds__(128) dt_pass_literal_kernel(const void* __restrict__ src, float* planes, MapDims dm,
                                                              EnvEntry* stack, int n, int n_lines, size_t elem_stride,
                                                              size_t line_stride) {
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    const int d = blockIdx.y;
    if (l >= n_lines) return;
    const size_t base = (size_t)d * dm.plane_elems + (size_t)l * line_stride;
    float* out = planes + base;
    const uint16_t* gin = kSrc == kSrcG16 ? reinterpret_cast<const uint16_t*>(src) + base : nullptr;
    // mask mode: scan line l is column l (elem_stride = pitch): bit (l & 31) of word (l >> 5) of every row
    const uint32_t* mrow = kSrc == kSrcMask ? reinterpret_cast<const uint32_t*>(src) + (size_t)d * dm.H * dm.wwords + (l >> 5) : nullptr;
    const uint32_t mbit = 1u << (l & 31);
    EnvEntry* st = stack + base;
    auto F = [&](int q) -> float {
        if (kSrc == kSrcG16) {
            const unsigned gv = gin[(size_t)q * elem_stride];
            return gv == kNoEdge16 ? FLT_MAX : (float)(gv * gv);
        }
        if (kSrc == kSrcMask) return (mrow[(size_t)q * dm.wwords] & mbit) ? 0.f : FLT_MAX;
        return out[(size_t)q * elem_stride];
    };
    // first loop: lower envelope (imgproc.h:101-121); top of stack cached in registers
    int k = 0, vk = 0;
    float fvk = F(0), zk = -INFINITY;
    st[0] = EnvEntry{0, -INFINITY};
    for (int q = 1; q < n; ++q) {
        const float fq = F(q);
        const float sqq = (float)((long long)q * q);
        while (true) {
            const float s = (fq + sqq - fvk - (float)((long long)vk * vk)) / (float)(2LL * q - 2LL * vk);
            if (s > zk) {
                ++k;
                st[(size_t)k * elem_stride] = EnvEntry{q, s};
                vk = q; fvk = fq; zk = s;
                break;
            }
            --k;
            const EnvEntry e = st[(size_t)k * elem_stride];
            vk = e.v; zk = e.z; fvk = F(vk);
        }
    }
    // second loop (imgproc.h:122-128), in place
    int k2 = 0, v = 0;
    float znext = (k >= 1) ? st[elem_stride].z : INFINITY;
    for (int q = 0; q < n; ++q) {
        while (znext < (float)q) {
            ++k2;
            v = st[(size_t)k2 * elem_stride].v;
            znext = (k2 + 1 <= k) ? st[(size_t)(k2 + 1) * elem_stride].z : INFINITY;
        }
        const long long dq = (long long)q - v;
        const float srcv = (kSrc != kSrcPlane && v >= q) ? F(v) : out[(size_t)v * elem_stride];
        out[(size_t)q * elem_stride] = srcv + (float)(dq * dq);
    }
}

// in-place transposition of the square W x W region of every plane (img.transposeInPlace(), imgproc.h:187,189):
// one CTA per pair of 32 x 32 tiles (i <= j), both staged through shared memory
__global__ void __launch_bounds__(256) transpose_square_kernel(float* __restrict__ planes, MapDims dm, int ntiles) {
    __shared__ float A[32][33], B[32][33];
    // linear index of the pair (ti <= tj) in the upper triangle, row by row
    int t = blockIdx.x, ti = 0;
    while (t >= ntiles - ti) { t -= ntiles - ti; ++ti; }
    const int tj = ti + t;
    float* P = planes + (size_t)blockIdx.y * dm.plane_elems;
    const int lx = threadIdx.x & 31, ly = threadIdx.x >> 5;   // 32 x 8 threads
    const int n = dm.W;
    for (int r = ly; r < 32; r += 8) {
        const int ya = ti * 32 + r, xa = tj * 32 + lx;        // tile (ti, tj): rows of ti, columns of tj
        const int yb = tj * 32 + r, xb = ti * 32 + lx;        // tile (tj, ti)
        A[r][lx] = (ya < n && xa < n) ? P[(size_t)ya * dm.pitch + xa] : 0.f;
        B[r][lx] = (yb < n && xb < n) ? P[(size_t)yb * dm.pitch + xb] : 0.f;
    }
    __syncthreads();
    for (int r = ly; r < 32; r += 8) {
        const int ya = ti * 32 + r, xa = tj * 32 + lx;
        const int yb = tj * 32 + r, xb = ti * 32 + lx;
        if (ya < n && xa < n) P[(size_t)ya * dm.pitch + xa] = B[lx][r];   // (ti, tj) <- transpose of (tj, ti)
        if (ti != tj && yb < n && xb < n) P[(size_t)yb * dm.pitch + xb] = A[lx][r];
    }
}

__global__ void __launch_bounds__(256) sqrt_kernel(float* __restrict__ planes, size_t total) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < total) planes[i] = sqrtf(planes[i]);
}

// =============================================================================================
// K3: propagateOrientation (matching/src/featuremaps/dt3cpu.cpp:77-107).  One thread per pixel keeps
// the D-long orientation vector in registers through the forward (ceil(1.5D)) and backward
// (D + floor(1.5D)) circular sweeps; P[c2] = min(P[c2], P[c1] + w_step).  sqrt_first fuses the final
// elementwise sqrt of the L2 transform (core/imgproc.h:191-192) into the load.
// =============================================================================================
template <int D>
__global__ void __launch_bounds__(128) propagate_kernel(float* __restrict__ planes, MapDims dm,
                                                        const __grid_constant__ PropParams pp, int sqrt_first) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= dm.plane_elems || (int)(i % dm.pitch) >= dm.W) return;
    float v[D];
#pragma unroll
    for (int d = 0; d < D; ++d) v[d] = planes[(size_t)d * dm.plane_elems + i];
    if (sqrt_first) {
#pragma unroll
        for (int d = 0; d < D; ++d) v[d] = sqrtf(v[d]);
    }
    constexpr int fwd = (3 * D + 1) / 2;
    constexpr int bwd = D + (3 * D) / 2;
#pragma unroll
    for (int c = 0; c < fwd; ++c) {
        const int c1 = (D + ((c - 1) % D)) % D;
        const int c2 = c % D;
        v[c2] = fminf(v[c2], v[c1] + pp.w[c]);
    }
#pragma unroll
    for (int j = 0; j < bwd; ++j) {
        const int c = D - j;
        const int c1 = (D + ((c + 1) % D)) % D;
        const int c2 = (D + (c % D)) % D;
        v[c2] = fminf(v[c2], v[c1] + pp.w[fwd + j]);
    }
#pragma unroll
    for (int d = 0; d < D; ++d) planes[(size_t)d * dm.plane_elems + i] = v[d];
}

// any depth (orientation vector in local memory)
__global__ void __launch_bounds__(128) propagate_generic_kernel(float* __restrict__ planes, MapDims dm,
                                                                const __grid_constant__ PropParams pp, int sqrt_first) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= dm.plane_elems || (int)(i % dm.pitch) >= dm.W) return;
    float v[kMaxDepthDev];
    for (int d = 0; d < dm.D; ++d) {
        const float x = planes[(size_t)d * dm.plane_elems + i];
        v[d] = sqrt_first ? sqrtf(x) : x;
    }
    for (int s = 0; s < pp.n_steps; ++s) {
        const int c1 = pp.c1[s], c2 = pp.c2[s];
        v[c2] = fminf(v[c2], v[c1] + pp.w[s]);
    }
    for (int d = 0; d < dm.D; ++d) planes[(size_t)d * dm.plane_elems + i] = v[d];
}

// =============================================================================================
// launchers
// =============================================================================================
static inline unsigned cdiv(size_t a, size_t b) { return (unsigned)((a + b - 1) / b); }

void launch_raster(const float* d_lines, const int32_t* d_bins, int n_lines, const MapDims& dm, uint32_t* d_mask,
                   cudaStream_t s) {
    if (n_lines <= 0) return;
    raster_kernel<<<cdiv((size_t)n_lines * 32, 256), 256, 0, s>>>(reinterpret_cast<const float4*>(d_lines), d_bins, n_lines,
                                                                   dm, d_mask);
}

// src_kind: 0 = the plane itself, 1 = the edge mask, 2 = explicit u16 distances
void launch_dt_pass_literal(int src_kind, bool along_rows, const void* d_src, float* d_planes, const MapDims& dm, void* d_stack,
                            cudaStream_t s) {
    const int n = along_rows ? dm.W : dm.H;
    const int n_lines = along_rows ? dm.H : dm.W;
    const size_t es = along_rows ? 1 : (size_t)dm.pitch;
    const size_t ls = along_rows ? (size_t)dm.pitch : 1;
    dim3 grid(cdiv(n_lines, 128), dm.D);
    if (src_kind == kSrcG16)
        dt_pass_literal_kernel<kSrcG16><<<grid, 128, 0, s>>>(d_src, d_planes, dm, (EnvEntry*)d_stack, n, n_lines, es, ls);
    else if (src_kind == kSrcMask)
        dt_pass_literal_kernel<kSrcMask><<<grid, 128, 0, s>>>(d_src, d_planes, dm, (EnvEntry*)d_stack, n, n_lines, es, ls);
    else
        dt_pass_literal_kernel<kSrcPlane><<<grid, 128, 0, s>>>(d_src, d_planes, dm, (EnvEntry*)d_stack, n, n_lines, es, ls);
}

void launch_transpose_square(float* d_planes, const MapDims& dm, cudaStream_t s) {
    const int nt = (dm.W + 31) / 32;
    dim3 grid((unsigned)((size_t)nt * (nt + 1) / 2), dm.D);
    transpose_square_kernel<<<grid, 256, 0, s>>>(d_planes, dm, nt);
}

void launch_sqrt(float* d_planes, const MapDims& dm, cudaStream_t s) {
    const size_t total = (size_t)dm.D * dm.plane_elems;
    sqrt_kernel<<<cdiv(total, 256), 256, 0, s>>>(d_planes, total);
}

void launch_propagate(float* d_planes, const MapDims& dm, const PropParams& pp, bool sqrt_first, cudaStream_t s) {
    const unsigned grid = cdiv(dm.plane_elems, 128);
    switch (dm.D) {
        case 30: propagate_kernel<30><<<grid, 128, 0, s>>>(d_planes, dm, pp, sqrt_first ? 1 : 0); break;
        case 4: propagate_kernel<4><<<grid, 128, 0, s>>>(d_planes, dm, pp, sqrt_first ? 1 : 0); break;
        default: propagate_generic_kernel<<<grid, 128, 0, s>>>(d_planes, dm, pp, sqrt_first ? 1 : 0); break;
    }
}

}   // namespace fdcm
