// search_kernels.cu — hot path 2: template search kernels (sm_100a).
//
// One warp per alignment hypothesis fuses the reference's
//   establishSearchStrategy<DefaultSearch>   (matching/src/searchstrategies/defaultsearch.cpp:29-49)
//   align / transform                        (core/math.h:387-406, 341-344)
//   optimize<BatchOptimize|DefaultOptimize>  (matching/src/optimizestrategies/batchoptimize.cpp:15-99)
//   minmaxTranslation / evaluate<Dt3Cpu>     (matching/src/featuremaps/dt3cpu.cpp:30-75, 126-179)
//   Match construction + penalty             (matching/src/matchstrategies/defaultmatch.cpp:76-86)
// Aligned templates are never materialised: every candidate re-applies the 2x3 transform to the
// template lines (broadcast loads) and gathers 2 values per line from the L2/HBM-resident DT3 map.
// Float arithmetic is non-fused and ordered as in the reference (scores use Eigen's packet-4 order).
#include <climits>
#include <cstdlib>

#include <cub/device/device_radix_sort.cuh>

#include "common.cuh"
#include "kernels.h"

namespace fdcm {

struct Rigid { float r00, r01, tx, r10, r11, ty; };

// colwise().normalized() (core/math.h:331-333; Eigen: z>0 ? v/sqrt(z) : v)
__device__ __forceinline__ void unit_vec_dev(const float4 l, float& ux, float& uy) {
    const float dx = l.z - l.x, dy = l.w - l.y;
    const float z = dx * dx + dy * dy;
    if (z > 0.f) {
        const float n = sqrtf(z);
        ux = dx / n;
        uy = dy / n;
    } else {
        ux = dx;
        uy = dy;
    }
}

// core/math.h:341-344: coefficient-based 2x2 product then + translation
__device__ __forceinline__ void xform(const Rigid& T, float x, float y, float& ox, float& oy) {
    ox = (T.r00 * x + T.r01 * y) + T.tx;
    oy = (T.r10 * x + T.r11 * y) + T.ty;
}

// core/math.h:387-406 align(); rev selects the second (180-degree) solution
__device__ __forceinline__ Rigid align_dev(const float4 tl, const float4 sl, int rev, float& avx, float& avy) {
    float tx, ty;
    unit_vec_dev(tl, tx, ty);
    unit_vec_dev(sl, avx, avy);
    float c = avx * tx + avy * ty;
    float s = avy * tx - avx * ty;
    const float cx = (sl.z + sl.x) / 2, cy = (sl.w + sl.y) / 2;
    float r00, r01, r10, r11;
    if (!rev) { r00 = c; r01 = -s; r10 = s; r11 = c; }
    else { r00 = -c; r01 = s; r10 = -s; r11 = -c; }
    const float p1x = r00 * tl.x + r01 * tl.y, p1y = r10 * tl.x + r11 * tl.y;
    const float p2x = r00 * tl.z + r01 * tl.w, p2y = r10 * tl.z + r11 * tl.w;
    const float mx = (p2x + p1x) / 2, my = (p2y + p1y) / 2;
    return Rigid{r00, r01, cx - mx, r10, r11, cy - my};
}

// minmaxTranslation (dt3cpu.cpp:30-75) given the bbox of the aligned template already shifted by the
// scene translation
__device__ void minmax_dev(float mnx, float mny, float mxx, float mxy, float sizex, float sizey, float vx, float vy,
                           float& lo, float& hi) {
    const float inf = INFINITY, nan = NAN;
    if (fabsf(vx) <= 1e-5f && fabsf(vy) <= 1e-5f) { lo = hi = inf; return; }
    if ((sizex - 1 - mxx) < 0 || (sizey - 1 - mxy) < 0 || mnx < 0 || mny < 0) { lo = hi = nan; return; }
    float E0[2], E1[2];
#pragma unroll
    for (int a = 0; a < 2; ++a) {
        const float mn = a ? mny : mnx, mx = a ? mxy : mxx, sz = a ? sizey : sizex, v = a ? vy : vx;
        const float m[4] = {(-mx) / v, (-mn) / v, (sz - mx - 1.f) / v, (sz - mn - 1.f) / v};
        float neg_max = -inf, pos_min = inf;
        bool neg_nan = false, pos_nan = false;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const bool sg = signbit(m[j]);
            const float pos = sg ? inf : m[j];
            const float neg = sg ? m[j] : -inf;
            pos_nan |= (pos != pos);
            neg_nan |= (neg != neg);
            if (neg > neg_max) neg_max = neg;
            if (pos < pos_min) pos_min = pos;
        }
        E0[a] = neg_nan ? nan : neg_max;
        E1[a] = pos_nan ? nan : pos_min;
    }
    const bool f0 = isfinite(E0[0]) && isfinite(E1[0]);
    const bool f1 = isfinite(E0[1]) && isfinite(E1[1]);
    if (f0 && f1) { lo = fmaxf(E0[0], E0[1]); hi = fminf(E1[0], E1[1]); }
    else if (f0) { lo = E0[0]; hi = E1[0]; }
    else { lo = E0[1]; hi = E1[1]; }
}

// (long) conversion of the reference (batchoptimize.cpp:51): truncation toward zero
__device__ __forceinline__ long long trunc_ll(float x) { return (long long)x; }

// hypothesis index -> (template, template line, scene line, reversed): establishSearchStrategy<DefaultSearch>
// (defaultsearch.cpp:29-49) evaluated for one combination
struct HypDecode { int t, l0, L, tline, sline, rev; };
__device__ __forceinline__ HypDecode decode_hypothesis(long long h, const TemplatesView& tv, const SceneView& sv, const SearchLaunch& sl) {
    HypDecode r;
    int lo = 0, hi = tv.n_tmpl;   // largest t with hyp_off[t] <= h
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (sl.hyp_off[mid] <= h) lo = mid; else hi = mid;
    }
    r.t = lo;
    const int loc = (int)(h - sl.hyp_off[r.t]);
    r.l0 = tv.offsets[r.t];
    r.L = tv.offsets[r.t + 1] - r.l0;
    const int nS = min(sv.n, sl.max_scene_lines);
    const int rank = loc / (2 * nS);
    const int slot = (loc >> 1) % nS;
    r.rev = loc & 1;
    r.tline = tv.argsort[r.l0 + rank];
    const float value = tv.line_len[r.l0 + r.tline];      // binarySearch with std::greater (core/math.h:138-146)
    int b0 = 0, b1 = sv.n;
    while (b0 < b1) {
        const int mid = (b0 + b1) >> 1;
        if (sv.sorted_len[mid] > value) b0 = mid + 1; else b1 = mid;
    }
    int closest;
    if (b0 == 0) closest = 0;
    else if (b0 == sv.n) closest = sv.n - 1;
    else closest = fabsf(value - sv.sorted_len[b0]) < fabsf(value - sv.sorted_len[b0 - 1]) ? b0 : b0 - 1;
    int rb = max(0, closest - sl.max_scene_lines / 2);   // getCenteredRange (defaultsearch.h:40-47)
    const int re = min(rb + sl.max_scene_lines, sv.n);
    rb = max(0, re - sl.max_scene_lines);
    r.sline = sv.sorted_idx[rb + slot];
    return r;
}

// Spatial sort key of a hypothesis: the cell (kSearchCellW x kSearchCellH pixels, row-major) of the centre of its scene line.  All
// hypotheses aligned on nearby scene lines gather from the same neighbourhood of the map, so processing them
// together keeps that neighbourhood (all D planes) resident in L2.  The order only affects scheduling; results
// are written at the hypothesis index.
__global__ void search_key_kernel(const __grid_constant__ TemplatesView tv, const __grid_constant__ SceneView sv,
                                  const __grid_constant__ SearchLaunch sl, float minx, float miny, int cells_x,
                                  uint32_t* __restrict__ keys, int32_t* __restrict__ idx, int4* __restrict__ hyp) {
    const long long h = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= sl.n_hyp) return;
    const HypDecode d = decode_hypothesis(h, tv, sv, sl);
    hyp[h] = make_int4(d.t + sl.tmpl_idx_base, d.tline, d.sline, d.rev);   // the search kernel reads it back
    const float4 s = sv.lines[d.sline];
    const int cx = min(max((int)(((s.x + s.z) * 0.5f - minx) * (1.f / (float)kSearchCellW)), 0), cells_x - 1);
    const int cy = min(max((int)(((s.y + s.w) * 0.5f - miny) * (1.f / (float)kSearchCellH)), 0), 4095);
    keys[h] = (uint32_t)(cy * cells_x + cx);
    idx[h] = (int32_t)h;
}

size_t search_order_temp_bytes(int64_t n_hyp) {
    size_t bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const uint32_t*)nullptr, (uint32_t*)nullptr, (const int32_t*)nullptr,
                                    (int32_t*)nullptr, (int)n_hyp);
    return bytes;
}

void launch_search_order(const TemplatesView& tv, const SceneView& sv, const SearchLaunch& sl, uint32_t* d_keys, uint32_t* d_keys_out,
                         int32_t* d_idx, int32_t* d_perm, void* d_temp, size_t temp_bytes, float minx, float miny, int cells_x,
                         int key_bits, int4* d_hyp, cudaStream_t s) {
    search_key_kernel<<<(unsigned)((sl.n_hyp + 255) / 256), 256, 0, s>>>(tv, sv, sl, minx, miny, cells_x, d_keys, d_idx, d_hyp);
    cub::DeviceRadixSort::SortPairs(d_temp, temp_bytes, d_keys, d_keys_out, d_idx, d_perm, (int)sl.n_hyp, 0, key_bits, s);
}

// =============================================================================================
// K5+K6, warp-per-hypothesis version: lanes = consecutive candidate translations.
// BatchOptimize scores the translations j * (svx, svy), j integer, and (svx, svy) has one unit component
// (rasterizeVector), so the candidates of a hypothesis lie on a discrete line and the lookups of all candidates for
// one template-line end point form a STREAK of adjacent pixels.  Lane l scores multiplier lo + l: one gather
// instruction then touches a handful of 128-byte lines instead of 32 unrelated ones (the L1TEX wavefront count is
// what bounds this kernel), and every lane runs Eigen's packet-4 / 2x-unrolled summation order on its own, so no
// cross-lane reduction is needed.  Scores are pure functions of the multiplier: a window of up to 32 multipliers
// around 0 is scored up front (it contains the first batch of either direction, which the reference always
// evaluates), further ranges on demand; the control flow of batchoptimize.cpp:51-94 then consumes them in order.
// =============================================================================================
__global__ void __launch_bounds__(128, 6) search_warp_kernel(const __grid_constant__ MapView map,
                                                          const __grid_constant__ SlopeTableDev table,
                                                          const __grid_constant__ TemplatesView tv,
                                                          const __grid_constant__ SceneView sv,
                                                          const __grid_constant__ SearchLaunch sl,
                                                          const __grid_constant__ SearchOutputs out) {
    extern __shared__ __align__(16) uint8_t s_raw[];   // per warp: aligned end points float4[max_lines], planes u8[max_lines]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long slot_idx = (long long)blockIdx.x * (blockDim.x >> 5) + warp;
    if (slot_idx >= sl.n_hyp) return;     // whole warp
    const long long h = sl.perm ? (long long)sl.perm[slot_idx] : slot_idx;
    const size_t per_warp = (size_t)tv.max_lines * 16 + (((size_t)tv.max_lines + 15) & ~(size_t)15);
    float4* apts = reinterpret_cast<float4*>(s_raw + (size_t)warp * per_warp);   // transform(T, line) (core/math.h:341-344)
    uint8_t* bins = reinterpret_cast<uint8_t*>(apts + tv.max_lines);
    unsigned long long n_eval = 0;
    bool valid = false;

    int t, l0, L;
    float avx, avy;
    Rigid T;
    if (sl.direct_align) {
        // optimize<BatchOptimize>(templates, alignments, featuremap) (batchoptimize.cpp:6-123): template h as given
        t = (int)h;
        l0 = tv.offsets[t];
        L = tv.offsets[t + 1] - l0;
        T = Rigid{1.f, 0.f, 0.f, 0.f, 1.f, 0.f};      // x*1 + y*0 + 0 is exact: coordinates pass through unchanged
        avx = sl.direct_align[h].x;
        avy = sl.direct_align[h].y;
    } else {
        HypDecode d;
        if (sl.hyp_ready) {                   // decoded by the ordering pass
            const int4 q = sl.hyp_ready[h];
            d.t = q.x - sl.tmpl_idx_base; d.tline = q.y; d.sline = q.z; d.rev = q.w;
            d.l0 = tv.offsets[d.t];
            d.L = tv.offsets[d.t + 1] - d.l0;
        } else {
            d = decode_hypothesis(h, tv, sv, sl);
            if (lane == 0) out.hyp[h] = make_int4(d.t + sl.tmpl_idx_base, d.tline, d.sline, d.rev);
        }
        t = d.t; l0 = d.l0; L = d.L;
        T = align_dev(tv.lines[l0 + d.tline], sv.lines[d.sline], d.rev, avx, avy);   // defaultmatch.cpp:57-69
    }
    const float4* TL = tv.lines + l0;
    const float asum = fabsf(avx) + fabsf(avy);
    const bool null_vec = (double)asum <= (double)FLT_EPSILON + 1e-10 * (double)asum;   // batchoptimize.cpp:20
    if (!null_vec) {
        float svx, svy;
        rasterize_vector_dev(avx, avy, svx, svy);
        // bbox of the aligned template + orientation plane of every line (lane takes lines lane, lane+32, ...)
        float mnx = INFINITY, mny = INFINITY, mxx = -INFINITY, mxy = -INFINITY;
        for (int i = lane; i < L; i += 32) {
            const float4 p = __ldg(TL + i);
            float ax, ay, bx, by;
            xform(T, p.x, p.y, ax, ay);
            xform(T, p.z, p.w, bx, by);
            mnx = fminf(mnx, fminf(ax, bx)); mxx = fmaxf(mxx, fmaxf(ax, bx));
            mny = fminf(mny, fminf(ay, by)); mxy = fmaxf(mxy, fmaxf(ay, by));
            apts[i] = make_float4(ax, ay, bx, by);     // the aligned template: identical for every candidate translation
            bins[i] = (uint8_t)bin_of_slope_dev(table, (by - ay) / (bx - ax));
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            mnx = fminf(mnx, __shfl_xor_sync(0xffffffffu, mnx, o)); mxx = fmaxf(mxx, __shfl_xor_sync(0xffffffffu, mxx, o));
            mny = fminf(mny, __shfl_xor_sync(0xffffffffu, mny, o)); mxy = fmaxf(mxy, __shfl_xor_sync(0xffffffffu, mxy, o));
        }
        __syncwarp();
        float min_mul, max_mul;
        minmax_dev(mnx + map.shift_x, mny + map.shift_y, mxx + map.shift_x, mxy + map.shift_y, (float)map.dm.W,
                   (float)map.dm.H, svx, svy, min_mul, max_mul);
        if (isfinite(min_mul) && isfinite(max_mul)) {
            const float* planes = map.planes;
            const unsigned pitch = (unsigned)map.dm.pitch;
            const unsigned last = (unsigned)(map.dm.plane_elems - 1);
            // (long) conversions of batchoptimize.cpp:51,74; |multiplier| < map side <= 65534, so int arithmetic is exact
            const int maxm = (int)min(max(trunc_ll(max_mul), -70000LL), 70000LL), minm = (int)min(max(trunc_ll(min_mul), -70000LL), 70000LL);
            // score of multiplier m on this lane (dt3cpu.cpp:126-179)
            auto score_of = [&](int mult) -> float {
                const float m = (float)mult;
                const float offx = map.shift_x + m * svx, offy = map.shift_y + m * svy;   // sceneTranslation + translation
                return eigen_sum_lazy(L, [&](int i) {
                    const float4 a = apts[i];
                    const int x1 = (int)(a.x + offx), y1 = (int)(a.y + offy), x2 = (int)(a.z + offx), y2 = (int)(a.w + offy);
                    // inside the minmaxTranslation bounds every index is in range; the clamp only guards non-finite input
                    const unsigned i1 = min((unsigned)y1 * pitch + (unsigned)x1, last), i2 = min((unsigned)y2 * pitch + (unsigned)x2, last);
                    const float* P = planes + (size_t)bins[i] * map.dm.plane_elems;
                    return fabsf(__ldg(P + i1) - __ldg(P + i2));
                });
            };
            // cached range of scores: lane l holds the score of multiplier c_lo + l, l < c_n
            int c_lo = 0, c_n = 0;
            float c_score = 0.f;
            auto fill_cache = [&](int lo, int hi) {   // lo <= hi, hi - lo < 32, both inside [minm, maxm]
                c_lo = lo;
                c_n = hi - lo + 1;
                if (lane < c_n) c_score = score_of(lo + lane);
                __syncwarp();
            };
            // score of multiplier j (uniform); dir = direction in which further multipliers will be asked for
            // Ranges are as wide as one batch (every candidate of a started batch is evaluated by the reference) or, for
            // small batches, as wide as the warp: a few speculative scores cost less than idle lanes.
            const int B = sl.batch;
            const int span = B >= 8 ? min(B, 32) : 32;
            auto score_at = [&](int j, int dir) -> float {
                if (j < c_lo || j >= c_lo + c_n) {
                    if (dir > 0) fill_cache(j, min(maxm, j + span - 1));
                    else fill_cache(max(minm, j - span + 1), j);
                }
                return __shfl_sync(0xffffffffu, c_score, j - c_lo);
            };
            {   // first window: 0 and the first batch of both directions when they fit into the warp
                int lo, hi;
                if (2 * span + 1 <= 32) { lo = max(minm, -span); hi = min(maxm, span); }
                else if (span >= 16) { lo = 0; hi = min(maxm, min(span, 31)); }     // 0 and the whole first batch upwards when it fits
                else { lo = max(minm, -15); hi = min(maxm, 16); }
                if (lo > 0) lo = 0;            // (limits always include 0: the template is inside the map at t = 0)
                if (hi < 0) hi = 0;
                fill_cache(lo, hi);
            }
            float back = score_at(0, 1);                  // scores.back()
            n_eval += 1;
            float best = back, best_tx = 0.f, best_ty = 0.f;
            for (int dir = 1; dir >= -1; dir -= 2) {
                // batchoptimize.cpp:51-71 (dir = +1) and :74-94 (dir = -1)
                const int lim = dir > 0 ? maxm : -minm;           // multipliers run 1..lim in units of dir
                for (int kk = 1; kk <= lim; kk += B) {
                    const int jend = min(kk + B - 1, lim);
                    float bmin = 0.f, blast = 0.f;
                    int barg = kk;
                    (void)score_at(dir * kk, dir);                    // makes the cached range start at this batch if needed
                    const int la = dir * kk - c_lo, lb = dir * jend - c_lo;          // lanes of the first / last candidate
                    const bool inside = min(la, lb) >= 0 && max(la, lb) < c_n;
                    const unsigned bmask = inside ? (0xFFFFFFFFu >> (31 - max(la, lb))) & (0xFFFFFFFFu << min(la, lb)) : 0u;
                    const bool in_batch = (bmask >> lane) & 1u;
                    // scores are sums of absolute values: non-negative floats order like their bit patterns; NaN (an
                    // empty plane under a line) takes the sequential path so that `s < bmin` keeps its exact meaning
                    if (inside && __ballot_sync(0xffffffffu, in_batch && !(c_score >= 0.f)) == 0u) {
                        const unsigned key = in_batch ? __float_as_uint(c_score) : 0xFFFFFFFFu;
                        const unsigned kmin = __reduce_min_sync(0xffffffffu, key);
                        const unsigned hit = __ballot_sync(0xffffffffu, in_batch && key == kmin);
                        const int lmin = dir > 0 ? __ffs(hit) - 1 : 31 - __clz(hit);   // first minimum in evaluation order
                        bmin = __uint_as_float(kmin);
                        barg = dir * (c_lo + lmin);
                        blast = __shfl_sync(0xffffffffu, c_score, lb);
                    } else {
                        for (int j = kk; j <= jend; ++j) {
                            const float sj = score_at(dir * j, dir);
                            if (j == kk || sj < bmin) { bmin = sj; barg = j; }   // std::min_element: first minimum
                            blast = sj;
                        }
                    }
                    n_eval += (unsigned long long)(jend - kk + 1);
                    if (bmin > back) break;
                    back = bmin;
                    if (bmin < best) {
                        best = bmin;
                        best_tx = (float)(dir * barg) * svx;
                        best_ty = (float)(dir * barg) * svy;
                    }
                    if (bmin < blast) break;
                }
            }
            valid = true;
            if (lane == 0) {
                fdcm_match m;   // Match{tmplIdx, score, combine(translation, T)} (defaultmatch.cpp:82-84)
                m.tmpl_idx = t + sl.tmpl_idx_base;
                m.score = tv.denom ? best / tv.denom[t] : best;
                m.transform[0] = T.r00; m.transform[1] = T.r01; m.transform[2] = T.tx + best_tx;
                m.transform[3] = T.r10; m.transform[4] = T.r11; m.transform[5] = T.ty + best_ty;
                out.rec[h] = m;
            }
        }
    }
    if (lane == 0) {
        out.valid[h] = valid ? 1 : 0;
        atomicAdd(out.counters + 0, n_eval);
        atomicAdd(out.counters + 1, n_eval * 2ull * (unsigned long long)L);
        atomicAdd(out.counters + 2, valid ? 1ull : 0ull);
    }
}

// shared memory one warp of search_warp_kernel stages a template of max_lines lines in
static size_t search_smem_per_warp(int max_lines) { return (size_t)max_lines * 16 + (((size_t)max_lines + 15) & ~(size_t)15); }

int search_max_template_lines(int smem_optin) {
    int L = smem_optin / 17;
    while (search_smem_per_warp(L + 1) <= (size_t)smem_optin) ++L;
    while (L > 0 && search_smem_per_warp(L) > (size_t)smem_optin) --L;
    return L;
}

cudaError_t launch_search(const MapView& map, const SlopeTableDev& table, const TemplatesView& tv, const SceneView& sv,
                          const SearchLaunch& sl, const SearchOutputs& out, int smem_optin, cudaStream_t s) {
    if (sl.n_hyp <= 0) return cudaSuccess;
    // 4 warps per block; long templates halve that until the block's staging fits the device's opt-in shared memory
    const size_t per_warp = search_smem_per_warp(tv.max_lines);
    int hyps = 4;
    while (hyps > 1 && (size_t)hyps * per_warp > (size_t)smem_optin) hyps >>= 1;
    const size_t smem = (size_t)hyps * per_warp;
    if (smem > (size_t)smem_optin) return cudaErrorInvalidValue;   // callers reject such templates first
    if (smem > 48 * 1024) {
        const cudaError_t e = cudaFuncSetAttribute(search_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    const unsigned grid = (unsigned)((sl.n_hyp + hyps - 1) / hyps);
    search_warp_kernel<<<grid, hyps * 32, smem, s>>>(map, table, tv, sv, sl, out);
    return cudaGetLastError();
}

// fdcm_search_scales rule 4: a valid record of copy v = t * scales + k becomes a record of template t posed at scale s_k
__global__ void search_scale_remap_kernel(const __grid_constant__ ScaleRemapLaunch p) {
    const long long h = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= p.n_hyp || !p.valid[h]) return;
    fdcm_match m = p.rec[h];
    const int v = m.tmpl_idx - p.tmpl_idx_base, t = v / p.scales, k = v - t * p.scales;
    const float s = p.scale[k];
    m.tmpl_idx = t + p.tmpl_idx_base;
    m.transform[0] = s * m.transform[0];
    m.transform[1] = s * m.transform[1];
    m.transform[3] = s * m.transform[3];
    m.transform[4] = s * m.transform[4];
    p.rec[h] = m;
    p.rec_scale[h] = s;
}

void launch_search_scale_remap(const ScaleRemapLaunch& p, cudaStream_t s) {
    if (p.n_hyp <= 0) return;
    search_scale_remap_kernel<<<(unsigned)((p.n_hyp + 255) / 256), 256, 0, s>>>(p);
}

// =============================================================================================
// K7: top-K.  K rounds of a block-wide arg-min over keys (score, index) strictly greater than the
// previously selected key: deterministic, ties broken by hypothesis order.
// =============================================================================================
struct Key { float s; long long i; };
__device__ __forceinline__ bool key_less(const Key& a, const Key& b) { return a.s < b.s || (a.s == b.s && a.i < b.i); }

__device__ Key block_min_key(Key k, Key* s_keys) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        Key other;
        other.s = __shfl_down_sync(0xffffffffu, k.s, o);
        other.i = __shfl_down_sync(0xffffffffu, k.i, o);
        if (key_less(other, k)) k = other;
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) s_keys[warp] = k;
    __syncthreads();
    if (warp == 0) {
        const int nw = blockDim.x >> 5;
        k = lane < nw ? s_keys[lane] : Key{INFINITY, LLONG_MAX};
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            Key other;
            other.s = __shfl_down_sync(0xffffffffu, k.s, o);
            other.i = __shfl_down_sync(0xffffffffu, k.i, o);
            if (key_less(other, k)) k = other;
        }
        if (lane == 0) s_keys[0] = k;
    }
    __syncthreads();
    k = s_keys[0];
    __syncthreads();
    return k;
}

// level 1: block b scans records [b*chunk, (b+1)*chunk) -> k keys per block
__global__ void __launch_bounds__(1024) topk_level1_kernel(const fdcm_match* __restrict__ rec, const uint8_t* __restrict__ valid,
                                                           long long n, long long chunk, int k, float* __restrict__ ws_score,
                                                           long long* __restrict__ ws_idx) {
    __shared__ Key s_keys[32];
    const long long begin = (long long)blockIdx.x * chunk;
    const long long end = min(n, begin + chunk);
    Key last{-INFINITY, -1};
    for (int r = 0; r < k; ++r) {
        Key best{INFINITY, LLONG_MAX};
        for (long long i = begin + threadIdx.x; i < end; i += blockDim.x) {
            if (!valid[i]) continue;
            float s = rec[i].score;
            if (s != s) s = INFINITY;
            const Key c{s, i};
            if (key_less(last, c) && key_less(c, best)) best = c;
        }
        best = block_min_key(best, s_keys);
        if (threadIdx.x == 0) {
            ws_score[(size_t)blockIdx.x * k + r] = best.s;
            ws_idx[(size_t)blockIdx.x * k + r] = best.i;
        }
        last = best;
        if (best.i == LLONG_MAX) {   // exhausted: pad the rest
            for (int q = r + 1 + threadIdx.x; q < k; q += blockDim.x) {
                ws_score[(size_t)blockIdx.x * k + q] = INFINITY;
                ws_idx[(size_t)blockIdx.x * k + q] = LLONG_MAX;
            }
            break;
        }
    }
}

// level 2: one block merges the per-block lists and gathers the winning records
__global__ void __launch_bounds__(1024) topk_level2_kernel(const fdcm_match* __restrict__ rec, const float* __restrict__ ws_score,
                                                           const long long* __restrict__ ws_idx, int n_cand, int k,
                                                           fdcm_match* __restrict__ out, int* __restrict__ n_out) {
    __shared__ Key s_keys[32];
    Key last{-INFINITY, -1};
    int produced = 0;
    for (int r = 0; r < k; ++r) {
        Key best{INFINITY, LLONG_MAX};
        for (int i = threadIdx.x; i < n_cand; i += blockDim.x) {
            const Key c{ws_score[i], ws_idx[i]};
            if (c.i == LLONG_MAX) continue;
            if (key_less(last, c) && key_less(c, best)) best = c;
        }
        best = block_min_key(best, s_keys);
        if (best.i == LLONG_MAX) break;
        if (threadIdx.x == 0) out[r] = rec[best.i];
        last = best;
        ++produced;
    }
    // unused slots: invalid records (tmpl_idx -1, score +inf), so that the k-record buffer can be exchanged as it is
    for (int q = produced + threadIdx.x; q < k; q += blockDim.x) {
        fdcm_match m;
        m.tmpl_idx = -1;
        m.score = INFINITY;
        for (int i = 0; i < 6; ++i) m.transform[i] = 0.f;
        out[q] = m;
    }
    if (threadIdx.x == 0) *n_out = produced;
}

// merge of the ranks' top-k lists (all-gathered, rank-major): the k best of R*k records, ascending score, ties by
// (rank, position in the rank's list) = global hypothesis order when templates are sharded in contiguous blocks
__global__ void __launch_bounds__(256) topk_merge_kernel(const fdcm_match* __restrict__ gathered, int n_cand, int k,
                                                         fdcm_match* __restrict__ out, int* __restrict__ n_out) {
    __shared__ Key s_keys[32];
    Key last{-INFINITY, -1};
    int produced = 0;
    for (int r = 0; r < k; ++r) {
        Key best{INFINITY, LLONG_MAX};
        for (int i = threadIdx.x; i < n_cand; i += blockDim.x) {
            if (gathered[i].tmpl_idx < 0) continue;
            float s = gathered[i].score;
            if (s != s) s = INFINITY;
            const Key c{s, (long long)i};
            if (key_less(last, c) && key_less(c, best)) best = c;
        }
        best = block_min_key(best, s_keys);
        if (best.i == LLONG_MAX) break;
        if (threadIdx.x == 0) out[r] = gathered[best.i];
        last = best;
        ++produced;
    }
    if (threadIdx.x == 0) *n_out = produced;
}

void launch_topk_merge(const fdcm_match* d_gathered, int n_cand, int k, fdcm_match* d_out, int* d_n_out, cudaStream_t s) {
    topk_merge_kernel<<<1, 256, 0, s>>>(d_gathered, n_cand, k, d_out, d_n_out);
}

// an empty shard still takes part in the exchange: k invalid records
__global__ void topk_invalid_kernel(fdcm_match* __restrict__ out, int k, int* __restrict__ n_out) {
    for (int q = threadIdx.x; q < k; q += blockDim.x) {
        fdcm_match m;
        m.tmpl_idx = -1;
        m.score = INFINITY;
        for (int i = 0; i < 6; ++i) m.transform[i] = 0.f;
        out[q] = m;
    }
    if (threadIdx.x == 0) *n_out = 0;
}
void launch_topk_invalid(fdcm_match* d_out, int k, int* d_n_out, cudaStream_t s) { topk_invalid_kernel<<<1, 256, 0, s>>>(d_out, k, d_n_out); }

int topk_ws_blocks(int64_t n) {
    const int64_t per_block = 1024 * 2;
    int64_t b = (n + per_block - 1) / per_block;
    if (b < 1) b = 1;
    if (b > 592) b = 592;   // 4 x 148 SMs
    return (int)b;
}

void launch_topk(const fdcm_match* d_rec, const uint8_t* d_valid, int64_t n, int k, float* d_ws_score, int64_t* d_ws_idx,
                 int ws_blocks, fdcm_match* d_out, int* d_n_out, cudaStream_t s) {
    const long long chunk = (n + ws_blocks - 1) / ws_blocks;
    topk_level1_kernel<<<ws_blocks, 1024, 0, s>>>(d_rec, d_valid, n, chunk, k, d_ws_score, (long long*)d_ws_idx);
    topk_level2_kernel<<<1, 1024, 0, s>>>(d_rec, d_ws_score, (const long long*)d_ws_idx, ws_blocks * k, k, d_out, d_n_out);
}

// =============================================================================================
// Distinct top-K (fdcm_search_select, beyond the reference): greedy walk of the valid matches in (score, h) order that
// caps the matches per template and suppresses matches whose anchors lie within a radius (and a rotation) of an accepted
// one.  Semantics in include/fdcm_b200.h; the keys below order exactly like the top-K kernels' (score, h) comparison.
// =============================================================================================
constexpr uint32_t kInvalidKey = 0xFFFFFFFFu;

// order-preserving 32-bit key of a score: NaN as +inf (0xFF800000, still below kInvalidKey), -0 as +0
__device__ __forceinline__ uint32_t score_key(float s) {
    if (s != s) s = INFINITY;
    if (s == 0.f) s = 0.f;
    const uint32_t u = __float_as_uint(s);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// anchor of a match and the first column of its rotation: (px, py, T0, T3)
__device__ __forceinline__ float4 match_anchor(const fdcm_match& m, float2 a) {
    return make_float4((m.transform[0] * a.x + m.transform[1] * a.y) + m.transform[2],
                       (m.transform[3] * a.x + m.transform[4] * a.y) + m.transform[5], m.transform[0], m.transform[3]);
}

// near(a, b) of the header (the build has no FMA contraction, so this is the fp32 expression as written)
__device__ __forceinline__ bool anchors_near(const float4 a, const float4 b, const SelectLaunch& p) {
    const float dx = a.x - b.x, dy = a.y - b.y;
    if (!(dx * dx + dy * dy <= p.r2)) return false;
    return p.any_angle || a.z * b.z + a.w * b.w >= p.cos_thr;
}
// near(a, b) of the scaled dense search: the angle test against cos_thr * (s_a * s_b), s_a and s_b the grid scales
template <bool kScaled>
__device__ __forceinline__ bool anchors_near(const float4 a, float sa, const float4 b, float sb, const SelectLaunch& p) {
    if constexpr (!kScaled) return anchors_near(a, b, p);
    const float dx = a.x - b.x, dy = a.y - b.y;
    if (!(dx * dx + dy * dy <= p.r2)) return false;
    return p.any_angle || a.z * b.z + a.w * b.w >= p.cos_thr * (sa * sb);
}

__device__ __forceinline__ void write_invalid(fdcm_match* out) {
    fdcm_match m;
    m.tmpl_idx = -1;
    m.score = INFINITY;
    for (int i = 0; i < 6; ++i) m.transform[i] = 0.f;
    *out = m;
}

__global__ void select_key_kernel(const __grid_constant__ SelectLaunch p, bool by_template, uint64_t* __restrict__ keys,
                                  int32_t* __restrict__ vals) {
    const long long h = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= p.n_hyp) return;
    const uint32_t k = p.valid[h] ? score_key(p.rec[h].score) : kInvalidKey;
    uint64_t t = 0;
    if (by_template) {   // largest t with hyp_off[t] <= h
        int lo = 0, hi = p.n_tmpl;
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (p.hyp_off[mid] <= h) lo = mid; else hi = mid;
        }
        t = (uint64_t)lo;
    }
    keys[h] = t << 32 | k;
    vals[h] = (int32_t)h;
}

size_t select_temp_bytes(int64_t n_hyp) {
    size_t b64 = 0, b32 = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, b64, (const uint64_t*)nullptr, (uint64_t*)nullptr, (const int32_t*)nullptr,
                                    (int32_t*)nullptr, (int)n_hyp);
    cub::DeviceRadixSort::SortPairs(nullptr, b32, (const uint32_t*)nullptr, (uint32_t*)nullptr, (const int32_t*)nullptr,
                                    (int32_t*)nullptr, (int)n_hyp);
    return b64 > b32 ? b64 : b32;
}

void launch_select_sort(const SelectLaunch& p, bool by_template, uint64_t* keys_in, uint64_t* keys_out, int32_t* vals_in,
                        int32_t* vals_out, void* d_temp, size_t temp_bytes, cudaStream_t s) {
    select_key_kernel<<<(unsigned)((p.n_hyp + 255) / 256), 256, 0, s>>>(p, by_template, keys_in, vals_in);
    int end_bit = 32;
    if (by_template)
        while (p.n_tmpl > 1 && ((int64_t)1 << (end_bit - 32)) < p.n_tmpl) ++end_bit;
    // radix sort is stable: equal keys keep ascending h
    cub::DeviceRadixSort::SortPairs(d_temp, temp_bytes, keys_in, keys_out, vals_in, vals_out, (int)p.n_hyp, 0, end_bit, s);
}

// One warp per template.  Every rule of the walk involves matches of one template only when across_templates == 0, so
// walking each template's range on its own and keeping the survivors' global (score, h) order (launch_select_topk) gives
// exactly the walk over the global order.  The warp takes its sorted range 32 candidates at a time: each lane tests its
// candidate against the template's accepted anchors, then the chunk is settled in order (the first live lane is accepted
// and removes the live lanes near it).  The walk ends at min(cap, top_k) accepted or at the first invalid key.
// kScaled: the grid scales of the accepted anchors follow the n_hyp anchors of acc
template <bool kScaled>
__global__ void __launch_bounds__(128) select_greedy_kernel(const __grid_constant__ SelectLaunch p, const uint64_t* __restrict__ skeys,
                                                            const int32_t* __restrict__ sh, uint32_t* __restrict__ surv_keys,
                                                            float4* __restrict__ acc) {
    float* __restrict__ acc_s = reinterpret_cast<float*>(acc + p.n_hyp);
    const int lane = threadIdx.x & 31;
    const int t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (t >= p.n_tmpl) return;   // whole warp
    const long long b = p.hyp_off[t], e = p.hyp_off[t + 1];
    const int lim = p.cap > 0 ? min(p.cap, p.top_k) : p.top_k;
    const float2 anchor = p.anchors[t];
    int n_acc = 0;
    for (long long base = b; base < e && n_acc < lim; base += 32) {
        const long long i = base + lane;
        const uint32_t key = i < e ? (uint32_t)skeys[i] : kInvalidKey;
        bool live = key != kInvalidKey;
        const bool last_chunk = __ballot_sync(0xffffffffu, i < e && !live) != 0u;
        const int h = live ? sh[i] : 0;
        float4 me = make_float4(0.f, 0.f, 0.f, 0.f);
        float me_s = 1.f;
        if (live && p.radius_on) {
            me = match_anchor(p.rec[h], anchor);
            if constexpr (kScaled) me_s = p.rec_scale[h];
            for (int j = 0; j < n_acc && live; ++j) live = !anchors_near<kScaled>(acc[b + j], kScaled ? acc_s[b + j] : 1.f, me, me_s, p);
        }
        for (;;) {
            const unsigned alive = __ballot_sync(0xffffffffu, live);
            if (alive == 0u || n_acc == lim) break;
            const int ld = __ffs(alive) - 1;
            const float4 a = make_float4(__shfl_sync(0xffffffffu, me.x, ld), __shfl_sync(0xffffffffu, me.y, ld),
                                         __shfl_sync(0xffffffffu, me.z, ld), __shfl_sync(0xffffffffu, me.w, ld));
            const float a_s = kScaled ? __shfl_sync(0xffffffffu, me_s, ld) : 1.f;
            if (lane == ld) {
                surv_keys[h] = key;
                if (p.radius_on) {
                    acc[b + n_acc] = me;
                    if constexpr (kScaled) acc_s[b + n_acc] = me_s;
                }
                live = false;
            } else if (live && p.radius_on && anchors_near<kScaled>(a, a_s, me, me_s, p)) {
                live = false;
            }
            ++n_acc;
        }
        __syncwarp();   // the accepted anchors written above are read by every lane in the next chunk
        if (last_chunk) break;
    }
}

void launch_select_greedy(const SelectLaunch& p, const uint64_t* sorted_keys, const int32_t* sorted_h, uint32_t* surv_keys, float4* acc,
                          cudaStream_t s) {
    cudaMemsetAsync(surv_keys, 0xFF, (size_t)p.n_hyp * 4, s);
    if (p.rec_scale) select_greedy_kernel<true><<<(unsigned)((p.n_tmpl + 3) / 4), 128, 0, s>>>(p, sorted_keys, sorted_h, surv_keys, acc);
    else select_greedy_kernel<false><<<(unsigned)((p.n_tmpl + 3) / 4), 128, 0, s>>>(p, sorted_keys, sorted_h, surv_keys, acc);
}

__global__ void select_gather_kernel(const uint32_t* __restrict__ skeys, const int32_t* __restrict__ sh, long long n,
                                     const fdcm_match* __restrict__ rec, int k, fdcm_match* __restrict__ out, int* __restrict__ n_out) {
    __shared__ int s_n;
    if (threadIdx.x == 0) s_n = 0;
    __syncthreads();
    int mine = 0;
    for (int q = threadIdx.x; q < k; q += blockDim.x) {
        if (q < n && skeys[q] != kInvalidKey) {
            out[q] = rec[sh[q]];
            ++mine;
        } else {
            write_invalid(out + q);
        }
    }
    atomicAdd(&s_n, mine);
    __syncthreads();
    if (threadIdx.x == 0) *n_out = s_n;
}

void launch_select_topk(const SelectLaunch& p, const uint32_t* surv_keys, uint32_t* keys_out, const int32_t* vals_in, int32_t* vals_out,
                        void* d_temp, size_t temp_bytes, fdcm_match* d_out, int* d_n_out, cudaStream_t s) {
    cub::DeviceRadixSort::SortPairs(d_temp, temp_bytes, surv_keys, keys_out, vals_in, vals_out, (int)p.n_hyp, 0, 32, s);
    select_gather_kernel<<<1, 256, 0, s>>>(keys_out, vals_out, p.n_hyp, p.rec, p.top_k, d_out, d_n_out);
}

// across_templates != 0: one block walks the global (score, h) order blockDim candidates at a time.  Every thread tests its
// candidate against the accepted list in shared memory (anchor, rotation, template: the per-template count for the cap is
// taken in the same pass), then the chunk is settled in order like the warp version above.  Worst case H x top_k tests.
template <bool kScaled>
__global__ void __launch_bounds__(1024) select_walk_kernel(const __grid_constant__ SelectLaunch p, const uint64_t* __restrict__ skeys,
                                                           const int32_t* __restrict__ sh, fdcm_match* __restrict__ out,
                                                           int* __restrict__ n_out) {
    __shared__ float4 s_acc[kSelectMaxAcross];
    __shared__ float s_acc_s[kScaled ? kSelectMaxAcross : 1];   // grid scales of the accepted records
    __shared__ int s_tmpl[kSelectMaxAcross];
    __shared__ unsigned s_live[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, n_warps = blockDim.x >> 5;
    int n_acc = 0;   // uniform
    for (long long base = 0; base < p.n_hyp && n_acc < p.top_k; base += blockDim.x) {
        const long long i = base + tid;
        const uint32_t key = i < p.n_hyp ? (uint32_t)skeys[i] : kInvalidKey;
        bool live = key != kInvalidKey;
        const bool last_chunk = __syncthreads_or(!live) != 0;
        int h = 0, t = -1, same = 0;
        float4 me = make_float4(0.f, 0.f, 0.f, 0.f);
        float me_s = 1.f;
        if (live) {
            h = sh[i];
            const fdcm_match m = p.rec[h];
            t = m.tmpl_idx - p.tmpl_idx_base;
            me = match_anchor(m, p.anchors[t]);
            if constexpr (kScaled) me_s = p.rec_scale[h];
            for (int j = 0; j < n_acc && live; ++j) {
                same += s_tmpl[j] == t;
                live = !(p.radius_on && anchors_near<kScaled>(s_acc[j], kScaled ? s_acc_s[j] : 1.f, me, me_s, p));
            }
            if (p.cap > 0 && same >= p.cap) live = false;
        }
        for (;;) {
            const unsigned m = __ballot_sync(0xffffffffu, live);
            if (lane == 0) s_live[warp] = m;
            __syncthreads();
            int ld = -1;
            for (int w = 0; w < n_warps; ++w)
                if (s_live[w]) { ld = w * 32 + __ffs(s_live[w]) - 1; break; }
            if (ld < 0) break;   // uniform
            if (tid == ld) {
                s_acc[n_acc] = me;
                if constexpr (kScaled) s_acc_s[n_acc] = me_s;
                s_tmpl[n_acc] = t;
                out[n_acc] = p.rec[h];
                live = false;
            }
            __syncthreads();
            const float4 a = s_acc[n_acc];
            const float a_s = kScaled ? s_acc_s[n_acc] : 1.f;
            const int at = s_tmpl[n_acc];
            ++n_acc;
            if (n_acc == p.top_k) break;   // uniform
            if (live) {
                same += at == t;
                if ((p.cap > 0 && same >= p.cap) || (p.radius_on && anchors_near<kScaled>(a, a_s, me, me_s, p))) live = false;
            }
        }
        __syncthreads();   // s_live is rewritten by the next chunk
        if (last_chunk) break;
    }
    for (int q = n_acc + tid; q < p.top_k; q += blockDim.x) write_invalid(out + q);
    if (tid == 0) *n_out = n_acc;
}

void launch_select_walk(const SelectLaunch& p, const uint64_t* sorted_keys, const int32_t* sorted_h, fdcm_match* d_out, int* d_n_out,
                        cudaStream_t s) {
    if (p.rec_scale) select_walk_kernel<true><<<1, 1024, 0, s>>>(p, sorted_keys, sorted_h, d_out, d_n_out);
    else select_walk_kernel<false><<<1, 1024, 0, s>>>(p, sorted_keys, sorted_h, d_out, d_n_out);
}

// =============================================================================================
// Pose refinement (fdcm_refine_matches / fdcm_search_refine, beyond the reference): rules in include/fdcm_b200.h.
// One block per (match, rotation i): the rotated template and its orientation bins are staged in shared memory once, then
// thread (k, j) scores the translation (j h, k h), so that with h = 1 the lanes of a row gather runs of adjacent pixels as
// in the search kernel.  Every thread sums its own candidate in Eigen's order (evaluate<Dt3Cpu>).  The walk's argmin is
// the minimum of a 64-bit key (score, grid order) over all candidates of a match, taken with one atomicMin per warp.
// =============================================================================================
constexpr unsigned long long kNoPose = ~0ull;

// Block-wide (every thread calls it): stage the L lines of a template rotated by (r0 r1; r3 r4), or as given when as_given
// (no multiply touches the coordinates, so no zero changes sign), with their orientation bins in shared memory; then every
// warp reduces the bounding box of the staged end points itself (no cross-warp exchange, no static shared memory).
// nan: some staged end point is NaN.
struct StagedBox { float mnx, mny, mxx, mxy; bool nan; };
__device__ __forceinline__ StagedBox stage_rotated(const float4* __restrict__ lines, int L, float r0, float r1, float r3, float r4,
                                                   bool as_given, const SlopeTableDev& table, float4* apts, uint8_t* bins) {
    const int tid = threadIdx.x, lane = tid & 31;
    bool nan = false;
    for (int q = tid; q < L; q += blockDim.x) {
        const float4 v = __ldg(lines + q);
        float x1 = v.x, y1 = v.y, x2 = v.z, y2 = v.w;
        if (!as_given) {
            x1 = r0 * v.x + r1 * v.y; y1 = r3 * v.x + r4 * v.y;
            x2 = r0 * v.z + r1 * v.w; y2 = r3 * v.z + r4 * v.w;
        }
        nan |= x1 != x1 || y1 != y1 || x2 != x2 || y2 != y2;
        apts[q] = make_float4(x1, y1, x2, y2);
        bins[q] = (uint8_t)bin_of_slope_dev(table, (y2 - y1) / (x2 - x1));
    }
    StagedBox b;
    b.nan = __syncthreads_or(nan) != 0;   // also publishes apts / bins
    b.mnx = INFINITY; b.mny = INFINITY; b.mxx = -INFINITY; b.mxy = -INFINITY;
    for (int q = lane; q < L; q += 32) {
        const float4 e = apts[q];
        b.mnx = fminf(b.mnx, fminf(e.x, e.z)); b.mxx = fmaxf(b.mxx, fmaxf(e.x, e.z));
        b.mny = fminf(b.mny, fminf(e.y, e.w)); b.mxy = fmaxf(b.mxy, fmaxf(e.y, e.w));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        b.mnx = fminf(b.mnx, __shfl_xor_sync(0xffffffffu, b.mnx, o)); b.mxx = fmaxf(b.mxx, __shfl_xor_sync(0xffffffffu, b.mxx, o));
        b.mny = fminf(b.mny, __shfl_xor_sync(0xffffffffu, b.mny, o)); b.mxy = fmaxf(b.mxy, __shfl_xor_sync(0xffffffffu, b.mxy, o));
    }
    return b;
}

// sum of |plane(x1, y1) - plane(x2, y2)| over the staged lines in Eigen's order, every end point offset by (offx, offy)
__device__ __forceinline__ float staged_score(const MapView& map, const float4* apts, const uint8_t* bins, int L, float offx, float offy) {
    const float* planes = map.planes;
    const size_t pitch = (size_t)map.dm.pitch, pe = map.dm.plane_elems;
    return eigen_sum_lazy(L, [&](int q) {
        const float4 e = apts[q];
        return line_cost(planes, pitch, pe, bins[q], e.x + offx, e.y + offy, e.z + offx, e.w + offy);
    });
}

__global__ void refine_init_kernel(const __grid_constant__ RefineLaunch p) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= (p.d_n ? *p.d_n : p.n)) return;
    RefineState st;
    for (int q = 0; q < 6; ++q) st.c[q] = p.in[m].transform[q];
    st.raw = NAN;
    st.valid = 0;
    p.state[m] = st;
    p.keys[m] = kNoPose;
}

void launch_refine_init(const RefineLaunch& p, cudaStream_t s) {
    refine_init_kernel<<<(unsigned)((p.n + 127) / 128), 128, 0, s>>>(p);
}

__global__ void __launch_bounds__(1024) refine_eval_kernel(const __grid_constant__ MapView map,
                                                           const __grid_constant__ SlopeTableDev table,
                                                           const __grid_constant__ RefineLaunch p,
                                                           const __grid_constant__ RefineLevel lv) {
    // rotated end points float4[L], planes u8[L]: the search's staging size, and no static shared memory, so that every
    // template the search accepts fits the opt-in limit
    extern __shared__ __align__(16) uint8_t s_raw[];
    const int NR = 2 * p.n_r + 1, NT = 2 * p.n_t + 1;
    const int m = blockIdx.x / NR, ir = blockIdx.x % NR;
    if (m >= (p.d_n ? *p.d_n : p.n)) return;   // whole block
    const int tid = threadIdx.x, lane = tid & 31;
    const RefineState st = p.state[m];
    const int t = p.in[m].tmpl_idx - p.tmpl_idx_base;
    const int l0 = p.offsets[t], L = p.offsets[t + 1] - l0;
    const float2 a = p.anchors[t];
    const RefineRot R = refine_rotation(st.c, a.x, a.y, ir - p.n_r, lv.ci[ir], lv.si[ir]);
    float4* apts = reinterpret_cast<float4*>(s_raw);
    uint8_t* bins = reinterpret_cast<uint8_t*>(apts + L);
    const StagedBox bb = stage_rotated(p.lines + l0, L, R.r0, R.r1, R.r3, R.r4, false, table, apts, bins);
    unsigned long long key = kNoPose;
    if (tid < NT * NT) {
        const int kk = tid / NT, jj = tid - kk * NT;
        const float P2 = R.bx + (float)(jj - p.n_t) * lv.h, P5 = R.by + (float)(kk - p.n_t) * lv.h;
        const float offx = map.shift_x + P2, offy = map.shift_y + P5;
        // the rounding of r + off is monotonic in r, so the bounding box decides for every end point
        bool valid = !bb.nan && !(R.r0 != R.r0 || R.r1 != R.r1 || R.r3 != R.r3 || R.r4 != R.r4 || P2 != P2 || P5 != P5);
        if (valid && L > 0)
            valid = 0.f <= bb.mnx + offx && bb.mxx + offx <= (float)(map.dm.W - 1) && 0.f <= bb.mny + offy &&
                    bb.mxy + offy <= (float)(map.dm.H - 1);
        if (valid) {
            const float sc = staged_score(map, apts, bins, L, offx, offy);
            // walk order: squared grid distance from the centre (0 only for the centre), then (i, k, j)
            const int di = ir - p.n_r, dk = kk - p.n_t, dj = jj - p.n_t;
            const unsigned order = (unsigned)(di * di + dk * dk + dj * dj) << 15 | (unsigned)((ir * NT + kk) * NT + jj);
            const bool is_nan = sc != sc;
            key = (unsigned long long)(is_nan ? 0x7F800000u : __float_as_uint(sc)) << 32 | (unsigned long long)(order << 1 | (is_nan ? 1u : 0u));
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
        key = other < key ? other : key;
    }
    if (lane == 0 && key != kNoPose) atomicMin(p.keys + m, key);
}

static size_t refine_smem_bytes(int max_lines) { return (size_t)max_lines * 16 + (((size_t)max_lines + 15) & ~(size_t)15); }

cudaError_t launch_refine_eval(const MapView& map, const SlopeTableDev& table, const RefineLaunch& p, const RefineLevel& lv,
                               int max_lines, int smem_optin, cudaStream_t s) {
    const int NR = 2 * p.n_r + 1, NT = 2 * p.n_t + 1;
    const int threads = ((NT * NT + 31) / 32) * 32;
    const size_t smem = refine_smem_bytes(max_lines > 0 ? max_lines : 1);
    if (smem > (size_t)smem_optin) return cudaErrorInvalidValue;   // callers reject such templates first
    if (smem > 48 * 1024) {
        const cudaError_t e = cudaFuncSetAttribute(refine_eval_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    refine_eval_kernel<<<(unsigned)((int64_t)p.n * NR), threads, smem, s>>>(map, table, p, lv);
    return cudaGetLastError();
}

__global__ void refine_advance_kernel(const __grid_constant__ RefineLaunch p, const __grid_constant__ RefineLevel lv,
                                      fdcm_match* out) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= (p.d_n ? *p.d_n : p.n)) return;
    const int tmpl_idx = p.in[m].tmpl_idx;   // (out may be in)
    const int t = tmpl_idx - p.tmpl_idx_base;
    RefineState st = p.state[m];
    const unsigned long long key = p.keys[m];
    if (key != kNoPose) {
        const unsigned order = (unsigned)key >> 1;
        if ((order >> 15) != 0u) {   // not the centre: recompute the winning pose exactly as refine_eval_kernel did
            const int NT = 2 * p.n_t + 1, g = (int)(order & 0x7FFFu);
            const int jj = g % NT, kk = (g / NT) % NT, ir = g / (NT * NT);
            const float2 a = p.anchors[t];
            const RefineRot R = refine_rotation(st.c, a.x, a.y, ir - p.n_r, lv.ci[ir], lv.si[ir]);
            st.c[0] = R.r0; st.c[1] = R.r1; st.c[2] = R.bx + (float)(jj - p.n_t) * lv.h;
            st.c[3] = R.r3; st.c[4] = R.r4; st.c[5] = R.by + (float)(kk - p.n_t) * lv.h;
        }
        st.raw = (key & 1ull) ? NAN : __uint_as_float((unsigned)(key >> 32));
        st.valid = 1;
        p.state[m] = st;
        p.keys[m] = kNoPose;
    }
    if (out) {
        fdcm_match r;
        r.tmpl_idx = tmpl_idx;
        r.score = st.valid ? (p.denom ? st.raw / p.denom[t] : st.raw) : NAN;
        for (int q = 0; q < 6; ++q) r.transform[q] = st.c[q];
        out[m] = r;
    }
}

void launch_refine_advance(const RefineLaunch& p, const RefineLevel& lv, fdcm_match* out, cudaStream_t s) {
    refine_advance_kernel<<<(unsigned)((p.n + 127) / 128), 128, 0, s>>>(p, lv, out);
}

// =============================================================================================
// Dense pose-grid search (fdcm_search_dense, beyond the reference): rules in include/fdcm_b200.h.
// One block per (template, rotation, band of cell rows) stages the rotated template once (stage_rotated, as refinement
// does).  The valid poses of a rotation form a rectangle of the grid: the bounding-box test is monotonic in u and in v, so
// the block finds the valid u and v intervals by bisection and its warps visit only those.  A warp item is 32 consecutive
// u (adjacent pixels at stride 1) by up to kDenseRowGroup rows of one cell row; each lane keeps the minimum key of its
// column, then a segmented shuffle reduction takes the minimum over the lanes of one cell and the first lane of every
// cell does one atomicMin on the cell's record key.
// =============================================================================================
constexpr int kDenseThreads = 256;
constexpr int kDenseRowGroup = 8;

// first i in [0, n) with pred(i) for a predicate that is false, then true; n when there is none
template <class Pred>
__device__ __forceinline__ int first_true(int n, Pred pred) {
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (pred(mid)) hi = mid; else lo = mid + 1;
    }
    return lo;
}

__global__ void __launch_bounds__(kDenseThreads) dense_eval_kernel(const __grid_constant__ MapView map,
                                                                   const __grid_constant__ SlopeTableDev table,
                                                                   const __grid_constant__ DenseLaunch p) {
    extern __shared__ __align__(16) uint8_t s_raw[];   // rotated end points float4[L], planes u8[L], as refinement
    const long long tr = blockIdx.x / p.n_bands;   // (t * scales + k) * rotations + r
    const int band = (int)(blockIdx.x - tr * p.n_bands);
    const int per_t = p.scales * p.rotations;
    const int kr = (int)(tr % per_t), t = (int)(tr / per_t);   // kr = k * rotations + r
    const int l0 = p.offsets[t], L = p.offsets[t + 1] - l0;
    if (L == 0) return;   // whole block: an empty template has no records
    const float2 cs = p.rot[kr], a = p.anchors[t];
    const float c = cs.x, s = cs.y;
    float4* apts = reinterpret_cast<float4*>(s_raw);
    uint8_t* bins = reinterpret_cast<uint8_t*>(apts + L);
    const StagedBox bb = stage_rotated(p.lines + l0, L, c, -s, s, c, c == 1.f && s == 0.f, table, apts, bins);
    if (bb.nan) return;   // uniform
    // shift + tx(u) is non-decreasing in u (every rounding step is monotonic): the x test holds on an interval of u, the y
    // test on an interval of v (NaN translations fail everywhere)
    const float Wm1 = (float)(map.dm.W - 1), Hm1 = (float)(map.dm.H - 1);
    const float shx = map.shift_x, shy = map.shift_y, ax = a.x, ay = a.y;
    const int lo_x = p.lo_x, lo_y = p.lo_y, stride = p.stride;
    auto offx = [=](int u) { return shx + dense_tx(c, s, ax, ay, lo_x + u * stride, shx); };
    auto offy = [=](int v) { return shy + dense_ty(c, s, ax, ay, lo_y + v * stride, shy); };
    const float mnx = bb.mnx, mxx = bb.mxx, mny = bb.mny, mxy = bb.mxy;
    const int ulo = first_true(p.nx, [=](int u) { return 0.f <= mnx + offx(u); });
    const int uhi = first_true(p.nx, [=](int u) { return !(mxx + offx(u) <= Wm1); }) - 1;
    const int vlo = first_true(p.ny, [=](int v) { return 0.f <= mny + offy(v); });
    const int vhi = first_true(p.ny, [=](int v) { return !(mxy + offy(v) <= Hm1); }) - 1;
    if (ulo > uhi || vlo > vhi) return;   // uniform
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    const int n_chunks = (uhi - ulo + 32) / 32;
    const long long rec0 = tr * p.cells_y;
    const int cv1 = min(p.cells_y, (band + 1) * p.band);
    for (int cv = band * p.band; cv < cv1; ++cv) {
        const int ra = max(cv * p.cell, vlo), rb = min(cv * p.cell + (p.cell - 1), vhi);
        if (ra > rb) continue;
        const int n_items = ((rb - ra) / kDenseRowGroup + 1) * n_chunks;
        for (int item = warp; item < n_items; item += n_warps) {   // warp-uniform
            const int grp = item / n_chunks, ch = item - grp * n_chunks;
            const int u = ulo + ch * 32 + lane;
            const int va = ra + grp * kDenseRowGroup, vb = min(va + kDenseRowGroup - 1, rb);
            unsigned long long key = kNoPose;
            if (u <= uhi) {
                const float ox = offx(u);
                for (int v = va; v <= vb; ++v) {
                    const float sc = staged_score(map, apts, bins, L, ox, offy(v));
                    const bool is_nan = sc != sc;
                    const unsigned g = (unsigned)v * (unsigned)p.nx + (unsigned)u;   // grid index (row-major)
                    const unsigned long long k =
                        (unsigned long long)(is_nan ? 0x7F800000u : __float_as_uint(sc)) << 32 | (unsigned long long)(g << 1 | (is_nan ? 1u : 0u));
                    key = k < key ? k : key;
                }
            }
            // segmented minimum: after the step of offset o, lane l holds the minimum over lanes [l, l + 2o) of its cell
            const int cu = u / p.cell;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long other = __shfl_down_sync(0xffffffffu, key, o);
                const int ocu = __shfl_down_sync(0xffffffffu, cu, o);
                if (lane + o < 32 && ocu == cu && other < key) key = other;
            }
            const int pcu = __shfl_up_sync(0xffffffffu, cu, 1);
            if ((lane == 0 || pcu != cu) && key != kNoPose) atomicMin(p.keys + (rec0 + cv) * p.cells_x + cu, key);
        }
    }
}

cudaError_t launch_dense_eval(const MapView& map, const SlopeTableDev& table, const DenseLaunch& p, int max_lines, int smem_optin,
                              cudaStream_t s) {
    const size_t smem = refine_smem_bytes(max_lines > 0 ? max_lines : 1);
    if (smem > (size_t)smem_optin) return cudaErrorInvalidValue;   // callers reject such templates first
    if (smem > 48 * 1024) {
        const cudaError_t e = cudaFuncSetAttribute(dense_eval_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    const long long blocks = (long long)p.n_tmpl * p.scales * p.rotations * p.n_bands;   // <= n_rec < 2^31
    dense_eval_kernel<<<(unsigned)blocks, kDenseThreads, smem, s>>>(map, table, p);
    return cudaGetLastError();
}

__global__ void dense_finish_kernel(const __grid_constant__ MapView map, const __grid_constant__ DenseLaunch p) {
    const long long h = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= p.n_rec) return;
    const unsigned long long key = p.keys[h];
    if (key == kNoPose) {
        p.valid[h] = 0;
        return;
    }
    const long long tr = h / ((long long)p.cells_y * p.cells_x);   // (t * scales + k) * rotations + r
    const int r = (int)(tr % p.rotations), tk = (int)(tr / p.rotations), t = tk / p.scales, k = tk - t * p.scales;
    const unsigned g = (unsigned)key >> 1;
    const int u = (int)(g % (unsigned)p.nx), v = (int)(g / (unsigned)p.nx);
    const float2 cs = p.rot[k * p.rotations + r], a = p.anchors[t];
    fdcm_match m;
    m.tmpl_idx = t + p.tmpl_idx_base;
    const float raw = (key & 1ull) ? NAN : __uint_as_float((unsigned)(key >> 32));
    m.score = p.denom ? raw / p.denom[tk] : raw;
    if (p.rec_scale) p.rec_scale[h] = p.scale[k];
    // the pose dense_eval_kernel scored, recomputed from its grid index
    dense_pose(cs.x, cs.y, a.x, a.y, p.lo_x + u * p.stride, p.lo_y + v * p.stride, map.shift_x, map.shift_y, m.transform);
    p.rec[h] = m;
    p.valid[h] = 1;
}

void launch_dense_finish(const MapView& map, const DenseLaunch& p, cudaStream_t s) {
    dense_finish_kernel<<<(unsigned)((p.n_rec + 255) / 256), 256, 0, s>>>(map, p);
}

// =============================================================================================
// evaluate<Dt3Cpu> (dt3cpu.cpp:126-179) as a standalone entry point: one thread per (template, translation)
// =============================================================================================
__global__ void __launch_bounds__(128) evaluate_kernel(const __grid_constant__ MapView map,
                                                       const __grid_constant__ SlopeTableDev table,
                                                       const float4* __restrict__ lines, const int32_t* __restrict__ toff,
                                                       const float2* __restrict__ transl, const int32_t* __restrict__ owner,
                                                       long long n_scores, float* __restrict__ scores) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_scores) return;
    const int t = owner[i];
    const float4* TL = lines + toff[t];
    const int L = toff[t + 1] - toff[t];
    const float2 tr = transl[i];
    const float offx = map.shift_x + tr.x, offy = map.shift_y + tr.y;
    const Rigid I{1.f, 0.f, 0.f, 0.f, 1.f, 0.f};
    scores[i] = eigen_sum_lazy(L, [&](int j) {
        const float4 p = __ldg(TL + j);
        const int bin = bin_of_slope_dev(table, (p.w - p.y) / (p.z - p.x));
        // identity transform written out so that no arithmetic touches the coordinates
        int x1 = (int)(p.x + offx), y1 = (int)(p.y + offy), x2 = (int)(p.z + offx), y2 = (int)(p.w + offy);
        x1 = min(max(x1, 0), map.dm.W - 1); x2 = min(max(x2, 0), map.dm.W - 1);
        y1 = min(max(y1, 0), map.dm.H - 1); y2 = min(max(y2, 0), map.dm.H - 1);
        const float* P = map.planes + (size_t)bin * map.dm.plane_elems;
        return fabsf(__ldg(P + (size_t)y1 * map.dm.pitch + x1) - __ldg(P + (size_t)y2 * map.dm.pitch + x2));
    });
    (void)I;
}

void launch_evaluate(const MapView& map, const SlopeTableDev& table, const float4* d_lines, const int32_t* d_toff,
                     const float2* d_transl, const int32_t* d_troff, const int32_t* d_owner, int64_t n_scores,
                     float* d_scores, cudaStream_t s) {
    (void)d_troff;
    if (n_scores <= 0) return;
    evaluate_kernel<<<(unsigned)((n_scores + 127) / 128), 128, 0, s>>>(map, table, d_lines, d_toff, d_transl, d_owner,
                                                                        n_scores, d_scores);
}

__global__ void classify_kernel(const __grid_constant__ SlopeTableDev table, const float4* __restrict__ lines, int n,
                                int32_t* __restrict__ bins) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 p = lines[i];
    bins[i] = bin_of_slope_dev(table, (p.w - p.y) / (p.z - p.x));
}

void launch_classify(const SlopeTableDev& table, const float4* d_lines, int n, int32_t* d_bins, cudaStream_t s) {
    if (n <= 0) return;
    classify_kernel<<<(n + 127) / 128, 128, 0, s>>>(table, d_lines, n, d_bins);
}

}   // namespace fdcm
