// fdcm_api.cu — C ABI of libfdcm_b200 (declared in include/fdcm_b200.h): handle management, the
// O(#lines) host preparation the reference also does on the host (scene shift, orientation bins via
// the host libm, std::sort orderings), stream / workspace plumbing and per-kernel CUDA-event timing.
// There is deliberately no CPU compute path here: if CUDA is unavailable every entry point fails.
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "host_math.hpp"
#include "kernels.h"

using namespace fdcm;

// =============================================================================================
// error handling
// =============================================================================================
static thread_local std::string g_last_error;

static fdcm_status fail(fdcm_status st, const std::string& msg) {
    g_last_error = msg;
    return st;
}

#define CUDA_TRY(expr)                                                                                     \
    do {                                                                                                   \
        cudaError_t _e = (expr);                                                                           \
        if (_e != cudaSuccess)                                                                             \
            return fail(_e == cudaErrorMemoryAllocation ? FDCM_ERR_NOMEM : FDCM_ERR_CUDA,                  \
                        std::string(#expr) + ": " + cudaGetErrorString(_e));                              \
    } while (0)

extern "C" const char* fdcm_last_error(void) { return g_last_error.c_str(); }
extern "C" int32_t fdcm_abi_version(void) { return FDCM_B200_ABI_VERSION; }

extern "C" fdcm_status fdcm_device_count(int32_t* n) {
    if (!n) return fail(FDCM_ERR_INVALID, "n is null");
    int c = 0;
    cudaError_t e = cudaGetDeviceCount(&c);
    if (e != cudaSuccess) {
        *n = 0;
        return fail(FDCM_ERR_CUDA, std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e));
    }
    *n = c;
    return FDCM_OK;
}

// =============================================================================================
// streams, launch counter, per-kernel event timing
// =============================================================================================
static std::mutex g_mutex;
static std::map<int, cudaStream_t> g_own_streams, g_user_streams;
static std::atomic<long long> g_launches{0};

static fdcm_status get_stream(int device, cudaStream_t* s) {
    std::lock_guard<std::mutex> lk(g_mutex);
    auto u = g_user_streams.find(device);
    if (u != g_user_streams.end()) { *s = u->second; return FDCM_OK; }
    auto o = g_own_streams.find(device);
    if (o == g_own_streams.end()) {
        cudaStream_t ns;
        CUDA_TRY(cudaStreamCreateWithFlags(&ns, cudaStreamNonBlocking));
        o = g_own_streams.emplace(device, ns).first;
    }
    *s = o->second;
    return FDCM_OK;
}

// side stream for host-to-device uploads that may overlap kernels of the main stream (template sets)
static std::map<int, cudaStream_t> g_copy_streams;
static fdcm_status get_copy_stream(int device, cudaStream_t* s) {
    std::lock_guard<std::mutex> lk(g_mutex);
    auto o = g_copy_streams.find(device);
    if (o == g_copy_streams.end()) {
        cudaStream_t ns;
        CUDA_TRY(cudaStreamCreateWithFlags(&ns, cudaStreamNonBlocking));
        o = g_copy_streams.emplace(device, ns).first;
    }
    *s = o->second;
    return FDCM_OK;
}

// second stream of a device for kernels that run beside the main stream inside one build
static std::map<int, cudaStream_t> g_aux_streams;
static fdcm_status get_aux_stream(int device, cudaStream_t* s) {
    std::lock_guard<std::mutex> lk(g_mutex);
    auto o = g_aux_streams.find(device);
    if (o == g_aux_streams.end()) {
        // highest priority: what runs here (the scene bands' envelopes and their resolve pass) is the long pole of a build,
        // its CTAs must not queue behind the pending CTAs of the far rows' fill on the main stream
        cudaStream_t ns;
        int prio_lo = 0, prio_hi = 0;
        CUDA_TRY(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        CUDA_TRY(cudaStreamCreateWithPriority(&ns, cudaStreamNonBlocking, prio_hi));
        o = g_aux_streams.emplace(device, ns).first;
    }
    *s = o->second;
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_set_stream(int32_t device, void* cuda_stream) {
    std::lock_guard<std::mutex> lk(g_mutex);
    if (cuda_stream) g_user_streams[device] = (cudaStream_t)cuda_stream;
    else g_user_streams.erase(device);
    return FDCM_OK;
}

struct ProfEntry { double total_ms = 0; long long launches = 0; double bytes = 0; };
struct ProfPending { const char* name; cudaEvent_t a, b; double bytes; int device; };
static bool g_prof_on = false;
static std::vector<std::string> g_prof_order;
static std::map<std::string, ProfEntry> g_prof;
static std::vector<ProfPending> g_prof_pending;
// timing events are recycled (per device): creating and destroying two events per kernel scope cost ~0.1 ms of driver calls
// per profiled step, most of it after the step's host synchronisation
static std::map<int, std::vector<cudaEvent_t>> g_prof_events;
static cudaEvent_t prof_event_get(int device) {   // (g_mutex held)
    auto& pool = g_prof_events[device];
    cudaEvent_t e = nullptr;
    if (!pool.empty()) {
        e = pool.back();
        pool.pop_back();
    } else {
        cudaEventCreate(&e);
    }
    return e;
}
static void prof_event_put(int device, cudaEvent_t e) { g_prof_events[device].push_back(e); }   // (g_mutex held)

struct KernelScope {   // brackets one kernel launch
    cudaStream_t s;
    bool on;
    ProfPending p;
    KernelScope(const char* name, double bytes, cudaStream_t stream, int n_kernels = 1) : s(stream), on(g_prof_on) {
        g_launches.fetch_add(n_kernels, std::memory_order_relaxed);
        if (on) {
            p.name = name;                                  // (string literals)
            p.bytes = bytes;
            p.device = 0;
            cudaGetDevice(&p.device);
            {
                std::lock_guard<std::mutex> lk(g_mutex);
                p.a = prof_event_get(p.device);
                p.b = prof_event_get(p.device);
            }
            cudaEventRecord(p.a, s);
        }
    }
    ~KernelScope() {
        if (on) {
            cudaEventRecord(p.b, s);
            std::lock_guard<std::mutex> lk(g_mutex);
            g_prof_pending.push_back(p);
        }
    }
};

extern "C" fdcm_status fdcm_profile_enable(int32_t on) { g_prof_on = on != 0; return FDCM_OK; }
extern "C" fdcm_status fdcm_profile_reset(void) {
    std::lock_guard<std::mutex> lk(g_mutex);
    g_prof.clear();
    g_prof_order.clear();
    return FDCM_OK;
}
// Accounts the scopes that have finished and keeps the others pending, with their events out of the pool: a call resolves
// after synchronising its own stream, while scopes of other streams may still run (the next scene's build of a SceneBatch,
// calls of other threads, asynchronous rebuilds).
static void prof_resolve() {
    std::lock_guard<std::mutex> lk(g_mutex);
    std::vector<ProfPending> keep;
    bool not_ready = false;
    for (auto& p : g_prof_pending) {
        if (cudaEventQuery(p.b) != cudaSuccess) { keep.push_back(p); not_ready = true; continue; }
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) {
            if (!g_prof.count(p.name)) g_prof_order.push_back(p.name);
            auto& e = g_prof[p.name];
            e.total_ms += ms;
            e.launches += 1;
            e.bytes = p.bytes;
        }
        prof_event_put(p.device, p.a);
        prof_event_put(p.device, p.b);
    }
    g_prof_pending.swap(keep);
    // a query of a running scope is not a failure of the caller: it must not surface at its next cudaGetLastError
    if (not_ready && cudaPeekAtLastError() == cudaErrorNotReady) cudaGetLastError();
}

extern "C" fdcm_status fdcm_profile_count(int32_t* n) {
    if (!n) return fail(FDCM_ERR_INVALID, "n is null");
    prof_resolve();
    std::lock_guard<std::mutex> lk(g_mutex);
    *n = (int32_t)g_prof_order.size();
    return FDCM_OK;
}
extern "C" fdcm_status fdcm_profile_get(int32_t index, char* name, int32_t name_cap, double* total_ms, int64_t* launches,
                                        double* bytes_per_launch) {
    std::lock_guard<std::mutex> lk(g_mutex);
    if (index < 0 || index >= (int32_t)g_prof_order.size()) return fail(FDCM_ERR_INVALID, "profile index out of range");
    const std::string& nm = g_prof_order[index];
    const ProfEntry& e = g_prof[nm];
    if (name && name_cap > 0) {
        std::strncpy(name, nm.c_str(), name_cap - 1);
        name[name_cap - 1] = 0;
    }
    if (total_ms) *total_ms = e.total_ms;
    if (launches) *launches = e.launches;
    if (bytes_per_launch) *bytes_per_launch = e.bytes;
    return FDCM_OK;
}
extern "C" int64_t fdcm_kernel_launch_count(void) { return g_launches.load(); }

// =============================================================================================
// device buffer with grow-only capacity
// =============================================================================================
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

// =============================================================================================
// feature map handle
// =============================================================================================
struct fdcm_dt3 {
    std::atomic<int> refs{1};
    fdcm_dt3_params params{};
    int device = 0;
    int stage = 0;
    MapDims dm{};
    float shift[2] = {0.f, 0.f};
    bool exact = true;
    int col_lo = 0, col_hi = 0;  // column range that can hold edge pixels (bbox of the shifted scene)
    int row_lo = 0, row_hi = 0;  // row range likewise
    int tables_depth = -1;       // (depth, coeff) the slope table / propagation schedule / integral directions were built for
    float tables_coeff = 0.f;
    int n_lines = 0;
    std::vector<float> keys;
    std::vector<int32_t> scene_bins;
    SlopeTable table;
    SlopeTableDev table_dev{};
    PropParams prop{};
    IntegralParams integ{};
    DevBuf planes, mask, stack, lines, bins, band_info, band_spill, integ_items;
    // lineIntegral plan (shift table, work items, tensor maps): a function of the map geometry and the planes pointer
    IntegralPlanDev integ_plan{};
    int plan_W = -1, plan_H = -1, plan_D = -1, plan_pitch = -1;
    const void* plan_planes = nullptr;
    int plan_tables_depth = -1;
    int n_sms = 148;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;   // fork / join of the second stream inside a build
    // recorded after everything that writes the map (build, rebuild, rerun, SceneBatch slot build, broadcast); every call that
    // reads or writes the map makes its stream wait on it, so work queued on another stream stays ordered before it
    cudaEvent_t ev_written = nullptr;
    bool band_path = false, band_l1 = false;   // which distance-transform formulation this map uses (set by prepare)
    // search workspace (mutable state of the last search on this map)
    mutable std::mutex search_mutex;
    mutable DevBuf s_scene, s_sorted_len, s_sorted_idx, s_hyp_off, s_rec, s_valid, s_hyp, s_counters, s_topk_score, s_topk_idx,
        s_topk_out, s_topk_n, s_keys, s_keys2, s_idx, s_perm, s_sort_tmp;
    mutable DevBuf s_sel_keys, s_sel_keys2, s_sel_vals, s_sel_vals2, s_sel_surv, s_sel_acc, s_sel_tmp;   // distinct top-K
    mutable DevBuf s_ref_state, s_ref_keys, s_ref_io;   // pose refinement
    // penalty denominators of the last template set searched on this map, for (the set's load_id, kind, tau): per map and
    // not per set, because every use of a map is serialised by search_mutex and ends in a host synchronisation, while
    // searches of other maps sharing the set may still be queued
    mutable DevBuf s_denom;
    mutable uint64_t denom_set = 0;
    mutable int denom_kind = -1;
    mutable float denom_tau = 0.f;
    mutable DevBuf s_dense_keys, s_dense_rot;   // dense pose-grid search (records: s_rec / s_valid / s_hyp_off)
    mutable float s_scene_min[2] = {0.f, 0.f}, s_scene_max[2] = {0.f, 0.f};   // bbox of the resident search scene
    mutable std::mutex host_tset_mutex;
    mutable fdcm_templates* host_tset = nullptr;   // reusable template set of fdcm_search_host
    mutable int32_t s_scene_n = 0;      // scene lines currently resident for the search (original, un-shifted)
    mutable int32_t s_sorted_n = 0;     // entries of the resident length ordering (== s_scene_n unless radius-filtered)
    mutable bool s_resident_is_build = false;   // the resident search scene is the scene the map was built from
    mutable bool s_filter_on = false;
    mutable float s_filter[4] = {0.f, 0.f, 0.f, 0.f};
    std::vector<float> h_build_scene;   // host copy of the build scene (for scene == NULL searches with a new filter)
    mutable int64_t last_n_hyp = 0;
    mutable fdcm_search_stats last_stats{};
    mutable void* h_scene_stage = nullptr;   // pinned staging for the search-scene upload (truly asynchronous copies)
    mutable size_t h_scene_stage_cap = 0;
    mutable cudaEvent_t scene_stage_ev = nullptr;
    mutable void* h_pinned = nullptr;   // pinned staging for match download
    mutable size_t h_pinned_cap = 0;

    ~fdcm_dt3() {
        cudaSetDevice(device);
        for (DevBuf* b : {&planes, &mask, &stack, &lines, &bins, &band_info, &band_spill, &integ_items, &s_scene, &s_sorted_len, &s_sorted_idx, &s_hyp_off, &s_rec,
                          &s_valid, &s_hyp, &s_counters, &s_topk_score, &s_topk_idx, &s_topk_out, &s_topk_n, &s_keys, &s_keys2, &s_idx,
                          &s_perm, &s_sort_tmp, &s_sel_keys, &s_sel_keys2, &s_sel_vals, &s_sel_vals2, &s_sel_surv, &s_sel_acc,
                          &s_sel_tmp, &s_ref_state, &s_ref_keys, &s_ref_io, &s_denom, &s_dense_keys, &s_dense_rot})
            b->release();
        if (h_pinned) cudaFreeHost(h_pinned);
        if (ev_fork) cudaEventDestroy(ev_fork);
        if (ev_join) cudaEventDestroy(ev_join);
        if (ev_written) cudaEventDestroy(ev_written);
        if (h_scene_stage) cudaFreeHost(h_scene_stage);
        if (scene_stage_ev) cudaEventDestroy(scene_stage_ev);
        destroy_host_tset();
    }
    void destroy_host_tset();
};

// largest supported map side: the band kernels keep one column of band records per CTA in shared memory (H <= 17056)
// and u16 fields hold column indices; 16384^2 x 30 planes is already a 32 GB map
constexpr int64_t kMaxSide = 16384;

struct SceneFilter { bool on; float cx, cy, lo, hi; };

// Ordering of the work on one map across streams: the caller's stream may change between calls (fdcm_set_stream), and a
// SceneBatch builds on a stream of its own, so stream order alone does not put a call after a queued build of the same map.
// The caller holds m->search_mutex.
static fdcm_status map_wait(const fdcm_dt3* m, cudaStream_t s) {
    if (m->ev_written) CUDA_TRY(cudaStreamWaitEvent(s, m->ev_written, 0));
    return FDCM_OK;
}
// (the first call comes from the map's first build, before the handle is visible to any other call)
static fdcm_status map_written(fdcm_dt3* m, cudaStream_t s) {
    if (!m->ev_written) CUDA_TRY(cudaEventCreateWithFlags(&m->ev_written, cudaEventDisableTiming));
    CUDA_TRY(cudaEventRecord(m->ev_written, s));
    return FDCM_OK;
}

// filterInRange (searchstrategies/concentricrange.h:73-84)
static std::vector<int32_t> filter_in_range(const float* lines, int32_t n, const SceneFilter& f) {
    std::vector<int32_t> idx;
    for (int32_t i = 0; i < n; ++i) {
        const float* l = lines + 4 * (size_t)i;
        const float mx = (l[2] + l[0]) / 2 - f.cx, my = (l[3] + l[1]) / 2 - f.cy;
        const float rad = std::sqrt(mx * mx + my * my);
        if (rad > (f.lo - std::numeric_limits<float>::epsilon()) && rad < f.hi) idx.push_back(i);
    }
    return idx;
}

// scene length ordering of establishSearchStrategy (defaultsearch.cpp:32-36; concentricrange.cpp:33-45 when a radius
// filter is given: ordering of the filtered lines, indices mapped back to the original scene) + upload of the scene
static fdcm_status upload_search_scene(const fdcm_dt3* m, const float* scene, int32_t n_scene, const SceneFilter& flt, cudaStream_t s) {
    std::vector<int32_t> subset;
    if (flt.on) subset = filter_in_range(scene, n_scene, flt);
    else {
        subset.resize((size_t)n_scene);
        for (int i = 0; i < n_scene; ++i) subset[(size_t)i] = i;
    }
    const int ns = (int)subset.size();
    std::vector<float> slen((size_t)ns);
    for (int i = 0; i < ns; ++i) slen[(size_t)i] = line_length(scene + 4 * (size_t)subset[(size_t)i]);
    const std::vector<long> sidx = argsort_desc(slen.data(), ns);
    std::vector<float> sorted_len((size_t)ns);
    std::vector<int32_t> sorted_idx((size_t)ns);
    for (int i = 0; i < ns; ++i) {
        sorted_len[(size_t)i] = slen[(size_t)sidx[(size_t)i]];
        sorted_idx[(size_t)i] = subset[(size_t)sidx[(size_t)i]];
    }
    m->s_scene_n = 0;
    m->s_sorted_n = 0;
    m->s_scene_min[0] = m->s_scene_max[0] = scene[0];
    m->s_scene_min[1] = m->s_scene_max[1] = scene[1];
    for (int64_t i = 0; i < 2 * (int64_t)n_scene; ++i)
        for (int a = 0; a < 2; ++a) {
            const float v = scene[2 * i + a];
            if (v < m->s_scene_min[a]) m->s_scene_min[a] = v;
            if (v > m->s_scene_max[a]) m->s_scene_max[a] = v;
        }
    CUDA_TRY(m->s_scene.reserve((size_t)n_scene * 16));
    CUDA_TRY(m->s_sorted_len.reserve(std::max<size_t>(4, (size_t)ns * 4)));
    CUDA_TRY(m->s_sorted_idx.reserve(std::max<size_t>(4, (size_t)ns * 4)));
    // through pinned staging: the copies queue behind whatever runs on the stream (e.g. the map build) without making the
    // host wait for it, which a copy from pageable memory would
    const size_t need = (size_t)n_scene * 16 + (size_t)ns * 8;
    if (!m->scene_stage_ev) CUDA_TRY(cudaEventCreateWithFlags(&m->scene_stage_ev, cudaEventDisableTiming));
    else CUDA_TRY(cudaEventSynchronize(m->scene_stage_ev));   // the staging buffer may still feed the previous upload
    if (m->h_scene_stage_cap < need) {
        if (m->h_scene_stage) cudaFreeHost(m->h_scene_stage);
        m->h_scene_stage = nullptr;
        m->h_scene_stage_cap = 0;
        CUDA_TRY(cudaMallocHost(&m->h_scene_stage, need));
        m->h_scene_stage_cap = need;
    }
    unsigned char* st = static_cast<unsigned char*>(m->h_scene_stage);
    std::memcpy(st, scene, (size_t)n_scene * 16);
    CUDA_TRY(cudaMemcpyAsync(m->s_scene.p, st, (size_t)n_scene * 16, cudaMemcpyHostToDevice, s));
    if (ns) {
        std::memcpy(st + (size_t)n_scene * 16, sorted_len.data(), (size_t)ns * 4);
        std::memcpy(st + (size_t)n_scene * 16 + (size_t)ns * 4, sorted_idx.data(), (size_t)ns * 4);
        CUDA_TRY(cudaMemcpyAsync(m->s_sorted_len.p, st + (size_t)n_scene * 16, (size_t)ns * 4, cudaMemcpyHostToDevice, s));
        CUDA_TRY(cudaMemcpyAsync(m->s_sorted_idx.p, st + (size_t)n_scene * 16 + (size_t)ns * 4, (size_t)ns * 4, cudaMemcpyHostToDevice, s));
    }
    CUDA_TRY(cudaEventRecord(m->scene_stage_ev, s));
    m->s_scene_n = n_scene;
    m->s_sorted_n = ns;
    m->s_filter_on = flt.on;
    m->s_filter[0] = flt.cx; m->s_filter[1] = flt.cy; m->s_filter[2] = flt.lo; m->s_filter[3] = flt.hi;
    return FDCM_OK;
}

static fdcm_status run_build_kernels(fdcm_dt3* m, cudaStream_t s);

// ---- TMA tensor maps: cuTensorMapEncodeTiled through the runtime's driver entry point (no link against libcuda) ----
namespace fdcm {
bool encode_planes_map(CUtensorMap* out, const void* planes, int W, int H, int D, int pitch, int bx, int by, int bz) {
    typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static EncodeFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
            p = nullptr;
        return (EncodeFn)p;
    }();
    if (!fn) return false;
    const cuuint64_t dims[3] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D};
    const cuuint64_t strides[2] = {(cuuint64_t)pitch * 4, (cuuint64_t)pitch * 4 * (cuuint64_t)H};
    const cuuint32_t box[3] = {(cuuint32_t)bx, (cuuint32_t)by, (cuuint32_t)bz};
    const cuuint32_t estr[3] = {1, 1, 1};
    return fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(planes), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
}   // namespace fdcm

// lineIntegral plan: R(i) = (long)roundf(float(i) * r) (imgproc.h:55,72; same IEEE operations as the reference, on the
// host), the (plane, strip) work items in decreasing order of work, and the tensor maps of the planes.
static fdcm_status build_integral_plan(fdcm_dt3* m, cudaStream_t s) {
    const MapDims& dm = m->dm;
    const bool same = m->plan_W == dm.W && m->plan_H == dm.H && m->plan_D == dm.D && m->plan_pitch == dm.pitch &&
                      m->plan_planes == m->planes.p && m->plan_tables_depth == m->tables_depth;
    if (same) return FDCM_OK;
    m->plan_W = -1;
    const int rlen = std::max(dm.W, dm.H);
    std::vector<int32_t> rtab((size_t)dm.D * rlen);
    struct Item { int work; int4 it; };
    std::vector<Item> items;
    const int CW = integral_strip_chains(), RB = integral_tile_steps();
    for (int d = 0; d < dm.D; ++d) {
        const int mode = m->integ.mode[d];
        const float r = mode == 1 ? m->integ.ry[d] : m->integ.rx[d];
        int32_t* R = rtab.data() + (size_t)d * rlen;
        for (int i = 0; i < rlen; ++i) R[i] = (int32_t)(long long)std::round((float)i * r);
        if (mode != 1 && mode != 2) continue;
        const int n_major = mode == 1 ? dm.W : dm.H, n_minor = mode == 1 ? dm.H : dm.W;
        const int Rend = R[n_major - 1];
        const int cmin = Rend > 0 ? -Rend : 0, cmax = (Rend < 0 ? -Rend : 0) + n_minor - 1;
        const int nblk = (n_major + RB - 1) / RB;
        for (int c0 = cmin; c0 <= cmax; c0 += CW) {
            // tiles in which some chain of the strip lies inside the image (R is monotone: they form one range)
            int b_lo = nblk, b_hi = 0;
            for (int b = 0; b < nblk; ++b) {
                const int i0 = b * RB, i1 = std::min(n_major, i0 + RB);
                const int rlo = std::min(R[i0], R[i1 - 1]), rhi = std::max(R[i0], R[i1 - 1]);
                if (c0 + CW - 1 + rhi >= 0 && c0 + rlo <= n_minor - 1) { b_lo = std::min(b_lo, b); b_hi = std::max(b_hi, b + 1); }
            }
            if (b_lo < b_hi) items.push_back(Item{b_hi - b_lo, make_int4(d, c0, b_lo, b_hi)});
        }
    }
    std::stable_sort(items.begin(), items.end(), [](const Item& a, const Item& b) { return a.work > b.work; });
    std::vector<int4> flat(items.size());
    for (size_t i = 0; i < items.size(); ++i) flat[i] = items[i].it;
    CUDA_TRY(m->integ_items.reserve(std::max<size_t>(16, flat.size() * sizeof(int4))));
    if (!flat.empty()) CUDA_TRY(cudaMemcpyAsync(m->integ_items.p, flat.data(), flat.size() * sizeof(int4), cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaStreamSynchronize(s));   // the host vectors go out of scope (rare: only when the geometry changes)
    IntegralPlanDev& pl = m->integ_plan;
    pl.items4 = m->integ_items.as<int4>();
    pl.n_items = (int)flat.size();
    if (!integral_tma_encode(m->planes.p, dm, &pl.map_y, &pl.map_x))
        return fail(FDCM_ERR_CUDA, "cuTensorMapEncodeTiled failed for the feature-map planes");
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, m->device) == cudaSuccess && sms > 0) m->n_sms = sms;
    m->plan_W = dm.W; m->plan_H = dm.H; m->plan_D = dm.D; m->plan_pitch = dm.pitch;
    m->plan_planes = m->planes.p;
    m->plan_tables_depth = m->tables_depth;
    return FDCM_OK;
}

// host preparation: shift, size, keys, bins (reference dt3cpu.h:180-193), then upload
static fdcm_status prepare_and_upload(fdcm_dt3* m, const float* scene, int32_t n_lines, cudaStream_t s) {
    m->n_lines = n_lines;
    m->scene_bins.clear();
    if (n_lines == 0) {   // dt3cpu.h:180-181: empty map, translation (0,0), size (0,0)
        m->s_scene_n = 0;
        m->s_sorted_n = 0;
        m->h_build_scene.clear();
        m->dm = MapDims{0, 0, 0, 0, 0, 0};
        m->shift[0] = m->shift[1] = 0.f;
        m->keys.clear();
        return FDCM_OK;
    }
    int64_t size[2];
    scene_centered_translation(scene, n_lines, m->params.padding, m->shift, size);
    if (size[0] <= 0 || size[0] > kMaxSide || size[1] != size[0])
        return fail(FDCM_ERR_INVALID, "feature size out of the supported range (1.." + std::to_string(kMaxSide) + "): " + std::to_string(size[0]));
    m->keys = angle_keys(m->params.depth);
    const int D = (int)m->keys.size();
    MapDims dm;
    dm.D = D;
    dm.W = (int)size[0];
    dm.H = (int)size[1];
    dm.pitch = (dm.W + 31) / 32 * 32;
    dm.wwords = dm.pitch / 32;
    dm.plane_elems = (size_t)dm.H * dm.pitch;
    m->dm = dm;
    // every intermediate of the reference's first/second L2 pass is an exact integer iff 2*(side-1)^2 < 2^24
    m->exact = 2.0 * (double)(dm.W - 1) * (double)(dm.W - 1) < 16777216.0;

    // translated scene (core/math.h:352-354) and orientation bins with the host libm (dt3cpu.h:123-134)
    std::vector<float> ts((size_t)4 * n_lines);
    m->scene_bins.resize(n_lines);
    for (int64_t i = 0; i < 2 * (int64_t)n_lines; ++i) {
        ts[2 * i] = scene[2 * i] + m->shift[0];
        ts[2 * i + 1] = scene[2 * i + 1] + m->shift[1];
    }
    for (int i = 0; i < n_lines; ++i) m->scene_bins[i] = bin_of_line(m->keys.data(), D, &ts[4 * (size_t)i]);
    {
        // clipping only moves end points inwards and pixels are round()ed coordinates: every edge pixel column lies in
        // [floor(min x), ceil(max x)] of the shifted scene
        float mnx = ts[0], mxx = ts[0], mny = ts[1], mxy = ts[1];
        for (int64_t i = 0; i < 2 * (int64_t)n_lines; ++i) {
            mnx = std::min(mnx, ts[2 * i]);
            mxx = std::max(mxx, ts[2 * i]);
            mny = std::min(mny, ts[2 * i + 1]);
            mxy = std::max(mxy, ts[2 * i + 1]);
        }
        {
            const double lo = std::floor((double)mny) - 1.0, hi = std::ceil((double)mxy) + 1.0;
            m->row_lo = (lo < 0.0 || !(lo == lo)) ? 0 : (lo > dm.H - 1 ? dm.H - 1 : (int)lo);
            m->row_hi = (!(hi == hi) || hi > dm.H - 1) ? dm.H - 1 : (hi < 0.0 ? 0 : (int)hi);
        }
        const double lo = std::floor((double)mnx) - 1.0, hi = std::ceil((double)mxx) + 1.0;
        m->col_lo = (lo < 0.0 || !(lo == lo)) ? 0 : (lo > dm.W - 1 ? dm.W - 1 : (int)lo);
        m->col_hi = (!(hi == hi) || hi > dm.W - 1) ? dm.W - 1 : (hi < 0.0 ? 0 : (int)hi);
    }

    // tables: functions of (depth, coeff) only, kept across rebuilds of the same map
    if (m->tables_depth != D || m->tables_coeff != m->params.dt3_coeff) {
    m->table = build_slope_table(m->keys.data(), D);
    if ((int)m->table.thr.size() > kMaxDepthDev + 8) return fail(FDCM_ERR_INVALID, "slope table too large");
    m->table_dev.n_thr = (int)m->table.thr.size();
    m->table_dev.nan_bin = m->table.nan_bin;
    for (size_t i = 0; i < m->table.thr.size(); ++i) m->table_dev.thr[i] = m->table.thr[i];
    for (size_t i = 0; i < m->table.piece_bin.size(); ++i) m->table_dev.piece_bin[i] = (uint8_t)m->table.piece_bin[i];
    const std::vector<PropStep> steps = propagation_schedule(m->keys, m->params.dt3_coeff);
    m->prop.n_steps = (int)steps.size();
    for (size_t i = 0; i < steps.size(); ++i) {
        m->prop.w[i] = steps[i].w;
        m->prop.c1[i] = (uint8_t)steps[i].c1;
        m->prop.c2[i] = (uint8_t)steps[i].c2;
    }
    for (int d = 0; d < D; ++d) {
        const IntegralDir id = integral_direction(m->keys[d]);
        m->integ.rx[d] = id.rx;
        m->integ.ry[d] = id.ry;
        m->integ.mode[d] = id.mode;
    }
    m->tables_depth = D;
    m->tables_coeff = m->params.dt3_coeff;
    }

    // device allocations (grow-only)
    const size_t n_px = (size_t)D * dm.plane_elems;
    CUDA_TRY(m->planes.reserve(n_px * sizeof(float)));
    CUDA_TRY(m->mask.reserve((size_t)D * dm.H * dm.wwords * sizeof(uint32_t) + 256));   // + the work counters of the build kernels
    if (dt_band_smem_bytes(dm) > 200 * 1024) return fail(FDCM_ERR_INVALID, "feature size too large for the band kernels");
    const bool band_path = m->exact && m->params.distance != FDCM_L1;     // L2 / L2^2, exact regime
    const bool band_l1 = m->params.distance == FDCM_L1;                   // L1, any size
    m->band_path = band_path;
    m->band_l1 = band_l1;
    if (band_path || band_l1) CUDA_TRY(m->band_info.reserve(dt_band_info_bytes(dm)));
    if (band_path) CUDA_TRY(m->band_spill.reserve(dt_band_spill_bytes(dm, m->col_hi - m->col_lo + 1)));
    if (m->params.distance != FDCM_L1 && !band_path) CUDA_TRY(m->stack.reserve(n_px * 8));
    CUDA_TRY(m->lines.reserve((size_t)n_lines * 16));
    CUDA_TRY(m->bins.reserve((size_t)n_lines * 4));
    CUDA_TRY(cudaMemcpyAsync(m->lines.p, ts.data(), (size_t)n_lines * 16, cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(m->bins.p, m->scene_bins.data(), (size_t)n_lines * 4, cudaMemcpyHostToDevice, s));
    // (copies from pageable memory return once the source has been staged: ts may go out of scope)
    return build_integral_plan(m, s);
}

// second half of the host preparation, queued AFTER the build kernels so that its host work (length ordering of the
// scene lines) overlaps the device build: keep the original scene resident for searches that pass scene == NULL
static fdcm_status upload_build_scene(fdcm_dt3* m, const float* scene, int32_t n_lines, cudaStream_t s) {
    if (n_lines == 0) return FDCM_OK;   // (the caller holds m->search_mutex)
    m->h_build_scene.assign(scene, scene + 4 * (size_t)n_lines);
    m->s_resident_is_build = true;
    return upload_search_scene(m, scene, n_lines, SceneFilter{false, 0, 0, 0, 0}, s);
}

static fdcm_status run_build_kernels(fdcm_dt3* m, cudaStream_t s) {
    if (m->n_lines == 0) return FDCM_OK;
    const MapDims& dm = m->dm;
    const double N = (double)dm.D * dm.H * dm.W * 4.0;   // algorithmic plane bytes
    const size_t mask_bytes = (size_t)dm.D * dm.H * dm.wwords * sizeof(uint32_t);
    {
        KernelScope k("mask_clear", (double)mask_bytes, s, 0);   // cudaMemsetAsync, not one of our kernels
        CUDA_TRY(cudaMemsetAsync(m->mask.p, 0, mask_bytes + 256, s));   // (+ the work counters behind the mask)
    }
    {
        KernelScope k("raster", 0.0, s);
        launch_raster(m->lines.as<float>(), m->bins.as<int32_t>(), m->n_lines, dm, m->mask.as<uint32_t>(), s);
    }
    const int dist = m->params.distance;
    bool fused_propagate = false;
    if (m->band_l1) {
        {
            KernelScope k("dt_col_band", (double)mask_bytes + (double)dt_band_info_bytes(dm), s);
            launch_dt_col_band(m->mask.as<uint32_t>(), dm, m->band_info.p, s);
        }
        fused_propagate = m->stage != 1 && dt_fill_propagate_supported(dm);
        if (fused_propagate) {
            KernelScope k("dt_l1_propagate", (double)dt_band_info_bytes(dm) + N, s);
            launch_dt_l1_propagate(m->band_info.p, m->planes.as<float>(), dm, m->prop, s);
        } else {
            KernelScope k("dt_row_l1_band", (double)dt_band_info_bytes(dm) + N, s);
            launch_dt_row_l1_band(m->band_info.p, m->planes.as<float>(), dm, s);
        }
    } else if (m->band_path) {
        {
            KernelScope k("dt_col_band", (double)mask_bytes + (double)dt_band_info_bytes(dm), s);
            launch_dt_col_band(m->mask.as<uint32_t>(), dm, m->band_info.p, s);
        }
        fused_propagate = m->stage != 1 && dt_fill_propagate_supported(dm);
        int ys0 = 0, ys1 = dm.H;                     // image rows of the bands that overlap the scene's rows
        dt_band_scene_rows(dm, m->row_lo, m->row_hi, &ys0, &ys1);
        const bool split = fused_propagate && (ys0 > 0 || ys1 < dm.H) && ys1 > ys0;
        if (split) {
            // The envelopes of the bands that hold the scene's edge rows are the long pole of the build (serial column chains,
            // ~half of the issue slots idle); the rows of the other (far) bands only need the cheap far envelopes.  So the scene
            // envelopes, their resolve pass and their fill run on a second stream while the main stream fills + propagates the
            // far rows under them.
            cudaStream_t sa;
            if (fdcm_status st = get_aux_stream(m->device, &sa)) return st;
            if (!m->ev_fork) CUDA_TRY(cudaEventCreateWithFlags(&m->ev_fork, cudaEventDisableTiming));
            if (!m->ev_join) CUDA_TRY(cudaEventCreateWithFlags(&m->ev_join, cudaEventDisableTiming));
            CUDA_TRY(cudaEventRecord(m->ev_fork, s));
            CUDA_TRY(cudaStreamWaitEvent(sa, m->ev_fork, 0));
            {
                KernelScope k("dt_row_envelope", (double)dt_band_info_bytes(dm), sa);
                launch_dt_row_envelope(m->band_info.p, nullptr, dm, m->band_spill.p, m->col_lo, m->col_hi, m->row_lo, m->row_hi, 1, sa);
            }
            {
                KernelScope k("dt_resolve", 2.0 * (double)dt_band_info_bytes(dm), sa);
                launch_dt_resolve(dm, m->band_spill.p, m->col_lo, m->col_hi, ys0, ys1, 0, 0, sa);
            }
            {
                // (same stream: the scene rows' fill starts as soon as their envelopes are resolved and shares the GPU with the
                // tail of the far rows' fill instead of waiting behind it)
                KernelScope k("dt_fill_propagate", N * (double)(ys1 - ys0) / dm.H, sa);
                launch_dt_fill_propagate(m->planes.as<float>(), dm, m->band_spill.p, m->col_lo, m->col_hi, m->prop, dist == FDCM_L2, ys0, ys1, 0,
                                         0, sa);
            }
            CUDA_TRY(cudaEventRecord(m->ev_join, sa));
            {
                KernelScope k("dt_row_envelope_far", (double)dt_band_info_bytes(dm), s);
                launch_dt_row_envelope(m->band_info.p, nullptr, dm, m->band_spill.p, m->col_lo, m->col_hi, m->row_lo, m->row_hi, 2, s);
            }
            {
                KernelScope k("dt_resolve_far", 2.0 * (double)dt_band_info_bytes(dm), s);
                launch_dt_resolve(dm, m->band_spill.p, m->col_lo, m->col_hi, 0, ys0, ys1, dm.H, s);
            }
            {
                KernelScope k("dt_fill_propagate_far", N * (double)(dm.H - (ys1 - ys0)) / dm.H, s);
                launch_dt_fill_propagate(m->planes.as<float>(), dm, m->band_spill.p, m->col_lo, m->col_hi, m->prop, dist == FDCM_L2, 0, ys0, ys1,
                                         dm.H, s);
            }
            CUDA_TRY(cudaStreamWaitEvent(s, m->ev_join, 0));
        } else {
            {
                KernelScope k("dt_row_envelope", (double)dt_band_info_bytes(dm), s);
                launch_dt_row_envelope(m->band_info.p, nullptr, dm, m->band_spill.p, m->col_lo, m->col_hi, m->row_lo, m->row_hi, 0, s);
            }
            if (fused_propagate) {
                {
                    KernelScope k("dt_resolve", 2.0 * (double)dt_band_info_bytes(dm), s);
                    launch_dt_resolve(dm, m->band_spill.p, m->col_lo, m->col_hi, 0, dm.H, 0, 0, s);
                }
                KernelScope k("dt_fill_propagate", N, s);
                launch_dt_fill_propagate(m->planes.as<float>(), dm, m->band_spill.p, m->col_lo, m->col_hi, m->prop, dist == FDCM_L2, 0, dm.H, 0, 0,
                                         s);
            } else {
                KernelScope k("dt_row_fill", N, s);
                launch_dt_row_fill(m->planes.as<float>(), dm, m->band_spill.p, m->col_lo, m->col_hi, s);
            }
        }
    } else {
        // side > 2897, L2 / L2^2: float(q^2) rounds, the reference's float arithmetic is replayed literally.  Like the
        // reference (imgproc.h:186-190): column pass, transpose, column pass, transpose -- every pass coalesced.
        {
            KernelScope k("dt_col_literal", (double)mask_bytes + N, s);
            launch_dt_pass_literal(1, false, m->mask.p, m->planes.as<float>(), dm, m->stack.p, s);
        }
        {
            KernelScope k("transpose", 2 * N, s);
            launch_transpose_square(m->planes.as<float>(), dm, s);
        }
        {
            KernelScope k("dt_row_literal", 2 * N, s);
            launch_dt_pass_literal(0, false, nullptr, m->planes.as<float>(), dm, m->stack.p, s);
        }
        {
            KernelScope k("transpose", 2 * N, s);
            launch_transpose_square(m->planes.as<float>(), dm, s);
        }
    }
    const bool need_sqrt = dist == FDCM_L2;
    if (m->stage == 1) {
        if (need_sqrt) {
            KernelScope k("sqrt", 2 * N, s);
            launch_sqrt(m->planes.as<float>(), dm, s);
        }
    } else {
        if (!fused_propagate) {
            KernelScope k("propagate", 2 * N, s);
            launch_propagate(m->planes.as<float>(), dm, m->prop, need_sqrt, s);
        }
        if (m->stage == 0) {
            KernelScope k("integral", 2 * N, s, 1);
            IntegralPlanDev pl = m->integ_plan;
            pl.counter = reinterpret_cast<int*>(m->mask.as<unsigned char>() + mask_bytes);
            launch_integral_tma(m->planes.as<float>(), dm, m->integ, pl, m->n_sms, s);
        }
    }
    CUDA_TRY(cudaGetLastError());
    return FDCM_OK;
}

static fdcm_status validate_params(const fdcm_dt3_params* p) {
    if (!p) return fail(FDCM_ERR_INVALID, "params is null");
    if (p->depth < 1 || p->depth > kMaxDepth) return fail(FDCM_ERR_INVALID, "depth must be in 1..64");
    if (p->distance < 0 || p->distance > 2) return fail(FDCM_ERR_INVALID, "unknown distance");
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_dt3_build(const float* scene_xyxy, int32_t n_lines, const fdcm_dt3_params* params, int32_t device,
                                      int32_t stage, fdcm_dt3** out) {
    if (!out) return fail(FDCM_ERR_INVALID, "out is null");
    *out = nullptr;
    if (fdcm_status st = validate_params(params)) return st;
    if (n_lines < 0 || (n_lines > 0 && !scene_xyxy)) return fail(FDCM_ERR_INVALID, "bad scene");
    if (stage < 0 || stage > 2) return fail(FDCM_ERR_INVALID, "bad stage");
    CUDA_TRY(cudaSetDevice(device));
    cudaStream_t s;
    if (fdcm_status st = get_stream(device, &s)) return st;
    fdcm_dt3* m = new (std::nothrow) fdcm_dt3();
    if (!m) return fail(FDCM_ERR_NOMEM, "host allocation failed");
    m->params = *params;
    m->device = device;
    m->stage = stage;
    fdcm_status st = prepare_and_upload(m, scene_xyxy, n_lines, s);
    if (st == FDCM_OK) st = run_build_kernels(m, s);
    if (st == FDCM_OK) st = upload_build_scene(m, scene_xyxy, n_lines, s);
    if (st == FDCM_OK) st = map_written(m, s);
    if (st == FDCM_OK) {
        cudaError_t e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) st = fail(FDCM_ERR_CUDA, std::string("build: ") + cudaGetErrorString(e));
    }
    prof_resolve();
    if (st != FDCM_OK) {
        delete m;
        return st;
    }
    *out = m;
    return FDCM_OK;
}

// A rebuild that fails half way (size check, allocation) must not leave a handle that mixes the old map with the new
// scene: the map becomes the empty map (dt3cpu.h:180-181 state), which every entry point handles.
static void invalidate_map(fdcm_dt3* m) {
    m->n_lines = 0;
    m->scene_bins.clear();
    m->keys.clear();
    m->dm = MapDims{0, 0, 0, 0, 0, 0};
    m->shift[0] = m->shift[1] = 0.f;
    m->s_scene_n = 0;
    m->s_sorted_n = 0;
    m->s_resident_is_build = false;
    m->h_build_scene.clear();
    m->last_n_hyp = 0;
}

static fdcm_status rebuild_impl(fdcm_dt3* m, const float* scene_xyxy, int32_t n_lines, bool wait) {
    if (!m) return fail(FDCM_ERR_INVALID, "map is null");
    if (n_lines < 0 || (n_lines > 0 && !scene_xyxy)) return fail(FDCM_ERR_INVALID, "bad scene");
    CUDA_TRY(cudaSetDevice(m->device));
    cudaStream_t s;
    if (fdcm_status st = get_stream(m->device, &s)) return st;
    std::lock_guard<std::mutex> lk(m->search_mutex);   // a search on this handle must not see a half-replaced map
    fdcm_status st = map_wait(m, s);   // an earlier build of this map queued on another stream must not overlap this one
    if (st == FDCM_OK) st = prepare_and_upload(m, scene_xyxy, n_lines, s);
    if (st == FDCM_OK) st = run_build_kernels(m, s);
    if (st == FDCM_OK) st = upload_build_scene(m, scene_xyxy, n_lines, s);
    if (st == FDCM_OK) st = map_written(m, s);
    if (st != FDCM_OK) {
        const std::string msg = g_last_error;
        cudaStreamSynchronize(s);
        invalidate_map(m);
        g_last_error = msg;
    }
    if (st == FDCM_OK && wait) {
        cudaError_t e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) st = fail(FDCM_ERR_CUDA, std::string("rebuild: ") + cudaGetErrorString(e));
        prof_resolve();
    }
    return st;
}

extern "C" fdcm_status fdcm_dt3_rebuild(fdcm_dt3* m, const float* scene_xyxy, int32_t n_lines) {
    return rebuild_impl(m, scene_xyxy, n_lines, true);
}

// Same as fdcm_dt3_rebuild but returns as soon as the build kernels are queued on the current stream: the host can
// prepare the next call (e.g. the template ordering of fdcm_search_host) while the device builds the map.  Every later
// call on this map is ordered after the build, on whichever stream it runs (ev_written); errors of the build surface at
// the next synchronising call.
extern "C" fdcm_status fdcm_dt3_rebuild_async(fdcm_dt3* m, const float* scene_xyxy, int32_t n_lines) {
    return rebuild_impl(m, scene_xyxy, n_lines, false);
}

extern "C" fdcm_status fdcm_dt3_rerun(fdcm_dt3* m) {
    if (!m) return fail(FDCM_ERR_INVALID, "map is null");
    CUDA_TRY(cudaSetDevice(m->device));
    cudaStream_t s;
    if (fdcm_status st = get_stream(m->device, &s)) return st;
    std::lock_guard<std::mutex> lk(m->search_mutex);
    fdcm_status st = map_wait(m, s);
    if (st == FDCM_OK) st = run_build_kernels(m, s);
    if (st == FDCM_OK) st = map_written(m, s);
    if (st == FDCM_OK) {
        cudaError_t e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) st = fail(FDCM_ERR_CUDA, std::string("rerun: ") + cudaGetErrorString(e));
    }
    prof_resolve();
    return st;
}

extern "C" fdcm_status fdcm_dt3_rerun_async(fdcm_dt3* m) {
    if (!m) return fail(FDCM_ERR_INVALID, "map is null");
    CUDA_TRY(cudaSetDevice(m->device));
    cudaStream_t s;
    if (fdcm_status st = get_stream(m->device, &s)) return st;
    std::lock_guard<std::mutex> lk(m->search_mutex);
    if (fdcm_status st = map_wait(m, s)) return st;
    if (fdcm_status st = run_build_kernels(m, s)) return st;
    return map_written(m, s);
}

extern "C" fdcm_status fdcm_dt3_retain(fdcm_dt3* m) {
    if (!m) return fail(FDCM_ERR_INVALID, "map is null");
    m->refs.fetch_add(1);
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_dt3_release(fdcm_dt3* m) {
    if (!m) return FDCM_OK;
    if (m->refs.fetch_sub(1) == 1) delete m;
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_dt3_get_info(const fdcm_dt3* m, fdcm_dt3_info* info) {
    if (!m || !info) return fail(FDCM_ERR_INVALID, "null argument");
    info->depth = m->dm.D;
    info->width = m->dm.W;
    info->height = m->dm.H;
    info->pitch = m->dm.pitch;
    info->scene_translation[0] = m->shift[0];
    info->scene_translation[1] = m->shift[1];
    info->distance = m->params.distance;
    info->device = m->device;
    info->n_scene_lines = m->n_lines;
    info->exact_dt_path = m->exact ? 1 : 0;
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_dt3_angles(const fdcm_dt3* m, float* keys) {
    if (!m || !keys) return fail(FDCM_ERR_INVALID, "null argument");
    std::memcpy(keys, m->keys.data(), m->keys.size() * sizeof(float));
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_dt3_download_plane(const fdcm_dt3* m, int32_t plane, float* dst) {
    if (!m || !dst) return fail(FDCM_ERR_INVALID, "null argument");
    if (plane < 0 || plane >= m->dm.D) return fail(FDCM_ERR_INVALID, "plane out of range");
    CUDA_TRY(cudaSetDevice(m->device));
    cudaStream_t s;   // a legacy-stream copy would not be ordered after an async rebuild
    if (fdcm_status st = get_stream(m->device, &s)) return st;
    std::lock_guard<std::mutex> lk(m->search_mutex);
    if (fdcm_status st = map_wait(m, s)) return st;
    const float* src = m->planes.as<float>() + (size_t)plane * m->dm.plane_elems;
    CUDA_TRY(cudaMemcpy2DAsync(dst, (size_t)m->dm.W * 4, src, (size_t)m->dm.pitch * 4, (size_t)m->dm.W * 4, m->dm.H,
                               cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_dt3_download_mask(const fdcm_dt3* m, int32_t plane, uint8_t* dst) {
    if (!m || !dst) return fail(FDCM_ERR_INVALID, "null argument");
    if (plane < 0 || plane >= m->dm.D) return fail(FDCM_ERR_INVALID, "plane out of range");
    CUDA_TRY(cudaSetDevice(m->device));
    cudaStream_t s;
    if (fdcm_status st = get_stream(m->device, &s)) return st;
    std::lock_guard<std::mutex> lk(m->search_mutex);
    if (fdcm_status st = map_wait(m, s)) return st;
    std::vector<uint32_t> w((size_t)m->dm.H * m->dm.wwords);
    CUDA_TRY(cudaMemcpyAsync(w.data(), m->mask.as<uint32_t>() + (size_t)plane * m->dm.H * m->dm.wwords, w.size() * 4,
                             cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    for (int y = 0; y < m->dm.H; ++y)
        for (int x = 0; x < m->dm.W; ++x)
            dst[(size_t)y * m->dm.W + x] = (w[(size_t)y * m->dm.wwords + (x >> 5)] >> (x & 31)) & 1u;
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_dt3_scene_bins(const fdcm_dt3* m, int32_t* bins) {
    if (!m || !bins) return fail(FDCM_ERR_INVALID, "null argument");
    std::memcpy(bins, m->scene_bins.data(), m->scene_bins.size() * sizeof(int32_t));
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_dt3_device_ptr(const fdcm_dt3* m, void** planes, uint64_t* n_bytes) {
    if (!m || !planes) return fail(FDCM_ERR_INVALID, "null argument");
    *planes = m->planes.p;
    if (n_bytes) *n_bytes = (uint64_t)m->dm.D * m->dm.plane_elems * 4;
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_dt3_minmax_translation(const fdcm_dt3* m, const float* tmpl, int32_t n_lines, const float align_vec[2],
                                                   float out[2]) {
    if (!m || !align_vec || !out || (n_lines > 0 && !tmpl)) return fail(FDCM_ERR_INVALID, "null argument");
    const int64_t fs[2] = {m->dm.W, m->dm.H};
    minmax_translation(tmpl, n_lines, align_vec, fs, m->shift, out);
    return FDCM_OK;
}

static MapView map_view(const fdcm_dt3* m) {
    MapView v;
    v.planes = m->planes.as<float>();
    v.dm = m->dm;
    v.shift_x = m->shift[0];
    v.shift_y = m->shift[1];
    return v;
}

extern "C" fdcm_status fdcm_dt3_evaluate(const fdcm_dt3* m, const float* tmpl_lines, const int32_t* tmpl_offsets, int32_t n_tmpl,
                                         const float* translations, const int32_t* transl_offsets, float* scores) {
    if (!m || !tmpl_offsets || !transl_offsets) return fail(FDCM_ERR_INVALID, "null argument");
    if (n_tmpl <= 0) return FDCM_OK;
    const int64_t n_lines = tmpl_offsets[n_tmpl], n_scores = transl_offsets[n_tmpl];
    if (n_scores <= 0) return FDCM_OK;
    if (!scores || !translations || (n_lines > 0 && !tmpl_lines)) return fail(FDCM_ERR_INVALID, "null argument");
    if (m->dm.D == 0) return fail(FDCM_ERR_INVALID, "evaluate on an empty feature map");
    CUDA_TRY(cudaSetDevice(m->device));
    cudaStream_t s;
    if (fdcm_status st = get_stream(m->device, &s)) return st;
    std::lock_guard<std::mutex> lk(m->search_mutex);
    if (fdcm_status st = map_wait(m, s)) return st;
    std::vector<int32_t> owner((size_t)n_scores);
    for (int t = 0; t < n_tmpl; ++t)
        for (int i = transl_offsets[t]; i < transl_offsets[t + 1]; ++i) owner[i] = t;
    DevBuf dl, doff, dtr, down, dsc;
    auto cleanup = [&]() { for (DevBuf* b : {&dl, &doff, &dtr, &down, &dsc}) b->release(); };
    cudaError_t e = cudaSuccess;
    if (e == cudaSuccess) e = dl.reserve(std::max<size_t>(16, (size_t)n_lines * 16));
    if (e == cudaSuccess) e = doff.reserve((size_t)(n_tmpl + 1) * 4);
    if (e == cudaSuccess) e = dtr.reserve((size_t)n_scores * 8);
    if (e == cudaSuccess) e = down.reserve((size_t)n_scores * 4);
    if (e == cudaSuccess) e = dsc.reserve((size_t)n_scores * 4);
    if (e == cudaSuccess && n_lines) e = cudaMemcpyAsync(dl.p, tmpl_lines, (size_t)n_lines * 16, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(doff.p, tmpl_offsets, (size_t)(n_tmpl + 1) * 4, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dtr.p, translations, (size_t)n_scores * 8, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(down.p, owner.data(), (size_t)n_scores * 4, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) {
        KernelScope k("evaluate", 0.0, s);
        launch_evaluate(map_view(m), m->table_dev, dl.as<float4>(), doff.as<int32_t>(), dtr.as<float2>(), nullptr, down.as<int32_t>(),
                        n_scores, dsc.as<float>(), s);
    }
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(scores, dsc.p, (size_t)n_scores * 4, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    prof_resolve();
    cleanup();
    if (e != cudaSuccess) return fail(FDCM_ERR_CUDA, std::string("evaluate: ") + cudaGetErrorString(e));
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_dt3_classify(const fdcm_dt3* m, const float* lines, int32_t n, int32_t* bins) {
    if (!m || (n > 0 && (!lines || !bins))) return fail(FDCM_ERR_INVALID, "null argument");
    if (n <= 0) return FDCM_OK;
    if (m->dm.D == 0) return fail(FDCM_ERR_INVALID, "classify on an empty feature map");
    CUDA_TRY(cudaSetDevice(m->device));
    cudaStream_t s;
    if (fdcm_status st = get_stream(m->device, &s)) return st;
    std::lock_guard<std::mutex> lk(m->search_mutex);
    if (fdcm_status st = map_wait(m, s)) return st;
    DevBuf dl, db;
    cudaError_t e = dl.reserve((size_t)n * 16);
    if (e == cudaSuccess) e = db.reserve((size_t)n * 4);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dl.p, lines, (size_t)n * 16, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) {
        KernelScope k("classify", 0.0, s);
        launch_classify(m->table_dev, dl.as<float4>(), n, db.as<int32_t>(), s);
    }
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(bins, db.p, (size_t)n * 4, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    prof_resolve();
    dl.release();
    db.release();
    if (e != cudaSuccess) return fail(FDCM_ERR_CUDA, std::string("classify: ") + cudaGetErrorString(e));
    return FDCM_OK;
}

// =============================================================================================
// template sets
// =============================================================================================
// grow-only page-locked host array: what the library uploads every search is written straight into pinned memory, so the
// cudaMemcpyAsync of it neither stages through the driver nor holds the calling thread
template <class T>
struct PinnedVec {
    T* p = nullptr;
    size_t cap = 0;
    cudaError_t resize(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        const size_t want = n + n / 4 + 64;
        cudaError_t e = cudaMallocHost(reinterpret_cast<void**>(&p), want * sizeof(T));
        if (e == cudaSuccess) cap = want;
        return e;
    }
    T* data() { return p; }
    ~PinnedVec() { if (p) cudaFreeHost(p); }
};

struct fdcm_templates {
    int device = 0;
    int32_t n_tmpl = 0;
    int32_t max_lines = 0;
    int64_t n_lines = 0;
    std::vector<int32_t> offsets;     // host copy
    std::vector<float> lengths;       // getTemplateLengths
    PinnedVec<float> h_line_len;      // host scratch kept for reloads (pinned: uploaded every fdcm_search_host)
    PinnedVec<int32_t> h_argsort;
    PinnedVec<float> h_anchors;       // 2 per template (fdcm_template_anchors)
    DevBuf lines, offs, argsort, line_len, anchors;
    uint64_t load_id = 0;             // unique over all loads of all sets: keys the maps' denominator caches
    std::mutex mu;
    // uploads run on the copy stream (they overlap a map build in flight on the main stream); consumers wait on `ready`
    cudaEvent_t ready = nullptr;
    std::atomic<bool> upload_pending{false};   // (read by searches of other maps sharing the set)
    void* h_stage = nullptr;          // pinned staging for the small per-search uploads (denominators, hypothesis offsets)
    size_t h_stage_cap = 0;
    cudaError_t stage_reserve(size_t bytes) {
        if (bytes <= h_stage_cap) return cudaSuccess;
        if (h_stage) cudaFreeHost(h_stage);
        h_stage = nullptr;
        h_stage_cap = 0;
        cudaError_t e = cudaMallocHost(&h_stage, bytes);
        if (e == cudaSuccess) h_stage_cap = bytes;
        return e;
    }
    ~fdcm_templates() {
        cudaSetDevice(device);
        if (ready) cudaEventDestroy(ready);
        if (h_stage) cudaFreeHost(h_stage);
        for (DevBuf* b : {&lines, &offs, &argsort, &line_len, &anchors}) b->release();
    }
};

// small persistent worker pool for the O(#templates) host preparation (std::sort per template)
class HostPool {
    std::vector<std::thread> workers_;
    std::mutex mu_;
    std::condition_variable cv_, done_cv_;
    std::function<void(int, int)> job_;
    int n_items_ = 0, chunk_ = 1, generation_ = 0, pending_ = 0;
    std::atomic<int> next_{0};
    bool stop_ = false;

    void run() {
        int seen = 0;
        for (;;) {
            std::function<void(int, int)> job;
            int n, chunk;
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [&] { return stop_ || generation_ != seen; });
                if (stop_) return;
                seen = generation_;
                job = job_;
                n = n_items_;
                chunk = chunk_;
            }
            for (;;) {
                const int b = next_.fetch_add(chunk);
                if (b >= n) break;
                job(b, std::min(n, b + chunk));
            }
            std::lock_guard<std::mutex> lk(mu_);
            if (--pending_ == 0) done_cv_.notify_all();
        }
    }

public:
    explicit HostPool(int n) {
        for (int i = 0; i < n; ++i) workers_.emplace_back([this] { run(); });
    }
    ~HostPool() {
        {
            std::lock_guard<std::mutex> lk(mu_);
            stop_ = true;
        }
        cv_.notify_all();
        for (auto& t : workers_) t.join();
    }
    // fn(begin, end) over [0, n) in chunks; the calling thread participates
    void parallel_for(int n, int chunk, const std::function<void(int, int)>& fn) {
        if (workers_.empty() || n <= chunk) { fn(0, n); return; }
        {
            std::lock_guard<std::mutex> lk(mu_);
            job_ = fn;
            n_items_ = n;
            chunk_ = chunk;
            next_.store(0);
            pending_ = (int)workers_.size();
            ++generation_;
        }
        cv_.notify_all();
        for (;;) {
            const int b = next_.fetch_add(chunk);
            if (b >= n) break;
            fn(b, std::min(n, b + chunk));
        }
        std::unique_lock<std::mutex> lk(mu_);
        done_cv_.wait(lk, [&] { return pending_ == 0; });
    }
};

static int g_host_threads = 0;   // 0: default (min(16, cores)); takes effect before the first template preparation
static HostPool& host_pool() {
    // workers besides the calling thread; fdcm_set_host_threads / fdcm_comm_init bound it (one process per GPU shares a host)
    static HostPool pool(std::max(0, std::min(15, (g_host_threads > 0 ? g_host_threads : (int)std::max(1u, std::thread::hardware_concurrency())) - 1)));
    return pool;
}
static std::mutex g_pool_mutex;   // one parallel_for at a time

void fdcm_dt3::destroy_host_tset() {
    delete host_tset;
    host_tset = nullptr;
}

// anchor of a template for the distinct top-K: centre of the bounding box of its 2 L end points, (0, 0) when empty
static void template_anchor(const float* lines, int L, float* xy) {
    if (L <= 0) { xy[0] = xy[1] = 0.f; return; }
    float mnx = lines[0], mxx = lines[0], mny = lines[1], mxy = lines[1];
    for (int i = 0; i < 2 * L; ++i) {
        const float x = lines[2 * (size_t)i], y = lines[2 * (size_t)i + 1];
        mnx = std::min(mnx, x); mxx = std::max(mxx, x);
        mny = std::min(mny, y); mxy = std::max(mxy, y);
    }
    xy[0] = (mnx + mxx) * 0.5f;
    xy[1] = (mny + mxy) * 0.5f;
}

// need_ranks: how many leading entries of every template's length order the caller will read (DefaultSearch only aligns the
// max_tmpl_lines longest lines, defaultsearch.cpp:35-38); <= 0: the whole order.  When the need_ranks + 1 largest lengths
// of a template are pairwise distinct, the leading ranks of ANY correct descending sort are the same as std::sort's, and a
// selection scan yields them at a tenth of the cost; ties (or NaN) take the reference's std::sort, whose result for equal
// keys depends on the algorithm.  (Host cores are shared by all ranks of a node: at 8 GPUs per 16 cores the full sort of
// 5000 templates per step no longer hid behind the map build.)
static void template_host_prep(const float* tl, const int32_t* off, int32_t T, float* line_len /* off[T] */,
                               int32_t* argsort /* off[T] */, float* anchors /* 2 T */, std::vector<float>& lengths, int need_ranks = 0) {
    lengths.resize((size_t)T);
    auto work = [&](int t0, int t1) {
        for (int t = t0; t < t1; ++t) {
            const int l0 = off[t], L = off[t + 1] - off[t];
            template_anchor(tl + 4 * (size_t)l0, L, anchors + 2 * (size_t)t);
            float* len = line_len + l0;
            int32_t* idx = argsort + l0;
            for (int i = 0; i < L; ++i) {
                len[i] = line_length(tl + 4 * ((size_t)l0 + i));
                idx[i] = i;
            }
            lengths[(size_t)t] = eigen_sum(len, L);   // math.h:319-324
            constexpr int kMaxSel = 8;
            if (need_ranks > 0 && need_ranks < kMaxSel && need_ranks + 1 < L) {
                // the need_ranks + 1 largest lengths, descending, by insertion into a short list
                const int k = need_ranks + 1;
                float top[kMaxSel];
                int32_t at[kMaxSel];
                int n = 0;
                bool bad = false;                  // NaN among the lengths: no order to speak of
                for (int i = 0; i < L; ++i) {
                    const float v = len[i];
                    if (v != v) { bad = true; break; }
                    if (n == k && !(v > top[k - 1])) continue;    // (ties at or below the extra, k-th value do not touch the leading ranks)
                    int j = n < k ? n : k - 1;
                    while (j > 0 && v > top[j - 1]) { top[j] = top[j - 1]; at[j] = at[j - 1]; --j; }
                    top[j] = v;
                    at[j] = i;
                    if (n < k) ++n;
                }
                bool distinct = !bad && n == k;
                for (int j = 0; distinct && j + 1 < k; ++j) distinct = top[j] > top[j + 1];
                if (distinct) {
                    // ranks [0, need_ranks) as std::sort would give them; the remaining slots hold the other indices in
                    // natural order (never read by a search with this max_tmpl_lines)
                    int w = 0;
                    for (int j = 0; j < need_ranks; ++j) idx[w++] = at[j];
                    for (int i = 0; i < L; ++i) {
                        bool used = false;
                        for (int j = 0; j < need_ranks; ++j) used |= at[j] == i;
                        if (!used) idx[w++] = i;
                    }
                    continue;
                }
            }
            // argsort(tmpl_lengths, std::greater<>()) (defaultsearch.cpp:35, math.h:107-116): same std::sort, same comparator
            std::sort(idx, idx + L, [len](int32_t const i1, int32_t const i2) { return len[i1] > len[i2]; });
        }
    };
    if (T < 256) { work(0, T); return; }
    std::lock_guard<std::mutex> lk(g_pool_mutex);
    host_pool().parallel_for(T, 64, work);
}

// (re)load a template set into an existing object: device buffers grow only, host scratch is reused
// make the main stream wait for a template upload in flight on the copy stream
static fdcm_status templates_ready(fdcm_templates* t, cudaStream_t s) {
    if (t->upload_pending) {
        CUDA_TRY(cudaStreamWaitEvent(s, t->ready, 0));
        t->upload_pending = false;
    }
    return FDCM_OK;
}

static std::atomic<uint64_t> g_tset_loads{0};

// Only fdcm_templates_create (a new set) and fdcm_search_host (the map's own set, under its host_tset_mutex, after the
// previous search of that map has synchronised) load a set, so no kernel can still be reading the device arrays here.
static fdcm_status templates_load(fdcm_templates* t, const float* tmpl_lines, const int32_t* tmpl_offsets, int32_t n_tmpl,
                                  cudaStream_t main_stream, int need_ranks = 0) {
    (void)main_stream;
    cudaStream_t s;
    if (fdcm_status st = get_copy_stream(t->device, &s)) return st;
    if (!t->ready) CUDA_TRY(cudaEventCreateWithFlags(&t->ready, cudaEventDisableTiming));
    if (n_tmpl < 0 || !tmpl_offsets) return fail(FDCM_ERR_INVALID, "bad template offsets");
    for (int i = 0; i < n_tmpl; ++i)
        if (tmpl_offsets[i + 1] < tmpl_offsets[i]) return fail(FDCM_ERR_INVALID, "template offsets must be non-decreasing");
    const int64_t n = tmpl_offsets[n_tmpl];
    if (n > 0 && !tmpl_lines) return fail(FDCM_ERR_INVALID, "tmpl_lines is null");
    t->n_tmpl = n_tmpl;
    t->n_lines = n;
    t->max_lines = 0;
    t->load_id = g_tset_loads.fetch_add(1) + 1;
    t->offsets.assign(tmpl_offsets, tmpl_offsets + n_tmpl + 1);
    for (int i = 0; i < n_tmpl; ++i) t->max_lines = std::max(t->max_lines, tmpl_offsets[i + 1] - tmpl_offsets[i]);
    CUDA_TRY(t->h_line_len.resize((size_t)std::max<int64_t>(n, 1)));
    CUDA_TRY(t->h_argsort.resize((size_t)std::max<int64_t>(n, 1)));
    CUDA_TRY(t->h_anchors.resize((size_t)std::max<int32_t>(2 * n_tmpl, 2)));
    template_host_prep(tmpl_lines, tmpl_offsets, n_tmpl, t->h_line_len.data(), t->h_argsort.data(), t->h_anchors.data(), t->lengths,
                       need_ranks);
    cudaError_t e = t->lines.reserve(std::max<size_t>(16, (size_t)n * 16));
    if (e == cudaSuccess) e = t->offs.reserve((size_t)(n_tmpl + 1) * 4);
    if (e == cudaSuccess) e = t->argsort.reserve(std::max<size_t>(4, (size_t)n * 4));
    if (e == cudaSuccess) e = t->line_len.reserve(std::max<size_t>(4, (size_t)n * 4));
    if (e == cudaSuccess) e = t->anchors.reserve(std::max<size_t>(8, (size_t)n_tmpl * 8));
    if (e == cudaSuccess && n) e = cudaMemcpyAsync(t->lines.p, tmpl_lines, (size_t)n * 16, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(t->offs.p, tmpl_offsets, (size_t)(n_tmpl + 1) * 4, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess && n) e = cudaMemcpyAsync(t->argsort.p, t->h_argsort.data(), (size_t)n * 4, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess && n) e = cudaMemcpyAsync(t->line_len.p, t->h_line_len.data(), (size_t)n * 4, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess && n_tmpl) e = cudaMemcpyAsync(t->anchors.p, t->h_anchors.data(), (size_t)n_tmpl * 8, cudaMemcpyHostToDevice, s);
    // no host synchronisation needed: pageable sources are staged by the runtime before the call returns
    if (e == cudaSuccess) e = cudaEventRecord(t->ready, s);
    if (e != cudaSuccess)
        return fail(e == cudaErrorMemoryAllocation ? FDCM_ERR_NOMEM : FDCM_ERR_CUDA,
                    std::string("templates_load: ") + cudaGetErrorString(e));
    t->upload_pending = true;
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_templates_create(const float* tmpl_lines, const int32_t* tmpl_offsets, int32_t n_tmpl, int32_t device,
                                             fdcm_templates** out) {
    if (!out) return fail(FDCM_ERR_INVALID, "out is null");
    *out = nullptr;
    CUDA_TRY(cudaSetDevice(device));
    cudaStream_t s;
    if (fdcm_status st = get_stream(device, &s)) return st;
    fdcm_templates* t = new (std::nothrow) fdcm_templates();
    if (!t) return fail(FDCM_ERR_NOMEM, "host allocation failed");
    t->device = device;
    fdcm_status st = templates_load(t, tmpl_lines, tmpl_offsets, n_tmpl, s);
    if (st == FDCM_OK && cudaEventSynchronize(t->ready) != cudaSuccess) st = fail(FDCM_ERR_CUDA, "templates_create: upload failed");
    if (st == FDCM_OK) t->upload_pending = false;
    if (st != FDCM_OK) {
        delete t;
        return st;
    }
    *out = t;
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_templates_release(fdcm_templates* t) {
    delete t;
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_templates_lengths(const fdcm_templates* t, float* lengths) {
    if (!t || !lengths) return fail(FDCM_ERR_INVALID, "null argument");
    std::memcpy(lengths, t->lengths.data(), t->lengths.size() * sizeof(float));
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_template_anchors(const float* tl, const int32_t* off, int32_t T, float* anchors_xy) {
    if (T < 0 || !off || (T > 0 && !anchors_xy)) return fail(FDCM_ERR_INVALID, "null argument");
    for (int t = 0; t < T; ++t) {
        if (off[t + 1] < off[t]) return fail(FDCM_ERR_INVALID, "template offsets must be non-decreasing");
        if (off[t + 1] > off[t] && !tl) return fail(FDCM_ERR_INVALID, "tmpl_lines is null");
    }
    for (int t = 0; t < T; ++t) template_anchor(tl + 4 * (size_t)off[t], off[t + 1] - off[t], anchors_xy + 2 * (size_t)t);
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_template_lengths(const float* tl, const int32_t* off, int32_t T, float* lengths) {
    if (T < 0 || !off || !lengths) return fail(FDCM_ERR_INVALID, "null argument");
    for (int t = 0; t < T; ++t) {
        const int L = off[t + 1] - off[t];
        std::vector<float> len((size_t)L);
        for (int i = 0; i < L; ++i) len[(size_t)i] = line_length(tl + 4 * ((size_t)off[t] + i));
        lengths[t] = eigen_sum(len.data(), L);
    }
    return FDCM_OK;
}


// =============================================================================================
// multi-GPU: one process per GPU, NCCL resolved at run time (dlopen: the library has no hard NCCL dependency, and a
// process that already loaded torch's NCCL shares that copy through the SONAME)
// =============================================================================================
#include <dlfcn.h>
#include <nccl.h>   // types only

struct NcclApi {
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
};
static const NcclApi& nccl_api() {
    static const NcclApi api = [] {
        NcclApi a;
        void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!h) return a;
        a.GetUniqueId = (decltype(a.GetUniqueId))dlsym(h, "ncclGetUniqueId");
        a.CommInitRank = (decltype(a.CommInitRank))dlsym(h, "ncclCommInitRank");
        a.CommDestroy = (decltype(a.CommDestroy))dlsym(h, "ncclCommDestroy");
        a.AllGather = (decltype(a.AllGather))dlsym(h, "ncclAllGather");
        a.Broadcast = (decltype(a.Broadcast))dlsym(h, "ncclBroadcast");
        a.GetErrorString = (decltype(a.GetErrorString))dlsym(h, "ncclGetErrorString");
        a.ok = a.GetUniqueId && a.CommInitRank && a.CommDestroy && a.AllGather && a.Broadcast && a.GetErrorString;
        return a;
    }();
    return api;
}
#define NCCL_TRY(expr)                                                                                     \
    do {                                                                                                   \
        ncclResult_t _r = (expr);                                                                          \
        if (_r != ncclSuccess) return fail(FDCM_ERR_CUDA, std::string(#expr) + ": " + nccl_api().GetErrorString(_r)); \
    } while (0)

struct fdcm_comm {
    ncclComm_t comm = nullptr;
    int rank = 0, world = 1, device = 0;
    DevBuf gather, merged, merged_n;
    ~fdcm_comm() {
        cudaSetDevice(device);
        for (DevBuf* b : {&gather, &merged, &merged_n}) b->release();
        if (comm) nccl_api().CommDestroy(comm);
    }
};

extern "C" fdcm_status fdcm_comm_unique_id(uint8_t id[FDCM_COMM_ID_BYTES]) {
    if (!id) return fail(FDCM_ERR_INVALID, "id is null");
    static_assert(FDCM_COMM_ID_BYTES == NCCL_UNIQUE_ID_BYTES, "id size");
    if (!nccl_api().ok) return fail(FDCM_ERR_CUDA, "NCCL (libnccl.so.2) is not available");
    ncclUniqueId u;
    NCCL_TRY(nccl_api().GetUniqueId(&u));
    std::memcpy(id, u.internal, NCCL_UNIQUE_ID_BYTES);
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_set_host_threads(int32_t n) {
    if (n < 0) return fail(FDCM_ERR_INVALID, "bad thread count");
    g_host_threads = n;
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_comm_init(const uint8_t id[FDCM_COMM_ID_BYTES], int32_t rank, int32_t world, int32_t device, fdcm_comm** out) {
    if (!out) return fail(FDCM_ERR_INVALID, "out is null");
    *out = nullptr;
    if (!id || world < 1 || rank < 0 || rank >= world) return fail(FDCM_ERR_INVALID, "bad communicator arguments");
    if (!nccl_api().ok) return fail(FDCM_ERR_CUDA, "NCCL (libnccl.so.2) is not available");
    CUDA_TRY(cudaSetDevice(device));
    fdcm_comm* c = new (std::nothrow) fdcm_comm();
    if (!c) return fail(FDCM_ERR_NOMEM, "host allocation failed");
    c->rank = rank; c->world = world; c->device = device;
    ncclUniqueId u;
    std::memcpy(u.internal, id, NCCL_UNIQUE_ID_BYTES);
    ncclResult_t r = nccl_api().CommInitRank(&c->comm, world, u, rank);
    if (r != ncclSuccess) {
        c->comm = nullptr;
        delete c;
        return fail(FDCM_ERR_CUDA, std::string("ncclCommInitRank: ") + nccl_api().GetErrorString(r));
    }
    // one process per GPU on one host: share the host cores between the ranks' template-preparation pools
    if (g_host_threads == 0) g_host_threads = std::max(1, (int)std::thread::hardware_concurrency() / world);
    *out = c;
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_comm_destroy(fdcm_comm* c) {
    delete c;
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_comm_info(const fdcm_comm* c, int32_t* rank, int32_t* world) {
    if (!c) return fail(FDCM_ERR_INVALID, "comm is null");
    if (rank) *rank = c->rank;
    if (world) *world = c->world;
    return FDCM_OK;
}

// contiguous template block of a rank (global tmpl_idx = begin + local index; ties of the merged top-k then resolve
// in global hypothesis order)
extern "C" fdcm_status fdcm_comm_shard(int32_t n_items, int32_t rank, int32_t world, int32_t* begin, int32_t* end) {
    if (!begin || !end || n_items < 0 || world < 1 || rank < 0 || rank >= world) return fail(FDCM_ERR_INVALID, "bad argument");
    const int64_t q = n_items / world, r = n_items % world;
    *begin = (int32_t)(rank * q + std::min<int64_t>(rank, r));
    *end = (int32_t)(*begin + q + (rank < r ? 1 : 0));
    return FDCM_OK;
}

// device-side exchange of the ranks' top-k: ncclAllGather of the k x 32-byte buffer the top-K kernels just wrote, on the
// compute stream, then an R*k -> k merge kernel; the caller downloads the merged list
static fdcm_status comm_merge_topk(fdcm_comm* c, const fdcm_dt3* m, int k, cudaStream_t s, const fdcm_match** d_result, const int** d_n) {
    if (c->device != m->device) return fail(FDCM_ERR_INVALID, "communicator and feature map live on different devices");
    CUDA_TRY(c->gather.reserve((size_t)c->world * k * sizeof(fdcm_match)));
    CUDA_TRY(c->merged.reserve((size_t)k * sizeof(fdcm_match)));
    CUDA_TRY(c->merged_n.reserve(4));
    NCCL_TRY(nccl_api().AllGather(m->s_topk_out.p, c->gather.p, (size_t)k * sizeof(fdcm_match), ncclChar, c->comm, s));
    {
        KernelScope ks("topk_merge", 0.0, s, 1);
        launch_topk_merge(c->gather.as<fdcm_match>(), c->world * k, k, c->merged.as<fdcm_match>(), c->merged_n.as<int>(), s);
    }
    *d_result = c->merged.as<fdcm_match>();
    *d_n = c->merged_n.as<int>();
    return FDCM_OK;
}

// =============================================================================================
// search
// =============================================================================================
static float penalty_denominator(int kind, float tau, float length) {
    const float len = std::max(length, 1e-6f);                    // exponentialpenalty.cpp:42
    return kind == FDCM_PENALTY_DEFAULT ? len : std::pow(len, tau);   // defaultpenalty.cpp:39 / exponentialpenalty.cpp:43
}

// download of the (possibly merged) top-k list at the end of a search
static fdcm_status finish_topk(const fdcm_dt3* m, fdcm_comm* comm, int k, cudaStream_t s, unsigned long long* counters, fdcm_match* out,
                               int64_t capacity, int64_t* n_out) {
    const fdcm_match* d_result = m->s_topk_out.as<fdcm_match>();
    const int* d_n = m->s_topk_n.as<int>();
    if (comm)
        if (fdcm_status st = comm_merge_topk(comm, m, k, s, &d_result, &d_n)) return st;
    int n_sel = 0;
    std::vector<fdcm_match> sel((size_t)k);
    CUDA_TRY(cudaMemcpyAsync(&n_sel, d_n, 4, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(sel.data(), d_result, (size_t)k * sizeof(fdcm_match), cudaMemcpyDeviceToHost, s));
    if (counters) CUDA_TRY(cudaMemcpyAsync(counters, m->s_counters.p, 3 * 8, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    *n_out = n_sel;
    if (n_sel > capacity || (n_sel > 0 && !out)) return fail(FDCM_ERR_CAPACITY, "output buffer too small");
    if (n_sel > 0) std::memcpy(out, sel.data(), (size_t)n_sel * sizeof(fdcm_match));
    return FDCM_OK;
}

// a rank whose shard yields no hypothesis still takes part in the exchange
static fdcm_status exchange_empty(const fdcm_dt3* m, fdcm_comm* comm, int k, fdcm_match* out, int64_t capacity, int64_t* n_out) {
    CUDA_TRY(cudaSetDevice(m->device));
    cudaStream_t s;
    if (fdcm_status st = get_stream(m->device, &s)) return st;
    CUDA_TRY(m->s_topk_out.reserve((size_t)k * sizeof(fdcm_match)));
    CUDA_TRY(m->s_topk_n.reserve(4));
    launch_topk_invalid(m->s_topk_out.as<fdcm_match>(), k, m->s_topk_n.as<int>(), s);
    return finish_topk(m, comm, k, s, nullptr, out, capacity, n_out);
}

// Penalty denominators of set t for (kind, tau) (host powf like the reference) in the map's buffer: written through the
// pinned staging `stage` on the copy stream `cs` unless the map holds them already.  Nothing else reads that buffer: every
// earlier use of the map has synchronised (m->search_mutex held), and other maps sharing the set have their own.
static fdcm_status map_denominators(const fdcm_dt3* m, const fdcm_templates* t, int kind, float tau, float* stage, cudaStream_t cs,
                                    const float** d_denom) {
    *d_denom = nullptr;
    if (kind == FDCM_PENALTY_NONE) return FDCM_OK;
    if (m->denom_set != t->load_id || m->denom_kind != kind || m->denom_tau != tau) {
        m->denom_set = 0;
        CUDA_TRY(m->s_denom.reserve(std::max<size_t>(4, (size_t)t->n_tmpl * 4)));
        for (int i = 0; i < t->n_tmpl; ++i) stage[i] = penalty_denominator(kind, tau, t->lengths[(size_t)i]);
        CUDA_TRY(cudaMemcpyAsync(m->s_denom.p, stage, (size_t)t->n_tmpl * 4, cudaMemcpyHostToDevice, cs));
        m->denom_set = t->load_id;
        m->denom_kind = kind;
        m->denom_tau = tau;
    }
    *d_denom = m->s_denom.as<float>();
    return FDCM_OK;
}

// Small per-call uploads (n_off hypothesis offsets to m->s_hyp_off, the penalty denominators) go through the set's pinned
// staging on the copy stream, and `s` waits for them: a pageable copy on `s` would first wait for everything queued there,
// e.g. a map build in flight.  (m->search_mutex held)
static fdcm_status stage_uploads(const fdcm_dt3* m, fdcm_templates* t, const int64_t* hyp_off, size_t n_off, int kind, float tau,
                                 cudaStream_t s, const float** d_denom) {
    std::lock_guard<std::mutex> lk(t->mu);
    cudaStream_t cs;
    if (fdcm_status st = get_copy_stream(m->device, &cs)) return st;
    if (!t->ready) CUDA_TRY(cudaEventCreateWithFlags(&t->ready, cudaEventDisableTiming));
    else CUDA_TRY(cudaEventSynchronize(t->ready));   // the staging buffer may still feed an earlier upload (other threads)
    const size_t off_bytes = n_off * 8, den_bytes = (size_t)t->n_tmpl * 4;
    CUDA_TRY(t->stage_reserve(std::max<size_t>(16, off_bytes + den_bytes)));
    unsigned char* stage = static_cast<unsigned char*>(t->h_stage);
    if (off_bytes) {
        std::memcpy(stage, hyp_off, off_bytes);
        CUDA_TRY(cudaMemcpyAsync(m->s_hyp_off.p, stage, off_bytes, cudaMemcpyHostToDevice, cs));
    }
    if (fdcm_status st = map_denominators(m, t, kind, tau, reinterpret_cast<float*>(stage + off_bytes), cs, d_denom)) return st;
    CUDA_TRY(cudaEventRecord(t->ready, cs));
    CUDA_TRY(cudaStreamWaitEvent(s, t->ready, 0));
    t->upload_pending = false;   // (this event is recorded after any template upload on the same copy stream)
    return FDCM_OK;
}

// The search kernel stages the longest template of a set in shared memory, at least one warp's worth per block: a set
// holding a template longer than one warp can stage within the device's per-block opt-in limit cannot be searched.
static fdcm_status search_smem_optin(int device, int max_lines, int* smem_optin) {
    CUDA_TRY(cudaDeviceGetAttribute(smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
    const int limit = search_max_template_lines(*smem_optin);
    if (max_lines > limit)
        return fail(FDCM_ERR_INVALID, "template of " + std::to_string(max_lines) + " lines: the search takes at most " +
                                          std::to_string(limit) + " lines per template on this device (" +
                                          std::to_string(*smem_optin) + " bytes of shared memory per block)");
    return FDCM_OK;
}

// parameters of the distinct top-K (fdcm_search_select)
static fdcm_status check_select(const fdcm_select_params* q, int32_t top_k, bool comm) {
    if (top_k < 1) return fail(FDCM_ERR_INVALID, "distinct top-K: top_k must be >= 1");
    if (q->max_per_template < 0) return fail(FDCM_ERR_INVALID, "distinct top-K: max_per_template must be >= 0");
    if (!(q->radius >= 0.f) || !std::isfinite(q->radius)) return fail(FDCM_ERR_INVALID, "distinct top-K: radius must be finite and >= 0");
    if (!(q->max_angle >= 0.f)) return fail(FDCM_ERR_INVALID, "distinct top-K: max_angle must be >= 0 (and not NaN)");
    if (q->across_templates && comm)
        return fail(FDCM_ERR_INVALID, "distinct top-K: across_templates is not supported by the multi-GPU search (it does not decompose over template shards)");
    if (q->across_templates && top_k > FDCM_SELECT_MAX_ACROSS)
        return fail(FDCM_ERR_INVALID, "distinct top-K: across_templates takes top_k <= " + std::to_string(FDCM_SELECT_MAX_ACROSS));
    return FDCM_OK;
}

// Distinct top-K over the records the search kernel just queued on `s`: writes s_topk_out / s_topk_n like the top-K kernels
static fdcm_status run_select(const fdcm_dt3* m, const fdcm_templates* t, const fdcm_search_params* p, const fdcm_select_params* q,
                              int64_t H, cudaStream_t s) {
    if (H >= ((int64_t)1 << 31)) return fail(FDCM_ERR_INVALID, "distinct top-K: more than 2^31 - 1 hypotheses");
    SelectLaunch sp;
    sp.rec = m->s_rec.as<fdcm_match>();
    sp.valid = m->s_valid.as<uint8_t>();
    sp.hyp_off = m->s_hyp_off.as<int64_t>();
    sp.anchors = t->anchors.as<float2>();
    sp.n_hyp = H;
    sp.n_tmpl = t->n_tmpl;
    sp.tmpl_idx_base = p->tmpl_idx_base;
    sp.top_k = p->top_k;
    sp.cap = q->max_per_template;
    sp.radius_on = q->radius > 0.f;
    sp.r2 = q->radius * q->radius;
    sp.any_angle = q->max_angle >= 3.14159274f;
    sp.cos_thr = (float)std::cos((double)q->max_angle);
    const bool within = q->across_templates == 0;
    const size_t tmp = select_temp_bytes(H);
    CUDA_TRY(m->s_sel_keys.reserve((size_t)H * 8));
    CUDA_TRY(m->s_sel_keys2.reserve((size_t)H * 8));
    CUDA_TRY(m->s_sel_vals.reserve((size_t)H * 4));
    CUDA_TRY(m->s_sel_vals2.reserve((size_t)H * 4));
    CUDA_TRY(m->s_sel_tmp.reserve(std::max<size_t>(tmp, 16)));
    uint64_t* keys = m->s_sel_keys.as<uint64_t>();
    uint64_t* sorted_keys = m->s_sel_keys2.as<uint64_t>();
    int32_t* iota = m->s_sel_vals.as<int32_t>();
    int32_t* sorted_h = m->s_sel_vals2.as<int32_t>();
    {
        KernelScope k("select_sort", 0.0, s, 1);   // our key kernel; the CUB radix-sort launches are library code
        launch_select_sort(sp, within, keys, sorted_keys, iota, sorted_h, m->s_sel_tmp.p, tmp, s);
    }
    fdcm_match* d_out = m->s_topk_out.as<fdcm_match>();
    int* d_n = m->s_topk_n.as<int>();
    if (within) {
        CUDA_TRY(m->s_sel_surv.reserve((size_t)H * 4));
        if (sp.radius_on) CUDA_TRY(m->s_sel_acc.reserve((size_t)H * 16));
        {
            KernelScope k("select_greedy", 0.0, s);
            launch_select_greedy(sp, sorted_keys, sorted_h, m->s_sel_surv.as<uint32_t>(), m->s_sel_acc.as<float4>(), s);
        }
        // the unsorted keys and the per-template order are free again: they take the global sort of the survivors
        KernelScope k("select_topk", 0.0, s, 1);
        launch_select_topk(sp, m->s_sel_surv.as<uint32_t>(), reinterpret_cast<uint32_t*>(keys), iota, sorted_h, m->s_sel_tmp.p, tmp, d_out,
                           d_n, s);
    } else {
        KernelScope k("select_walk", 0.0, s);
        launch_select_walk(sp, sorted_keys, sorted_h, d_out, d_n, s);
    }
    CUDA_TRY(cudaGetLastError());
    return FDCM_OK;
}

// parameters of the pose refinement (fdcm_refine_matches, fdcm_search_refine)
static fdcm_status check_refine(const fdcm_refine_params* r) {
    if (!r) return fail(FDCM_ERR_INVALID, "refine is null");
    if (r->levels < 1) return fail(FDCM_ERR_INVALID, "pose refinement: levels must be >= 1");
    if (r->rot_steps < 0 || r->rot_steps > FDCM_REFINE_MAX_STEPS || r->trans_steps < 0 || r->trans_steps > FDCM_REFINE_MAX_STEPS)
        return fail(FDCM_ERR_INVALID, "pose refinement: rot_steps and trans_steps must be in 0.." + std::to_string(FDCM_REFINE_MAX_STEPS));
    if (!(r->rot_step >= 0.f) || !std::isfinite(r->rot_step) || !(r->trans_step >= 0.f) || !std::isfinite(r->trans_step))
        return fail(FDCM_ERR_INVALID, "pose refinement: rot_step and trans_step must be finite and >= 0");
    return FDCM_OK;
}

// the host table of one level: ci, si of every rotation index and the translation step
static void refine_level_table(const fdcm_refine_params* r, int level, RefineLevel* lv) {
    const double step = (double)r->rot_step / std::ldexp(1.0, level);
    for (int i = -r->rot_steps; i <= r->rot_steps; ++i) {
        lv->ci[i + r->rot_steps] = (float)std::cos((double)i * step);
        lv->si[i + r->rot_steps] = (float)std::sin((double)i * step);
    }
    lv->h = r->trans_step * std::ldexp(1.0f, -level);
}

// at most this many matches per call: the evaluation grid has (2 rot_steps + 1) blocks per match
static constexpr int64_t kRefineMaxMatches = ((int64_t)1 << 31) / kRefineSide;

// Refinement of the n (or *d_n <= n) matches at d_in, queued on `s`; the refined records go to d_out (which may be d_in)
static fdcm_status run_refine(const fdcm_dt3* m, const fdcm_templates* t, int32_t tmpl_idx_base, const float* d_denom,
                              const fdcm_refine_params* r, const fdcm_match* d_in, const int* d_n, int n, fdcm_match* d_out,
                              int smem_optin, cudaStream_t s) {
    CUDA_TRY(m->s_ref_state.reserve((size_t)n * sizeof(RefineState)));
    CUDA_TRY(m->s_ref_keys.reserve((size_t)n * 8));
    RefineLaunch rl;
    rl.in = d_in;
    rl.d_n = d_n;
    rl.n = n;
    rl.lines = t->lines.as<float4>();
    rl.offsets = t->offs.as<int32_t>();
    rl.anchors = t->anchors.as<float2>();
    rl.denom = d_denom;
    rl.tmpl_idx_base = tmpl_idx_base;
    rl.n_r = r->rot_steps;
    rl.n_t = r->trans_steps;
    rl.state = m->s_ref_state.as<RefineState>();
    rl.keys = m->s_ref_keys.as<unsigned long long>();
    {
        KernelScope k("refine_init", 0.0, s);
        launch_refine_init(rl, s);
    }
    for (int level = 0; level < r->levels; ++level) {
        RefineLevel lv{};
        refine_level_table(r, level, &lv);
        {
            KernelScope k("refine_eval", 0.0, s);
            CUDA_TRY(launch_refine_eval(map_view(m), m->table_dev, rl, lv, t->max_lines, smem_optin, s));
        }
        KernelScope k("refine_advance", 0.0, s);
        launch_refine_advance(rl, lv, level + 1 == r->levels ? d_out : nullptr, s);
    }
    CUDA_TRY(cudaGetLastError());
    return FDCM_OK;
}

// sel: distinct top-K (fdcm_search_select); ref: pose refinement of the top-K (fdcm_search_refine); nullptr when not asked
static fdcm_status search_impl(const fdcm_dt3* m, const fdcm_templates* tc, const float* scene, int32_t n_scene,
                               const fdcm_search_params* p, fdcm_match* out, int64_t capacity, int64_t* n_out, fdcm_comm* comm,
                               const fdcm_select_params* sel, const fdcm_refine_params* ref = nullptr) {
    if (!m || !tc || !p || !n_out) return fail(FDCM_ERR_INVALID, "null argument");
    *n_out = 0;
    if (sel)
        if (fdcm_status st = check_select(sel, p->top_k, comm != nullptr)) return st;
    // caps and radius both off: the selection is the plain top-K
    if (sel && sel->max_per_template == 0 && !(sel->radius > 0.f)) sel = nullptr;
    if (comm && p->top_k <= 0) return fail(FDCM_ERR_INVALID, "the multi-GPU search needs top_k > 0");
#define FDCM_NO_LOCAL_MATCHES() do { if (comm) return exchange_empty(m, comm, p->top_k, out, capacity, n_out); return FDCM_OK; } while (0)
    if (p->max_tmpl_lines < 0 || p->max_scene_lines < 0 || p->batch_size < 0 || p->top_k < 0 || p->penalty_kind < 0 ||
        p->penalty_kind > 2)
        return fail(FDCM_ERR_INVALID, "bad search parameters");
    if (tc->device != m->device) return fail(FDCM_ERR_INVALID, "templates and feature map live on different devices");
    fdcm_templates* t = const_cast<fdcm_templates*>(tc);
    std::lock_guard<std::mutex> lk(m->search_mutex);
    m->last_n_hyp = 0;
    m->last_stats = fdcm_search_stats{0, 0, 0, 0};
    // defaultmatch.cpp:40-41
    // n_scene == FDCM_SCENE_RESIDENT: the scene the map was built from (already on the device); an EMPTY scene
    // (n_scene == 0, whatever the pointer) yields no matches like the reference (defaultmatch.cpp:40)
    const bool resident_scene = n_scene == FDCM_SCENE_RESIDENT;
    if (n_scene < 0 && !resident_scene) return fail(FDCM_ERR_INVALID, "bad scene size");
    if (n_scene > 0 && !scene) return fail(FDCM_ERR_INVALID, "scene is null");
    if (resident_scene) {
        scene = m->h_build_scene.data();
        n_scene = (int32_t)(m->h_build_scene.size() / 4);
    }
    if (t->n_tmpl == 0 || n_scene <= 0 || (m->dm.W == 0 && m->dm.H == 0)) FDCM_NO_LOCAL_MATCHES();
    if (m->stage != 0) return fail(FDCM_ERR_INVALID, "feature map was built with a debug stage");
    CUDA_TRY(cudaSetDevice(m->device));
    cudaStream_t s;
    if (fdcm_status st = get_stream(m->device, &s)) return st;
    if (fdcm_status st = map_wait(m, s)) return st;
    if (fdcm_status st = templates_ready(t, s)) return st;
    int smem_optin = 0;
    if (fdcm_status st = search_smem_optin(m->device, t->max_lines, &smem_optin)) return st;

    // ---- host prep: scene length order (defaultsearch.cpp:32-36) and hypothesis offsets ----
    const SceneFilter flt{p->concentric != 0, p->center_x, p->center_y, p->low_radius, p->high_radius};
    const bool same_filter = flt.on == m->s_filter_on && (!flt.on || (flt.cx == m->s_filter[0] && flt.cy == m->s_filter[1] &&
                                                                      flt.lo == m->s_filter[2] && flt.hi == m->s_filter[3]));
    if (!(resident_scene && m->s_resident_is_build && same_filter)) {
        if (fdcm_status st = upload_search_scene(m, scene, n_scene, flt, s)) return st;
        m->s_resident_is_build = resident_scene;
    }
    n_scene = m->s_sorted_n;   // the lines that take part in the length matching
    if (n_scene <= 0) FDCM_NO_LOCAL_MATCHES();   // concentricrange.cpp:37-38
    const int nS = std::min<int>(n_scene, p->max_scene_lines);
    std::vector<int64_t> hyp_off((size_t)t->n_tmpl + 1, 0);
    for (int i = 0; i < t->n_tmpl; ++i) {
        const int L = t->offsets[(size_t)i + 1] - t->offsets[(size_t)i];
        hyp_off[(size_t)i + 1] = hyp_off[(size_t)i] + 2LL * std::min(L, p->max_tmpl_lines) * nS;
    }
    const int64_t H = hyp_off[(size_t)t->n_tmpl];
    m->last_n_hyp = H;
    m->last_stats.n_hypotheses = H;
    if (H == 0) FDCM_NO_LOCAL_MATCHES();
#undef FDCM_NO_LOCAL_MATCHES

    // ---- workspace ----
    CUDA_TRY(m->s_hyp_off.reserve(hyp_off.size() * 8));
    CUDA_TRY(m->s_rec.reserve((size_t)H * sizeof(fdcm_match)));
    CUDA_TRY(m->s_valid.reserve((size_t)H));
    CUDA_TRY(m->s_hyp.reserve((size_t)H * 16));
    CUDA_TRY(m->s_counters.reserve(3 * 8));

    const float* d_denom = nullptr;
    if (fdcm_status st = stage_uploads(m, t, hyp_off.data(), hyp_off.size(), p->penalty_kind, p->penalty_tau, s, &d_denom)) return st;
    CUDA_TRY(cudaMemsetAsync(m->s_counters.p, 0, 3 * 8, s));

    TemplatesView tv;
    tv.lines = t->lines.as<float4>();
    tv.offsets = t->offs.as<int32_t>();
    tv.argsort = t->argsort.as<int32_t>();
    tv.line_len = t->line_len.as<float>();
    tv.denom = d_denom;
    tv.n_tmpl = t->n_tmpl;
    tv.max_lines = std::max(1, t->max_lines);
    SceneView sv;
    sv.lines = m->s_scene.as<float4>();
    sv.sorted_len = m->s_sorted_len.as<float>();
    sv.sorted_idx = m->s_sorted_idx.as<int32_t>();
    sv.n = n_scene;   // number of length-ordered (possibly radius-filtered) lines; lines[] holds the whole scene
    SearchLaunch sl;
    sl.max_tmpl_lines = p->max_tmpl_lines;
    sl.max_scene_lines = p->max_scene_lines;
    sl.batch = p->batch_size > 0 ? p->batch_size : 1;   // DefaultOptimize == batches of one (defaultoptimize.cpp:49-64)
    sl.tmpl_idx_base = p->tmpl_idx_base;
    sl.hyp_off = m->s_hyp_off.as<int64_t>();
    sl.n_hyp = H;
    sl.direct_align = nullptr;
    SearchOutputs so;
    so.rec = m->s_rec.as<fdcm_match>();
    so.valid = m->s_valid.as<uint8_t>();
    so.hyp = m->s_hyp.as<int4>();
    so.counters = m->s_counters.as<unsigned long long>();
    sl.perm = nullptr;
    sl.hyp_ready = nullptr;
    if (H >= 4096 && H < (int64_t)1 << 31) {
        // process the hypotheses in the spatial order of their scene lines (L2 locality of the map gathers)
        const float ex = m->s_scene_max[0] - m->s_scene_min[0], ey = m->s_scene_max[1] - m->s_scene_min[1];
        const int cells_x = std::min(4096, std::max(1, (int)(ex / (float)kSearchCellW) + 1));
        const int cells_y = std::min(4096, std::max(1, (int)(ey / (float)kSearchCellH) + 1));
        int key_bits = 1;
        while (((int64_t)1 << key_bits) < (int64_t)cells_x * cells_y) ++key_bits;
        const size_t tmp = search_order_temp_bytes(H);
        CUDA_TRY(m->s_keys.reserve((size_t)H * 4));
        CUDA_TRY(m->s_keys2.reserve((size_t)H * 4));
        CUDA_TRY(m->s_idx.reserve((size_t)H * 4));
        CUDA_TRY(m->s_perm.reserve((size_t)H * 4));
        CUDA_TRY(m->s_sort_tmp.reserve(std::max<size_t>(tmp, 16)));
        KernelScope k("search_order", 0.0, s, 1);   // our key kernel; the 3 CUB radix-sort launches are library code
        launch_search_order(tv, sv, sl, m->s_keys.as<uint32_t>(), m->s_keys2.as<uint32_t>(), m->s_idx.as<int32_t>(),
                            m->s_perm.as<int32_t>(), m->s_sort_tmp.p, tmp, m->s_scene_min[0], m->s_scene_min[1], cells_x, key_bits,
                            so.hyp, s);
        sl.perm = m->s_perm.as<int32_t>();
        sl.hyp_ready = so.hyp;
    }
    {
        KernelScope k("search", 0.0, s);
        CUDA_TRY(launch_search(map_view(m), m->table_dev, tv, sv, sl, so, smem_optin, s));
    }

    unsigned long long counters[3] = {0, 0, 0};
    fdcm_status result = FDCM_OK;
    if (p->top_k > 0) {
        const int k = p->top_k;
        if (sel) {
            CUDA_TRY(m->s_topk_out.reserve((size_t)k * sizeof(fdcm_match)));
            CUDA_TRY(m->s_topk_n.reserve(4));
            if (fdcm_status st = run_select(m, t, p, sel, H, s)) return st;
        } else {
            const int blocks = topk_ws_blocks(H);
            CUDA_TRY(m->s_topk_score.reserve((size_t)blocks * k * 4));
            CUDA_TRY(m->s_topk_idx.reserve((size_t)blocks * k * 8));
            CUDA_TRY(m->s_topk_out.reserve((size_t)k * sizeof(fdcm_match)));
            CUDA_TRY(m->s_topk_n.reserve(4));
            {
                KernelScope ks("topk", 0.0, s, 2);   // two kernels in this scope
                launch_topk(so.rec, so.valid, H, k, m->s_topk_score.as<float>(), m->s_topk_idx.as<int64_t>(), blocks,
                            m->s_topk_out.as<fdcm_match>(), m->s_topk_n.as<int>(), s);
            }
            CUDA_TRY(cudaGetLastError());
        }
        if (ref)
            if (fdcm_status st = run_refine(m, t, p->tmpl_idx_base, d_denom, ref, m->s_topk_out.as<fdcm_match>(), m->s_topk_n.as<int>(), k,
                                            m->s_topk_out.as<fdcm_match>(), smem_optin, s))
                return st;
        result = finish_topk(m, comm, k, s, counters, out, capacity, n_out);
        if (result != FDCM_OK && result != FDCM_ERR_CAPACITY) return result;
    } else {
        // every match in hypothesis order: download records + flags, compact on the host
        const size_t need = (size_t)H * sizeof(fdcm_match) + (size_t)H;
        if (m->h_pinned_cap < need) {
            if (m->h_pinned) cudaFreeHost(m->h_pinned);
            m->h_pinned = nullptr;
            m->h_pinned_cap = 0;
            CUDA_TRY(cudaMallocHost(&m->h_pinned, need));
            m->h_pinned_cap = need;
        }
        fdcm_match* h_rec = (fdcm_match*)m->h_pinned;
        uint8_t* h_valid = (uint8_t*)m->h_pinned + (size_t)H * sizeof(fdcm_match);
        CUDA_TRY(cudaMemcpyAsync(h_rec, so.rec, (size_t)H * sizeof(fdcm_match), cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaMemcpyAsync(h_valid, so.valid, (size_t)H, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaMemcpyAsync(counters, m->s_counters.p, 3 * 8, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaStreamSynchronize(s));
        int64_t n = 0;
        for (int64_t h = 0; h < H; ++h) n += h_valid[h] ? 1 : 0;
        *n_out = n;
        if (n > capacity || (n > 0 && !out)) result = fail(FDCM_ERR_CAPACITY, "output buffer too small");
        else {
            int64_t w = 0;
            for (int64_t h = 0; h < H; ++h)
                if (h_valid[h]) out[w++] = h_rec[h];
        }
    }
    prof_resolve();
    m->last_stats.n_evaluations = (int64_t)counters[0];
    m->last_stats.n_lookups = (int64_t)counters[1];
    m->last_stats.n_valid = (int64_t)counters[2];
    return result;
}

extern "C" fdcm_status fdcm_search(const fdcm_dt3* m, const fdcm_templates* tc, const float* scene, int32_t n_scene,
                                   const fdcm_search_params* p, fdcm_match* out, int64_t capacity, int64_t* n_out) {
    return search_impl(m, tc, scene, n_scene, p, out, capacity, n_out, nullptr, nullptr);
}

extern "C" fdcm_status fdcm_search_select(const fdcm_dt3* m, const fdcm_templates* tc, const float* scene, int32_t n_scene,
                                          const fdcm_search_params* p, const fdcm_select_params* select, fdcm_match* out, int64_t capacity,
                                          int64_t* n_out) {
    if (!select) return fail(FDCM_ERR_INVALID, "select is null");
    return search_impl(m, tc, scene, n_scene, p, out, capacity, n_out, nullptr, select);
}

extern "C" fdcm_status fdcm_search_refine(const fdcm_dt3* m, const fdcm_templates* tc, const float* scene, int32_t n_scene,
                                          const fdcm_search_params* p, const fdcm_select_params* select, const fdcm_refine_params* refine,
                                          fdcm_match* out, int64_t capacity, int64_t* n_out) {
    if (fdcm_status st = check_refine(refine)) return st;
    if (!p) return fail(FDCM_ERR_INVALID, "null argument");
    if (p->top_k < 1 || p->top_k > kRefineMaxMatches)
        return fail(FDCM_ERR_INVALID, "pose refinement: top_k must be in 1.." + std::to_string(kRefineMaxMatches));
    return search_impl(m, tc, scene, n_scene, p, out, capacity, n_out, nullptr, select, refine);
}

extern "C" fdcm_status fdcm_refine_matches(const fdcm_dt3* m, const fdcm_templates* tc, int32_t tmpl_idx_base, int32_t penalty_kind,
                                           float penalty_tau, const fdcm_refine_params* refine, const fdcm_match* in, int64_t n,
                                           fdcm_match* out) {
    if (fdcm_status st = check_refine(refine)) return st;
    if (!m || !tc || n < 0) return fail(FDCM_ERR_INVALID, "bad argument");
    if (penalty_kind < 0 || penalty_kind > 2) return fail(FDCM_ERR_INVALID, "bad penalty kind");
    if (n == 0) return FDCM_OK;
    if (!in || !out) return fail(FDCM_ERR_INVALID, "null argument");
    if (n > kRefineMaxMatches) return fail(FDCM_ERR_INVALID, "pose refinement: at most " + std::to_string(kRefineMaxMatches) + " matches per call");
    if (tc->device != m->device) return fail(FDCM_ERR_INVALID, "templates and feature map live on different devices");
    if (m->stage != 0) return fail(FDCM_ERR_INVALID, "feature map was built with a debug stage");
    if (m->dm.D == 0) return fail(FDCM_ERR_INVALID, "refine on an empty feature map");
    for (int64_t i = 0; i < n; ++i) {
        const int64_t t = (int64_t)in[i].tmpl_idx - tmpl_idx_base;
        if (t < 0 || t >= tc->n_tmpl)
            return fail(FDCM_ERR_OUT_OF_RANGE, "match " + std::to_string(i) + ": tmpl_idx " + std::to_string(in[i].tmpl_idx) +
                                                   " outside the template set");
    }
    fdcm_templates* t = const_cast<fdcm_templates*>(tc);
    std::lock_guard<std::mutex> lk(m->search_mutex);
    CUDA_TRY(cudaSetDevice(m->device));
    cudaStream_t s;
    if (fdcm_status st = get_stream(m->device, &s)) return st;
    if (fdcm_status st = map_wait(m, s)) return st;
    if (fdcm_status st = templates_ready(t, s)) return st;
    int smem_optin = 0;
    if (fdcm_status st = search_smem_optin(m->device, t->max_lines, &smem_optin)) return st;
    CUDA_TRY(m->s_ref_io.reserve((size_t)n * sizeof(fdcm_match)));
    CUDA_TRY(cudaMemcpyAsync(m->s_ref_io.p, in, (size_t)n * sizeof(fdcm_match), cudaMemcpyHostToDevice, s));
    const float* d_denom = nullptr;   // the search's denominators
    if (fdcm_status st = stage_uploads(m, t, nullptr, 0, penalty_kind, penalty_tau, s, &d_denom)) return st;
    fdcm_match* d_io = m->s_ref_io.as<fdcm_match>();
    if (fdcm_status st = run_refine(m, t, tmpl_idx_base, d_denom, refine, d_io, nullptr, (int)n, d_io, smem_optin, s)) return st;
    CUDA_TRY(cudaMemcpyAsync(out, d_io, (size_t)n * sizeof(fdcm_match), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    prof_resolve();
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_refine_poses(const float transform[6], const float anchor[2], const fdcm_refine_params* refine, int32_t level,
                                         float* out) {
    if (fdcm_status st = check_refine(refine)) return st;
    if (!transform || !anchor || !out) return fail(FDCM_ERR_INVALID, "null argument");
    if (level < 0 || level >= refine->levels) return fail(FDCM_ERR_INVALID, "level must be in 0..levels - 1");
    RefineLevel lv{};
    refine_level_table(refine, level, &lv);
    const int n_r = refine->rot_steps, n_t = refine->trans_steps, NT = 2 * n_t + 1;
    for (int ir = 0; ir < 2 * n_r + 1; ++ir) {
        const RefineRot R = refine_rotation(transform, anchor[0], anchor[1], ir - n_r, lv.ci[ir], lv.si[ir]);
        for (int kk = 0; kk < NT; ++kk)
            for (int jj = 0; jj < NT; ++jj) {
                float* P = out + 6 * (size_t)((ir * NT + kk) * NT + jj);
                if (ir == n_r && kk == n_t && jj == n_t) {   // the grid point (0, 0, 0) is C itself
                    for (int q = 0; q < 6; ++q) P[q] = transform[q];
                    continue;
                }
                P[0] = R.r0; P[1] = R.r1; P[2] = R.bx + (float)(jj - n_t) * lv.h;
                P[3] = R.r3; P[4] = R.r4; P[5] = R.by + (float)(kk - n_t) * lv.h;
            }
    }
    return FDCM_OK;
}

// =============================================================================================
// dense pose-grid search (rules in include/fdcm_b200.h)
// =============================================================================================
static fdcm_status check_dense(const fdcm_dense_params* d) {
    if (!d) return fail(FDCM_ERR_INVALID, "dense is null");
    if (d->rotations < 1 || d->rotations > FDCM_DENSE_MAX_ROTATIONS)
        return fail(FDCM_ERR_INVALID, "dense search: rotations must be in 1.." + std::to_string(FDCM_DENSE_MAX_ROTATIONS));
    if (d->stride < 1 || d->cell < 1) return fail(FDCM_ERR_INVALID, "dense search: stride and cell must be >= 1");
    if (!std::isfinite(d->rot_start) || !std::isfinite(d->rot_step))
        return fail(FDCM_ERR_INVALID, "dense search: rot_start and rot_step must be finite");
    if (d->roi_on) {
        bool ok = d->roi[0] <= d->roi[2] && d->roi[1] <= d->roi[3];
        for (int q = 0; q < 4; ++q) ok = ok && std::isfinite(d->roi[q]);
        if (!ok) return fail(FDCM_ERR_INVALID, "dense search: the region must be finite with x0 <= x1 and y0 <= y1");
    }
    return FDCM_OK;
}

// rule 1: cosine and sine of rotation r
static void dense_rotation(const fdcm_dense_params* d, int r, float* c, float* s) {
    const double th = (double)d->rot_start + (double)r * (double)d->rot_step;
    *c = (float)std::cos(th);
    *s = (float)std::sin(th);
}

// rule 2: the grid points of a W x H map with scene translation shift (nx = ny = 0: none)
struct DenseGrid { int lo_x, lo_y, nx, ny; };
static DenseGrid dense_grid(const fdcm_dense_params* d, const float shift[2], int W, int H) {
    double lo[2] = {0.0, 0.0}, hi[2] = {(double)W - 1.0, (double)H - 1.0};
    if (d->roi_on)
        for (int a = 0; a < 2; ++a) {
            lo[a] = std::max(lo[a], std::ceil((double)d->roi[a] + (double)shift[a]));
            hi[a] = std::min(hi[a], std::floor((double)d->roi[a + 2] + (double)shift[a]));
        }
    if (lo[0] > hi[0] || lo[1] > hi[1]) return DenseGrid{0, 0, 0, 0};
    const int lx = (int)lo[0], ly = (int)lo[1];
    return DenseGrid{lx, ly, ((int)hi[0] - lx) / d->stride + 1, ((int)hi[1] - ly) / d->stride + 1};
}

extern "C" fdcm_status fdcm_search_dense(const fdcm_dt3* m, const fdcm_templates* tc, const fdcm_dense_params* dense, int32_t penalty_kind,
                                         float penalty_tau, int32_t top_k, int32_t tmpl_idx_base, const fdcm_select_params* sel,
                                         const fdcm_refine_params* ref, fdcm_match* out, int64_t capacity, int64_t* n_out) {
    if (!m || !tc || !n_out) return fail(FDCM_ERR_INVALID, "null argument");
    *n_out = 0;
    if (fdcm_status st = check_dense(dense)) return st;
    if (penalty_kind < 0 || penalty_kind > 2) return fail(FDCM_ERR_INVALID, "bad penalty kind");
    if (top_k < 1) return fail(FDCM_ERR_INVALID, "dense search: top_k must be >= 1");
    if (sel)
        if (fdcm_status st = check_select(sel, top_k, false)) return st;
    if (sel && sel->max_per_template == 0 && !(sel->radius > 0.f)) sel = nullptr;   // the plain top-K
    if (ref) {
        if (fdcm_status st = check_refine(ref)) return st;
        if (top_k > kRefineMaxMatches) return fail(FDCM_ERR_INVALID, "pose refinement: top_k must be in 1.." + std::to_string(kRefineMaxMatches));
    }
    if (tc->device != m->device) return fail(FDCM_ERR_INVALID, "templates and feature map live on different devices");
    if (m->stage != 0) return fail(FDCM_ERR_INVALID, "feature map was built with a debug stage");
    fdcm_templates* t = const_cast<fdcm_templates*>(tc);
    if (t->n_tmpl == 0 || m->dm.D == 0 || m->dm.W == 0 || m->dm.H == 0) return FDCM_OK;
    // The records, their valid flags and the per-template offsets go to the search's buffers, so that the selection runs
    // unchanged; the hypothesis list and the counters of the last fdcm_search (s_hyp, last_n_hyp, last_stats) stay as they are.
    std::lock_guard<std::mutex> lk(m->search_mutex);
    CUDA_TRY(cudaSetDevice(m->device));
    cudaStream_t s;
    if (fdcm_status st = get_stream(m->device, &s)) return st;
    if (fdcm_status st = map_wait(m, s)) return st;
    if (fdcm_status st = templates_ready(t, s)) return st;
    int smem_optin = 0;
    if (fdcm_status st = search_smem_optin(m->device, t->max_lines, &smem_optin)) return st;
    const DenseGrid g = dense_grid(dense, m->shift, m->dm.W, m->dm.H);
    if (g.nx == 0 || g.ny == 0) return FDCM_OK;
    const int cell = std::min(dense->cell, std::max(g.nx, g.ny));   // (a larger cell holds the same points)
    const int cells_x = (g.nx + cell - 1) / cell, cells_y = (g.ny + cell - 1) / cell;
    const int64_t per_tmpl = (int64_t)dense->rotations * cells_y * cells_x;
    const int64_t limit = ((int64_t)1 << 31) - 1;
    if (per_tmpl > limit || per_tmpl * t->n_tmpl > limit)
        return fail(FDCM_ERR_INVALID, "dense search: " + std::to_string(per_tmpl) + " records per template x " + std::to_string(t->n_tmpl) +
                                          " templates; at most 2^31 - 1 records (use fewer rotations or templates, a larger cell or stride, or a region)");
    const int64_t H = per_tmpl * t->n_tmpl;

    std::vector<int64_t> hyp_off((size_t)t->n_tmpl + 1);
    for (int i = 0; i <= t->n_tmpl; ++i) hyp_off[(size_t)i] = (int64_t)i * per_tmpl;
    std::vector<float> rot(2 * (size_t)dense->rotations);
    for (int r = 0; r < dense->rotations; ++r) dense_rotation(dense, r, &rot[2 * (size_t)r], &rot[2 * (size_t)r + 1]);
    CUDA_TRY(m->s_rec.reserve((size_t)H * sizeof(fdcm_match)));
    CUDA_TRY(m->s_valid.reserve((size_t)H));
    CUDA_TRY(m->s_hyp_off.reserve(hyp_off.size() * 8));
    CUDA_TRY(m->s_dense_keys.reserve((size_t)H * 8));
    CUDA_TRY(m->s_dense_rot.reserve(rot.size() * 4));
    CUDA_TRY(cudaMemcpyAsync(m->s_dense_rot.p, rot.data(), rot.size() * 4, cudaMemcpyHostToDevice, s));
    const float* d_denom = nullptr;   // the search's denominators
    if (fdcm_status st = stage_uploads(m, t, hyp_off.data(), hyp_off.size(), penalty_kind, penalty_tau, s, &d_denom)) return st;
    DenseLaunch dl;
    dl.lines = t->lines.as<float4>();
    dl.offsets = t->offs.as<int32_t>();
    dl.anchors = t->anchors.as<float2>();
    dl.rot = m->s_dense_rot.as<float2>();
    dl.denom = d_denom;
    dl.n_tmpl = t->n_tmpl;
    dl.rotations = dense->rotations;
    dl.tmpl_idx_base = tmpl_idx_base;
    dl.lo_x = g.lo_x;
    dl.lo_y = g.lo_y;
    dl.stride = dense->stride;
    dl.nx = g.nx;
    dl.ny = g.ny;
    dl.cell = cell;
    dl.cells_x = cells_x;
    dl.cells_y = cells_y;
    // at least 32 grid rows per block where the cells allow it: the staging of the rotated template is paid once per block
    const int cell_rows = std::min(cell, g.ny);
    dl.band = std::max(1, std::min(cells_y, (32 + cell_rows - 1) / cell_rows));
    dl.n_bands = (cells_y + dl.band - 1) / dl.band;
    dl.n_rec = H;
    dl.keys = m->s_dense_keys.as<unsigned long long>();
    dl.rec = m->s_rec.as<fdcm_match>();
    dl.valid = m->s_valid.as<uint8_t>();
    CUDA_TRY(cudaMemsetAsync(dl.keys, 0xFF, (size_t)H * 8, s));
    {
        KernelScope k("dense_eval", 0.0, s);
        CUDA_TRY(launch_dense_eval(map_view(m), m->table_dev, dl, t->max_lines, smem_optin, s));
    }
    {
        KernelScope k("dense_finish", (double)H * (8 + sizeof(fdcm_match) + 1), s);
        launch_dense_finish(map_view(m), dl, s);
    }
    const int k = top_k;
    CUDA_TRY(m->s_topk_out.reserve((size_t)k * sizeof(fdcm_match)));
    CUDA_TRY(m->s_topk_n.reserve(4));
    if (sel) {
        fdcm_search_params sp{};
        sp.top_k = k;
        sp.tmpl_idx_base = tmpl_idx_base;
        if (fdcm_status st = run_select(m, t, &sp, sel, H, s)) return st;
    } else {
        const int blocks = topk_ws_blocks(H);
        CUDA_TRY(m->s_topk_score.reserve((size_t)blocks * k * 4));
        CUDA_TRY(m->s_topk_idx.reserve((size_t)blocks * k * 8));
        KernelScope ks("topk", 0.0, s, 2);   // two kernels in this scope
        launch_topk(dl.rec, dl.valid, H, k, m->s_topk_score.as<float>(), m->s_topk_idx.as<int64_t>(), blocks, m->s_topk_out.as<fdcm_match>(),
                    m->s_topk_n.as<int>(), s);
    }
    CUDA_TRY(cudaGetLastError());
    if (ref)
        if (fdcm_status st = run_refine(m, t, tmpl_idx_base, d_denom, ref, m->s_topk_out.as<fdcm_match>(), m->s_topk_n.as<int>(), k,
                                        m->s_topk_out.as<fdcm_match>(), smem_optin, s))
            return st;
    const fdcm_status result = finish_topk(m, nullptr, k, s, nullptr, out, capacity, n_out);
    prof_resolve();
    return result;
}

extern "C" fdcm_status fdcm_dense_poses(const fdcm_dense_params* dense, const float anchor[2], const float shift[2], int32_t width,
                                        int32_t height, int32_t rotation, float* out, int64_t capacity, int64_t* n_out, int32_t grid_wh[2]) {
    if (fdcm_status st = check_dense(dense)) return st;
    if (!anchor || !shift || !n_out || !grid_wh) return fail(FDCM_ERR_INVALID, "null argument");
    if (width < 0 || height < 0) return fail(FDCM_ERR_INVALID, "width and height must be >= 0");
    if (rotation < 0 || rotation >= dense->rotations) return fail(FDCM_ERR_INVALID, "rotation must be in 0..rotations - 1");
    const DenseGrid g = dense_grid(dense, shift, width, height);
    grid_wh[0] = g.nx;
    grid_wh[1] = g.ny;
    const int64_t n = (int64_t)g.nx * g.ny;
    *n_out = n;
    if (n > capacity || (n > 0 && !out)) return fail(FDCM_ERR_CAPACITY, "output buffer too small");
    float c, s;
    dense_rotation(dense, rotation, &c, &s);
    for (int v = 0; v < g.ny; ++v)
        for (int u = 0; u < g.nx; ++u)
            dense_pose(c, s, anchor[0], anchor[1], g.lo_x + u * dense->stride, g.lo_y + v * dense->stride, shift[0], shift[1],
                       out + 6 * ((size_t)v * g.nx + u));
    return FDCM_OK;
}

// fdcm_search of this rank's template shard (params->tmpl_idx_base = first global index of the shard) followed by the
// device-side exchange: every rank returns the same global top-k.  Collective: every rank of the communicator must call it.
extern "C" fdcm_status fdcm_comm_search_topk(fdcm_comm* comm, const fdcm_dt3* m, const fdcm_templates* shard, const float* scene,
                                             int32_t n_scene, const fdcm_search_params* p, fdcm_match* out, int64_t capacity,
                                             int64_t* n_out) {
    if (!comm) return fail(FDCM_ERR_INVALID, "comm is null");
    return search_impl(m, shard, scene, n_scene, p, out, capacity, n_out, comm, nullptr);
}

extern "C" fdcm_status fdcm_comm_search_select(fdcm_comm* comm, const fdcm_dt3* m, const fdcm_templates* shard, const float* scene,
                                               int32_t n_scene, const fdcm_search_params* p, const fdcm_select_params* select,
                                               fdcm_match* out, int64_t capacity, int64_t* n_out) {
    if (!comm) return fail(FDCM_ERR_INVALID, "comm is null");
    if (!select) return fail(FDCM_ERR_INVALID, "select is null");
    return search_impl(m, shard, scene, n_scene, p, out, capacity, n_out, comm, select);
}

// Scene feature map on every rank without building it everywhere: all ranks run the O(#lines) host preparation of the same
// scene, `root` runs the build kernels, the planes travel by ncclBroadcast (NVLink).  Collective.  north_star: "each rank
// builds the scene's feature map itself, or it is NCCL-broadcast over NVLink, whichever measures faster".
extern "C" fdcm_status fdcm_comm_rebuild_broadcast(fdcm_comm* comm, fdcm_dt3* m, const float* scene_xyxy, int32_t n_lines, int32_t root) {
    if (!comm || !m) return fail(FDCM_ERR_INVALID, "null argument");
    if (root < 0 || root >= comm->world) return fail(FDCM_ERR_INVALID, "bad root");
    if (n_lines < 0 || (n_lines > 0 && !scene_xyxy)) return fail(FDCM_ERR_INVALID, "bad scene");
    if (m->stage != 0) return fail(FDCM_ERR_INVALID, "feature map was built with a debug stage");
    CUDA_TRY(cudaSetDevice(m->device));
    cudaStream_t s;
    if (fdcm_status st = get_stream(m->device, &s)) return st;
    std::lock_guard<std::mutex> lk(m->search_mutex);
    fdcm_status st = map_wait(m, s);
    if (st == FDCM_OK) st = prepare_and_upload(m, scene_xyxy, n_lines, s);
    if (st == FDCM_OK && comm->rank == root) st = run_build_kernels(m, s);
    if (st == FDCM_OK && n_lines > 0) {
        const size_t bytes = (size_t)m->dm.D * m->dm.plane_elems * sizeof(float);
        ncclResult_t r = nccl_api().Broadcast(m->planes.p, m->planes.p, bytes, ncclChar, root, comm->comm, s);
        if (r != ncclSuccess) st = fail(FDCM_ERR_CUDA, std::string("ncclBroadcast: ") + nccl_api().GetErrorString(r));
    }
    if (st == FDCM_OK) st = upload_build_scene(m, scene_xyxy, n_lines, s);
    if (st == FDCM_OK) st = map_written(m, s);
    if (st == FDCM_OK && cudaStreamSynchronize(s) != cudaSuccess) st = fail(FDCM_ERR_CUDA, "rebuild_broadcast: stream failed");
    prof_resolve();
    if (st != FDCM_OK) {
        const std::string msg = g_last_error;
        invalidate_map(m);
        g_last_error = msg;
    }
    return st;
}


// =============================================================================================
// multi-scene batches (BASELINE config 5; SURVEY 8(f3)): per scene a map build + a search of one resident template set
// + fused penalty + top-k.  Two maps alternate: the build of scene s+1 is queued on a second stream before the host
// blocks in the search of scene s, so the latency-bound build kernels run under the gather-bound search kernel.
// =============================================================================================
struct fdcm_scene_batch {
    int device = 0;
    fdcm_dt3_params params{};
    fdcm_dt3* maps[2] = {nullptr, nullptr};
    cudaStream_t build_stream = nullptr;
    ~fdcm_scene_batch() {
        cudaSetDevice(device);
        for (int i = 0; i < 2; ++i)
            if (maps[i]) fdcm_dt3_release(maps[i]);
        if (build_stream) cudaStreamDestroy(build_stream);
    }
};

extern "C" fdcm_status fdcm_scene_batch_create(const fdcm_dt3_params* params, int32_t device, fdcm_scene_batch** out) {
    if (!out) return fail(FDCM_ERR_INVALID, "out is null");
    *out = nullptr;
    if (fdcm_status st = validate_params(params)) return st;
    CUDA_TRY(cudaSetDevice(device));
    fdcm_scene_batch* b = new (std::nothrow) fdcm_scene_batch();
    if (!b) return fail(FDCM_ERR_NOMEM, "host allocation failed");
    b->device = device;
    b->params = *params;
    cudaError_t e = cudaStreamCreateWithFlags(&b->build_stream, cudaStreamNonBlocking);
    for (int i = 0; i < 2 && e == cudaSuccess; ++i) {
        b->maps[i] = new (std::nothrow) fdcm_dt3();
        if (!b->maps[i]) { delete b; return fail(FDCM_ERR_NOMEM, "host allocation failed"); }
        b->maps[i]->params = *params;
        b->maps[i]->device = device;
        b->maps[i]->stage = 0;
    }
    if (e != cudaSuccess) {
        delete b;
        return fail(FDCM_ERR_CUDA, std::string("scene_batch_create: ") + cudaGetErrorString(e));
    }
    *out = b;
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_scene_batch_destroy(fdcm_scene_batch* b) {
    delete b;
    return FDCM_OK;
}

// queue the whole build of one scene on the batch's build stream
static fdcm_status batch_queue_build(fdcm_scene_batch* b, int slot, const float* scene, int32_t n_lines) {
    fdcm_dt3* m = b->maps[slot];
    std::lock_guard<std::mutex> lk(m->search_mutex);
    fdcm_status st = map_wait(m, b->build_stream);
    if (st == FDCM_OK) st = prepare_and_upload(m, scene, n_lines, b->build_stream);
    if (st == FDCM_OK) st = run_build_kernels(m, b->build_stream);
    if (st == FDCM_OK) st = upload_build_scene(m, scene, n_lines, b->build_stream);
    if (st == FDCM_OK) st = map_written(m, b->build_stream);
    if (st != FDCM_OK) {
        const std::string msg = g_last_error;
        cudaStreamSynchronize(b->build_stream);
        invalidate_map(m);
        g_last_error = msg;
        return st;
    }
    return FDCM_OK;
}

static fdcm_status search_scenes_impl(fdcm_scene_batch* b, const float* scene_lines, const int32_t* scene_offsets, int32_t n_scenes,
                                      const fdcm_templates* templates, const fdcm_search_params* p, const fdcm_select_params* sel,
                                      fdcm_match* out, int32_t* n_out) {
    if (!b || !p || n_scenes < 0) return fail(FDCM_ERR_INVALID, "bad argument");
    if (n_scenes == 0) return FDCM_OK;
    if (!scene_offsets || !templates || !out || !n_out) return fail(FDCM_ERR_INVALID, "null argument");
    if (p->top_k <= 0) return fail(FDCM_ERR_INVALID, "fdcm_search_scenes needs top_k > 0 (fixed-size result per scene)");
    for (int s = 0; s < n_scenes; ++s)
        if (scene_offsets[s + 1] < scene_offsets[s]) return fail(FDCM_ERR_INVALID, "scene offsets must be non-decreasing");
    if (scene_offsets[n_scenes] > 0 && !scene_lines) return fail(FDCM_ERR_INVALID, "scene_lines is null");
    CUDA_TRY(cudaSetDevice(b->device));
    auto scene_ptr = [&](int s) { return scene_lines + 4 * (size_t)scene_offsets[s]; };
    auto scene_n = [&](int s) { return scene_offsets[s + 1] - scene_offsets[s]; };
    // the build stream must not overtake a search still running on the map it is about to overwrite: searches are
    // host-synchronous, so every earlier search has completed when its slot comes round again
    if (fdcm_status st = batch_queue_build(b, 0, scene_ptr(0), scene_n(0))) return st;
    for (int s = 0; s < n_scenes; ++s) {
        const int slot = s & 1;
        if (s + 1 < n_scenes)
            if (fdcm_status st = batch_queue_build(b, slot ^ 1, scene_ptr(s + 1), scene_n(s + 1))) return st;
        int64_t n = 0;   // (the search waits for the slot's build: map_wait)
        fdcm_search_params ps = *p;
        const fdcm_status st = search_impl(b->maps[slot], templates, nullptr, FDCM_SCENE_RESIDENT, &ps, out + (size_t)s * p->top_k, p->top_k, &n, nullptr,
                                           sel);
        if (st != FDCM_OK) return st;
        n_out[s] = (int32_t)n;
    }
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_search_scenes(fdcm_scene_batch* b, const float* scene_lines, const int32_t* scene_offsets, int32_t n_scenes,
                                          const fdcm_templates* templates, const fdcm_search_params* p, fdcm_match* out, int32_t* n_out) {
    return search_scenes_impl(b, scene_lines, scene_offsets, n_scenes, templates, p, nullptr, out, n_out);
}

extern "C" fdcm_status fdcm_search_scenes_select(fdcm_scene_batch* b, const float* scene_lines, const int32_t* scene_offsets, int32_t n_scenes,
                                                 const fdcm_templates* templates, const fdcm_search_params* p, const fdcm_select_params* select,
                                                 fdcm_match* out, int32_t* n_out) {
    if (!select) return fail(FDCM_ERR_INVALID, "select is null");
    if (p)
        if (fdcm_status st = check_select(select, p->top_k, false)) return st;
    return search_scenes_impl(b, scene_lines, scene_offsets, n_scenes, templates, p, select, out, n_out);
}

// optimize(optimizer, templates, alignments, featuremap) (matching/optimizestrategy.h:62-64;
// batchoptimize.cpp:6-123 / defaultoptimize.cpp:6-93): the templates are taken as given (already aligned).
extern "C" fdcm_status fdcm_optimize(const fdcm_dt3* m, const float* tmpl_lines, const int32_t* tmpl_offsets, int32_t n_tmpl,
                                     const float* alignments, int32_t batch_size, uint8_t* has_value, float* scores,
                                     float* translations) {
    if (!m || n_tmpl < 0 || batch_size < 0) return fail(FDCM_ERR_INVALID, "bad argument");
    if (n_tmpl == 0) return FDCM_OK;
    if (!tmpl_offsets || !alignments || !has_value || !scores || !translations) return fail(FDCM_ERR_INVALID, "null argument");
    if (m->dm.D == 0) return fail(FDCM_ERR_INVALID, "optimize on an empty feature map");
    if (m->stage != 0) return fail(FDCM_ERR_INVALID, "feature map was built with a debug stage");
    const int64_t n_lines = tmpl_offsets[n_tmpl];
    if (n_lines > 0 && !tmpl_lines) return fail(FDCM_ERR_INVALID, "tmpl_lines is null");
    CUDA_TRY(cudaSetDevice(m->device));
    cudaStream_t s;
    if (fdcm_status st = get_stream(m->device, &s)) return st;
    std::lock_guard<std::mutex> lk(m->search_mutex);
    if (fdcm_status st = map_wait(m, s)) return st;
    int max_lines = 1;
    for (int t = 0; t < n_tmpl; ++t) max_lines = std::max(max_lines, tmpl_offsets[t + 1] - tmpl_offsets[t]);
    int smem_optin = 0;
    if (fdcm_status st = search_smem_optin(m->device, max_lines, &smem_optin)) return st;
    DevBuf dl, doff, dal, drec, dval, dcnt;
    auto cleanup = [&]() { for (DevBuf* b : {&dl, &doff, &dal, &drec, &dval, &dcnt}) b->release(); };
    std::vector<fdcm_match> rec((size_t)n_tmpl);
    cudaError_t e = dl.reserve(std::max<size_t>(16, (size_t)n_lines * 16));
    if (e == cudaSuccess) e = doff.reserve((size_t)(n_tmpl + 1) * 4);
    if (e == cudaSuccess) e = dal.reserve((size_t)n_tmpl * 8);
    if (e == cudaSuccess) e = drec.reserve((size_t)n_tmpl * sizeof(fdcm_match));
    if (e == cudaSuccess) e = dval.reserve((size_t)n_tmpl);
    if (e == cudaSuccess) e = dcnt.reserve(3 * 8);
    if (e == cudaSuccess && n_lines) e = cudaMemcpyAsync(dl.p, tmpl_lines, (size_t)n_lines * 16, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(doff.p, tmpl_offsets, (size_t)(n_tmpl + 1) * 4, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dal.p, alignments, (size_t)n_tmpl * 8, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemsetAsync(dcnt.p, 0, 3 * 8, s);
    if (e == cudaSuccess) {
        TemplatesView tv{};
        tv.lines = dl.as<float4>();
        tv.offsets = doff.as<int32_t>();
        tv.n_tmpl = n_tmpl;
        tv.max_lines = max_lines;
        SceneView sv{};
        SearchLaunch sl{};
        sl.batch = batch_size > 0 ? batch_size : 1;
        sl.n_hyp = n_tmpl;
        sl.perm = nullptr;
        sl.direct_align = dal.as<float2>();
        SearchOutputs so{};
        so.rec = drec.as<fdcm_match>();
        so.valid = dval.as<uint8_t>();
        so.counters = dcnt.as<unsigned long long>();
        KernelScope k("optimize", 0.0, s);
        e = launch_search(map_view(m), m->table_dev, tv, sv, sl, so, smem_optin, s);
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(rec.data(), drec.p, (size_t)n_tmpl * sizeof(fdcm_match), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(has_value, dval.p, (size_t)n_tmpl, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    prof_resolve();
    cleanup();
    if (e != cudaSuccess) return fail(FDCM_ERR_CUDA, std::string("optimize: ") + cudaGetErrorString(e));
    for (int t = 0; t < n_tmpl; ++t) {
        if (has_value[t]) {
            scores[t] = rec[(size_t)t].score;
            translations[2 * t] = rec[(size_t)t].transform[2];       // identity transform + translation
            translations[2 * t + 1] = rec[(size_t)t].transform[5];
        } else {
            scores[t] = 0.f;
            translations[2 * t] = translations[2 * t + 1] = 0.f;
        }
    }
    return FDCM_OK;
}

static fdcm_status search_host_impl(const fdcm_dt3* m, const float* tmpl_lines, const int32_t* tmpl_offsets, int32_t n_tmpl,
                                    const float* scene, int32_t n_scene, const fdcm_search_params* p, fdcm_match* out,
                                    int64_t capacity, int64_t* n_out, fdcm_comm* comm) {
    if (!m || !n_out) return fail(FDCM_ERR_INVALID, "null argument");
    *n_out = 0;
    if (n_tmpl < 0) return fail(FDCM_ERR_INVALID, "bad template count");
    if (n_tmpl == 0 && !comm) return FDCM_OK;
    CUDA_TRY(cudaSetDevice(m->device));
    cudaStream_t s;
    if (fdcm_status st = get_stream(m->device, &s)) return st;
    std::lock_guard<std::mutex> lk(m->host_tset_mutex);
    if (!m->host_tset) {   // one reusable template set per map: no allocation in steady state
        m->host_tset = new (std::nothrow) fdcm_templates();
        if (!m->host_tset) return fail(FDCM_ERR_NOMEM, "host allocation failed");
        m->host_tset->device = m->device;
    }
    static const int32_t zero_off[1] = {0};
    // (this template set lives for this one search: only the ranks DefaultSearch / ConcentricRange will read are ordered)
    if (fdcm_status st = templates_load(m->host_tset, tmpl_lines, n_tmpl ? tmpl_offsets : zero_off, n_tmpl, s, p ? p->max_tmpl_lines : 0)) return st;
    return search_impl(m, m->host_tset, scene, n_scene, p, out, capacity, n_out, comm, nullptr);
}

extern "C" fdcm_status fdcm_search_host(const fdcm_dt3* m, const float* tmpl_lines, const int32_t* tmpl_offsets, int32_t n_tmpl,
                                        const float* scene, int32_t n_scene, const fdcm_search_params* p, fdcm_match* out,
                                        int64_t capacity, int64_t* n_out) {
    return search_host_impl(m, tmpl_lines, tmpl_offsets, n_tmpl, scene, n_scene, p, out, capacity, n_out, nullptr);
}

// fdcm_comm_search_topk taking this rank's shard as host templates (uploaded into the map's reusable template set)
extern "C" fdcm_status fdcm_comm_search_host_topk(fdcm_comm* comm, const fdcm_dt3* m, const float* tmpl_lines, const int32_t* tmpl_offsets,
                                                  int32_t n_tmpl, const float* scene, int32_t n_scene, const fdcm_search_params* p,
                                                  fdcm_match* out, int64_t capacity, int64_t* n_out) {
    if (!comm) return fail(FDCM_ERR_INVALID, "comm is null");
    return search_host_impl(m, tmpl_lines, tmpl_offsets, n_tmpl, scene, n_scene, p, out, capacity, n_out, comm);
}

extern "C" fdcm_status fdcm_search_last_hypotheses(const fdcm_dt3* m, int32_t* out, int64_t capacity, int64_t* n_out) {
    if (!m || !n_out) return fail(FDCM_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> lk(m->search_mutex);
    *n_out = m->last_n_hyp;
    if (m->last_n_hyp == 0) return FDCM_OK;
    if (capacity < m->last_n_hyp || !out) return fail(FDCM_ERR_CAPACITY, "output buffer too small");
    CUDA_TRY(cudaSetDevice(m->device));
    cudaStream_t s;
    if (fdcm_status st = get_stream(m->device, &s)) return st;
    CUDA_TRY(cudaMemcpyAsync(out, m->s_hyp.p, (size_t)m->last_n_hyp * 16, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_search_last_stats(const fdcm_dt3* m, fdcm_search_stats* stats) {
    if (!m || !stats) return fail(FDCM_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> lk(m->search_mutex);
    *stats = m->last_stats;
    return FDCM_OK;
}

// =============================================================================================
// host-side helpers mirroring the remaining concept entry points (no device work)
// =============================================================================================
extern "C" fdcm_status fdcm_default_search(const float* tmpl, int32_t L, const float* scene, int32_t M, int32_t maxT, int32_t maxS,
                                           int32_t* out_pairs, int32_t capacity, int32_t* n_out) {
    if (!n_out || L < 0 || M < 0 || maxT < 0 || maxS < 0) return fail(FDCM_ERR_INVALID, "bad argument");
    *n_out = 0;
    if (L == 0 || M == 0) return FDCM_OK;
    if (!tmpl || !scene) return fail(FDCM_ERR_INVALID, "null argument");
    std::vector<float> sl((size_t)M), tl((size_t)L);
    for (int i = 0; i < M; ++i) sl[(size_t)i] = line_length(scene + 4 * (size_t)i);
    for (int i = 0; i < L; ++i) tl[(size_t)i] = line_length(tmpl + 4 * (size_t)i);
    const std::vector<long> ss = argsort_desc(sl.data(), M), st = argsort_desc(tl.data(), L);
    std::vector<float> sorted_len((size_t)M);
    for (int i = 0; i < M; ++i) sorted_len[(size_t)i] = sl[(size_t)ss[(size_t)i]];
    int32_t n = 0;
    for (int r = 0; r < std::min(L, maxT); ++r) {
        const long ti = st[(size_t)r];
        const int64_t c = closest_in_descending(sorted_len.data(), M, tl[(size_t)ti]);
        int64_t b, e;
        centered_range(c, M, maxS, b, e);
        for (int64_t i = b; i < e; ++i) {
            if (n < capacity && out_pairs) {
                out_pairs[2 * n] = (int32_t)ti;
                out_pairs[2 * n + 1] = (int32_t)ss[(size_t)i];
            }
            ++n;
        }
    }
    *n_out = n;
    if (n > capacity) return fail(FDCM_ERR_CAPACITY, "output buffer too small");
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_concentric_search(const float* tmpl, int32_t L, const float* scene, int32_t M, int32_t maxT, int32_t maxS,
                                              float cx, float cy, float lo, float hi, int32_t* out_pairs, int32_t capacity, int32_t* n_out) {
    if (!n_out || L < 0 || M < 0) return fail(FDCM_ERR_INVALID, "bad argument");
    *n_out = 0;
    if (L == 0 || M == 0) return FDCM_OK;
    if (!tmpl || !scene) return fail(FDCM_ERR_INVALID, "null argument");
    const std::vector<int32_t> subset = filter_in_range(scene, M, SceneFilter{true, cx, cy, lo, hi});
    if (subset.empty()) return FDCM_OK;
    std::vector<float> fs;
    for (int32_t i : subset) fs.insert(fs.end(), scene + 4 * (size_t)i, scene + 4 * (size_t)i + 4);
    int32_t n = 0;
    std::vector<int32_t> pairs((size_t)std::max(1, capacity) * 2);
    fdcm_status st = fdcm_default_search(tmpl, L, fs.data(), (int32_t)subset.size(), maxT, maxS, pairs.data(), capacity, &n);
    *n_out = n;
    if (st != FDCM_OK) return st;
    for (int32_t i = 0; i < n; ++i) {
        out_pairs[2 * i] = pairs[2 * (size_t)i];
        out_pairs[2 * i + 1] = subset[(size_t)pairs[2 * (size_t)i + 1]];
    }
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_debug_sqrt_check(int32_t device, int64_t* n_mismatches, uint32_t* first_mismatch) {
    if (!n_mismatches || !first_mismatch) return fail(FDCM_ERR_INVALID, "null output");
    CUDA_TRY(cudaSetDevice(device));
    cudaStream_t s;
    if (fdcm_status st = get_stream(device, &s)) return st;
    unsigned long long bad = 0;
    uint32_t first = 0;
    CUDA_TRY(run_sqrt_check(&bad, &first, s));
    *n_mismatches = (int64_t)bad;
    *first_mismatch = first;
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_debug_dt_rows(const uint16_t* g_rows, int32_t n_rows, int32_t n, int32_t literal, int32_t device, float* out) {
    if (!g_rows || !out || n_rows <= 0 || n <= 0 || n > 4000 || (literal != 1 && literal != 2)) return fail(FDCM_ERR_INVALID, "bad argument");
    CUDA_TRY(cudaSetDevice(device));
    cudaStream_t s;
    if (fdcm_status st = get_stream(device, &s)) return st;
    MapDims dm;
    dm.D = 1; dm.H = n_rows; dm.W = n; dm.pitch = (n + 31) / 32 * 32; dm.wwords = dm.pitch / 32;
    dm.plane_elems = (size_t)dm.H * dm.pitch;
    DevBuf dg, dp, ds;
    cudaError_t e = dg.reserve(dm.plane_elems * 2);
    if (e == cudaSuccess) e = dp.reserve(dm.plane_elems * 4);
    if (e == cudaSuccess) e = ds.reserve(literal == 2 ? dt_band_spill_bytes(dm, dm.W) : dm.plane_elems * 8);
    // same stream as the kernel: legacy-stream copies do not order against a non-blocking stream
    if (e == cudaSuccess) e = cudaMemsetAsync(dg.p, 0xFF, dm.plane_elems * 2, s);
    if (e == cudaSuccess) e = cudaMemcpy2DAsync(dg.p, (size_t)dm.pitch * 2, g_rows, (size_t)n * 2, (size_t)n * 2, n_rows, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) {
        KernelScope k(literal == 2 ? "dt_row_band" : "dt_row_literal", 0.0, s);
        if (literal == 2) {
            launch_dt_row_envelope(nullptr, dg.as<uint16_t>(), dm, ds.p, 0, dm.W - 1, 0, dm.H - 1, 0, s);
            launch_dt_row_fill(dp.as<float>(), dm, ds.p, 0, dm.W - 1, s);
        } else {
            launch_dt_pass_literal(2, true, dg.as<uint16_t>(), dp.as<float>(), dm, ds.p, s);
        }
    }
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpy2DAsync(out, (size_t)n * 4, dp.p, (size_t)dm.pitch * 4, (size_t)n * 4, n_rows, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    prof_resolve();
    dg.release(); dp.release(); ds.release();
    if (e != cudaSuccess) return fail(FDCM_ERR_CUDA, std::string("debug_dt_rows: ") + cudaGetErrorString(e));
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_orientation_bins(int32_t depth, const float* lines, int32_t n, int32_t* bins_atanf, int32_t* bins_table) {
    if (depth < 1 || depth > kMaxDepth || n < 0 || (n > 0 && !lines)) return fail(FDCM_ERR_INVALID, "bad argument");
    const std::vector<float> keys = angle_keys(depth);
    const SlopeTable table = build_slope_table(keys.data(), (int)keys.size());
    for (int i = 0; i < n; ++i) {
        const float* l = lines + 4 * (size_t)i;
        const float slope = (l[3] - l[1]) / (l[2] - l[0]);
        if (bins_atanf) bins_atanf[i] = bin_of_slope(keys.data(), (int)keys.size(), slope);
        if (bins_table) bins_table[i] = slope_table_lookup(table, slope);
    }
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_penalize(int32_t kind, float tau, fdcm_match* matches, int64_t n, const float* lengths, int64_t n_lengths) {
    if (n < 0 || (n > 0 && !matches)) return fail(FDCM_ERR_INVALID, "bad matches");
    if (kind != FDCM_PENALTY_DEFAULT && kind != FDCM_PENALTY_EXPONENTIAL) return fail(FDCM_ERR_INVALID, "unknown penalty");
    for (int64_t i = 0; i < n; ++i)
        if ((uint64_t)(uint32_t)matches[i].tmpl_idx >= (uint64_t)n_lengths || matches[i].tmpl_idx < 0)
            return fail(FDCM_ERR_OUT_OF_RANGE,
                        "In penalize, the size of templatelengths is not consistent with match template indices");
    for (int64_t i = 0; i < n; ++i) matches[i].score = matches[i].score / penalty_denominator(kind, tau, lengths[matches[i].tmpl_idx]);
    return FDCM_OK;
}

extern "C" fdcm_status fdcm_sort_matches(fdcm_match* matches, int64_t n) {
    if (n < 0 || (n > 0 && !matches)) return fail(FDCM_ERR_INVALID, "bad matches");
    std::sort(matches, matches + n, [](const fdcm_match& a, const fdcm_match& b) { return a.score < b.score; });
    return FDCM_OK;
}
