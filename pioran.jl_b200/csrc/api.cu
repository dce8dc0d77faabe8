// api.cu — C ABI of libpioran_b200.so (include/pioran_b200.h): contexts, resident series, launch logic.
// No CPU fallback anywhere: every entry point either runs the sm_100a kernels or fails with an error code.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <new>
#include <exception>
#include <string>
#include <thread>
#include <tuple>
#include <vector>

#include "../../include/pioran_b200.h"
#include "approx.cuh"
#include "celerite.cuh"
#include "blocked.cuh"
#include "common.cuh"
#include "dense.cuh"
#include "scan.cuh"
#include "posterior.cuh"
#include "postvar.cuh"
#include "table.cuh"
#include "grad.cuh"
#include "grad_pipe.cuh"
#include "blocked_grad.cuh"
#include "blocked_wide.cuh"
#include "wide.cuh"
#include "prior.cuh"
#include "wide_grad.cuh"
#include "scan_wide.cuh"
#include "scan_blocked.cuh"
#include "jvp.cuh"
#include "vjp.cuh"

using namespace pioran;

// ------------------------------------------------------------------------------------------------ errors
static thread_local std::string g_err;
static int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

// The C ABI never lets an exception escape (include/pioran_b200.h): every extern "C" entry is a function-try-block ending here.
static int guard_fail() {
    try { throw; }
    catch (const std::bad_alloc&) { return fail(PIORAN_ENOMEM, "out of host memory"); }
    catch (const std::exception& e) { return fail(PIORAN_EINVAL, "unexpected exception: %s", e.what()); }
    catch (...) { return fail(PIORAN_EINVAL, "unexpected exception"); }
}
#define CUDA_TRY(expr)                                                                                     \
    do {                                                                                                   \
        cudaError_t e__ = (expr);                                                                          \
        if (e__ != cudaSuccess)                                                                            \
            return fail(e__ == cudaErrorMemoryAllocation ? PIORAN_ENOMEM : PIORAN_ECUDA, "%s failed: %s",  \
                        #expr, cudaGetErrorString(e__));                                                   \
    } while (0)

extern "C" const char* pioran_last_error(void) { return g_err.c_str(); }
extern "C" int pioran_version(void) { return 303; }   // 0.3.3: pioran_celerite_predict_var

// ------------------------------------------------------------------------------------------------ context
namespace {

struct DevBuf {  // grow-only device workspace
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return 0;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = std::max(bytes, (size_t)4096);
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) return fail(PIORAN_ENOMEM, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
        cap = want;
        return 0;
    }
    template <typename T> T* as() { return reinterpret_cast<T*>(p); }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

using TableKey = std::tuple<int, int, double, double>;  // basis, J, f0, fM
struct Table { double* d = nullptr; int rpad = 0; int64_t npad = 0; uint64_t last_use = 0; };
constexpr size_t MAX_TABLES_PER_SERIES = 8;   // per kind; least recently used first out (a table of N = 1e6 at rank 60 is 3.9 GB)

struct Series {
    int64_t N = 0;
    double *t = nullptr, *y = nullptr, *s2 = nullptr;
    std::map<TableKey, Table> tables;
    std::map<TableKey, Table> btables;   // block tables of the tensor-pipe kernel (blocked.cuh)
};

using PlanKey = std::tuple<int, int, int, int, double, double, double, double>;

// The most recent main-kernel launch (pioran_ctx_last_kernel_name): a kernel family and its template integers, formatted
// only when queried so that the launch path stores four ints.
enum KernelFamily : int {
    KF_NONE = 0, KF_BLOCKED, KF_BLOCKED_WIDE, KF_SHARED, KF_SHARED_PAIR, KF_GENERIC, KF_WIDE_REG, KF_WIDE_REG_STORE, KF_WIDE_REG_SIM,
    KF_WIDE, KF_BLOCKED_GRAD, KF_GRAD, KF_GRAD_PIPE, KF_WIDE_GRAD, KF_JVP, KF_PREDICT, KF_GENERIC_SIM, KF_SCAN_FINISH,
    KF_SCAN_PARTIAL, KF_DENSE_FINISH, KF_VJP, KF_POSTVAR
};
struct KernelTag { int family = KF_NONE; int p[4] = {0, 0, 0, 0}; };

}  // namespace

struct pioran_ctx {
    int device = 0;
    int num_sms = 0;
    cudaStream_t own = nullptr, stream = nullptr;
    cudaStream_t side = nullptr, hi = nullptr;   // K4: the bulk trailing updates (side) run beside the panel chain (hi: highest stream priority, so its
                                                 // small kernels take the SM slots the bulk's CTAs free); created on first use
    cudaEvent_t ev_fact = nullptr, ev_bulk = nullptr, ev_join = nullptr, ev_fill = nullptr, ev_col[8] = {};
    int64_t launches = 0;
    std::vector<Series*> series;
    std::map<PlanKey, ApproxPlan*> plans;  // device pointers
    DevBuf theta, amp, suma, out, work, coef, rows, misc, post, gradws, gwork, stab;   // stab: per-θ block table of the K3 fold
    DevBuf vjpws;   // K5r: per-step values and T checkpoints of one θ-chunk
    // device time of the most recent main-kernel launch (K2/K3/K4), for bench.py's roofline line
    cudaEvent_t ev_beg = nullptr, ev_end = nullptr;
    bool ev_valid = false;
    KernelTag last_kernel;   // which kernel that launch ran (note_kernel)
    // the work-item list of the last fused call, kept on the device while the call shape repeats (a sampler
    // evaluates the same series × batch-size shape ~1e5 times)
    std::vector<int64_t> work_key;
    int work_items = 0, work_tpi = 0;
    std::vector<int64_t> gwork_key;   // same for the gradient path's work items
    int gwork_items = 0, gwork_tpi = 0;
    int scan_chunks = 0;   // K3: chunks per parameter vector (0 = automatic)
    size_t vjp_ws_bytes = 0;   // K5r: workspace cap per θ-chunk (0 = 1 GiB; pioran_ctx_set_vjp_workspace)
    bool auto_scan = true; // route few-evaluation calls on long series to K3 (pioran_ctx_set_auto_scan)
    int sweep_kernel = PIORAN_SWEEP_AUTO;   // pioran_ctx_set_sweep_kernel
    // pioran_ctx_create_multi: a group context owns one child context per device and no CUDA state of its own; the batched
    // host-pointer entries split their parameter vectors over the children, everything else runs on children[0]
    std::vector<pioran_ctx*> children;
    std::vector<std::vector<int>> group_series;   // group series id -> series id on each child (empty = freed)
    uint64_t epoch = 0;    // bumped by every entry that uses the shared workspaces (a pending scan range checks it)
    uint64_t use_clock = 0;   // LRU stamp source of the per-series table caches
    double scan_tol = 1e-10;       // K3 self-check: tolerated deviation estimate, relative to max(1, |log L|); <= 0: no check
    double scan_floor_cap = 1e-7;  // K3: largest stalled estimate of a converged Newton iteration that is accepted as rounding floor; <= 0: never
    std::vector<std::vector<double>> scan_hist_est, scan_hist_val;   // per parameter vector of the last K3 call: estimate and value after every pass
    double scan_last_est = 0.0;    // largest relative estimate of the last K3 call
    int scan_last_fallback = 0;    // parameter vectors of the last K3 call that were re-evaluated by the sequential sweep
    int scan_last_refined = 0;     // … that were accepted after a run-up pass
    double scan_range_chk[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // pioran_celerite_scan_range_check
    std::mutex mu;
};

// Entry points that launch work or touch the context's workspaces: take the lock and invalidate a range left pending by
// pioran_celerite_scan_range_begin (its record points into those workspaces).
#define PIORAN_COMPUTE_LOCK(c) std::lock_guard<std::mutex> lk((c)->mu); (c)->epoch++
// Every main-kernel launch site: the events around it are valid, and the kernel is named for pioran_ctx_last_kernel_name.
static void note_kernel(pioran_ctx* c, int family, int p0 = 0, int p1 = 0, int p2 = 0, int p3 = 0) {
    c->ev_valid = true;
    c->last_kernel.family = family;
    c->last_kernel.p[0] = p0; c->last_kernel.p[1] = p1; c->last_kernel.p[2] = p2; c->last_kernel.p[3] = p3;
}
static int make_term_rows(int B, int Jt, const double* b, const double* d, std::vector<int>& term_row);

static int bs_for_rank(int R) {
    int bs = (R + G - 1) / G;
    if (bs < 4) bs = 4;
    return bs;
}

// A handful of evaluations of one long series is latency-bound in the sequential sweep (≈ 0.9 µs per step whatever the rank);
// from a few thousand steps on the parallel-in-time path K3 is faster (tools/scan_vs_seq.py: 2.0–2.2 vs 3.9–8.2 ms at N = 4 096, 2.5–2.9 vs 7.8–16 ms at N = 8 192,
// 5–6 vs 62–130 ms at N = 65 536), so the plain entries route such calls to it.  Same value as the sequential sweep: every
// routed call verifies itself and ill-conditioned parameter vectors are re-evaluated sequentially (scan_logl_locked).
constexpr int64_t AUTO_SCAN_MIN_STEPS = 4096;
constexpr int AUTO_SCAN_MAX_BATCH = 4;
// Thresholds from tools/scan_threshold.py (one evaluation): the fused path's sequential sweep (shared table, pre-decayed state)
// costs 0.5–0.66 µs per step and is overtaken at 2 048 (rank ≤ 32) / 4 096 steps; the explicit-coefficient sweep builds its
// own table (0.65–1.5 µs per step) and is overtaken at 1 024 / 2 048 steps.
static bool auto_scan(const pioran_ctx* c, int64_t N, int B, int R, bool explicit_coefficients = false) {
    int64_t min_steps = R <= 32 ? AUTO_SCAN_MIN_STEPS / 2 : AUTO_SCAN_MIN_STEPS;
    if (explicit_coefficients) min_steps /= 2;
    // from 4 column tiles on, one evaluation runs as a CTA of four warps on the tensor pipe (blocked_wide.cuh) at 0.18–0.23 µs per
    // step, and the scan's fixed cost (Kogge–Stone levels) is overtaken later: tools/scan_threshold.py, round 2
    if (R >= 25 && R <= 63 && c->sweep_kernel != PIORAN_SWEEP_SCALAR) min_steps = R <= 32 ? 4096 : 8192;
    // wide ranks: the one-CTA blocked sweep runs 0.49 µs per step, the wide scan costs ≈ 9.7 ms + 0.02 µs per step (profiles/r02_reference_suite_mirror.jsonl)
    if (R > SCAN_LD) return c->auto_scan && N >= (c->sweep_kernel == PIORAN_SWEEP_SCALAR ? 4096 : 20480) && B <= AUTO_SCAN_MAX_BATCH && R <= SRW;
    return c->auto_scan && N >= min_steps && B <= AUTO_SCAN_MAX_BATCH && R <= SCAN_LD;
}
static int scan_logl_locked(pioran_ctx* c, Series* s, int series_id, int B, int Jt, const double* a, const double* b,
                            const double* cc, const double* d, const double* mu, const double* nu, double* logl_out);

static void scan_forget(pioran_ctx* c);   // drops the range-in-progress record of a context (K3 multi-GPU entries)
extern "C" int pioran_ctx_destroy(pioran_ctx* c);
extern "C" int pioran_ctx_create(int device, pioran_ctx** out) try {
    if (!out) return fail(PIORAN_EINVAL, "out is NULL");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(PIORAN_ECUDA, "no CUDA device available (%s); this backend has no CPU fallback",
                    e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return fail(PIORAN_EINVAL, "device %d out of range [0,%d)", device, ndev);
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(PIORAN_ECUDA, "device %d is sm_%d%d; libpioran_b200 carries sm_100a code only", device, prop.major,
                    prop.minor);
    CUDA_TRY(cudaSetDevice(device));
    pioran_ctx* c = new (std::nothrow) pioran_ctx();
    if (!c) return fail(PIORAN_ENOMEM, "out of host memory");
    c->device = device;
    c->num_sms = prop.multiProcessorCount;
    e = cudaStreamCreateWithFlags(&c->own, cudaStreamNonBlocking);
    if (e != cudaSuccess) { delete c; return fail(PIORAN_ECUDA, "cudaStreamCreate failed: %s", cudaGetErrorString(e)); }
    c->stream = c->own;
    if (cudaEventCreate(&c->ev_beg) != cudaSuccess || cudaEventCreate(&c->ev_end) != cudaSuccess) {
        pioran_ctx_destroy(c);
        return fail(PIORAN_ECUDA, "cudaEventCreate failed");
    }
    *out = c;
    return PIORAN_OK;
} catch (...) { return guard_fail(); }


// ------------------------------------------------------------------------------------------------ device groups
// Single-process multi-GPU (SURVEY 8b/8e; reference examples/ultranest/single_pl.jl:113-117 runs ONE process and one
// callback): the parameter batch is cut into contiguous slices, one per device; each slice goes through the ordinary
// single-device entry on its own host thread (cudaSetDevice is per thread) and writes straight into the caller's output
// rows.  No data-path collective: the slices are independent, and host pointers need no all-gather.
static bool is_group(const pioran_ctx* c) { return c && !c->children.empty(); }
static int group_series_id(pioran_ctx* g, int gid, size_t child, int* out) {
    if (gid < 0 || gid >= (int)g->group_series.size() || g->group_series[gid].empty())
        return fail(PIORAN_EINVAL, "unknown series id %d", gid);
    *out = g->group_series[gid][child];
    return 0;
}
// Runs fn(child index, first row, row count) for every non-empty slice of B rows, one thread per slice.
template <typename F>
static int group_split(pioran_ctx* g, int B, F fn) {
    const int nd = (int)g->children.size();
    std::vector<int> rcs(nd, 0);
    std::vector<std::string> errs(nd);
    std::vector<std::thread> th;
    for (int k = 0; k < nd; k++) {
        const int beg = (int)((long long)B * k / nd), end = (int)((long long)B * (k + 1) / nd);
        if (end <= beg) continue;
        th.emplace_back([&, k, beg, end] {
            rcs[k] = fn(k, beg, end - beg);
            if (rcs[k]) errs[k] = pioran_last_error();     // the message is thread-local: carry it back
        });
    }
    for (auto& t : th) t.join();
    for (int k = 0; k < nd; k++)
        if (rcs[k]) return fail(rcs[k], "device %d: %s", g->children[k]->device, errs[k].c_str());
    return 0;
}
// The batched host-pointer entries of a group: the S series ids are resolved on every child under the group lock, then
// fn(child, the child's S ids, N, first row, row count) runs for every slice of B rows.  N is the length of the first series,
// for slicing per-row data of N steps.
template <typename F>
static int group_fanout(pioran_ctx* g, int S, const int* series_ids, int B, F fn) {
    std::vector<int> cid(g->children.size() * S);
    {
        std::lock_guard<std::mutex> lk(g->mu);
        for (size_t k = 0; k < g->children.size(); k++)
            for (int q = 0; q < S; q++) { const int rc = group_series_id(g, series_ids[q], k, &cid[k * S + q]); if (rc) return rc; }
    }
    int64_t N = 0;
    const int rc = pioran_series_length(g->children[0], cid[0], &N);
    if (rc) return rc;
    return group_split(g, B, [&](int k, int beg, int nb) { return fn(g->children[k], cid.data() + (size_t)k * S, N, beg, nb); });
}
template <typename F>
static int group_fanout(pioran_ctx* g, int series_id, int B, F fn) {
    return group_fanout(g, 1, &series_id, B, [&](pioran_ctx* ch, const int* cid, int64_t N, int beg, int nb) { return fn(ch, *cid, N, beg, nb); });
}
// Single-device work of a group runs on its first device: fn(children[0], the series id on it).
template <typename F>
static int group_first(pioran_ctx* g, int series_id, F fn) {
    int cid;
    { std::lock_guard<std::mutex> lk(g->mu); const int rc = group_series_id(g, series_id, 0, &cid); if (rc) return rc; }
    return fn(g->children[0], cid);
}
// Settings of a group apply to every child.
template <typename F>
static int group_each(pioran_ctx* g, F fn) {
    for (pioran_ctx* ch : g->children) { const int rc = fn(ch); if (rc) return rc; }
    return PIORAN_OK;
}
// An optional array at an offset: the slices of a group split and the θ-chunks of one call.
template <typename T>
static T* at(T* p, size_t off) { return p ? p + off : nullptr; }

extern "C" int pioran_ctx_create_multi(const int* devices, int ndev, pioran_ctx** out) try {
    if (!devices || !out) return fail(PIORAN_EINVAL, "NULL argument");
    if (ndev < 1 || ndev > 64) return fail(PIORAN_EINVAL, "ndev must be in [1, 64] (got %d)", ndev);
    for (int i = 0; i < ndev; i++)
        for (int j = 0; j < i; j++)
            if (devices[i] == devices[j]) return fail(PIORAN_EINVAL, "device %d listed twice", devices[i]);
    pioran_ctx* g = new (std::nothrow) pioran_ctx();
    if (!g) return fail(PIORAN_ENOMEM, "out of host memory");
    for (int i = 0; i < ndev; i++) {
        pioran_ctx* ch = nullptr;
        const int rc = pioran_ctx_create(devices[i], &ch);
        if (rc) {
            const std::string msg = pioran_last_error();
            for (pioran_ctx* x : g->children) pioran_ctx_destroy(x);
            delete g;
            return fail(rc, "%s", msg.c_str());
        }
        g->children.push_back(ch);
    }
    g->device = devices[0];
    g->num_sms = g->children[0]->num_sms;
    *out = g;
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

extern "C" int pioran_ctx_device_count(pioran_ctx* c) { return !c ? 0 : is_group(c) ? (int)c->children.size() : 1; }

static void free_series(Series* s) {
    if (!s) return;
    cudaFree(s->t); cudaFree(s->y); cudaFree(s->s2);
    for (auto& kv : s->tables) cudaFree(kv.second.d);
    for (auto& kv : s->btables) cudaFree(kv.second.d);
    delete s;
}

extern "C" int pioran_ctx_destroy(pioran_ctx* c) try {
    if (!c) return PIORAN_OK;
    if (is_group(c)) {
        for (pioran_ctx* ch : c->children) pioran_ctx_destroy(ch);
        delete c;
        return PIORAN_OK;
    }
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    scan_forget(c);
    for (Series* s : c->series) free_series(s);
    for (auto& kv : c->plans) cudaFree(kv.second);
    c->theta.release(); c->amp.release(); c->suma.release(); c->out.release(); c->work.release();
    c->coef.release(); c->rows.release(); c->misc.release(); c->post.release(); c->gradws.release(); c->gwork.release(); c->stab.release(); c->vjpws.release();
    if (c->ev_beg) cudaEventDestroy(c->ev_beg);
    if (c->ev_end) cudaEventDestroy(c->ev_end);
    if (c->ev_fact) cudaEventDestroy(c->ev_fact);
    if (c->ev_bulk) cudaEventDestroy(c->ev_bulk);
    if (c->ev_join) cudaEventDestroy(c->ev_join);
    if (c->ev_fill) cudaEventDestroy(c->ev_fill);
    for (cudaEvent_t e : c->ev_col) if (e) cudaEventDestroy(e);
    if (c->side) cudaStreamDestroy(c->side);
    if (c->hi) cudaStreamDestroy(c->hi);
    if (c->own) cudaStreamDestroy(c->own);
    delete c;
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

extern "C" int pioran_ctx_set_stream(pioran_ctx* c, void* s) try {
    if (!c) return fail(PIORAN_EINVAL, "ctx is NULL");
    if (is_group(c)) return fail(PIORAN_EUNSUPPORTED, "a device group has one stream per device; set streams on single-device contexts");
    std::lock_guard<std::mutex> lk(c->mu);
    cudaStream_t next = s ? reinterpret_cast<cudaStream_t>(s) : c->own;
    if (next != c->stream) {
        // the workspaces and the cached work items are ordered on the old stream only: drain it before switching
        CUDA_TRY(cudaSetDevice(c->device));
        CUDA_TRY(cudaStreamSynchronize(c->stream));
        c->stream = next;
    }
    return PIORAN_OK;
} catch (...) { return guard_fail(); }
extern "C" int pioran_ctx_synchronize(pioran_ctx* c) try {
    if (!c) return fail(PIORAN_EINVAL, "ctx is NULL");
    if (is_group(c)) return group_each(c, [](pioran_ctx* ch) { return pioran_ctx_synchronize(ch); });
    CUDA_TRY(cudaSetDevice(c->device));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return PIORAN_OK;
} catch (...) { return guard_fail(); }
extern "C" int64_t pioran_ctx_launch_count(pioran_ctx* c) {
    if (!c) return 0;
    if (is_group(c)) { int64_t n = 0; for (pioran_ctx* ch : c->children) n += pioran_ctx_launch_count(ch); return n; }
    std::lock_guard<std::mutex> lk(c->mu);
    return c->launches;
}
extern "C" int pioran_ctx_last_kernel_ms(pioran_ctx* c, double* ms) try {
    if (!c || !ms) return fail(PIORAN_EINVAL, "NULL argument");
    if (is_group(c)) {   // the slowest device bounds the call
        double worst = 0.0;
        for (pioran_ctx* ch : c->children) { double v = 0.0; if (pioran_ctx_last_kernel_ms(ch, &v) == 0 && v > worst) worst = v; }
        *ms = worst;
        return PIORAN_OK;
    }
    if (!c->ev_valid) return fail(PIORAN_EINVAL, "no main kernel has been launched on this context yet");
    CUDA_TRY(cudaSetDevice(c->device));
    CUDA_TRY(cudaEventSynchronize(c->ev_end));
    float f = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&f, c->ev_beg, c->ev_end));
    *ms = (double)f;
    return PIORAN_OK;
} catch (...) { return guard_fail(); }
extern "C" int pioran_ctx_last_kernel_name(pioran_ctx* c, char* buf, int len) try {
    if (!c || !buf) return fail(PIORAN_EINVAL, "NULL argument");
    if (is_group(c)) return fail(PIORAN_EUNSUPPORTED, "a device group launches on several devices; ask a single-device context");
    KernelTag k;
    { std::lock_guard<std::mutex> lk(c->mu); k = c->last_kernel; }
    const int* p = k.p;
    char name[64];
    switch (k.family) {
        case KF_BLOCKED: snprintf(name, sizeof name, "blocked<%d,%d,%s,%d>", p[0], p[1], p[2] ? "true" : "false", p[3]); break;
        case KF_BLOCKED_WIDE: snprintf(name, sizeof name, "blocked_wide<%d,%d,%d>", p[0], p[1], p[2]); break;
        case KF_SHARED: snprintf(name, sizeof name, "shared<%d,%d>", p[0], p[1]); break;
        case KF_SHARED_PAIR: snprintf(name, sizeof name, "shared_pair<%d,%d>", p[0], p[1]); break;
        case KF_GENERIC: snprintf(name, sizeof name, "generic<%d,%d>", p[0], p[1]); break;
        case KF_WIDE_REG: snprintf(name, sizeof name, "wide_reg<%d>", p[0]); break;
        case KF_WIDE_REG_STORE: snprintf(name, sizeof name, "wide_reg_store<%d>", p[0]); break;
        case KF_WIDE_REG_SIM: snprintf(name, sizeof name, "wide_reg_sim<%d>", p[0]); break;
        case KF_WIDE: snprintf(name, sizeof name, "wide"); break;
        case KF_BLOCKED_GRAD: snprintf(name, sizeof name, "blocked_grad<%d,%d,%s,%d>", p[0], p[1], p[2] ? "true" : "false", p[3]); break;
        case KF_GRAD: snprintf(name, sizeof name, "grad<%d,%d>", p[0], p[1]); break;
        case KF_GRAD_PIPE: snprintf(name, sizeof name, "grad_pipe<%d,%d>", p[0], p[1]); break;
        case KF_WIDE_GRAD: snprintf(name, sizeof name, "wide_grad<%d>", p[0]); break;
        case KF_JVP: snprintf(name, sizeof name, "jvp<%d>", p[0]); break;
        case KF_VJP: snprintf(name, sizeof name, "vjp<%d>", p[0]); break;
        case KF_PREDICT: snprintf(name, sizeof name, "predict<%d>", p[0]); break;
        case KF_POSTVAR: snprintf(name, sizeof name, "postvar<%d>", p[0]); break;
        case KF_GENERIC_SIM: snprintf(name, sizeof name, "generic_sim<%d,%d>", p[0], p[1]); break;
        case KF_SCAN_FINISH: snprintf(name, sizeof name, "scan_finish"); break;
        case KF_SCAN_PARTIAL: snprintf(name, sizeof name, "scan_partial"); break;
        case KF_DENSE_FINISH: snprintf(name, sizeof name, "dense_finish"); break;
        default: name[0] = '\0'; break;
    }
    const int need = (int)strlen(name) + 1;
    if (len < need) return fail(PIORAN_EINVAL, "buffer of %d bytes is too small for the %d-byte kernel name", len, need);
    memcpy(buf, name, need);
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

extern "C" int pioran_series_upload(pioran_ctx* c, int64_t N, const double* t, const double* y, const double* s2,
                                    int* series_id) try {
    if (!c || !t || !y || !s2 || !series_id) return fail(PIORAN_EINVAL, "NULL argument");
    if (N < 1) return fail(PIORAN_EINVAL, "N must be >= 1 (got %lld)", (long long)N);
    if (is_group(c)) {
        std::vector<int> ids(c->children.size(), -1);
        for (size_t k = 0; k < c->children.size(); k++) {
            const int rc = pioran_series_upload(c->children[k], N, t, y, s2, &ids[k]);
            if (rc) { for (size_t q = 0; q < k; q++) pioran_series_free(c->children[q], ids[q]); return rc; }
        }
        std::lock_guard<std::mutex> lk(c->mu);
        int gid = -1;
        for (size_t k = 0; k < c->group_series.size(); k++)
            if (c->group_series[k].empty()) { gid = (int)k; break; }
        if (gid < 0) { c->group_series.emplace_back(); gid = (int)c->group_series.size() - 1; }
        c->group_series[gid] = ids;
        *series_id = gid;
        return PIORAN_OK;
    }
    for (int64_t n = 1; n < N; n++)
        if (!(t[n] > t[n - 1])) return fail(PIORAN_EINVAL, "t must be strictly increasing (t[%lld] <= t[%lld])", (long long)n, (long long)(n - 1));
    std::lock_guard<std::mutex> lk(c->mu);
    CUDA_TRY(cudaSetDevice(c->device));
    Series* s = new (std::nothrow) Series();
    if (!s) return fail(PIORAN_ENOMEM, "out of host memory");
    s->N = N;
    const size_t bytes = sizeof(double) * (size_t)N;
    if (cudaMalloc(&s->t, bytes) != cudaSuccess || cudaMalloc(&s->y, bytes) != cudaSuccess ||
        cudaMalloc(&s->s2, bytes) != cudaSuccess) {
        free_series(s);
        return fail(PIORAN_ENOMEM, "cudaMalloc of a %lld-point series failed", (long long)N);
    }
    cudaMemcpyAsync(s->t, t, bytes, cudaMemcpyHostToDevice, c->stream);
    cudaMemcpyAsync(s->y, y, bytes, cudaMemcpyHostToDevice, c->stream);
    cudaMemcpyAsync(s->s2, s2, bytes, cudaMemcpyHostToDevice, c->stream);
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) { free_series(s); return fail(PIORAN_ECUDA, "series upload failed: %s", cudaGetErrorString(e)); }
    int id = -1;
    for (size_t k = 0; k < c->series.size(); k++)
        if (!c->series[k]) { id = (int)k; break; }
    if (id < 0) { c->series.push_back(nullptr); id = (int)c->series.size() - 1; }
    c->series[id] = s;
    *series_id = id;
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

static Series* get_series(pioran_ctx* c, int id) {
    if (id < 0 || id >= (int)c->series.size()) return nullptr;
    return c->series[id];
}

extern "C" int pioran_series_free(pioran_ctx* c, int id) try {
    if (!c) return fail(PIORAN_EINVAL, "ctx is NULL");
    if (is_group(c)) {
        std::lock_guard<std::mutex> lk(c->mu);
        if (id < 0 || id >= (int)c->group_series.size() || c->group_series[id].empty()) return fail(PIORAN_EINVAL, "unknown series id %d", id);
        for (size_t k = 0; k < c->children.size(); k++) pioran_series_free(c->children[k], c->group_series[id][k]);
        c->group_series[id].clear();
        return PIORAN_OK;
    }
    PIORAN_COMPUTE_LOCK(c);
    Series* s = get_series(c, id);
    if (!s) return fail(PIORAN_EINVAL, "unknown series id %d", id);
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    free_series(s);
    c->series[id] = nullptr;
    c->work_key.clear();    // cached work items hold the freed series' device pointers
    c->gwork_key.clear();
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

extern "C" int pioran_series_length(pioran_ctx* c, int id, int64_t* N) try {
    if (!c || !N) return fail(PIORAN_EINVAL, "NULL argument");
    if (is_group(c)) return group_first(c, id, [&](pioran_ctx* ch, int cid) { return pioran_series_length(ch, cid, N); });
    std::lock_guard<std::mutex> lk(c->mu);
    Series* s = get_series(c, id);
    if (!s) return fail(PIORAN_EINVAL, "unknown series id %d", id);
    *N = s->N;
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

// ------------------------------------------------------------------------------------------------ approx plan
static int n_psd_par_of(int model) { return model == PIORAN_PSD_SBPL ? 3 : model == PIORAN_PSD_DBPL ? 5 : -1; }

static int check_spec(const pioran_approx_spec& sp) {
    if (n_psd_par_of(sp.psd_model) < 0) return fail(PIORAN_EINVAL, "unknown psd_model %d", sp.psd_model);
    if (sp.basis != PIORAN_BASIS_SHO && sp.basis != PIORAN_BASIS_DRWCELERITE)
        return fail(PIORAN_EINVAL, "unknown basis %d (src/psd.jl:285 errors likewise)", sp.basis);
    if (sp.n_components < 2 || sp.n_components > MAXJ)
        return fail(PIORAN_EINVAL, "n_components must be in [2,%d] (got %d)", MAXJ, sp.n_components);
    if (!(sp.f_min > 0) || !(sp.f_max > sp.f_min) || !(sp.S_low > 0) || !(sp.S_high > 0))
        return fail(PIORAN_EINVAL, "need 0 < f_min < f_max and positive S_low, S_high");
    return 0;
}

// Builds (or fetches) the device plan: grid (src/psd.jl:81-83), spectral matrix (:86-97), LU with partial pivoting.
static int get_plan(pioran_ctx* c, const pioran_approx_spec& sp, ApproxPlan** out) {
    PlanKey key{sp.psd_model, sp.n_components, sp.basis, sp.is_integrated_power, sp.f_min, sp.f_max, sp.S_low, sp.S_high};
    auto it = c->plans.find(key);
    if (it != c->plans.end()) { *out = it->second; return 0; }
    static thread_local ApproxPlan hp;
    std::memset(&hp, 0, sizeof hp);
    const int J = sp.n_components;
    const double f0 = sp.f_min / sp.S_low, fM = sp.f_max * sp.S_high;
    for (int j = 0; j < J; j++) hp.fj[j] = f0 * std::pow(fM / f0, (double)j / (double)(J - 1));
    double* A = hp.lu;
    for (int j = 0; j < J; j++)
        for (int k = 0; k < J; k++) {
            const double r = hp.fj[j] / hp.fj[k], r2 = r * r;
            A[j + k * J] = 1.0 / (1.0 + (sp.basis == PIORAN_BASIS_SHO ? r2 * r2 : r2 * r2 * r2));
        }
    for (int k = 0; k < J; k++) {  // right-looking LU, partial pivoting
        int p = k;
        double best = std::fabs(A[k + k * J]);
        for (int r = k + 1; r < J; r++)
            if (std::fabs(A[r + k * J]) > best) { best = std::fabs(A[r + k * J]); p = r; }
        if (best == 0.0) return fail(PIORAN_ESINGULAR, "spectral matrix is singular at column %d", k);
        hp.piv[k] = p;
        if (p != k)
            for (int col = 0; col < J; col++) std::swap(A[k + col * J], A[p + col * J]);
        const double inv = 1.0 / A[k + k * J];
        for (int r = k + 1; r < J; r++) A[r + k * J] *= inv;
        for (int col = k + 1; col < J; col++) {
            const double akc = A[k + col * J];
            for (int r = k + 1; r < J; r++) A[r + col * J] -= A[r + k * J] * akc;
        }
    }
    hp.J = J; hp.basis = sp.basis; hp.model = sp.psd_model; hp.n_psd_par = n_psd_par_of(sp.psd_model);
    hp.is_integrated_power = sp.is_integrated_power ? 1 : 0;
    hp.f_min = sp.f_min; hp.f_max = sp.f_max;
    ApproxPlan* dp = nullptr;
    CUDA_TRY(cudaMalloc(&dp, sizeof(ApproxPlan)));
    cudaError_t e = cudaMemcpyAsync(dp, &hp, sizeof(ApproxPlan), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);  // hp is reused by the next call
    if (e != cudaSuccess) { cudaFree(dp); return fail(PIORAN_ECUDA, "plan upload failed: %s", cudaGetErrorString(e)); }
    c->plans[key] = dp;
    *out = dp;
    return 0;
}

static int rank_of(int basis, int J) { return basis == PIORAN_BASIS_SHO ? 2 * J : 3 * J; }

// Row descriptors of the shared table for a spec (rows: cos/sin pairs of the J complex terms, then — DRWCelerite
// only — the J real terms).  Coefficient formulas: src/psd.jl:250 (c = d = √2 π f) and :266-271 (c = π f, d = √3 c; 2c).
static void make_rows(const pioran_approx_spec& sp, int RP, std::vector<RowDesc>& rows) {
    const int J = sp.n_components;
    const double f0 = sp.f_min / sp.S_low, fM = sp.f_max * sp.S_high;
    rows.assign(RP, RowDesc{0, 0, 0, ROW_PAD, 0});
    for (int j = 0; j < J; j++) {
        const double fj = f0 * std::pow(fM / f0, (double)j / (double)(J - 1));
        if (sp.basis == PIORAN_BASIS_SHO) {
            const double cj = std::sqrt(2.0) * M_PI * fj;
            rows[2 * j] = RowDesc{cj, cj, 1.0, ROW_COS, j};
            rows[2 * j + 1] = RowDesc{cj, cj, 1.0, ROW_SIN, j};
        } else {
            const double cj = M_PI * fj, dj = std::sqrt(3.0) * cj;
            rows[2 * j] = RowDesc{cj, dj, std::sqrt(3.0), ROW_COS, j};
            rows[2 * j + 1] = RowDesc{cj, dj, std::sqrt(3.0), ROW_SIN, j};
            rows[2 * J + j] = RowDesc{2.0 * cj, 0.0, 0.0, ROW_REAL, j};
        }
    }
}

// Cache discipline of the per-series tables: a hit refreshes the LRU stamp; an insert beyond MAX_TABLES_PER_SERIES evicts the
// least recently used table (after draining the stream: a kernel may still read it; cached work items hold its pointer).
static bool table_lookup(pioran_ctx* c, std::map<TableKey, Table>& cache, const TableKey& key, Table* out) {
    auto it = cache.find(key);
    if (it == cache.end()) return false;
    it->second.last_use = ++c->use_clock;
    *out = it->second;
    return true;
}
static void table_insert(pioran_ctx* c, std::map<TableKey, Table>& cache, const TableKey& key, Table& tb) {
    if (cache.size() >= MAX_TABLES_PER_SERIES) {
        auto victim = cache.begin();
        for (auto it = cache.begin(); it != cache.end(); ++it)
            if (it->second.last_use < victim->second.last_use) victim = it;
        cudaStreamSynchronize(c->stream);
        cudaFree(victim->second.d);
        cache.erase(victim);
        c->work_key.clear();
        c->gwork_key.clear();
    }
    tb.last_use = ++c->use_clock;
    cache[key] = tb;
}

static int get_table(pioran_ctx* c, Series* s, const pioran_approx_spec& sp, Table* out) {
    const double f0 = sp.f_min / sp.S_low, fM = sp.f_max * sp.S_high;
    TableKey key{sp.basis, sp.n_components, f0, fM};
    if (table_lookup(c, s->tables, key, out)) return 0;
    const int R = rank_of(sp.basis, sp.n_components);
    const int BS = bs_for_rank(R);
    if (BS > 8) return fail(PIORAN_EUNSUPPORTED, "rank %d needs block size %d > 8 (n_components too large for this build)", R, BS);
    const int RP = G * BS;            // logical rows; the table stores them in the padded layout of rps_of(BS)
    std::vector<RowDesc> rows;
    make_rows(sp, RP, rows);
    int rc = c->rows.ensure(sizeof(RowDesc) * RP);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->rows.p, rows.data(), sizeof(RowDesc) * RP, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));  // rows is a local
    Table tb;
    tb.rpad = RP;
    tb.npad = ((s->N + CHUNK_STEPS - 1) / CHUNK_STEPS) * CHUNK_STEPS;
    const size_t bytes = sizeof(double) * (size_t)tb.npad * table_step_doubles(rps_of(BS));
    CUDA_TRY(cudaMalloc(&tb.d, bytes));
    const int64_t total = tb.npad * rps_of(BS);
    const int tpb = 256;
    table_build_kernel<<<(unsigned)((total + tpb - 1) / tpb), tpb, 0, c->stream>>>(tb.d, s->t, s->y, s->s2, s->N, tb.npad,
                                                                                 c->rows.as<RowDesc>(), BS);
    c->launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { cudaFree(tb.d); return fail(PIORAN_ECUDA, "table_build_kernel launch failed: %s", cudaGetErrorString(e)); }
    table_insert(c, s->tables, key, tb);
    *out = tb;
    return 0;
}

// ------------------------------------------------------------------------------------------------ K2t (blocked.cuh)
// The tensor-pipe kernel serves the shared-table path at ranks <= 63 (64 needs a 9th row tile for the data row).
// pioran_ctx_set_sweep_kernel(ctx, PIORAN_SWEEP_SCALAR) or PIORAN_K2=scalar in the environment select the scalar-pipe kernel
// of celerite.cuh instead (A/B timing, tests of both paths).
static bool blocked_enabled(const pioran_ctx* c, int R) {
    static const int mode = [] { const char* e = getenv("PIORAN_K2"); return (e && (!strcmp(e, "scalar") || !strcmp(e, "0"))) ? 0 : 1; }();
    return mode != 0 && c->sweep_kernel != PIORAN_SWEEP_SCALAR && R >= 1 && blk_ntr(R) <= 8;
}
static int get_btable(pioran_ctx* c, Series* s, const pioran_approx_spec& sp, Table* out, bool grad = false) {
    const double f0 = sp.f_min / sp.S_low, fM = sp.f_max * sp.S_high;
    const int R = rank_of(sp.basis, sp.n_components);
    const BlkLayout lay = blk_layout(R, grad);
    const bool own = grad && lay.NTR != blk_layout(R, false).NTR;      // R ≡ 7 mod 8: the gradient's table has its own row layout
    TableKey key{sp.basis, own ? -sp.n_components : sp.n_components, f0, fM};
    if (table_lookup(c, s->btables, key, out)) return 0;
    const int NT = lay.NT, NTR = lay.NTR, RPT = 8 * NTR;
    std::vector<RowDesc> lrows, rows(RPT, RowDesc{0, 0, 0, ROW_PAD, 0});
    make_rows(sp, RPT, lrows);
    for (int r = 0; r < R; r++) {            // physical order; term = logical row index (the K_blk table is indexed by it)
        RowDesc rd = lrows[r];
        rd.term = r;
        rows[blk_phys_row(r, R)] = rd;
    }
    rows[lay.RG] = RowDesc{0, 0, 0, ROW_AUG, 0};
    if (lay.RM >= 0) rows[lay.RM] = RowDesc{0, 0, 0, ROW_AUG2, 0};   // ∂/∂μ row of the gradient kernel
    int rc = c->rows.ensure(sizeof(RowDesc) * RPT);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->rows.p, rows.data(), sizeof(RowDesc) * RPT, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));  // rows is a local
    Table tb;
    tb.rpad = RPT;
    const int64_t nblocks = (s->N + BLK - 1) / BLK;
    tb.npad = nblocks * BLK;
    const size_t bytes = sizeof(double) * (size_t)nblocks * blk_doubles(NT, NTR);
    CUDA_TRY(cudaMalloc(&tb.d, bytes));
    if (cudaMemsetAsync(tb.d, 0, bytes, c->stream) != cudaSuccess) { cudaFree(tb.d); return fail(PIORAN_ECUDA, "cudaMemsetAsync failed"); }
    const int64_t total = nblocks * RPT;
    const int tpb = 128;
    blocked_table_kernel<<<(unsigned)((total + tpb - 1) / tpb), tpb, 0, c->stream>>>(tb.d, s->t, s->y, s->s2, s->N, nblocks,
                                                                                    c->rows.as<RowDesc>(), NT, NTR);
    c->launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { cudaFree(tb.d); return fail(PIORAN_ECUDA, "blocked_table_kernel launch failed: %s", cudaGetErrorString(e)); }
    table_insert(c, s->btables, key, tb);
    *out = tb;
    return 0;
}
// Warps per CTA: the register budget of the state (NT(NT+1) doubles per lane) decides it.
#ifndef PIORAN_BLK_NW_LARGE
#define PIORAN_BLK_NW_LARGE 8     // warps per CTA at 7, 8 row tiles (255 registers per thread)
#endif
#ifndef PIORAN_BLK_NW_MID
#define PIORAN_BLK_NW_MID 12      // 5, 6 row tiles (168 registers)
#endif
static constexpr int blocked_nw_of(int NT) { return NT >= 7 ? PIORAN_BLK_NW_LARGE : NT >= 5 ? PIORAN_BLK_NW_MID : 16; }
static int blocked_force_nw() {   // PIORAN_BLK_NW=8: eight warps per CTA whatever the row tiles (experiments only)
    static const int force_nw = [] { const char* e = getenv("PIORAN_BLK_NW"); return e ? atoi(e) : 0; }();
    return force_nw;
}
static int blocked_nw(int NT) { return blocked_force_nw() == 8 ? 8 : blocked_nw_of(NT); }
template <int NT, int NTR, bool HALF, int NW>
static int launch_blocked_nw(pioran_ctx* c, const BatchArgs& args, int nitems, int R, int amp_stride) {
    auto kern = celerite_blocked_kernel<NT, NTR, HALF, NW, 1>;
    const size_t smem = sizeof(double) * ((size_t)BLK_NSTAGE * blk_doubles(NT, NTR) + (size_t)NW * (8 * NTR + 8 * NT)) +
                        BLK_NSTAGE * (sizeof(uint64_t) + sizeof(int)) + 16;
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaEventRecord(c->ev_beg, c->stream);
    kern<<<nitems, NW * 32, smem, c->stream>>>(args, R, amp_stride, blk_layout(R, false).RG);
    cudaEventRecord(c->ev_end, c->stream);
    note_kernel(c, KF_BLOCKED, NT, NTR, HALF, NW);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}
template <int NT, int NTR, bool HALF>
static int launch_blocked(pioran_ctx* c, const BatchArgs& args, int nitems, int tpi, int R, int amp_stride) {
    if (blocked_force_nw() == 8 && tpi > 4) return launch_blocked_nw<NT, NTR, HALF, 8>(c, args, nitems, R, amp_stride);
    if (tpi <= 4) return launch_blocked_nw<NT, NTR, HALF, 4>(c, args, nitems, R, amp_stride);
    if (tpi <= 8) return launch_blocked_nw<NT, NTR, HALF, 8>(c, args, nitems, R, amp_stride);
    return launch_blocked_nw<NT, NTR, HALF, blocked_nw_of(NT)>(c, args, nitems, R, amp_stride);
}
static int dispatch_blocked(pioran_ctx* c, const BatchArgs& a, int nitems, int tpi, int R, int amp_stride) {
    const int NT = blk_nt(R);
    const bool xrow = blk_ntr(R) != NT, half = blk_half(R);
#define PIORAN_BLK_CASE(nt)                                                                                   \
    case nt: return xrow ? launch_blocked<nt, nt + 1, false>(c, a, nitems, tpi, R, amp_stride)                \
                  : half ? launch_blocked<nt, nt, true>(c, a, nitems, tpi, R, amp_stride)                     \
                         : launch_blocked<nt, nt, false>(c, a, nitems, tpi, R, amp_stride);
    switch (NT) {
        PIORAN_BLK_CASE(1) PIORAN_BLK_CASE(2) PIORAN_BLK_CASE(3) PIORAN_BLK_CASE(4)
        PIORAN_BLK_CASE(5) PIORAN_BLK_CASE(6) PIORAN_BLK_CASE(7)
        case 8:
            if (xrow) break;
            return half ? launch_blocked<8, 8, true>(c, a, nitems, tpi, R, amp_stride)
                        : launch_blocked<8, 8, false>(c, a, nitems, tpi, R, amp_stride);
    }
#undef PIORAN_BLK_CASE
    return fail(PIORAN_EUNSUPPORTED, "rank %d not served by the blocked kernel", R);
}

// K2tw (blocked_wide.cuh): ranks 65 … 128 on the tensor pipe, one CTA of W warps per evaluation.  Small batches at 4 … 8
// column tiles run it too, one CTA per evaluation (PIORAN_K2_SMALL_CTA=0: the warp kernel instead).
static bool small_cta_enabled() {
    static const bool on = [] { const char* e = getenv("PIORAN_K2_SMALL_CTA"); return !(e && !strcmp(e, "0")); }();
    return on;
}
static bool blocked_wide_enabled(const pioran_ctx* c, int R) {
    static const int mode = [] { const char* e = getenv("PIORAN_K2W"); return (e && (!strcmp(e, "scalar") || !strcmp(e, "0"))) ? 0 : 1; }();
    return mode != 0 && c->sweep_kernel != PIORAN_SWEEP_SCALAR && R > 64 && R <= 128;
}
template <int NT, int NTR, int W>
static int launch_blocked_wide(pioran_ctx* c, const BatchArgs& args, int nitems, int R, int amp_stride) {
    auto kern = celerite_blocked_wide_kernel<NT, NTR, W>;
    const size_t smem = blkw_smem_bytes<NT, NTR, W>();
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaEventRecord(c->ev_beg, c->stream);
    kern<<<nitems, W * 32, smem, c->stream>>>(args, R, amp_stride, blk_layout(R, false).RG);
    cudaEventRecord(c->ev_end, c->stream);
    note_kernel(c, KF_BLOCKED_WIDE, NT, NTR, W);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}
static int dispatch_blocked_wide(pioran_ctx* c, const BatchArgs& a, int nitems, int R, int amp_stride) {
    const int NT = blk_nt(R);
    const bool xrow = blk_ntr(R) != NT;
#define PIORAN_BLKW_CASE(nt, w)                                                                       \
    case nt: return xrow ? launch_blocked_wide<nt, nt + 1, (nt + 1 > 12 ? 8 : w)>(c, a, nitems, R, amp_stride) \
                         : launch_blocked_wide<nt, nt, w>(c, a, nitems, R, amp_stride);
    switch (NT) {
        PIORAN_BLKW_CASE(4, 4) PIORAN_BLKW_CASE(5, 4) PIORAN_BLKW_CASE(6, 4) PIORAN_BLKW_CASE(7, 4) PIORAN_BLKW_CASE(8, 4)   // small batches (latency)
        PIORAN_BLKW_CASE(9, 4) PIORAN_BLKW_CASE(10, 4) PIORAN_BLKW_CASE(11, 4) PIORAN_BLKW_CASE(12, 4)
        PIORAN_BLKW_CASE(13, 8) PIORAN_BLKW_CASE(14, 8) PIORAN_BLKW_CASE(15, 8) PIORAN_BLKW_CASE(16, 8)
    }
#undef PIORAN_BLKW_CASE
    return fail(PIORAN_EUNSUPPORTED, "rank %d not served by the wide blocked kernel", R);
}

// ------------------------------------------------------------------------------------------------ K2 launchers
#ifndef PIORAN_NW_SMALL
#define PIORAN_NW_SMALL 12   // warps per CTA for block sizes <= 5 (register budget 168/thread)
#endif
#ifndef PIORAN_NW_LARGE
#define PIORAN_NW_LARGE 8    // block sizes 7, 8 (register budget 255/thread)
#endif
static constexpr int nw_for_bs(int BS) { return BS <= 5 ? PIORAN_NW_SMALL : BS == 6 ? 10 : PIORAN_NW_LARGE; }

// Calls f(std::integral_constant<int, v>{}): a launch site instantiates its kernel for LO … HI, and only for those.
template <int LO, int HI, class F>
static int with_int(int v, F f) {
    if constexpr (LO > HI) return fail(PIORAN_EUNSUPPORTED, "no kernel instantiated for %d", v);
    else return v == LO ? f(std::integral_constant<int, LO>{}) : with_int<LO + 1, HI>(v, f);
}

template <int BS>
static size_t generic_smem_bytes(int Jt) {
    constexpr int RPS = rps_of(BS), SD = table_step_doubles(RPS);
    return sizeof(double) * (size_t)nw_for_bs(BS) * ((size_t)GCH * SD + 2 * RPS + (size_t)(((GCH + 2) * Jt + 1) & ~1));
}

// Small batches (at most SMALL_NW parameter vectors per CTA, i.e. S·B ≤ 4 × SMs — a nested sampler's few hundred live
// points): a CTA of 4 warps, one per SM sub-partition.  The full-size CTA would fill its surplus warps with redundant
// sweeps that share the FP64 pipe of the useful ones and roughly double the latency of the call.
constexpr int SMALL_NW = 4;
template <int BS, int NW = nw_for_bs(BS)>
static int launch_shared(pioran_ctx* c, const BatchArgs& args, int nitems) {
    constexpr int RPS = rps_of(BS), SD = table_step_doubles(RPS);
    auto kern = celerite_shared_kernel<BS, NW>;
    const size_t smem = sizeof(double) * (2 * (size_t)CHUNK_STEPS * SD + (size_t)NW * 2 * RPS) + 2 * sizeof(uint64_t) + 16;
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaEventRecord(c->ev_beg, c->stream);
    kern<<<nitems, NW * 32, smem, c->stream>>>(args);
    cudaEventRecord(c->ev_end, c->stream);
    note_kernel(c, KF_SHARED, BS, NW);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}
// Two parameter vectors per warp for block sizes <= 5 (celerite_shared_pair_kernel); PIORAN_PAIR=0 falls back to one.
#ifndef PIORAN_NW_PAIR
#define PIORAN_NW_PAIR 8
#endif
static bool pair_enabled(int BS) {
    static const int env = [] { const char* e = getenv("PIORAN_PAIR"); return e ? atoi(e) : 1; }();
    return env != 0 && BS <= 5;
}
static int theta_per_item(int BS) { return pair_enabled(BS) ? 2 * PIORAN_NW_PAIR : nw_for_bs(BS); }
template <int BS>
static int launch_shared_pair(pioran_ctx* c, const BatchArgs& args, int nitems) {
    constexpr int RPS = rps_of(BS), SD = table_step_doubles(RPS), NW = PIORAN_NW_PAIR;
    auto kern = celerite_shared_pair_kernel<BS, NW>;
    const size_t smem = sizeof(double) * (2 * (size_t)CHUNK_STEPS * SD + (size_t)NW * 4 * RPS) + 2 * sizeof(uint64_t) + 16;
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaEventRecord(c->ev_beg, c->stream);
    kern<<<nitems, NW * 32, smem, c->stream>>>(args);
    cudaEventRecord(c->ev_end, c->stream);
    note_kernel(c, KF_SHARED_PAIR, BS, NW);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}
template <int BS, int NW = nw_for_bs(BS)>
static int launch_generic(pioran_ctx* c, const BatchArgs& args, int nitems) {
    constexpr int RPS = rps_of(BS), SD = table_step_doubles(RPS);
    auto kern = celerite_generic_kernel<BS, NW>;
    const size_t smem = sizeof(double) * (size_t)NW * ((size_t)GCH * SD + 2 * RPS + (size_t)(((GCH + 2) * args.Jt + 1) & ~1));
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaEventRecord(c->ev_beg, c->stream);
    kern<<<nitems, NW * 32, smem, c->stream>>>(args);
    cudaEventRecord(c->ev_end, c->stream);
    note_kernel(c, KF_GENERIC, BS, NW);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// K3 pass 3: the generic kernel in its chunked variant, 2 warps per CTA so that a few hundred chunks cover every SM.
constexpr int CHUNK_NW = 2;
template <int BS>
static int launch_chunked(pioran_ctx* c, const BatchArgs& args, int nctas) {
    constexpr int RPS = rps_of(BS), SD = table_step_doubles(RPS);
    auto kern = celerite_generic_kernel<BS, CHUNK_NW, true>;
    const size_t smem = sizeof(double) * (size_t)CHUNK_NW * ((size_t)GCH * SD + 2 * RPS + (size_t)(((GCH + 2) * args.Jt + 1) & ~1));
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<nctas, CHUNK_NW * 32, smem, c->stream>>>(args);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}
static int dispatch_chunked(pioran_ctx* c, int BS, const BatchArgs& a, int nctas) {
    return with_int<4, 8>(BS, [&](auto bs) { return launch_chunked<bs>(c, a, nctas); });
}

static int dispatch_shared(pioran_ctx* c, int BS, const BatchArgs& a, int nitems, int tpi) {
    if (tpi <= SMALL_NW) return with_int<4, 8>(BS, [&](auto bs) { return launch_shared<bs, SMALL_NW>(c, a, nitems); });
    if (tpi <= 8 && BS <= 6)    // two warps per sub-partition, one parameter vector each
        return with_int<4, 6>(BS, [&](auto bs) { return launch_shared<bs, 8>(c, a, nitems); });
    if (pair_enabled(BS)) return with_int<4, 5>(BS, [&](auto bs) { return launch_shared_pair<bs>(c, a, nitems); });
    return with_int<4, 8>(BS, [&](auto bs) { return launch_shared<bs>(c, a, nitems); });
}
static int dispatch_generic(pioran_ctx* c, int BS, const BatchArgs& a, int nitems, int tpi) {
    if (tpi <= SMALL_NW) return with_int<4, 8>(BS, [&](auto bs) { return launch_generic<bs, SMALL_NW>(c, a, nitems); });
    return with_int<4, 8>(BS, [&](auto bs) { return launch_generic<bs>(c, a, nitems); });
}

// generic kernel in STEP_STORE / STEP_SIM mode (posterior mean and GP draws)
template <int BS, int MODE>
static int launch_generic_mode(pioran_ctx* c, const BatchArgs& args, int nitems) {
    auto kern = celerite_generic_kernel<BS, nw_for_bs(BS), false, MODE>;
    const size_t smem = generic_smem_bytes<BS>(args.Jt);
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<nitems, nw_for_bs(BS) * 32, smem, c->stream>>>(args);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}
template <int MODE>
static int dispatch_generic_mode(pioran_ctx* c, int BS, const BatchArgs& a, int nitems) {
    return with_int<4, 8>(BS, [&](auto bs) { return launch_generic_mode<bs, MODE>(c, a, nitems); });
}

// Splits S series × B parameter vectors into CTA work items of at most NW vectors, sized so that the number of
// items is close to a multiple of the SM count (one CTA per SM is resident), longest series first.
struct ItemPlan { std::vector<WorkItem> items; int tpi = 0; };
static void plan_items(pioran_ctx* c, int S, Series* const* ser, const Table* tabs, int B, int NW, bool theta_per_series,
                       ItemPlan& ip, bool tail_items = false) {
    const long long E = (long long)S * B;
    if (tail_items && S == 1 && E > (long long)NW * c->num_sms) {
        // One series, more than one wave of full items: whole waves of NW-vector items, then the remainder spread evenly over
        // all SMs as ONE last wave of smaller items (their surplus warps exit, blocked.cuh), instead of a last wave that is
        // partly empty but runs at the full item's duration.
        const long long per_wave = (long long)NW * c->num_sms;
        const long long full = (E / per_wave) * per_wave;
        const long long rem = E - full;
        ip.tpi = NW;
        ip.items.clear();
        auto push = [&](long long beg, long long end) {
            WorkItem w;
            w.table = tabs ? tabs[0].d : nullptr;
            w.t = ser[0]->t; w.y = ser[0]->y; w.s2 = ser[0]->s2;
            w.N = ser[0]->N;
            w.theta_begin = (int)beg; w.par_begin = (int)beg; w.count = (int)(end - beg); w.out_begin = (int)beg;
            w.n_begin = 0; w.n_end = ser[0]->N; w.init = nullptr; w.part = nullptr;
            ip.items.push_back(w);
        };
        for (long long b0 = 0; b0 < full; b0 += NW) push(b0, b0 + NW);
        if (rem > 0) {
            const long long nit = std::min<long long>(c->num_sms, rem);
            for (long long k = 0; k < nit; k++) push(full + rem * k / nit, full + rem * (k + 1) / nit);
        }
        return;
    }
    int tpi = (int)std::min<long long>(NW, std::max<long long>(1, (E + c->num_sms - 1) / c->num_sms));
    long long items = 0;
    for (int s = 0; s < S; s++) items += (B + tpi - 1) / tpi;
    const long long waves = (items + c->num_sms - 1) / c->num_sms;
    const long long target = waves * c->num_sms;
    tpi = (int)std::min<long long>(NW, std::max<long long>(1, (E + target - 1) / target));
    ip.tpi = tpi;
    std::vector<int> order(S);
    for (int s = 0; s < S; s++) order[s] = s;
    std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return ser[x]->N > ser[y]->N; });
    ip.items.clear();
    for (int s : order) {
        const int nit = (B + tpi - 1) / tpi;
        for (int k = 0; k < nit; k++) {
            const int beg = (int)((long long)B * k / nit), end = (int)((long long)B * (k + 1) / nit);
            WorkItem w;
            w.table = tabs ? tabs[s].d : nullptr;
            w.t = ser[s]->t; w.y = ser[s]->y; w.s2 = ser[s]->s2;
            w.N = ser[s]->N;
            w.theta_begin = s * B + beg;
            w.par_begin = (theta_per_series ? s * B : 0) + beg;
            w.count = end - beg;
            w.out_begin = s * B + beg;
            w.n_begin = 0; w.n_end = ser[s]->N; w.init = nullptr; w.part = nullptr;
            ip.items.push_back(w);
        }
    }
}

// ------------------------------------------------------------------------------------------------ wide ranks (K2w)
// Ranks above 64 (block size > 8): state in shared memory, one CTA per parameter vector (wide.cuh).
template <int MODE = STEP_LOGL>
static int launch_wide(pioran_ctx* c, const BatchArgs& args, int nitems) {
    if (args.R > WIDE_MAX_RANK)
        return fail(PIORAN_EUNSUPPORTED, "rank %d exceeds this build's limit of %d", args.R, WIDE_MAX_RANK);
    if (args.R <= 128) {   // the state fits the register file of one CTA
        const int TS = std::max(5, (args.R + 15) / 16);
        cudaEventRecord(c->ev_beg, c->stream);
        with_int<5, 8>(TS, [&](auto ts) { celerite_wide_reg_kernel<ts, MODE><<<nitems, WIDE_THREADS, 0, c->stream>>>(args); return 0; });
        cudaEventRecord(c->ev_end, c->stream);
        note_kernel(c, MODE == STEP_STORE ? KF_WIDE_REG_STORE : MODE == STEP_SIM ? KF_WIDE_REG_SIM : KF_WIDE_REG, TS);
        c->launches++;
        CUDA_TRY(cudaGetLastError());
        return 0;
    }
    if (MODE != STEP_LOGL)
        return fail(PIORAN_EUNSUPPORTED, "posterior mean and draws are built for ranks up to 128 (rank %d)", args.R);
    const size_t smem = sizeof(double) * wide_smem_doubles(wide_geom(args.R));
    CUDA_TRY(cudaFuncSetAttribute(celerite_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaEventRecord(c->ev_beg, c->stream);
    celerite_wide_kernel<<<nitems, WIDE_THREADS, smem, c->stream>>>(args);
    cudaEventRecord(c->ev_end, c->stream);
    note_kernel(c, KF_WIDE);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}
// leading dimension of the factor a STEP_STORE sweep leaves behind: 8·BS logical rows (warp kernel) or 16·TS (register-file CTA kernel)
static int stored_factor_ld(int R) { const int BS = bs_for_rank(R); return BS <= 8 ? G * BS : 16 * std::max(5, (R + 15) / 16); }

// ------------------------------------------------------------------------------------------------ K1 entry
extern "C" int pioran_approx_coeffs(pioran_ctx* c, const pioran_approx_spec* spec, int B, const double* theta,
                                    double* a, double* b, double* cc, double* d) try {
    if (is_group(c)) return pioran_approx_coeffs(c->children[0], spec, B, theta, a, b, cc, d);
    if (!c || !spec || !theta || !a || !b || !cc || !d) return fail(PIORAN_EINVAL, "NULL argument");
    if (B < 1) return fail(PIORAN_EINVAL, "B must be >= 1");
    int rc = check_spec(*spec);
    if (rc) return rc;
    PIORAN_COMPUTE_LOCK(c);
    CUDA_TRY(cudaSetDevice(c->device));
    ApproxPlan* plan;
    if ((rc = get_plan(c, *spec, &plan))) return rc;
    const int npar = n_psd_par_of(spec->psd_model), ts = npar + 1;
    const int Jt = spec->basis == PIORAN_BASIS_SHO ? spec->n_components : 2 * spec->n_components;
    if ((rc = c->theta.ensure(sizeof(double) * (size_t)B * ts))) return rc;
    if ((rc = c->coef.ensure(sizeof(double) * (size_t)B * Jt * 4))) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->theta.p, theta, sizeof(double) * (size_t)B * ts, cudaMemcpyHostToDevice, c->stream));
    double* da = c->coef.as<double>();
    const size_t n = (size_t)B * Jt;
    approx_kernel<<<(B + 127) / 128, 128, 0, c->stream>>>(plan, B, c->theta.as<double>(), ts, da, da + n, da + 2 * n,
                                                         da + 3 * n, nullptr, 0, nullptr);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(a, da, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(b, da + n, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(cc, da + 2 * n, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(d, da + 3 * n, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

// ------------------------------------------------------------------------------------------------ fused entry
// theta_stride: doubles per θ row (0 = n_psd_par + 3; larger rows carry extra columns the sweep ignores).  y_batch / s2_batch:
// device [B × N] per-θ data replacing the resident y / σ² (single series, ranks ≤ 64) — the log-shift entry fills them.
static int approx_logl_dev_locked(pioran_ctx* c, int S, const int* series_ids, const pioran_approx_spec* specs, int B,
                                  const double* theta_dev, int theta_per_series, double* logl_dev, int theta_stride = 0,
                                  const double* y_batch = nullptr, const double* s2_batch = nullptr) {
    int rc;
    if (S < 1 || B < 1) return fail(PIORAN_EINVAL, "S and B must be >= 1");
    if ((long long)S * B > 0x7fffffffLL / 64) return fail(PIORAN_EINVAL, "S*B too large");
    std::vector<Series*> ser(S);
    std::vector<Table> tabs(S);
    for (int s = 0; s < S; s++) {
        if ((rc = check_spec(specs[s]))) return rc;
        if (specs[s].psd_model != specs[0].psd_model || specs[s].basis != specs[0].basis ||
            specs[s].n_components != specs[0].n_components)
            return fail(PIORAN_EINVAL, "all specs of one call must share psd_model, basis and n_components");
        ser[s] = get_series(c, series_ids[s]);
        if (!ser[s]) return fail(PIORAN_EINVAL, "unknown series id %d", series_ids[s]);
    }
    const int npar = n_psd_par_of(specs[0].psd_model), ts = theta_stride > 0 ? theta_stride : npar + 3;
    const int R = rank_of(specs[0].basis, specs[0].n_components);
    const int BS = bs_for_rank(R);
    if ((y_batch || s2_batch) && (S != 1 || BS > 8))
        return fail(PIORAN_EUNSUPPORTED, "per-parameter-vector data need a single series and a rank <= 64 (rank %d, %d series)", R, S);
    if (BS > 8 && blocked_wide_enabled(c, R)) {
        // ranks 65 … 128: the blocked sweep with one CTA per (series, θ) (blocked_wide.cuh) on the shared block table
        const int RPA = 8 * blk_nt(R);
        for (int s = 0; s < S; s++)
            if ((rc = get_btable(c, ser[s], specs[s], &tabs[s]))) return rc;
        if ((rc = c->amp.ensure(sizeof(double) * (size_t)S * B * RPA))) return rc;
        if ((rc = c->suma.ensure(sizeof(double) * (size_t)S * B))) return rc;
        for (int s = 0; s < S; s++) {
            ApproxPlan* plan;
            if ((rc = get_plan(c, specs[s], &plan))) return rc;
            const double* th = theta_dev + (theta_per_series ? (size_t)s * B * ts : 0);
            approx_kernel<<<(B + 127) / 128, 128, 0, c->stream>>>(plan, B, th, ts, nullptr, nullptr, nullptr, nullptr,
                                                                 c->amp.as<double>() + (size_t)s * B * RPA, RPA,
                                                                 c->suma.as<double>() + (size_t)s * B);
            c->launches++;
        }
        CUDA_TRY(cudaGetLastError());
        std::vector<int64_t> key;
        key.push_back(S); key.push_back(B); key.push_back(-1000 - R); key.push_back(theta_per_series != 0);
        for (int s = 0; s < S; s++) { key.push_back((int64_t)(intptr_t)tabs[s].d); key.push_back((int64_t)(intptr_t)ser[s]->t); key.push_back(ser[s]->N); }
        if (key != c->work_key) {
            ItemPlan ip;
            plan_items(c, S, ser.data(), tabs.data(), B, 1, theta_per_series != 0, ip);
            c->work_key.clear();
            if ((rc = c->work.ensure(sizeof(WorkItem) * ip.items.size()))) return rc;
            CUDA_TRY(cudaMemcpyAsync(c->work.p, ip.items.data(), sizeof(WorkItem) * ip.items.size(), cudaMemcpyHostToDevice, c->stream));
            CUDA_TRY(cudaStreamSynchronize(c->stream));
            c->work_key = key;
            c->work_items = (int)ip.items.size();
            c->work_tpi = ip.tpi;
        }
        BatchArgs args{};
        args.work = c->work.as<WorkItem>();
        args.amp = c->amp.as<double>(); args.suma = c->suma.as<double>();
        args.mu = theta_dev + npar + 2; args.nu = theta_dev + npar + 1; args.pstride = ts;
        args.out = logl_dev;
        return dispatch_blocked_wide(c, args, c->work_items, R, RPA);
    }
    if (BS > 8) {
        // ranks above 128 (and the scalar-pipe selection): K1 writes explicit coefficients, one CTA per (series, θ) (wide.cuh)
        if (R > WIDE_MAX_RANK) return fail(PIORAN_EUNSUPPORTED, "rank %d exceeds this build's limit of %d", R, WIDE_MAX_RANK);
        const int J = specs[0].n_components;
        const int Jt = specs[0].basis == PIORAN_BASIS_SHO ? J : 2 * J;
        std::vector<int> term_row(Jt);
        for (int m = 0; m < Jt; m++) term_row[m] = (m < J) ? 2 * m : -(2 * J + (m - J) + 1);   // src/psd.jl:264-275: DRW parts are real terms
        const size_t n = (size_t)B * Jt;
        if ((rc = c->coef.ensure(sizeof(double) * (size_t)S * n * 4))) return rc;
        if ((rc = c->rows.ensure(sizeof(int) * (Jt + 1)))) return rc;
        if ((rc = c->work.ensure(sizeof(WorkItem) * (size_t)S * B))) return rc;
        c->work_key.clear();
        std::vector<WorkItem> items;
        items.reserve((size_t)S * B);
        for (int s = 0; s < S; s++) {
            ItemPlan ip;
            plan_items(c, 1, &ser[s], nullptr, B, 1, false, ip);
            items.insert(items.end(), ip.items.begin(), ip.items.end());
        }
        CUDA_TRY(cudaMemcpyAsync(c->rows.p, term_row.data(), sizeof(int) * Jt, cudaMemcpyHostToDevice, c->stream));
        CUDA_TRY(cudaMemcpyAsync(c->work.p, items.data(), sizeof(WorkItem) * items.size(), cudaMemcpyHostToDevice, c->stream));
        CUDA_TRY(cudaStreamSynchronize(c->stream));   // term_row and items are locals
        for (int s = 0; s < S; s++) {
            ApproxPlan* plan;
            if ((rc = get_plan(c, specs[s], &plan))) return rc;
            const double* th = theta_dev + (theta_per_series ? (size_t)s * B * ts : 0);
            double* da = c->coef.as<double>() + (size_t)s * n * 4;
            approx_kernel<<<(B + 127) / 128, 128, 0, c->stream>>>(plan, B, th, ts, da, da + n, da + 2 * n, da + 3 * n, nullptr, 0,
                                                                 nullptr);
            c->launches++;
            CUDA_TRY(cudaGetLastError());
            BatchArgs args{};
            args.work = c->work.as<WorkItem>() + (size_t)s * B;
            args.a = da; args.b = da + n; args.c = da + 2 * n; args.d = da + 3 * n;
            args.Jt = Jt; args.term_row = c->rows.as<int>(); args.R = R;
            args.mu = th + npar + 2; args.nu = th + npar + 1; args.pstride = ts;
            args.out = logl_dev + (size_t)s * B;
            if ((rc = launch_wide(c, args, B))) return rc;
        }
        return 0;
    }
    const int RP = G * BS;
    const bool blocked = blocked_enabled(c, R);
    for (int s = 0; s < S; s++)
        if ((rc = blocked ? get_btable(c, ser[s], specs[s], &tabs[s]) : get_table(c, ser[s], specs[s], &tabs[s]))) return rc;
    // K1: amplitudes for every (series, θ)
    if ((rc = c->amp.ensure(sizeof(double) * (size_t)S * B * RP))) return rc;
    if ((rc = c->suma.ensure(sizeof(double) * (size_t)S * B))) return rc;
    for (int s = 0; s < S; s++) {
        ApproxPlan* plan;
        if ((rc = get_plan(c, specs[s], &plan))) return rc;
        const double* th = theta_dev + (theta_per_series ? (size_t)s * B * ts : 0);
        approx_kernel<<<(B + 127) / 128, 128, 0, c->stream>>>(plan, B, th, ts, nullptr, nullptr, nullptr, nullptr,
                                                             c->amp.as<double>() + (size_t)s * B * RP, RP,
                                                             c->suma.as<double>() + (size_t)s * B);
        c->launches++;
    }
    CUDA_TRY(cudaGetLastError());
    // K2
    std::vector<int64_t> key;
    key.reserve(4 + 3 * (size_t)S);
    // Small batches (at most 2 evaluations per SM: a handful of chains, the B = 1 drop-in) at 4 … 8 column tiles: one CTA of four warps
    // per evaluation (blocked_wide.cuh) — a block of 8 steps then costs a quarter of the products per warp: 0.22 instead of 0.48 ms per
    // 1 000 steps at rank 60 (tools/small_batch.py).  Beyond two CTAs per SM the register file holds no more of them and the warp kernel wins.
    const bool cta_per_theta = blocked && small_cta_enabled() && blk_nt(R) >= 4 && (long long)S * B <= 2LL * c->num_sms;
    key.push_back(S); key.push_back(B); key.push_back(blocked ? (cta_per_theta ? -2000 - R : -R) : BS); key.push_back(theta_per_series != 0);
    for (int s = 0; s < S; s++) { key.push_back((int64_t)(intptr_t)tabs[s].d); key.push_back((int64_t)(intptr_t)ser[s]->t); key.push_back(ser[s]->N); }
    if (key != c->work_key) {
        ItemPlan ip;
        plan_items(c, S, ser.data(), tabs.data(), B, cta_per_theta ? 1 : blocked ? blocked_nw(blk_nt(R)) : theta_per_item(BS), theta_per_series != 0, ip,
                   blocked && !cta_per_theta);
        c->work_key.clear();
        if ((rc = c->work.ensure(sizeof(WorkItem) * ip.items.size()))) return rc;
        CUDA_TRY(cudaMemcpyAsync(c->work.p, ip.items.data(), sizeof(WorkItem) * ip.items.size(), cudaMemcpyHostToDevice,
                                 c->stream));
        CUDA_TRY(cudaStreamSynchronize(c->stream));  // ip.items is a local; only when the call shape changes
        c->work_key = key;
        c->work_items = (int)ip.items.size();
        c->work_tpi = ip.tpi;
    }
    const int nitems = c->work_items;
    BatchArgs args{};
    args.work = c->work.as<WorkItem>();
    args.amp = c->amp.as<double>();
    args.suma = c->suma.as<double>();
    args.mu = theta_dev + npar + 2;
    args.nu = theta_dev + npar + 1;
    args.pstride = ts;
    args.y_batch = y_batch; args.s2_batch = s2_batch; args.ystride = ser[0]->N;
    args.out = logl_dev;
    if (cta_per_theta) return dispatch_blocked_wide(c, args, nitems, R, RP);
    if (blocked) return dispatch_blocked(c, args, nitems, c->work_tpi, R, RP);
    return dispatch_shared(c, BS, args, nitems, c->work_tpi);
}

// Log-normal time series (docs/src/timeseries.md:16-21, docs/src/ultranest.md:197-217): yn = log(y − c), σ² = σ²/(y − c)² per
// parameter vector (ν is applied by the sweep).  y − c <= 0 gives NaN, which the likelihood carries through as data.
__global__ void log_shift_kernel(const double* __restrict__ y, const double* __restrict__ s2, int64_t N, const double* __restrict__ theta,
                                 int ts, int c_col, int B, double* __restrict__ yb, double* __restrict__ sb) {
    const int64_t total = (int64_t)B * N;
    for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < total; k += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = k / N, n = k - i * N;
        const double dlt = y[n] - theta[i * ts + c_col];
        yb[k] = log(dlt);
        sb[k] = s2[n] / (dlt * dlt);
    }
}

// Parameter vectors per θ-chunk whose workspace of bytes_per_set each stays within cap (at least one).
static int theta_chunk(int B, size_t bytes_per_set, size_t cap = (size_t)1 << 30) {
    return (int)std::max<size_t>(1, std::min<size_t>((size_t)B, cap / bytes_per_set));
}

// The θ-chunk loop of the log-shift entries over the B × ts rows in c->theta: the chunk's transformed data, then
// fn(first row, row count, the chunk's θ rows, y batch, σ² batch).  16 N bytes of transformed data per parameter vector, at most
// 1 GiB at a time (written and read once: ≈ 0.3 ms per 65 536 × 1 000 block against tens of ms of sweep).
template <typename F>
static int logshift_chunks(pioran_ctx* c, Series* s, int B, int ts, F fn) {
    const int64_t N = s->N;
    const int chunk = theta_chunk(B, 16 * (size_t)N);
    int rc;
    if ((rc = c->post.ensure(sizeof(double) * 2 * (size_t)chunk * N))) return rc;
    double* yb = c->post.as<double>();
    double* sb = yb + (size_t)chunk * N;
    for (int off = 0; off < B; off += chunk) {
        const int nb = std::min(chunk, B - off);
        const double* th = c->theta.as<double>() + (size_t)off * ts;
        const int64_t total = (int64_t)nb * N;
        const int grid = (int)std::min<int64_t>((total + 255) / 256, (int64_t)c->num_sms * 16);
        log_shift_kernel<<<grid, 256, 0, c->stream>>>(s->y, s->s2, N, th, ts, ts - 1, nb, yb, sb);
        c->launches++;
        CUDA_TRY(cudaGetLastError());
        if ((rc = fn(off, nb, th, yb, sb))) return rc;
    }
    return 0;
}

extern "C" int pioran_approx_logl_logshift(pioran_ctx* c, int series_id, const pioran_approx_spec* spec, int B, const double* theta,
                                           double* logl_out) try {
    if (!c || !spec || !theta || !logl_out) return fail(PIORAN_EINVAL, "NULL argument");
    if (B < 1) return fail(PIORAN_EINVAL, "B must be >= 1");
    const int npar = n_psd_par_of(spec->psd_model);
    if (npar < 0) return fail(PIORAN_EINVAL, "unknown psd_model %d", spec->psd_model);
    const int ts = npar + 4;
    if (is_group(c))
        return group_fanout(c, series_id, B, [&](pioran_ctx* ch, int id, int64_t, int beg, int nb) {
            return pioran_approx_logl_logshift(ch, id, spec, nb, theta + (size_t)beg * ts, logl_out + beg);
        });
    PIORAN_COMPUTE_LOCK(c);
    CUDA_TRY(cudaSetDevice(c->device));
    int rc;
    if ((rc = check_spec(*spec))) return rc;
    Series* s = get_series(c, series_id);
    if (!s) return fail(PIORAN_EINVAL, "unknown series id %d", series_id);
    if ((rc = c->theta.ensure(sizeof(double) * (size_t)B * ts))) return rc;
    if ((rc = c->out.ensure(sizeof(double) * (size_t)B))) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->theta.p, theta, sizeof(double) * (size_t)B * ts, cudaMemcpyHostToDevice, c->stream));
    if ((rc = logshift_chunks(c, s, B, ts, [&](int off, int nb, const double* th, const double* yb, const double* sb) {
             return approx_logl_dev_locked(c, 1, &series_id, spec, nb, th, 0, c->out.as<double>() + off, ts, yb, sb);
         })))
        return rc;
    CUDA_TRY(cudaMemcpyAsync(logl_out, c->out.p, sizeof(double) * (size_t)B, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

extern "C" int pioran_approx_logl_dev(pioran_ctx* c, int S, const int* series_ids, const pioran_approx_spec* specs,
                                      int B, const double* theta_dev, int theta_per_series, double* logl_dev) try {
    if (is_group(c)) return fail(PIORAN_EUNSUPPORTED, "device-resident entries need a single-device context (a group spans devices)");
    if (!c || !series_ids || !specs || !theta_dev || !logl_dev) return fail(PIORAN_EINVAL, "NULL argument");
    PIORAN_COMPUTE_LOCK(c);
    CUDA_TRY(cudaSetDevice(c->device));
    return approx_logl_dev_locked(c, S, series_ids, specs, B, theta_dev, theta_per_series, logl_dev);
} catch (...) { return guard_fail(); }

extern "C" int pioran_approx_logl(pioran_ctx* c, int S, const int* series_ids, const pioran_approx_spec* specs, int B,
                                  const double* theta, int theta_per_series, double* logl_out) try {
    if (!c || !series_ids || !specs || !theta || !logl_out) return fail(PIORAN_EINVAL, "NULL argument");
    if (S < 1 || B < 1) return fail(PIORAN_EINVAL, "S and B must be >= 1");
    const int npar = n_psd_par_of(specs[0].psd_model);
    if (npar < 0) return fail(PIORAN_EINVAL, "unknown psd_model %d", specs[0].psd_model);
    const int ts = npar + 3;
    if (is_group(c))
        return group_fanout(c, S, series_ids, B, [&](pioran_ctx* ch, const int* ids, int64_t, int beg, int nb) -> int {
            if (S == 1) return pioran_approx_logl(ch, 1, ids, specs, nb, theta + (size_t)beg * ts, 0, logl_out + beg);
            // several series: the slice of every series' rows is gathered, evaluated and scattered back
            std::vector<double> th((size_t)(theta_per_series ? S : 1) * nb * ts), out((size_t)S * nb);
            for (int q = 0; q < (theta_per_series ? S : 1); q++)
                std::memcpy(th.data() + (size_t)q * nb * ts, theta + ((size_t)q * B + beg) * ts, sizeof(double) * (size_t)nb * ts);
            const int rc = pioran_approx_logl(ch, S, ids, specs, nb, th.data(), theta_per_series, out.data());
            if (rc) return rc;
            for (int q = 0; q < S; q++) std::memcpy(logl_out + (size_t)q * B + beg, out.data() + (size_t)q * nb, sizeof(double) * nb);
            return 0;
        });
    PIORAN_COMPUTE_LOCK(c);
    CUDA_TRY(cudaSetDevice(c->device));
    const size_t nth = (size_t)(theta_per_series ? S : 1) * B * ts;
    int rc;
    if (S == 1 && (rc = check_spec(specs[0])) == 0) {
        Series* s0 = get_series(c, series_ids[0]);
        const int R0 = rank_of(specs[0].basis, specs[0].n_components);
        if (s0 && auto_scan(c, s0->N, B, R0)) {
            // few parameter vectors, long series: K1 on the device, coefficients back to the host, parallel-in-time sweep
            ApproxPlan* plan;
            if ((rc = get_plan(c, specs[0], &plan))) return rc;
            const int J = specs[0].n_components, Jt = specs[0].basis == PIORAN_BASIS_SHO ? J : 2 * J;
            const size_t n = (size_t)B * Jt;
            if ((rc = c->theta.ensure(sizeof(double) * nth))) return rc;
            if ((rc = c->coef.ensure(sizeof(double) * n * 4))) return rc;
            CUDA_TRY(cudaMemcpyAsync(c->theta.p, theta, sizeof(double) * nth, cudaMemcpyHostToDevice, c->stream));
            double* da = c->coef.as<double>();
            approx_kernel<<<(B + 127) / 128, 128, 0, c->stream>>>(plan, B, c->theta.as<double>(), ts, da, da + n, da + 2 * n,
                                                                 da + 3 * n, nullptr, 0, nullptr);
            c->launches++;
            CUDA_TRY(cudaGetLastError());
            std::vector<double> co(4 * n), mu(B), nu(B);
            CUDA_TRY(cudaMemcpyAsync(co.data(), da, sizeof(double) * 4 * n, cudaMemcpyDeviceToHost, c->stream));
            CUDA_TRY(cudaStreamSynchronize(c->stream));
            for (int i = 0; i < B; i++) { nu[i] = theta[(size_t)i * ts + npar + 1]; mu[i] = theta[(size_t)i * ts + npar + 2]; }
            return scan_logl_locked(c, s0, series_ids[0], B, Jt, co.data(), co.data() + n, co.data() + 2 * n, co.data() + 3 * n,
                                    mu.data(), nu.data(), logl_out);
        }
    }
    if ((rc = c->theta.ensure(sizeof(double) * nth))) return rc;
    if ((rc = c->out.ensure(sizeof(double) * (size_t)S * B))) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->theta.p, theta, sizeof(double) * nth, cudaMemcpyHostToDevice, c->stream));
    if ((rc = approx_logl_dev_locked(c, S, series_ids, specs, B, c->theta.as<double>(), theta_per_series,
                                     c->out.as<double>())))
        return rc;
    CUDA_TRY(cudaMemcpyAsync(logl_out, c->out.p, sizeof(double) * (size_t)S * B, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

// ------------------------------------------------------------------------------------------------ prior transform
static_assert(sizeof(pioran_prior_spec) == sizeof(PriorSpec), "pioran_prior_spec layout");
static int prior_transform_dev_locked(pioran_ctx* c, int ncol, const pioran_prior_spec* priors, int B, const double* cube,
                                      double* theta_dev, int tstride) {
    if (ncol < 1 || ncol > PRIOR_MAX_COLS) return fail(PIORAN_EINVAL, "ncol must be in [1, %d]", PRIOR_MAX_COLS);
    for (int k = 0; k < ncol; k++) {
        const pioran_prior_spec& p = priors[k];
        if (p.kind < PIORAN_PRIOR_UNIFORM || p.kind > PIORAN_PRIOR_GAMMA) return fail(PIORAN_EINVAL, "column %d: unknown prior kind %d", k, p.kind);
        if (p.kind == PIORAN_PRIOR_UNIFORM_FROM && (p.ref_col < 0 || p.ref_col >= k))
            return fail(PIORAN_EINVAL, "column %d: ref_col %d must be an earlier column", k, p.ref_col);
        if (p.kind == PIORAN_PRIOR_LOGUNIFORM && !(p.p0 > 0.0 && p.p1 > 0.0)) return fail(PIORAN_EINVAL, "column %d: LogUniform needs positive bounds", k);
        if ((p.kind == PIORAN_PRIOR_NORMAL || p.kind == PIORAN_PRIOR_LOGNORMAL) && !(p.p1 > 0.0)) return fail(PIORAN_EINVAL, "column %d: sigma must be positive", k);
        if (p.kind == PIORAN_PRIOR_GAMMA && !(p.p0 >= 1.0 && p.p0 <= 32.0 && p.p0 == std::floor(p.p0) && p.p1 > 0.0))
            return fail(PIORAN_EUNSUPPORTED, "column %d: Gamma needs an integer shape in [1, 32] and a positive scale (shape %g)", k, p.p0);
    }
    int rc;
    const size_t ncube = (size_t)B * ncol;
    if ((rc = c->coef.ensure(sizeof(double) * ncube + sizeof(PriorSpec) * PRIOR_MAX_COLS))) return rc;
    double* cube_dev = c->coef.as<double>();
    PriorSpec* pr_dev = reinterpret_cast<PriorSpec*>(cube_dev + ncube);
    CUDA_TRY(cudaMemcpyAsync(cube_dev, cube, sizeof(double) * ncube, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaMemcpyAsync(pr_dev, priors, sizeof(PriorSpec) * ncol, cudaMemcpyHostToDevice, c->stream));
    prior_transform_kernel<<<(B + 127) / 128, 128, 0, c->stream>>>(pr_dev, ncol, B, cube_dev, theta_dev, tstride);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}
extern "C" int pioran_prior_transform(pioran_ctx* c, int ncol, const pioran_prior_spec* priors, int B, const double* cube,
                                      double* theta_out) try {
    if (is_group(c)) return pioran_prior_transform(c->children[0], ncol, priors, B, cube, theta_out);
    if (!c || !priors || !cube || !theta_out) return fail(PIORAN_EINVAL, "NULL argument");
    if (B < 1) return fail(PIORAN_EINVAL, "B must be >= 1");
    PIORAN_COMPUTE_LOCK(c);
    CUDA_TRY(cudaSetDevice(c->device));
    int rc;
    if ((rc = c->theta.ensure(sizeof(double) * (size_t)B * PRIOR_MAX_COLS))) return rc;
    if ((rc = prior_transform_dev_locked(c, ncol, priors, B, cube, c->theta.as<double>(), ncol))) return rc;
    CUDA_TRY(cudaMemcpyAsync(theta_out, c->theta.p, sizeof(double) * (size_t)B * ncol, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return PIORAN_OK;
} catch (...) { return guard_fail(); }
extern "C" int pioran_prior_transform_logl(pioran_ctx* c, int series_id, const pioran_approx_spec* spec, int ncol,
                                           const pioran_prior_spec* priors, int B, const double* cube, double* theta_out,
                                           double* logl_out) try {
    if (!c || !spec || !priors || !cube || !logl_out) return fail(PIORAN_EINVAL, "NULL argument");
    if (B < 1) return fail(PIORAN_EINVAL, "B must be >= 1");
    if (is_group(c))
        return group_fanout(c, series_id, B, [&](pioran_ctx* ch, int id, int64_t, int beg, int nb) {
            return pioran_prior_transform_logl(ch, id, spec, ncol, priors, nb, cube + (size_t)beg * ncol, at(theta_out, (size_t)beg * ncol),
                                               logl_out + beg);
        });
    const int npar = n_psd_par_of(spec->psd_model);
    if (npar < 0) return fail(PIORAN_EINVAL, "unknown psd_model %d", spec->psd_model);
    if (ncol != npar + 3) return fail(PIORAN_EINVAL, "ncol must be %d (psd parameters, norm, nu, mu) for this model, got %d", npar + 3, ncol);
    PIORAN_COMPUTE_LOCK(c);
    CUDA_TRY(cudaSetDevice(c->device));
    int rc;
    if ((rc = c->theta.ensure(sizeof(double) * (size_t)B * ncol))) return rc;
    if ((rc = c->out.ensure(sizeof(double) * (size_t)B))) return rc;
    if ((rc = prior_transform_dev_locked(c, ncol, priors, B, cube, c->theta.as<double>(), ncol))) return rc;
    if ((rc = approx_logl_dev_locked(c, 1, &series_id, spec, B, c->theta.as<double>(), 0, c->out.as<double>()))) return rc;
    if (theta_out) CUDA_TRY(cudaMemcpyAsync(theta_out, c->theta.p, sizeof(double) * (size_t)B * ncol, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(logl_out, c->out.p, sizeof(double) * (size_t)B, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

// ------------------------------------------------------------------------------------------------ gradient entry (K5)
constexpr int GRAD_NW = 8;
template <int BS, int NW>
static int launch_grad_nw(pioran_ctx* c, const GradArgs& args, int nitems) {
    auto kern = celerite_grad_kernel<BS, NW>;
    const size_t smem = grad_smem_bytes<BS, NW>();
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaEventRecord(c->ev_beg, c->stream);
    kern<<<nitems, NW * 32, smem, c->stream>>>(args);
    cudaEventRecord(c->ev_end, c->stream);
    note_kernel(c, KF_GRAD, BS, NW);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}
template <int BS, int NWARPS>
static int launch_grad_pipe(pioran_ctx* c, const GradArgs& args, int nitems) {
    constexpr int RPS = rps_of(BS), SD = table_step_doubles(RPS), nthreads = NWARPS * 32;
    auto kern = celerite_grad_pipe_kernel<BS, NWARPS>;
    const size_t smem = sizeof(double) * (2 * (size_t)PIPE_CS * SD + 3 * (size_t)pipe_slot_doubles<BS>() +
                                          (size_t)(args.ND + 1) * 2 * RPS + 2) + 2 * sizeof(uint64_t) + 16;
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaEventRecord(c->ev_beg, c->stream);
    kern<<<nitems, nthreads, smem, c->stream>>>(args);
    cudaEventRecord(c->ev_end, c->stream);
    note_kernel(c, KF_GRAD_PIPE, BS, NWARPS);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}
// a few chains (≤ 4 (θ, direction) pairs per CTA): one warp per SM sub-partition, as for the likelihood (SMALL_NW)
template <int BS>
static int launch_grad(pioran_ctx* c, const GradArgs& args, int nitems, int tpi) {
    return tpi <= SMALL_NW ? launch_grad_nw<BS, SMALL_NW>(c, args, nitems) : launch_grad_nw<BS, GRAD_NW>(c, args, nitems);
}
// K5t (blocked_grad.cuh): one CTA per parameter vector, value warp + one tangent warp per direction, all on the tensor pipe
template <int NT, int NTR, bool HALF, int NTAN>
static int launch_blocked_grad(pioran_ctx* c, const GradArgs& args, int nitems, int R, int amp_stride) {
    auto kern = celerite_blocked_grad_kernel<NT, NTR, HALF, NTAN>;
    const size_t smem = sizeof(double) * ((size_t)BLK_NSTAGE * blk_doubles(NT, NTR) + 2 * (size_t)blk_slot_doubles(NTR) +
                                          (size_t)(1 + NTAN) * (8 * NTR + 8 * NT) + 2) + BLK_NSTAGE * sizeof(uint64_t) + 16;
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaEventRecord(c->ev_beg, c->stream);
    kern<<<nitems, (1 + NTAN) * 32, smem, c->stream>>>(args, R, amp_stride, blk_layout(R, true).RG, blk_layout(R, true).RM);
    cudaEventRecord(c->ev_end, c->stream);
    note_kernel(c, KF_BLOCKED_GRAD, NT, NTR, HALF, NTAN);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}
template <int NTAN>
static int dispatch_blocked_grad(pioran_ctx* c, const GradArgs& a, int nitems, int R, int amp_stride) {
    const BlkLayout lay = blk_layout(R, true);
    const int NT = lay.NT;
    const bool xrow = lay.NTR != NT, half = lay.half;
#define PIORAN_BLKG_CASE(nt)                                                                                    \
    case nt: return xrow ? launch_blocked_grad<nt, nt + 1, false, NTAN>(c, a, nitems, R, amp_stride)            \
                  : half ? launch_blocked_grad<nt, nt, true, NTAN>(c, a, nitems, R, amp_stride)                 \
                         : launch_blocked_grad<nt, nt, false, NTAN>(c, a, nitems, R, amp_stride);
    switch (NT) {
        PIORAN_BLKG_CASE(1) PIORAN_BLKG_CASE(2) PIORAN_BLKG_CASE(3) PIORAN_BLKG_CASE(4)
        PIORAN_BLKG_CASE(5) PIORAN_BLKG_CASE(6) PIORAN_BLKG_CASE(7)
        case 8:
            if (xrow) break;
            return half ? launch_blocked_grad<8, 8, true, NTAN>(c, a, nitems, R, amp_stride)
                        : launch_blocked_grad<8, 8, false, NTAN>(c, a, nitems, R, amp_stride);
    }
#undef PIORAN_BLKG_CASE
    return fail(PIORAN_EUNSUPPORTED, "rank %d not served by the blocked gradient kernel", R);
}
static bool blocked_grad_enabled(const pioran_ctx* c, int R, int ND) {
    return blocked_enabled(c, R) && blk_layout(R, true).NTR <= 8 && (ND == 3 || ND == 5);
}

// logshift: θ rows carry a further column c and (y_batch, s2_batch) hold the per-θ transformed data; the gradient gains ∂/∂c.
// Gradient at ranks 65 … 96 (wide_grad.cuh): K1 tangents in row form, then one CTA per (parameter vector, direction).
static int wide_grad_locked(pioran_ctx* c, Series* ser, const pioran_approx_spec* spec, int B, const double* theta_dev,
                            double* logl_dev, double* grad_dev, int R, int npar, int ts) {
    int rc;
    const int ND = npar, J = spec->n_components, TS = std::max(5, (R + 15) / 16), RP = 16 * TS;
    const int Jt = spec->basis == PIORAN_BASIS_SHO ? J : 2 * J;
    ApproxPlan* plan;
    if ((rc = get_plan(c, *spec, &plan))) return rc;
    // term tables (θ-independent on the approx path): src/psd.jl:250 (c = d = √2 π f, b = a) and :266-271 (c = π f, d = √3 c, b = √3 a; 2c)
    std::vector<double> hv(3 * (size_t)Jt);
    std::vector<int> hrow(Jt);
    const double f0 = spec->f_min / spec->S_low, fM = spec->f_max * spec->S_high;
    for (int j = 0; j < J; j++) {
        const double fj = f0 * std::pow(fM / f0, (double)j / (double)(J - 1));
        if (spec->basis == PIORAN_BASIS_SHO) {
            hv[j] = hv[Jt + j] = std::sqrt(2.0) * M_PI * fj; hv[2 * Jt + j] = 1.0; hrow[j] = 2 * j;
        } else {
            const double cj = M_PI * fj;
            hv[j] = cj; hv[Jt + j] = std::sqrt(3.0) * cj; hv[2 * Jt + j] = std::sqrt(3.0); hrow[j] = 2 * j;
            hv[J + j] = 2.0 * cj; hv[Jt + J + j] = 0.0; hv[2 * Jt + J + j] = 0.0; hrow[J + j] = -(2 * J + j + 1);
        }
    }
    // workspace: amp [B×RP] | damp [B×ND×RP] | Σa [B] | dΣa [B×ND] | c, d, ρ [3·Jt] | term rows [Jt ints]
    const size_t n_amp = (size_t)B * RP, n_damp = (size_t)B * ND * RP;
    if ((rc = c->gradws.ensure(sizeof(double) * (n_amp + n_damp + (size_t)B + (size_t)B * ND + 3 * (size_t)Jt) + sizeof(int) * (size_t)(Jt + 2)))) return rc;
    double* amp = c->gradws.as<double>();
    double* damp = amp + n_amp;
    double* suma = damp + n_damp;
    double* dsuma = suma + B;
    double* tv = dsuma + (size_t)B * ND;
    int* trow = reinterpret_cast<int*>(tv + 3 * (size_t)Jt);
    std::vector<WorkItem> items(B, WorkItem{});
    for (int i = 0; i < B; i++) {
        WorkItem& w = items[i];
        w.t = ser->t; w.y = ser->y; w.s2 = ser->s2; w.N = ser->N;
        w.theta_begin = i; w.par_begin = i; w.count = 1; w.out_begin = i; w.n_begin = 0; w.n_end = ser->N;
    }
    c->gwork_key.clear();
    if ((rc = c->gwork.ensure(sizeof(WorkItem) * items.size()))) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->gwork.p, items.data(), sizeof(WorkItem) * items.size(), cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaMemcpyAsync(tv, hv.data(), sizeof(double) * hv.size(), cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaMemcpyAsync(trow, hrow.data(), sizeof(int) * hrow.size(), cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));      // the sources are locals
    const int nthr = B * ND;
    cudaEventRecord(c->ev_beg, c->stream);
    approx_grad_kernel<<<(nthr + 127) / 128, 128, 0, c->stream>>>(plan, B, theta_dev, ts, amp, damp, RP, suma, dsuma);
    WideGradArgs ga{};
    ga.work = c->gwork.as<WorkItem>();
    ga.amp = amp; ga.damp = damp; ga.suma = suma; ga.dsuma = dsuma;
    ga.c = tv; ga.d = tv + Jt; ga.rho = tv + 2 * Jt; ga.term_row = trow;
    ga.Jt = Jt; ga.R = R; ga.RP = RP; ga.ND = ND;
    ga.theta = theta_dev; ga.pstride = ts; ga.logl = logl_dev; ga.grad = grad_dev;
    if (TS == 5) celerite_wide_grad_kernel<5><<<B * (ND + 1), WIDE_THREADS, 0, c->stream>>>(ga);
    else celerite_wide_grad_kernel<6><<<B * (ND + 1), WIDE_THREADS, 0, c->stream>>>(ga);
    cudaEventRecord(c->ev_end, c->stream);
    note_kernel(c, KF_WIDE_GRAD, TS == 5 ? 5 : 6);
    c->launches += 2;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

static int approx_logl_grad_dev_locked(pioran_ctx* c, int series_id, const pioran_approx_spec* spec, int B,
                                       const double* theta_dev, double* logl_dev, double* grad_dev, bool logshift = false,
                                       const double* y_batch = nullptr, const double* s2_batch = nullptr) {
    int rc;
    if (B < 1) return fail(PIORAN_EINVAL, "B must be >= 1");
    if ((rc = check_spec(*spec))) return rc;
    Series* ser = get_series(c, series_id);
    if (!ser) return fail(PIORAN_EINVAL, "unknown series id %d", series_id);
    const int npar = n_psd_par_of(spec->psd_model), ts = npar + 3 + (logshift ? 1 : 0), ND = npar, P = ts;
    if ((long long)B * P > 0x7fffffffLL / 64) return fail(PIORAN_EINVAL, "B too large");
    const int R = rank_of(spec->basis, spec->n_components);
    const int BS = bs_for_rank(R);
    if (BS > 8) {
        if (R > 96 || logshift || y_batch || s2_batch)
            return fail(PIORAN_EUNSUPPORTED, "gradients are built for ranks <= 96 (log-shift model: <= 62); rank %d", R);
        return wide_grad_locked(c, ser, spec, B, theta_dev, logl_dev, grad_dev, R, npar, ts);
    }
    const int RP = G * BS;
    const bool blkg = blocked_grad_enabled(c, R, ND);
    if (logshift && !(blkg && ND == 3))
        return fail(PIORAN_EUNSUPPORTED, "the log-shift gradient is built for SingleBendingPowerLaw at ranks <= 62 (rank %d, %d PSD parameters)", R, ND);
    Table tab;
    if ((rc = blkg ? get_btable(c, ser, *spec, &tab, true) : get_table(c, ser, *spec, &tab))) return rc;
    ApproxPlan* plan;
    if ((rc = get_plan(c, *spec, &plan))) return rc;
    // workspace: amp [B×RP] | damp [B×ND×RP] | Σa [B] | dΣa [B×ND]
    const size_t n_amp = (size_t)B * RP, n_damp = (size_t)B * ND * RP;
    if ((rc = c->gradws.ensure(sizeof(double) * (n_amp + n_damp + (size_t)B + (size_t)B * ND)))) return rc;
    double* amp = c->gradws.as<double>();
    double* damp = amp + n_amp;
    double* suma = damp + n_damp;
    double* dsuma = suma + B;
    const int nthr = B * ND;
    approx_grad_kernel<<<(nthr + 127) / 128, 128, 0, c->stream>>>(plan, B, theta_dev, ts, amp, damp, RP, suma, dsuma);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    // one warp per (θ, direction): the work items run over the virtual batch of B·(n_psd_par + 1) entries
    const bool pipe = blkg || BS >= 6;   // one CTA per parameter vector: value warp + tangent-only warps (blocked_grad.cuh, grad_pipe.cuh)
    const int PW = pipe ? 1 : ND + 1;    // work-item entries per parameter vector (warps: psd parameters…, ν; ∂/∂μ rides along,
                                         // ∂/∂norm follows from ∂/∂ν)
    const std::vector<int64_t> key = {(int64_t)(intptr_t)tab.d, (int64_t)(intptr_t)ser->t, ser->N, (int64_t)B * PW, BS, (int64_t)pipe + 2 * (int64_t)blkg};
    if (key != c->gwork_key) {
        ItemPlan ip;
        Series* sp[1] = {ser};
        plan_items(c, 1, sp, &tab, B * PW, pipe ? 1 : GRAD_NW, false, ip);
        c->gwork_key.clear();
        if ((rc = c->gwork.ensure(sizeof(WorkItem) * ip.items.size()))) return rc;
        CUDA_TRY(cudaMemcpyAsync(c->gwork.p, ip.items.data(), sizeof(WorkItem) * ip.items.size(), cudaMemcpyHostToDevice,
                                 c->stream));
        CUDA_TRY(cudaStreamSynchronize(c->stream));   // ip.items is a local; only when the call shape changes
        c->gwork_key = key;
        c->gwork_items = (int)ip.items.size();
        c->gwork_tpi = ip.tpi;
    }
    GradArgs ga{};
    ga.work = c->gwork.as<WorkItem>();
    ga.amp = amp; ga.damp = damp; ga.suma = suma; ga.dsuma = dsuma;
    ga.theta = theta_dev; ga.pstride = ts; ga.ND = ND;
    ga.logl = logl_dev; ga.grad = grad_dev;
    ga.y_batch = y_batch; ga.s2_batch = s2_batch; ga.ystride = ser->N; ga.cdir = logshift ? 1 : 0;
    const int nitems = c->gwork_items;
    if (blkg && logshift) return dispatch_blocked_grad<5>(c, ga, nitems, R, RP);
    if (blkg) return ND == 3 ? dispatch_blocked_grad<4>(c, ga, nitems, R, RP) : dispatch_blocked_grad<6>(c, ga, nitems, R, RP);
    if (pipe) {
        const int nwarps = 1 + ND + 1;
        if (nwarps == 5) {
            switch (BS) {
                case 6: return launch_grad_pipe<6, 5>(c, ga, nitems);
                case 7: return launch_grad_pipe<7, 5>(c, ga, nitems);
                case 8: return launch_grad_pipe<8, 5>(c, ga, nitems);
            }
        } else if (nwarps == 7) {
            switch (BS) {
                case 6: return launch_grad_pipe<6, 7>(c, ga, nitems);
                case 7: return launch_grad_pipe<7, 7>(c, ga, nitems);
                case 8: return launch_grad_pipe<8, 7>(c, ga, nitems);
            }
        }
        return fail(PIORAN_EUNSUPPORTED, "no gradient kernel for %d PSD parameters", ND);
    }
    switch (BS) {
        case 4: return launch_grad<4>(c, ga, nitems, c->gwork_tpi);
        case 5: return launch_grad<5>(c, ga, nitems, c->gwork_tpi);
    }
    return fail(PIORAN_EUNSUPPORTED, "block size %d not compiled", BS);
}

// Gradient of the log-normal likelihood (docs/src/ultranest.md:197-217 differentiated like every other model of the reference,
// test/test_likelihood.jl:55): transform on the device, then K1 tangents + the blocked gradient kernel with per-θ data and the
// extra direction c.
extern "C" int pioran_approx_logl_logshift_grad(pioran_ctx* c, int series_id, const pioran_approx_spec* spec, int B,
                                                const double* theta, double* logl_out, double* grad_out) try {
    if (!c || !spec || !theta || !grad_out) return fail(PIORAN_EINVAL, "NULL argument");
    if (B < 1) return fail(PIORAN_EINVAL, "B must be >= 1");
    const int npar = n_psd_par_of(spec->psd_model);
    if (npar < 0) return fail(PIORAN_EINVAL, "unknown psd_model %d", spec->psd_model);
    const int ts = npar + 4;
    if (is_group(c))
        return group_fanout(c, series_id, B, [&](pioran_ctx* ch, int id, int64_t, int beg, int nb) {
            return pioran_approx_logl_logshift_grad(ch, id, spec, nb, theta + (size_t)beg * ts, at(logl_out, beg), grad_out + (size_t)beg * ts);
        });
    PIORAN_COMPUTE_LOCK(c);
    CUDA_TRY(cudaSetDevice(c->device));
    int rc;
    if ((rc = check_spec(*spec))) return rc;
    Series* s = get_series(c, series_id);
    if (!s) return fail(PIORAN_EINVAL, "unknown series id %d", series_id);
    if ((rc = c->theta.ensure(sizeof(double) * (size_t)B * ts))) return rc;
    if ((rc = c->out.ensure(sizeof(double) * (size_t)B * (ts + 1)))) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->theta.p, theta, sizeof(double) * (size_t)B * ts, cudaMemcpyHostToDevice, c->stream));
    double* gl = c->out.as<double>();
    double* gg = gl + B;
    if ((rc = logshift_chunks(c, s, B, ts, [&](int off, int nb, const double* th, const double* yb, const double* sb) {
             return approx_logl_grad_dev_locked(c, series_id, spec, nb, th, gl + off, gg + (size_t)off * ts, true, yb, sb);
         })))
        return rc;
    if (logl_out) CUDA_TRY(cudaMemcpyAsync(logl_out, gl, sizeof(double) * (size_t)B, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(grad_out, gg, sizeof(double) * (size_t)B * ts, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return PIORAN_OK;
} catch (...) { return guard_fail(); }


extern "C" int pioran_approx_logl_grad_dev(pioran_ctx* c, int series_id, const pioran_approx_spec* spec, int B,
                                           const double* theta_dev, double* logl_dev, double* grad_dev) try {
    if (is_group(c)) return fail(PIORAN_EUNSUPPORTED, "device-resident entries need a single-device context (a group spans devices)");
    if (!c || !spec || !theta_dev || !grad_dev) return fail(PIORAN_EINVAL, "NULL argument");
    PIORAN_COMPUTE_LOCK(c);
    CUDA_TRY(cudaSetDevice(c->device));
    return approx_logl_grad_dev_locked(c, series_id, spec, B, theta_dev, logl_dev, grad_dev);
} catch (...) { return guard_fail(); }

extern "C" int pioran_approx_logl_grad(pioran_ctx* c, int series_id, const pioran_approx_spec* spec, int B,
                                       const double* theta, double* logl_out, double* grad_out) try {
    if (!c || !spec || !theta || !grad_out) return fail(PIORAN_EINVAL, "NULL argument");
    if (B < 1) return fail(PIORAN_EINVAL, "B must be >= 1");
    const int npar = n_psd_par_of(spec->psd_model);
    if (npar < 0) return fail(PIORAN_EINVAL, "unknown psd_model %d", spec->psd_model);
    const int P = npar + 3;
    if (is_group(c))
        return group_fanout(c, series_id, B, [&](pioran_ctx* ch, int id, int64_t, int beg, int nb) {
            return pioran_approx_logl_grad(ch, id, spec, nb, theta + (size_t)beg * P, at(logl_out, beg), grad_out + (size_t)beg * P);
        });
    PIORAN_COMPUTE_LOCK(c);
    CUDA_TRY(cudaSetDevice(c->device));
    int rc;
    if ((rc = c->theta.ensure(sizeof(double) * (size_t)B * P))) return rc;
    if ((rc = c->out.ensure(sizeof(double) * (size_t)B * (P + 1)))) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->theta.p, theta, sizeof(double) * (size_t)B * P, cudaMemcpyHostToDevice, c->stream));
    double* gl = c->out.as<double>();
    double* gg = gl + B;
    if ((rc = approx_logl_grad_dev_locked(c, series_id, spec, B, c->theta.as<double>(), gl, gg))) return rc;
    if (logl_out) CUDA_TRY(cudaMemcpyAsync(logl_out, gl, sizeof(double) * (size_t)B, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(grad_out, gg, sizeof(double) * (size_t)B * P, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

// ------------------------------------------------------------------------------------------------ generic entry
// Uploads [B×Jt] coefficient arrays and per-θ scalars; returns device pointers inside ctx workspaces.
struct GenericInputs { double *a, *b, *c, *d, *mu, *nu, *yb, *sb; };
static int upload_generic(pioran_ctx* c, int B, int Jt, int64_t N, const double* a, const double* b, const double* cc,
                          const double* d, const double* mu, const double* nu, const double* y_batch,
                          const double* s2_batch, GenericInputs& gi) {
    int rc;
    const size_t n = (size_t)B * Jt;
    if ((rc = c->coef.ensure(sizeof(double) * (4 * n + 2 * (size_t)B)))) return rc;
    double* base = c->coef.as<double>();
    gi.a = base; gi.b = base + n; gi.c = base + 2 * n; gi.d = base + 3 * n;
    gi.mu = mu ? base + 4 * n : nullptr;
    gi.nu = nu ? base + 4 * n + B : nullptr;
    CUDA_TRY(cudaMemcpyAsync(gi.a, a, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaMemcpyAsync(gi.b, b, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaMemcpyAsync(gi.c, cc, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaMemcpyAsync(gi.d, d, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
    if (mu) CUDA_TRY(cudaMemcpyAsync(gi.mu, mu, sizeof(double) * B, cudaMemcpyHostToDevice, c->stream));
    if (nu) CUDA_TRY(cudaMemcpyAsync(gi.nu, nu, sizeof(double) * B, cudaMemcpyHostToDevice, c->stream));
    gi.yb = gi.sb = nullptr;
    const size_t ny = (size_t)B * N;
    if (y_batch || s2_batch) {
        if ((rc = c->misc.ensure(sizeof(double) * 2 * ny))) return rc;
        if (y_batch) {
            gi.yb = c->misc.as<double>();
            CUDA_TRY(cudaMemcpyAsync(gi.yb, y_batch, sizeof(double) * ny, cudaMemcpyHostToDevice, c->stream));
        }
        if (s2_batch) {
            gi.sb = c->misc.as<double>() + ny;
            CUDA_TRY(cudaMemcpyAsync(gi.sb, s2_batch, sizeof(double) * ny, cudaMemcpyHostToDevice, c->stream));
        }
    }
    return 0;
}

// The start of every explicit-coefficient entry; the caller holds the context's lock.  Looks the series up, reduces the rank
// (make_term_rows) and enforces the entry's rank limit: limit_fmt is formatted with the rank, Jt and max_rank as %1$d, %2$d
// and %3$d.  The caller uploads the coefficients (upload_generic): the likelihood first decides whether the scan path runs,
// and the posterior variance uploads one θ-chunk at a time.
struct ExplicitSet { Series* s = nullptr; std::vector<int> term_row; int R = 0; };
static const char* const LOGL_LIMIT = "rank %1$d (Jt = %2$d) exceeds this build's limit of %3$d";
static const char* const POSTERIOR_LIMIT = "rank %1$d (Jt = %2$d) exceeds the limit of %3$d of the posterior mean and the draws";
static int explicit_front(pioran_ctx* c, int series_id, int B, int Jt, const double* b, const double* d, int max_rank,
                          const char* limit_fmt, ExplicitSet& x) {
    CUDA_TRY(cudaSetDevice(c->device));
    x.s = get_series(c, series_id);
    if (!x.s) return fail(PIORAN_EINVAL, "unknown series id %d", series_id);
    x.R = make_term_rows(B, Jt, b, d, x.term_row);
    if (x.R > max_rank) return fail(PIORAN_EUNSUPPORTED, limit_fmt, x.R, Jt, max_rank);
    return 0;
}

// Row map and work items of the generic kernel (one CTA per parameter vector at wide ranks) for uploaded coefficients, and the
// launch arguments.  term_row may be the map of a larger batch this call is a θ-chunk of.
static int generic_setup(pioran_ctx* c, Series* s, int B, int Jt, const std::vector<int>& term_row, int R, const GenericInputs& gi,
                         BatchArgs& args, int& nitems, int& tpi) {
    int rc;
    if ((rc = c->rows.ensure(sizeof(int) * (Jt + 1)))) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->rows.p, term_row.data(), sizeof(int) * Jt, cudaMemcpyHostToDevice, c->stream));
    if ((rc = c->out.ensure(sizeof(double) * (size_t)B))) return rc;
    ItemPlan ip;
    const int BS = bs_for_rank(R);
    plan_items(c, 1, &s, nullptr, B, BS > 8 ? 1 : nw_for_bs(BS), false, ip);
    c->work_key.clear();  // the work buffer is shared with the fused path's cached plan
    if ((rc = c->work.ensure(sizeof(WorkItem) * ip.items.size()))) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->work.p, ip.items.data(), sizeof(WorkItem) * ip.items.size(), cudaMemcpyHostToDevice,
                             c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));   // term_row and ip are host sources
    nitems = (int)ip.items.size();
    tpi = ip.tpi;
    args = BatchArgs{};
    args.work = c->work.as<WorkItem>();
    args.a = gi.a; args.b = gi.b; args.c = gi.c; args.d = gi.d;
    args.Jt = Jt;
    args.term_row = c->rows.as<int>();
    args.R = R;
    args.mu = gi.mu; args.nu = gi.nu; args.pstride = 1;
    args.y_batch = gi.yb; args.s2_batch = gi.sb; args.ystride = s->N;
    args.out = c->out.as<double>();
    return 0;
}

// The sequential sweep on explicit coefficients (generic K2, K2w above rank 64) for the set-up of explicit_front; the context
// is locked by the caller.
static int generic_logl_locked(pioran_ctx* c, const ExplicitSet& x, int B, int Jt, const double* a, const double* b, const double* cc,
                               const double* d, const double* mu, const double* nu, const double* y_batch,
                               const double* s2_batch, double* logl_out) {
    Series* s = x.s;
    const int R = x.R;
    const std::vector<int>& term_row = x.term_row;
    int rc;
    GenericInputs gi;
    if ((rc = upload_generic(c, B, Jt, s->N, a, b, cc, d, mu, nu, y_batch, s2_batch, gi))) return rc;
    // Small batches at ranks <= 63, and 65 … 128 with the one-CTA-per-evaluation kernel (the B = 1 call a `:celerite_gpu` solver symbol makes per logpdf, a CARMA or QPO sampler's few
    // hundred points): per-θ block tables are built by a parallel kernel and every parameter vector runs the tensor-pipe sweep as a
    // one-warp item (0.48 ms per 1 000 steps) instead of building its trig/exp chunks inside a scalar-pipe sweep (1.2–1.8 ms).
    {
        const BlkLayout lay = blk_layout(R, false);
        const int64_t nblocks = (s->N + BLK - 1) / BLK;
        const size_t tbytes = sizeof(double) * (size_t)nblocks * blk_doubles(lay.NT, lay.NTR);
        if ((blocked_enabled(c, R) || blocked_wide_enabled(c, R)) && B <= 4 * c->num_sms && tbytes * (size_t)B <= ((size_t)2 << 30)) {
            const int RPT = 8 * lay.NTR, RPA = 8 * lay.NT;
            std::vector<BlkRowMap> prow(RPT, BlkRowMap{ROW_PAD, -1, 0});
            std::vector<int> lrow_term(std::max(R, 1), 0);
            for (int m = 0; m < Jt; m++) {
                const int tr = term_row[m];
                if (tr < 0) { const int lr = -tr - 1; prow[blk_phys_row(lr, R)] = BlkRowMap{ROW_REAL, m, lr}; lrow_term[lr] = m; }
                else {
                    prow[blk_phys_row(tr, R)] = BlkRowMap{ROW_COS, m, tr};
                    prow[blk_phys_row(tr + 1, R)] = BlkRowMap{ROW_SIN, m, tr + 1};
                    lrow_term[tr] = m; lrow_term[tr + 1] = m;
                }
            }
            prow[lay.RG] = BlkRowMap{ROW_AUG, -1, 0};
            const size_t meta = sizeof(BlkRowMap) * RPT + sizeof(int) * R;
            if ((rc = c->rows.ensure(meta))) return rc;
            if ((rc = c->post.ensure(tbytes * (size_t)B))) return rc;
            if ((rc = c->amp.ensure(sizeof(double) * (size_t)B * RPA))) return rc;
            if ((rc = c->suma.ensure(sizeof(double) * (size_t)B))) return rc;
            if ((rc = c->out.ensure(sizeof(double) * (size_t)B))) return rc;
            if ((rc = c->work.ensure(sizeof(WorkItem) * (size_t)B))) return rc;
            BlkRowMap* prow_d = c->rows.as<BlkRowMap>();
            int* lrow_d = reinterpret_cast<int*>(prow_d + RPT);
            double* tables = c->post.as<double>();
            const int64_t tstride = nblocks * blk_doubles(lay.NT, lay.NTR);
            std::vector<WorkItem> items(B);
            for (int i = 0; i < B; i++) {
                WorkItem w{};
                w.table = tables + (size_t)i * tstride;
                w.t = s->t; w.y = s->y; w.s2 = s->s2; w.N = s->N;
                w.theta_begin = i; w.par_begin = i; w.count = 1; w.out_begin = i;
                w.n_begin = 0; w.n_end = s->N; w.init = nullptr; w.part = nullptr;
                items[i] = w;
            }
            c->work_key.clear();
            CUDA_TRY(cudaMemcpyAsync(prow_d, prow.data(), sizeof(BlkRowMap) * RPT, cudaMemcpyHostToDevice, c->stream));
            CUDA_TRY(cudaMemcpyAsync(lrow_d, lrow_term.data(), sizeof(int) * R, cudaMemcpyHostToDevice, c->stream));
            CUDA_TRY(cudaMemcpyAsync(c->work.p, items.data(), sizeof(WorkItem) * (size_t)B, cudaMemcpyHostToDevice, c->stream));
            CUDA_TRY(cudaMemsetAsync(tables, 0, tbytes * (size_t)B, c->stream));
            const int64_t total = (int64_t)B * nblocks * RPT;
            blocked_table_theta_kernel<<<(unsigned)((total + 127) / 128), 128, 0, c->stream>>>(tables, tstride, B, s->t, s->y, s->s2, s->N,
                                                                                             nblocks, gi.a, gi.b, gi.c, gi.d, Jt, prow_d,
                                                                                             lay.NT, lay.NTR);
            blocked_amp_theta_kernel<<<(B + 127) / 128, 128, 0, c->stream>>>(c->amp.as<double>(), c->suma.as<double>(), B, RPA, R, gi.a,
                                                                            gi.b, Jt, lrow_d);
            c->launches += 2;
            CUDA_TRY(cudaGetLastError());
            CUDA_TRY(cudaStreamSynchronize(c->stream));      // prow, lrow_term and items are locals
            BatchArgs args{};
            args.work = c->work.as<WorkItem>();
            args.amp = c->amp.as<double>(); args.suma = c->suma.as<double>();
            args.mu = gi.mu; args.nu = gi.nu; args.pstride = 1;
            args.y_batch = gi.yb; args.s2_batch = gi.sb; args.ystride = s->N;
            args.out = c->out.as<double>();
            if ((rc = (R > 64 || (small_cta_enabled() && blk_nt(R) >= 4)) ? dispatch_blocked_wide(c, args, B, R, RPA) : dispatch_blocked(c, args, B, 1, R, RPA))) return rc;
            CUDA_TRY(cudaMemcpyAsync(logl_out, c->out.p, sizeof(double) * (size_t)B, cudaMemcpyDeviceToHost, c->stream));
            CUDA_TRY(cudaStreamSynchronize(c->stream));
            return PIORAN_OK;
        }
    }
    BatchArgs args;
    int nitems, tpi;
    if ((rc = generic_setup(c, s, B, Jt, term_row, R, gi, args, nitems, tpi))) return rc;
    const int BS = bs_for_rank(R);
    if ((rc = BS > 8 ? launch_wide(c, args, nitems) : dispatch_generic(c, BS, args, nitems, tpi))) return rc;
    CUDA_TRY(cudaMemcpyAsync(logl_out, c->out.p, sizeof(double) * (size_t)B, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return PIORAN_OK;
}

extern "C" int pioran_celerite_logl(pioran_ctx* c, int series_id, int B, int Jt, const double* a, const double* b,
                                    const double* cc, const double* d, const double* mu, const double* nu,
                                    const double* y_batch, const double* s2_batch, double* logl_out) try {
    if (!c || !a || !b || !cc || !d || !logl_out) return fail(PIORAN_EINVAL, "NULL argument");
    if (B < 1 || Jt < 1) return fail(PIORAN_EINVAL, "B and Jt must be >= 1");
    if (is_group(c))
        return group_fanout(c, series_id, B, [&](pioran_ctx* ch, int id, int64_t N, int beg, int nb) {
            const size_t o = (size_t)beg * Jt;
            return pioran_celerite_logl(ch, id, nb, Jt, a + o, b + o, cc + o, d + o, at(mu, beg), at(nu, beg), at(y_batch, beg * N),
                                        at(s2_batch, beg * N), logl_out + beg);
        });
    PIORAN_COMPUTE_LOCK(c);
    ExplicitSet x;
    int rc;
    if ((rc = explicit_front(c, series_id, B, Jt, b, d, WIDE_MAX_RANK, LOGL_LIMIT, x))) return rc;
    if (!y_batch && !s2_batch && auto_scan(c, x.s->N, B, x.R, true))
        return scan_logl_locked(c, x.s, series_id, B, Jt, a, b, cc, d, mu, nu, logl_out);
    return generic_logl_locked(c, x, B, Jt, a, b, cc, d, mu, nu, y_batch, s2_batch, logl_out);
} catch (...) { return guard_fail(); }


// ------------------------------------------------------------------------------------------------ PSD features (QPO)
// approx() of a continuum + QPO features (src/psd.jl:15-44, 221-243, 254-259, 277-282): K1 emits the Jt continuum terms followed
// by one celerite term per feature; their decay rates and frequencies depend on θ, so the sweep is the generic kernel.
static int approx_features_dev(pioran_ctx* c, const pioran_approx_spec* spec, int nf, int B, const double* theta, int ts,
                               int feat_off, int* Jout) {
    int rc;
    if ((rc = check_spec(*spec))) return rc;
    if (nf < 1 || nf > MAXFEAT) return fail(PIORAN_EINVAL, "n_features must be in [1, %d] (got %d)", MAXFEAT, nf);
    ApproxPlan* plan;
    if ((rc = get_plan(c, *spec, &plan))) return rc;
    const int Jt = (spec->basis == PIORAN_BASIS_SHO ? spec->n_components : 2 * spec->n_components) + nf;
    if ((rc = c->theta.ensure(sizeof(double) * (size_t)B * ts))) return rc;
    if ((rc = c->coef.ensure(sizeof(double) * (size_t)B * Jt * 4))) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->theta.p, theta, sizeof(double) * (size_t)B * ts, cudaMemcpyHostToDevice, c->stream));
    double* da = c->coef.as<double>();
    const size_t n = (size_t)B * Jt;
    approx_kernel<<<(B + 127) / 128, 128, 0, c->stream>>>(plan, B, c->theta.as<double>(), ts, da, da + n, da + 2 * n, da + 3 * n,
                                                         nullptr, 0, nullptr, nf, feat_off);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    *Jout = Jt;
    return 0;
}

extern "C" int pioran_approx_coeffs_features(pioran_ctx* c, const pioran_approx_spec* spec, int n_features, int B,
                                             const double* theta, double* a, double* b, double* cc, double* d) try {
    if (!c || !spec || !theta || !a || !b || !cc || !d) return fail(PIORAN_EINVAL, "NULL argument");
    if (B < 1) return fail(PIORAN_EINVAL, "B must be >= 1");
    if (is_group(c)) return pioran_approx_coeffs_features(c->children[0], spec, n_features, B, theta, a, b, cc, d);
    PIORAN_COMPUTE_LOCK(c);
    CUDA_TRY(cudaSetDevice(c->device));
    const int npar = n_psd_par_of(spec->psd_model);
    if (npar < 0) return fail(PIORAN_EINVAL, "unknown psd_model %d", spec->psd_model);
    int Jt, rc;
    if ((rc = approx_features_dev(c, spec, n_features, B, theta, npar + 1 + 3 * n_features, npar + 1, &Jt))) return rc;
    const size_t n = (size_t)B * Jt;
    const double* da = c->coef.as<double>();
    CUDA_TRY(cudaMemcpyAsync(a, da, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(b, da + n, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(cc, da + 2 * n, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(d, da + 3 * n, sizeof(double) * n, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

extern "C" int pioran_approx_features_logl(pioran_ctx* c, int series_id, const pioran_approx_spec* spec, int n_features, int B,
                                           const double* theta, double* logl_out) try {
    if (!c || !spec || !theta || !logl_out) return fail(PIORAN_EINVAL, "NULL argument");
    if (B < 1) return fail(PIORAN_EINVAL, "B must be >= 1");
    const int npar = n_psd_par_of(spec->psd_model);
    if (npar < 0) return fail(PIORAN_EINVAL, "unknown psd_model %d", spec->psd_model);
    const int ts = npar + 3 + 3 * n_features;
    if (is_group(c))
        return group_fanout(c, series_id, B, [&](pioran_ctx* ch, int id, int64_t, int beg, int nb) {
            return pioran_approx_features_logl(ch, id, spec, n_features, nb, theta + (size_t)beg * ts, logl_out + beg);
        });
    PIORAN_COMPUTE_LOCK(c);
    CUDA_TRY(cudaSetDevice(c->device));
    Series* s = get_series(c, series_id);
    if (!s) return fail(PIORAN_EINVAL, "unknown series id %d", series_id);
    int Jt, rc;
    if ((rc = approx_features_dev(c, spec, n_features, B, theta, ts, npar + 3, &Jt))) return rc;
    // coefficients back to the host (B × Jt × 4 doubles: a few hundred KB for a sampler's batch), then the generic sweep
    const size_t n = (size_t)B * Jt;
    std::vector<double> co(4 * n), mu(B), nu(B);
    CUDA_TRY(cudaMemcpyAsync(co.data(), c->coef.p, sizeof(double) * 4 * n, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    for (int i = 0; i < B; i++) { nu[i] = theta[(size_t)i * ts + npar + 1]; mu[i] = theta[(size_t)i * ts + npar + 2]; }
    ExplicitSet x;
    if ((rc = explicit_front(c, series_id, B, Jt, co.data() + n, co.data() + 3 * n, WIDE_MAX_RANK, LOGL_LIMIT, x))) return rc;
    return generic_logl_locked(c, x, B, Jt, co.data(), co.data() + n, co.data() + 2 * n, co.data() + 3 * n, mu.data(), nu.data(),
                               nullptr, nullptr, logl_out);
} catch (...) { return guard_fail(); }

// ------------------------------------------------------------------------------------------------ K5g: JVP on explicit coefficients
// Shared by pioran_celerite_logl_jvp and pioran_approx_features_logl_grad: `ja` holds the device pointers of the inputs and
// outputs (B parameter vectors, P directions); the series, term rows and shape are filled in here.  The context is locked by
// the caller; R <= JVP_MAX_RANK.
static int jvp_dev_locked(pioran_ctx* c, Series* s, int B, int Jt, int P, int R, const std::vector<int>& term_row, JvpArgs ja) {
    int rc;
    if ((rc = c->rows.ensure(sizeof(int) * (Jt + 1)))) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->rows.p, term_row.data(), sizeof(int) * Jt, cudaMemcpyHostToDevice, c->stream));
    ja.t = s->t; ja.y = s->y; ja.s2 = s->s2; ja.N = s->N;
    ja.term_row = c->rows.as<int>();
    ja.Jt = Jt; ja.P = P;
    const int TS = std::max(1, (R + 15) / 16);
    const unsigned grid = (unsigned)B * (unsigned)P;
    cudaEventRecord(c->ev_beg, c->stream);
    if ((rc = with_int<1, 6>(TS, [&](auto ts) { celerite_jvp_kernel<ts><<<grid, WIDE_THREADS, 0, c->stream>>>(ja); return 0; }))) return rc;
    cudaEventRecord(c->ev_end, c->stream);
    note_kernel(c, KF_JVP, TS);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    // term_row is the caller's host vector: the copy must have left it before the caller may drop it
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return 0;
}

extern "C" int pioran_celerite_logl_jvp(pioran_ctx* c, int series_id, int B, int Jt, int P, const double* a, const double* b,
                                        const double* cc, const double* d, const double* mu, const double* nu,
                                        const double* y_batch, const double* s2_batch, const double* da, const double* db,
                                        const double* dc, const double* dd, const double* dmu, const double* dnu,
                                        const double* dy, const double* ds2, double* logl_out, double* dlogl_out) try {
    if (!c || !a || !b || !cc || !d || !dlogl_out) return fail(PIORAN_EINVAL, "NULL argument");
    if (B < 1 || Jt < 1) return fail(PIORAN_EINVAL, "B and Jt must be >= 1");
    if (P < 1) return fail(PIORAN_EINVAL, "P must be >= 1 (got %d)", P);
    if ((long long)B * P > 0x7fffffffLL) return fail(PIORAN_EINVAL, "B * P too large");
    if (is_group(c))
        return group_fanout(c, series_id, B, [&](pioran_ctx* ch, int id, int64_t N, int beg, int nb) {
            const size_t o = (size_t)beg * Jt, op = (size_t)beg * P;
            return pioran_celerite_logl_jvp(ch, id, nb, Jt, P, a + o, b + o, cc + o, d + o, at(mu, beg), at(nu, beg), at(y_batch, beg * N),
                                            at(s2_batch, beg * N), at(da, op * Jt), at(db, op * Jt), at(dc, op * Jt), at(dd, op * Jt),
                                            at(dmu, op), at(dnu, op), at(dy, op * N), at(ds2, op * N), at(logl_out, beg), dlogl_out + op);
        });
    PIORAN_COMPUTE_LOCK(c);
    ExplicitSet x;
    int rc;
    if ((rc = explicit_front(c, series_id, B, Jt, b, d, JVP_MAX_RANK, "the JVP is built for ranks <= %3$d (rank %1$d, Jt = %2$d)", x))) return rc;
    GenericInputs gi;
    const int64_t N = x.s->N;
    if ((rc = upload_generic(c, B, Jt, N, a, b, cc, d, mu, nu, y_batch, s2_batch, gi))) return rc;
    // coefficient tangents [B × P × Jt] each, then dμ, dν [B × P]
    const size_t nt = (size_t)B * P * Jt, np = (size_t)B * P;
    if ((rc = c->gradws.ensure(sizeof(double) * (4 * nt + 2 * np)))) return rc;
    double* tb = c->gradws.as<double>();
    const double* hsrc[6] = {da, db, dc, dd, dmu, dnu};
    double* dsrc[6] = {tb, tb + nt, tb + 2 * nt, tb + 3 * nt, tb + 4 * nt, tb + 4 * nt + np};
    for (int q = 0; q < 6; q++) {
        if (!hsrc[q]) { dsrc[q] = nullptr; continue; }
        CUDA_TRY(cudaMemcpyAsync(dsrc[q], hsrc[q], sizeof(double) * (q < 4 ? nt : np), cudaMemcpyHostToDevice, c->stream));
    }
    if ((rc = c->out.ensure(sizeof(double) * (size_t)B * (P + 1)))) return rc;
    double* gl = c->out.as<double>();
    double* gg = gl + B;
    // data tangents [B × P × N]: θ-chunks of at most 1 GiB for dy and ds2 together
    const bool dt = dy || ds2;
    const int chunk = dt ? theta_chunk(B, 16 * (size_t)P * N) : B;
    const size_t nc = (size_t)chunk * P * N;
    if (dt && (rc = c->post.ensure(sizeof(double) * 2 * nc))) return rc;
    for (int off = 0; off < B; off += chunk) {
        const int nb = std::min(chunk, B - off);
        const size_t o = (size_t)off * Jt, op = (size_t)off * P, nd = (size_t)nb * P * N;
        JvpArgs ja{};
        ja.a = gi.a + o; ja.b = gi.b + o; ja.c = gi.c + o; ja.d = gi.d + o;
        ja.mu = at(gi.mu, off); ja.nu = at(gi.nu, off);
        ja.y_batch = at(gi.yb, (size_t)off * N); ja.s2_batch = at(gi.sb, (size_t)off * N);
        ja.da = at(dsrc[0], op * Jt); ja.db = at(dsrc[1], op * Jt); ja.dc = at(dsrc[2], op * Jt); ja.dd = at(dsrc[3], op * Jt);
        ja.dmu = at(dsrc[4], op); ja.dnu = at(dsrc[5], op);
        if (dy) {
            ja.dy = c->post.as<double>();
            CUDA_TRY(cudaMemcpyAsync(c->post.p, dy + op * N, sizeof(double) * nd, cudaMemcpyHostToDevice, c->stream));
        }
        if (ds2) {
            ja.ds2 = c->post.as<double>() + nc;
            CUDA_TRY(cudaMemcpyAsync(c->post.as<double>() + nc, ds2 + op * N, sizeof(double) * nd, cudaMemcpyHostToDevice, c->stream));
        }
        ja.logl = gl + off; ja.dlogl = gg + op;
        if ((rc = jvp_dev_locked(c, x.s, nb, Jt, P, x.R, x.term_row, ja))) return rc;
    }
    if (logl_out) CUDA_TRY(cudaMemcpyAsync(logl_out, gl, sizeof(double) * (size_t)B, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(dlogl_out, gg, sizeof(double) * np, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

// Gradients with PSD features, in forward mode (one K5g sweep with P = θ columns) and in reverse mode (one K5r sweep and the
// contraction kernel): K1 on pairs (approx_features_grad_kernel) writes the coefficients (co: a, b, c, d [B × Jt], μ, ν [B]) and
// their tangents along every θ column (tg: [B × P × Jt] each, then [B × P] each) in the JVP's device layout.  Nothing returns
// to the host in between.  features_grad_check validates what the group split needs; features_grad_setup runs under the
// caller's lock.
struct FeatureGrad { Series* s = nullptr; int Jt = 0, R = 0, P = 0; std::vector<int> term_row; double *co = nullptr, *tg = nullptr; };
static int features_grad_check(pioran_ctx* c, const pioran_approx_spec* spec, int n_features, int B, const double* theta,
                               const double* grad_out, int& ts) {
    if (!c || !spec || !theta || !grad_out) return fail(PIORAN_EINVAL, "NULL argument");
    if (B < 1) return fail(PIORAN_EINVAL, "B must be >= 1");
    const int npar = n_psd_par_of(spec->psd_model);
    if (npar < 0) return fail(PIORAN_EINVAL, "unknown psd_model %d", spec->psd_model);
    if (n_features < 1) return fail(PIORAN_EINVAL, "n_features must be >= 1 (got %d)", n_features);
    if (n_features > MAXFEAT) return fail(PIORAN_EUNSUPPORTED, "at most %d features (got %d)", MAXFEAT, n_features);
    ts = npar + 3 + 3 * n_features;
    if ((long long)B * ts > 0x7fffffffLL) return fail(PIORAN_EINVAL, "B too large");
    return 0;
}
static int features_grad_setup(pioran_ctx* c, int series_id, const pioran_approx_spec* spec, int nf, int B, const double* theta,
                               int ts, int max_rank, FeatureGrad& f) {
    CUDA_TRY(cudaSetDevice(c->device));
    int rc;
    if ((rc = check_spec(*spec))) return rc;
    f.s = get_series(c, series_id);
    if (!f.s) return fail(PIORAN_EINVAL, "unknown series id %d", series_id);
    const int J = spec->n_components;
    const int Jc = spec->basis == PIORAN_BASIS_SHO ? J : 2 * J, Rc = rank_of(spec->basis, J);
    f.Jt = Jc + nf; f.R = Rc + 2 * nf; f.P = ts;
    if (f.R > max_rank) return fail(PIORAN_EUNSUPPORTED, "gradients with features are built for ranks <= %d (rank %d)", max_rank, f.R);
    ApproxPlan* plan;
    if ((rc = get_plan(c, *spec, &plan))) return rc;
    // term rows: continuum as in the approx path (SHO complex; DRWCelerite complex ++ real), features complex
    f.term_row.assign(f.Jt + 1, 0);
    for (int j = 0; j < J; j++) {
        f.term_row[j] = 2 * j;
        if (spec->basis != PIORAN_BASIS_SHO) f.term_row[J + j] = -(2 * J + j + 1);
    }
    for (int q = 0; q < nf; q++) f.term_row[Jc + q] = Rc + 2 * q;
    const size_t n = (size_t)B * f.Jt, nt = (size_t)B * f.P * f.Jt, np = (size_t)B * f.P;
    if ((rc = c->theta.ensure(sizeof(double) * (size_t)B * ts))) return rc;
    if ((rc = c->coef.ensure(sizeof(double) * (4 * n + 2 * (size_t)B)))) return rc;
    if ((rc = c->gradws.ensure(sizeof(double) * (4 * nt + 2 * np)))) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->theta.p, theta, sizeof(double) * (size_t)B * ts, cudaMemcpyHostToDevice, c->stream));
    double* co = f.co = c->coef.as<double>();
    double* tg = f.tg = c->gradws.as<double>();
    approx_features_grad_kernel<<<(unsigned)((np + 127) / 128), 128, 0, c->stream>>>(
        plan, B, c->theta.as<double>(), ts, nf, ts - 3 * nf, co, co + n, co + 2 * n, co + 3 * n, co + 4 * n, co + 4 * n + B,
        tg, tg + nt, tg + 2 * nt, tg + 3 * nt, tg + 4 * nt, tg + 4 * nt + np);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int pioran_approx_features_logl_grad(pioran_ctx* c, int series_id, const pioran_approx_spec* spec, int n_features,
                                                int B, const double* theta, double* logl_out, double* grad_out) try {
    int ts, rc;
    if ((rc = features_grad_check(c, spec, n_features, B, theta, grad_out, ts))) return rc;
    if (is_group(c))
        return group_fanout(c, series_id, B, [&](pioran_ctx* ch, int id, int64_t, int beg, int nb) {
            return pioran_approx_features_logl_grad(ch, id, spec, n_features, nb, theta + (size_t)beg * ts, at(logl_out, beg),
                                                    grad_out + (size_t)beg * ts);
        });
    PIORAN_COMPUTE_LOCK(c);
    FeatureGrad f;
    if ((rc = features_grad_setup(c, series_id, spec, n_features, B, theta, ts, JVP_MAX_RANK, f))) return rc;
    const int Jt = f.Jt, P = f.P;
    const size_t n = (size_t)B * Jt, nt = (size_t)B * P * Jt, np = (size_t)B * P;
    if ((rc = c->out.ensure(sizeof(double) * (size_t)B * (P + 1)))) return rc;
    double* gl = c->out.as<double>();
    double* gg = gl + B;
    const double *co = f.co, *tg = f.tg;
    JvpArgs ja{};
    ja.a = co; ja.b = co + n; ja.c = co + 2 * n; ja.d = co + 3 * n; ja.mu = co + 4 * n; ja.nu = co + 4 * n + B;
    ja.da = tg; ja.db = tg + nt; ja.dc = tg + 2 * nt; ja.dd = tg + 3 * nt; ja.dmu = tg + 4 * nt; ja.dnu = tg + 4 * nt + np;
    ja.logl = gl; ja.dlogl = gg;
    if ((rc = jvp_dev_locked(c, f.s, B, Jt, P, f.R, f.term_row, ja))) return rc;
    if (logl_out) CUDA_TRY(cudaMemcpyAsync(logl_out, gl, sizeof(double) * (size_t)B, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(grad_out, gg, sizeof(double) * np, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

// ------------------------------------------------------------------------------------------------ K5r: VJP on explicit coefficients
// Shared by pioran_celerite_logl_vjp and pioran_approx_features_logl_grad_reverse.  `base` holds the device pointers of the
// inputs and outputs for all B sets (gy, gs2 ignored); the batch runs in θ-chunks whose workspace stays under the context's cap
// (1 GiB unless pioran_ctx_set_vjp_workspace says otherwise).  gy_host / gs2_host [B × N] (or NULL) receive the data gradients
// chunk by chunk.  The context is locked by the caller; R <= VJP_MAX_RANK.
static int vjp_dev_locked(pioran_ctx* c, Series* s, int B, int Jt, int R, const std::vector<int>& term_row, const VjpArgs& base,
                          double* gy_host, double* gs2_host) {
    int rc;
    const int64_t N = s->N;
    const int TS = std::max(1, (R + 15) / 16);
    if (TS > 6) return fail(PIORAN_EUNSUPPORTED, "the VJP is built for ranks <= %d (rank %d)", VJP_MAX_RANK, R);
    // K ≈ √N steps per checkpoint segment minimises the ⌈N/K⌉ + K tiles kept per set
    int64_t K = (int64_t)std::ceil(std::sqrt((double)N));
    K = (K + WIDE_CH - 1) / WIDE_CH * WIDE_CH;
    const size_t per = sizeof(double) * vjp_ws_doubles(TS, N, (int)K);
    const int chunk = c->vjp_ws_bytes ? theta_chunk(B, per, c->vjp_ws_bytes) : theta_chunk(B, per);
    if ((rc = c->vjpws.ensure(per * (size_t)chunk))) return rc;
    if ((rc = c->rows.ensure(sizeof(int) * (Jt + 1)))) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->rows.p, term_row.data(), sizeof(int) * Jt, cudaMemcpyHostToDevice, c->stream));
    const size_t nd = (size_t)chunk * N;
    if ((gy_host || gs2_host) && (rc = c->post.ensure(sizeof(double) * 2 * nd))) return rc;
    for (int off = 0; off < B; off += chunk) {
        const int nb = std::min(chunk, B - off);
        const size_t o = (size_t)off * Jt, on = (size_t)off * N;
        VjpArgs va = base;
        va.t = s->t; va.y = s->y; va.s2 = s->s2; va.N = N;
        va.term_row = c->rows.as<int>(); va.Jt = Jt; va.K = (int)K; va.ws = c->vjpws.as<double>();
        va.a = base.a + o; va.b = base.b + o; va.c = base.c + o; va.d = base.d + o;
        va.mu = at(base.mu, off); va.nu = at(base.nu, off);
        va.y_batch = at(base.y_batch, on); va.s2_batch = at(base.s2_batch, on);
        va.logl = at(base.logl, off);
        va.ga = at(base.ga, o); va.gb = at(base.gb, o); va.gc = at(base.gc, o); va.gd = at(base.gd, o);
        va.gmu = at(base.gmu, off); va.gnu = at(base.gnu, off);
        va.gy = gy_host ? c->post.as<double>() : nullptr;
        va.gs2 = gs2_host ? c->post.as<double>() + nd : nullptr;
        cudaEventRecord(c->ev_beg, c->stream);
        with_int<1, 6>(TS, [&](auto ts) { celerite_vjp_kernel<ts><<<nb, WIDE_THREADS, 0, c->stream>>>(va); return 0; });
        cudaEventRecord(c->ev_end, c->stream);
        note_kernel(c, KF_VJP, TS);
        c->launches++;
        CUDA_TRY(cudaGetLastError());
        if (gy_host) CUDA_TRY(cudaMemcpyAsync(gy_host + on, va.gy, sizeof(double) * nb * N, cudaMemcpyDeviceToHost, c->stream));
        if (gs2_host) CUDA_TRY(cudaMemcpyAsync(gs2_host + on, va.gs2, sizeof(double) * nb * N, cudaMemcpyDeviceToHost, c->stream));
    }
    // term_row is the caller's host vector: the copy must have left it before the caller may drop it
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return 0;
}

extern "C" int pioran_celerite_logl_vjp(pioran_ctx* c, int series_id, int B, int Jt, const double* a, const double* b,
                                        const double* cc, const double* d, const double* mu, const double* nu,
                                        const double* y_batch, const double* s2_batch, double* logl_out, double* ga, double* gb,
                                        double* gc, double* gd, double* gmu, double* gnu, double* gy, double* gs2) try {
    if (!c || !a || !b || !cc || !d) return fail(PIORAN_EINVAL, "NULL argument");
    if (!ga && !gb && !gc && !gd && !gmu && !gnu && !gy && !gs2) return fail(PIORAN_EINVAL, "no gradient output given");
    if (B < 1 || Jt < 1) return fail(PIORAN_EINVAL, "B and Jt must be >= 1");
    if (is_group(c))
        return group_fanout(c, series_id, B, [&](pioran_ctx* ch, int id, int64_t N, int beg, int nb) {
            const size_t o = (size_t)beg * Jt, on = (size_t)beg * N;
            return pioran_celerite_logl_vjp(ch, id, nb, Jt, a + o, b + o, cc + o, d + o, at(mu, beg), at(nu, beg), at(y_batch, on),
                                            at(s2_batch, on), at(logl_out, beg), at(ga, o), at(gb, o), at(gc, o), at(gd, o), at(gmu, beg),
                                            at(gnu, beg), at(gy, on), at(gs2, on));
        });
    PIORAN_COMPUTE_LOCK(c);
    ExplicitSet x;
    int rc;
    if ((rc = explicit_front(c, series_id, B, Jt, b, d, VJP_MAX_RANK, "the VJP is built for ranks <= %3$d (rank %1$d, Jt = %2$d)", x))) return rc;
    GenericInputs gi;
    if ((rc = upload_generic(c, B, Jt, x.s->N, a, b, cc, d, mu, nu, y_batch, s2_batch, gi))) return rc;
    // logL [B], ā … d̄ [B × Jt] each, μ̄, ν̄ [B]
    const size_t n = (size_t)B * Jt;
    if ((rc = c->out.ensure(sizeof(double) * (3 * (size_t)B + 4 * n)))) return rc;
    double* ob = c->out.as<double>();
    VjpArgs base{};
    base.a = gi.a; base.b = gi.b; base.c = gi.c; base.d = gi.d; base.mu = gi.mu; base.nu = gi.nu;
    base.y_batch = gi.yb; base.s2_batch = gi.sb;
    base.logl = ob; base.ga = ob + B; base.gb = ob + B + n; base.gc = ob + B + 2 * n; base.gd = ob + B + 3 * n;
    base.gmu = ob + B + 4 * n; base.gnu = ob + 2 * B + 4 * n;
    if ((rc = vjp_dev_locked(c, x.s, B, Jt, x.R, x.term_row, base, gy, gs2))) return rc;
    double* hdst[7] = {logl_out, ga, gb, gc, gd, gmu, gnu};
    const double* dsrc[7] = {base.logl, base.ga, base.gb, base.gc, base.gd, base.gmu, base.gnu};
    for (int q = 0; q < 7; q++)
        if (hdst[q]) CUDA_TRY(cudaMemcpyAsync(hdst[q], dsrc[q], sizeof(double) * (q >= 1 && q <= 4 ? n : (size_t)B), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

extern "C" int pioran_approx_features_logl_grad_reverse(pioran_ctx* c, int series_id, const pioran_approx_spec* spec, int n_features,
                                                        int B, const double* theta, double* logl_out, double* grad_out) try {
    int ts, rc;
    if ((rc = features_grad_check(c, spec, n_features, B, theta, grad_out, ts))) return rc;
    if (is_group(c))
        return group_fanout(c, series_id, B, [&](pioran_ctx* ch, int id, int64_t, int beg, int nb) {
            return pioran_approx_features_logl_grad_reverse(ch, id, spec, n_features, nb, theta + (size_t)beg * ts, at(logl_out, beg),
                                                            grad_out + (size_t)beg * ts);
        });
    PIORAN_COMPUTE_LOCK(c);
    FeatureGrad f;
    if ((rc = features_grad_setup(c, series_id, spec, n_features, B, theta, ts, VJP_MAX_RANK, f))) return rc;
    const int Jt = f.Jt, P = f.P;
    const size_t n = (size_t)B * Jt, nt = (size_t)B * P * Jt, np = (size_t)B * P;
    // logL [B], ā … d̄ [B × Jt] each, μ̄, ν̄ [B], ∂logL/∂θ [B × P]
    if ((rc = c->out.ensure(sizeof(double) * (3 * (size_t)B + 4 * n + np)))) return rc;
    double* ob = c->out.as<double>();
    const double *co = f.co, *tg = f.tg;
    VjpArgs base{};
    base.a = co; base.b = co + n; base.c = co + 2 * n; base.d = co + 3 * n; base.mu = co + 4 * n; base.nu = co + 4 * n + B;
    base.logl = ob; base.ga = ob + B; base.gb = ob + B + n; base.gc = ob + B + 2 * n; base.gd = ob + B + 3 * n;
    base.gmu = ob + B + 4 * n; base.gnu = ob + 2 * B + 4 * n;
    if ((rc = vjp_dev_locked(c, f.s, B, Jt, f.R, f.term_row, base, nullptr, nullptr))) return rc;
    double* gg = ob + 3 * (size_t)B + 4 * n;
    vjp_contract_kernel<<<(unsigned)((np + 127) / 128), 128, 0, c->stream>>>(
        B, P, Jt, base.ga, base.gb, base.gc, base.gd, base.gmu, base.gnu, tg, tg + nt, tg + 2 * nt, tg + 3 * nt, tg + 4 * nt,
        tg + 4 * nt + np, gg);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    if (logl_out) CUDA_TRY(cudaMemcpyAsync(logl_out, ob, sizeof(double) * (size_t)B, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(grad_out, gg, sizeof(double) * np, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

extern "C" int pioran_ctx_set_vjp_workspace(pioran_ctx* c, long long bytes) try {
    if (is_group(c)) return group_each(c, [&](pioran_ctx* ch) { return pioran_ctx_set_vjp_workspace(ch, bytes); });
    if (!c) return fail(PIORAN_EINVAL, "ctx is NULL");
    if (bytes < 0) return fail(PIORAN_EINVAL, "bytes must be >= 0 (0 = 1 GiB)");
    std::lock_guard<std::mutex> lk(c->mu);
    c->vjp_ws_bytes = (size_t)bytes;
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

// ------------------------------------------------------------------------------------------------ posterior mean, draws
// n₀ = searchsortedfirst(t, τ) − 1 (celerite_solver.jl:395): the series lives on the device, fetch its times once
static int prediction_gaps(pioran_ctx* c, const Series* s, int64_t M, const double* tau, std::vector<int>& n0) {
    std::vector<double> th(s->N);
    CUDA_TRY(cudaMemcpyAsync(th.data(), s->t, sizeof(double) * s->N, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    n0.resize(M);
    for (int64_t m = 0; m < M; m++) n0[m] = (int)(std::lower_bound(th.begin(), th.end(), tau[m]) - th.begin());
    return 0;
}
// backsolve and predict kernels of the posterior mean on a stored factor
static void launch_posterior_mean(pioran_ctx* c, const PostArgs& pa) {
    if (pa.Jt <= 64) {
        celerite_backsolve_kernel<2><<<(pa.B + 3) / 4, 128, 0, c->stream>>>(pa);
        celerite_predict_kernel<2><<<(pa.B + 3) / 4, 128, 0, c->stream>>>(pa);
    } else {
        celerite_backsolve_kernel<4><<<(pa.B + 3) / 4, 128, 0, c->stream>>>(pa);
        celerite_predict_kernel<4><<<(pa.B + 3) / 4, 128, 0, c->stream>>>(pa);
    }
    c->launches += 2;
}

extern "C" int pioran_celerite_predict(pioran_ctx* c, int series_id, int B, int Jt, const double* a, const double* b,
                                       const double* cc, const double* d, const double* mu, const double* nu, int64_t M,
                                       const double* tau, double* mean_out) try {
    if (is_group(c))
        return group_first(c, series_id, [&](pioran_ctx* ch, int id) { return pioran_celerite_predict(ch, id, B, Jt, a, b, cc, d, mu, nu, M, tau, mean_out); });
    if (!c || !a || !b || !cc || !d || !tau || !mean_out) return fail(PIORAN_EINVAL, "NULL argument");
    if (B < 1 || Jt < 1 || M < 1) return fail(PIORAN_EINVAL, "B, Jt and M must be >= 1");
    for (int64_t m = 1; m < M; m++)
        if (!(tau[m] >= tau[m - 1])) return fail(PIORAN_EINVAL, "tau must be ascending (tau[%lld] < tau[%lld])", (long long)m, (long long)m - 1);
    PIORAN_COMPUTE_LOCK(c);
    ExplicitSet x;
    int rc, nitems, tpi;
    if ((rc = explicit_front(c, series_id, B, Jt, b, d, 128, POSTERIOR_LIMIT, x))) return rc;
    Series* s = x.s;
    const int64_t N = s->N;
    std::vector<int> n0;
    if ((rc = prediction_gaps(c, s, M, tau, n0))) return rc;
    GenericInputs gi;
    BatchArgs args;
    if ((rc = upload_generic(c, B, Jt, N, a, b, cc, d, mu, nu, nullptr, nullptr, gi))) return rc;
    if ((rc = generic_setup(c, s, B, Jt, x.term_row, x.R, gi, args, nitems, tpi))) return rc;
    const int BS = bs_for_rank(x.R), RPL = stored_factor_ld(x.R);
    // workspace: W [B·N·RPL] | D [B·N] | z [B·N] | mean [B·M] | tau [M] | n0 [M ints]
    const size_t nW = (size_t)B * N * RPL, nBN = (size_t)B * N, nBM = (size_t)B * M;
    if ((rc = c->post.ensure(sizeof(double) * (nW + 2 * nBN + nBM + M) + sizeof(int) * (M + 2)))) return rc;
    double* W = c->post.as<double>();
    double* D = W + nW;
    double* z = D + nBN;
    double* mean = z + nBN;
    double* tau_dev = mean + nBM;
    int* n0_dev = reinterpret_cast<int*>(tau_dev + M);
    CUDA_TRY(cudaMemcpyAsync(tau_dev, tau, sizeof(double) * M, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaMemcpyAsync(n0_dev, n0.data(), sizeof(int) * M, cudaMemcpyHostToDevice, c->stream));
    args.W_out = W; args.D_out = D; args.zf_out = z;
    cudaEventRecord(c->ev_beg, c->stream);
    if ((rc = BS > 8 ? launch_wide<STEP_STORE>(c, args, nitems) : dispatch_generic_mode<STEP_STORE>(c, BS, args, nitems))) return rc;
    PostArgs pa{};
    pa.t = s->t; pa.tau = tau_dev; pa.n0 = n0_dev; pa.N = N; pa.M = M; pa.B = B; pa.Jt = Jt; pa.RPL = RPL;
    pa.a = gi.a; pa.b = gi.b; pa.c = gi.c; pa.d = gi.d; pa.term_row = c->rows.as<int>(); pa.mu = gi.mu;
    pa.W = W; pa.D = D; pa.z = z; pa.mean = mean;
    launch_posterior_mean(c, pa);
    cudaEventRecord(c->ev_end, c->stream);
    note_kernel(c, KF_PREDICT, Jt <= 64 ? 2 : 4);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(mean_out, mean, sizeof(double) * nBM, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));   // n0 is a local
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

extern "C" int pioran_celerite_simulate(pioran_ctx* c, int series_id, int B, int Jt, const double* a, const double* b,
                                        const double* cc, const double* d, const double* nu, const double* q,
                                        double* y_out) try {
    if (is_group(c))
        return group_first(c, series_id, [&](pioran_ctx* ch, int id) { return pioran_celerite_simulate(ch, id, B, Jt, a, b, cc, d, nu, q, y_out); });
    if (!c || !a || !b || !cc || !d || !q || !y_out) return fail(PIORAN_EINVAL, "NULL argument");
    if (B < 1 || Jt < 1) return fail(PIORAN_EINVAL, "B and Jt must be >= 1");
    PIORAN_COMPUTE_LOCK(c);
    ExplicitSet x;
    int rc, nitems, tpi;
    if ((rc = explicit_front(c, series_id, B, Jt, b, d, 128, POSTERIOR_LIMIT, x))) return rc;
    GenericInputs gi;
    BatchArgs args;
    if ((rc = upload_generic(c, B, Jt, x.s->N, a, b, cc, d, nullptr, nu, q, nullptr, gi))) return rc;
    if ((rc = generic_setup(c, x.s, B, Jt, x.term_row, x.R, gi, args, nitems, tpi))) return rc;
    const int BS = bs_for_rank(x.R);
    const size_t nBN = (size_t)B * x.s->N;
    if ((rc = c->post.ensure(sizeof(double) * nBN))) return rc;
    args.ysim_out = c->post.as<double>();
    cudaEventRecord(c->ev_beg, c->stream);
    if ((rc = BS > 8 ? launch_wide<STEP_SIM>(c, args, nitems) : dispatch_generic_mode<STEP_SIM>(c, BS, args, nitems))) return rc;
    cudaEventRecord(c->ev_end, c->stream);
    if (BS > 8) note_kernel(c, KF_WIDE_REG_SIM, std::max(5, (args.R + 15) / 16));
    else note_kernel(c, KF_GENERIC_SIM, BS, nw_for_bs(BS));
    CUDA_TRY(cudaMemcpyAsync(y_out, c->post.p, sizeof(double) * nBN, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

// ------------------------------------------------------------------------------------------------ posterior variance (K6)
static int launch_postvar(pioran_ctx* c, const PostVarArgs& pv, int B) {
    const int TS = (pv.R + 15) / 16;
    int rc;
    if ((rc = with_int<1, 8>(TS, [&](auto ts) { celerite_postvar_kernel<ts><<<B, WIDE_THREADS, 0, c->stream>>>(pv); return 0; }))) return rc;
    c->launches++;
    note_kernel(c, KF_POSTVAR, TS);
    CUDA_TRY(cudaGetLastError());
    return 0;
}

extern "C" int pioran_celerite_predict_var(pioran_ctx* c, int series_id, int B, int Jt, const double* a, const double* b,
                                           const double* cc, const double* d, const double* mu, const double* nu, int64_t M,
                                           const double* tau, double* mean_out, double* var_out) try {
    if (is_group(c))
        return group_first(c, series_id, [&](pioran_ctx* ch, int id) {
            return pioran_celerite_predict_var(ch, id, B, Jt, a, b, cc, d, mu, nu, M, tau, mean_out, var_out);
        });
    if (!c || !a || !b || !cc || !d || !tau || !var_out) return fail(PIORAN_EINVAL, "NULL argument");
    if (B < 1 || Jt < 1 || M < 1) return fail(PIORAN_EINVAL, "B, Jt and M must be >= 1");
    for (int64_t m = 1; m < M; m++)
        if (!(tau[m] >= tau[m - 1])) return fail(PIORAN_EINVAL, "tau must be ascending (tau[%lld] < tau[%lld])", (long long)m, (long long)m - 1);
    PIORAN_COMPUTE_LOCK(c);
    ExplicitSet x;   // the row map of the whole batch, shared by every θ-chunk
    int rc;
    if ((rc = explicit_front(c, series_id, B, Jt, b, d, 128, "rank %1$d (Jt = %2$d) exceeds the limit of %3$d of the posterior variance", x)))
        return rc;
    Series* s = x.s;
    const int R = x.R;
    const int64_t N = s->N;
    std::vector<int> n0;
    if ((rc = prediction_gaps(c, s, M, tau, n0))) return rc;

    // θ-chunks of at most 1 GiB: per set W [N·RPL] | D [N] | z [N] | mean [M] | g_τ, D_τ [M·(R + 1)] | var [M]
    const int RPL = stored_factor_ld(R);
    const size_t per_set = sizeof(double) * ((size_t)N * RPL + 2 * (size_t)N + (size_t)M * (R + 3));
    const int Bc = theta_chunk(B, per_set);
    if ((rc = c->post.ensure(per_set * Bc + sizeof(double) * M + sizeof(int) * (M + 2)))) return rc;
    double* W = c->post.as<double>();
    double* D = W + (size_t)Bc * N * RPL;
    double* z = D + (size_t)Bc * N;
    double* mean = z + (size_t)Bc * N;
    double* ws = mean + (size_t)Bc * M;
    double* var = ws + (size_t)Bc * M * (R + 1);
    double* tau_dev = var + (size_t)Bc * M;
    int* n0_dev = reinterpret_cast<int*>(tau_dev + M);
    CUDA_TRY(cudaMemcpyAsync(tau_dev, tau, sizeof(double) * M, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaMemcpyAsync(n0_dev, n0.data(), sizeof(int) * M, cudaMemcpyHostToDevice, c->stream));
    cudaEventRecord(c->ev_beg, c->stream);
    for (int b0 = 0; b0 < B; b0 += Bc) {
        const int Bk = std::min(Bc, B - b0);
        const size_t o = (size_t)b0 * Jt;
        int nitems, tpi;
        GenericInputs gi;
        BatchArgs args;
        if ((rc = upload_generic(c, Bk, Jt, N, a + o, b + o, cc + o, d + o, at(mu, b0), at(nu, b0), nullptr, nullptr, gi))) return rc;
        if ((rc = generic_setup(c, s, Bk, Jt, x.term_row, R, gi, args, nitems, tpi))) return rc;
        const int BS = bs_for_rank(R);
        args.W_out = W; args.D_out = D; args.zf_out = z;
        // the factor of pioran_celerite_predict, and its backsolve and predict kernels: mean_out is predict's, bit for bit
        if ((rc = BS > 8 ? launch_wide<STEP_STORE>(c, args, nitems) : dispatch_generic_mode<STEP_STORE>(c, BS, args, nitems))) return rc;
        if (mean_out) {
            PostArgs pa{};
            pa.t = s->t; pa.tau = tau_dev; pa.n0 = n0_dev; pa.N = N; pa.M = M; pa.B = Bk; pa.Jt = Jt; pa.RPL = RPL;
            pa.a = gi.a; pa.b = gi.b; pa.c = gi.c; pa.d = gi.d; pa.term_row = c->rows.as<int>(); pa.mu = gi.mu;
            pa.W = W; pa.D = D; pa.z = z; pa.mean = mean;
            launch_posterior_mean(c, pa);
            CUDA_TRY(cudaGetLastError());
        }
        PostVarArgs pv{};
        pv.t = s->t; pv.tau = tau_dev; pv.n0 = n0_dev; pv.N = N; pv.M = M; pv.Jt = Jt; pv.R = R; pv.RPL = RPL;
        pv.a = gi.a; pv.b = gi.b; pv.c = gi.c; pv.d = gi.d; pv.term_row = c->rows.as<int>();
        pv.W = W; pv.D = D; pv.ws = ws; pv.var = var;
        if ((rc = launch_postvar(c, pv, Bk))) return rc;
        if (mean_out)
            CUDA_TRY(cudaMemcpyAsync(mean_out + (size_t)b0 * M, mean, sizeof(double) * (size_t)Bk * M, cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(cudaMemcpyAsync(var_out + (size_t)b0 * M, var, sizeof(double) * (size_t)Bk * M, cudaMemcpyDeviceToHost, c->stream));
    }
    cudaEventRecord(c->ev_end, c->stream);
    CUDA_TRY(cudaStreamSynchronize(c->stream));   // n0 is a local
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

// ------------------------------------------------------------------------------------------------ K3 / K4 entries
// Rank reduction shared by the generic and the scan entry: a term that is real (b = d = 0) for every coefficient set of
// the batch needs one row, not two.  term_row[m] ≥ 0: complex term at rows (v, v+1); < 0: real term at row −v−1.
static int make_term_rows(int B, int Jt, const double* b, const double* d, std::vector<int>& term_row) {
    term_row.assign(Jt + 1, 0);
    int R = 0;
    for (int m = 0; m < Jt; m++) {
        bool real = true;
        for (int i = 0; i < B && real; i++) real = (b[(size_t)i * Jt + m] == 0.0 && d[(size_t)i * Jt + m] == 0.0);
        term_row[m] = real ? -(R + 1) : R;
        R += real ? 1 : 2;
    }
    return R;
}

extern "C" int pioran_ctx_set_auto_scan(pioran_ctx* c, int enabled) try {
    if (is_group(c)) return group_each(c, [&](pioran_ctx* ch) { return pioran_ctx_set_auto_scan(ch, enabled); });
    if (!c) return fail(PIORAN_EINVAL, "ctx is NULL");
    std::lock_guard<std::mutex> lk(c->mu);
    c->auto_scan = enabled != 0;
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

extern "C" int pioran_ctx_set_sweep_kernel(pioran_ctx* c, int which) try {
    if (is_group(c)) return group_each(c, [&](pioran_ctx* ch) { return pioran_ctx_set_sweep_kernel(ch, which); });
    if (!c) return fail(PIORAN_EINVAL, "ctx is NULL");
    if (which != PIORAN_SWEEP_AUTO && which != PIORAN_SWEEP_SCALAR) return fail(PIORAN_EINVAL, "unknown sweep kernel %d", which);
    std::lock_guard<std::mutex> lk(c->mu);
    c->sweep_kernel = which;
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

extern "C" int pioran_ctx_set_scan_tolerance(pioran_ctx* c, double tol) try {
    if (is_group(c)) return group_each(c, [&](pioran_ctx* ch) { return pioran_ctx_set_scan_tolerance(ch, tol); });
    if (!c) return fail(PIORAN_EINVAL, "ctx is NULL");
    if (tol != tol) return fail(PIORAN_EINVAL, "tol is NaN");
    std::lock_guard<std::mutex> lk(c->mu);
    c->scan_tol = tol;
    return PIORAN_OK;
} catch (...) { return guard_fail(); }
extern "C" int pioran_ctx_last_scan_check(pioran_ctx* c, double* estimate, int* n_fallback, int* n_refined) try {
    if (is_group(c)) return pioran_ctx_last_scan_check(c->children[0], estimate, n_fallback, n_refined);
    if (!c) return fail(PIORAN_EINVAL, "ctx is NULL");
    std::lock_guard<std::mutex> lk(c->mu);
    if (estimate) *estimate = c->scan_last_est;
    if (n_fallback) *n_fallback = c->scan_last_fallback;
    if (n_refined) *n_refined = c->scan_last_refined;
    return PIORAN_OK;
} catch (...) { return guard_fail(); }
extern "C" int pioran_ctx_set_scan_floor_cap(pioran_ctx* c, double cap) try {
    if (is_group(c)) return group_each(c, [&](pioran_ctx* ch) { return pioran_ctx_set_scan_floor_cap(ch, cap); });
    if (!c) return fail(PIORAN_EINVAL, "ctx is NULL");
    if (!(cap == cap)) return fail(PIORAN_EINVAL, "cap is NaN");
    std::lock_guard<std::mutex> lk(c->mu);
    c->scan_floor_cap = cap;
    return PIORAN_OK;
} catch (...) { return guard_fail(); }
extern "C" int pioran_ctx_last_scan_history(pioran_ctx* c, int index, int max_passes, double* estimates, double* values,
                                            int* n_passes) try {
    if (is_group(c)) return pioran_ctx_last_scan_history(c->children[0], index, max_passes, estimates, values, n_passes);
    if (!c) return fail(PIORAN_EINVAL, "ctx is NULL");
    std::lock_guard<std::mutex> lk(c->mu);
    if (index < 0 || (size_t)index >= c->scan_hist_est.size())
        return fail(PIORAN_EINVAL, "index %d outside the %zu parameter vectors of the last scan call", index, c->scan_hist_est.size());
    const std::vector<double>& e = c->scan_hist_est[index];
    const std::vector<double>& v = c->scan_hist_val[index];
    const int n = (int)e.size();
    if (n_passes) *n_passes = n;
    for (int k = 0; k < n && k < max_passes; k++) {
        if (estimates) estimates[k] = e[k];
        if (values) values[k] = v[k];
    }
    return PIORAN_OK;
} catch (...) { return guard_fail(); }
extern "C" int pioran_ctx_set_scan_chunks(pioran_ctx* c, int chunks) try {
    if (is_group(c)) return group_each(c, [&](pioran_ctx* ch) { return pioran_ctx_set_scan_chunks(ch, chunks); });
    if (!c) return fail(PIORAN_EINVAL, "ctx is NULL");
    if (chunks < 0) return fail(PIORAN_EINVAL, "chunks must be >= 0 (0 = automatic)");
    std::lock_guard<std::mutex> lk(c->mu);
    c->scan_chunks = chunks;
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

// One run of the parallel-in-time path over the step range [n_lo, n_hi) of a series: device buffers (inside ctx workspaces)
// and shapes, shared by the whole-series entry and by the two-phase range entries (time axis split across GPUs).
struct ScanRun {
    uint64_t epoch = 0;   // context epoch at range_begin; any later compute entry invalidates the record
    bool valid = false;
    int series_id = -1, B = 0, Jt = 0, R = 0, BS = 0, P = 0, G1 = 0, G2 = 0, SUB = 1;
    int64_t N = 0, n_lo = 0, n_hi = 0;
    std::vector<int64_t> bounds;
    std::vector<int> term_row_host;        // host sources of the asynchronous uploads: kept alive with the run
    std::vector<WorkItem> items_host;
    GenericInputs gi{};
    double *elems = nullptr, *pref = nullptr, *gstate = nullptr, *cstate = nullptr, *parts = nullptr, *out = nullptr;
    double *total = nullptr, *scratch = nullptr, *init = nullptr, *prev = nullptr, *sums = nullptr;
    double *subel = nullptr, *substate = nullptr, *tot0 = nullptr, *tot1 = nullptr, *tp = nullptr;
    double *chk = nullptr, *err = nullptr;   // self-check sums (4 per sub-chunk) and the per-θ deviation estimate
    double *ksbuf = nullptr;                 // second Kogge–Stone buffer (the fold's composites in `elems` stay intact for the Newton step)
    double *exits = nullptr, *tm = nullptr;  // Newton refinement: exit state of every chunk sweep, (T | m) of every chunk
    double *nel0 = nullptr, *nel1 = nullptr; // … and the two buffers of its affine scan (T | r | m | r^g per boundary)
    double check_scale = 1.0;
    int64_t* bounds_dev = nullptr;
    int* term_row_dev = nullptr;
    bool wide = false;                       // ranks 65 … 96: the kernels of scan_wide.cuh (leading dimension 96)
    bool bfold = false;                      // fold and pass 3 on the tensor pipe from the per-θ block table (scan_blocked.cuh)
    int NTs = 0; const double* stab = nullptr; int64_t stab_stride = 0;
    size_t sel() const { return wide ? (size_t)SELW : (size_t)SEL; }          // doubles per composite / state / (T | m)
    size_t sstate() const { return wide ? (size_t)SSTATEW : (size_t)SSTATE; }
    size_t snewt() const { return wide ? (size_t)SNEWTW : (size_t)SNEWT; }
    size_t snel() const { return wide ? (size_t)SNELW : (size_t)SNEL; }
    int rr() const { return wide ? std::min(SRW, (R + 3) & ~3) : std::min(SR, (R + 3) & ~3); }   // live rank, rounded up to a multiple of 4
    size_t smem() const { return wide ? scanw_smem_bytes(rr()) : SCAN_SMEM_BYTES; }
};
static int scan_live_rank(int R) { return std::min(SR, (R + 3) & ~3); }
// Steps of the self-check at a sub-chunk boundary: SCAN_CHECK_STEPS, or the (even part of the) sub-chunk when it is shorter.
constexpr int SCAN_CHECK_STEPS = 8;
constexpr int SCAN_MAX_NEWTON = 3;      // refinement ladder: up to three Newton steps on the chunk states, then the sequential sweep
static int scan_check_steps(int64_t sub_len) { return (int)std::min<int64_t>(SCAN_CHECK_STEPS, sub_len & ~(int64_t)1); }
static std::map<pioran_ctx*, ScanRun> g_scan;
static std::mutex g_scan_mu;
static void scan_forget(pioran_ctx* c) { std::lock_guard<std::mutex> g(g_scan_mu); g_scan.erase(c); }
static ScanRun* scan_slot(pioran_ctx* c) { std::lock_guard<std::mutex> g(g_scan_mu); return &g_scan[c]; }   // std::map nodes are stable

// Phase 1: coefficients, chunking, fold of every chunk into its composite, prefix composites inside the groups and — when
// want_total — the composite of the whole range.  max_prev = number of earlier-range composites phase 2 may receive.
static int scan_phase1(pioran_ctx* c, Series* s, int series_id, int B, int Jt, const double* a, const double* b,
                       const double* cc, const double* d, const double* mu, const double* nu, int64_t n_lo, int64_t n_hi,
                       bool want_total, int max_prev, ScanRun& run) {
    std::vector<int> term_row;
    const int R = make_term_rows(B, Jt, b, d, term_row);
    const int BS = bs_for_rank(R);
    const bool wide = R > SR;
    if (R > SRW)
        return fail(PIORAN_EUNSUPPORTED, "rank %d (Jt = %d) exceeds the scan path's limit of %d", R, Jt, SRW);
    if (wide && (want_total || max_prev > 0 || n_lo != 0 || n_hi != s->N))
        return fail(PIORAN_EUNSUPPORTED, "the time-axis split across devices is built for ranks <= %d (rank %d)", SR, R);
    const int64_t N = s->N, len = n_hi - n_lo;
    // chunking.  With log-depth scan levels the second pass costs little per extra chunk, so the optimum sits where the fold
    // runs as ONE round of CTAs: one chunk per SM for a single parameter vector (tools/scan_chunks_sweep.py: P = 148
    // is the best or within 3 % of it from 16 k to 1 M steps at ranks 4 … 60; two chunks per SM are 5 % slower), up to two
    // per SM in total when several parameter vectors share the device, and at least 64 steps per chunk.
    int P = c->scan_chunks;
    if (P <= 0) {
        P = std::min(c->num_sms, std::max(16, 2 * c->num_sms / std::max(1, B)));   // two fold CTAs fit an SM: B·P ≤ 2·SMs
        if (B == 1 && len / (2 * c->num_sms) >= 2048) P = 2 * c->num_sms;          // very long series: two chunks per SM (−7 % at 1e6 steps)
        if (wide) P = std::min(c->num_sms, std::max(16, c->num_sms / std::max(1, B)));   // the 512-thread fold: one CTA per SM
    }
    P = (int)std::max<int64_t>(1, std::min<int64_t>(P, len / 64));
    const int G2 = (int)std::ceil(std::sqrt((double)P));
    const int G1 = (P + G2 - 1) / G2;
    // pass 3 on SUB sub-chunks per chunk (states at the inner boundaries from the fold's running composite): worth one extra
    // apply per boundary once a chunk is a thousand steps long
    int SUB = (len / P >= 1024) ? 4 : 1;
    run = ScanRun{};
    run.series_id = series_id; run.B = B; run.Jt = Jt; run.R = R; run.BS = BS; run.P = P; run.G1 = G1; run.G2 = G2; run.SUB = SUB;
    run.N = N; run.n_lo = n_lo; run.n_hi = n_hi; run.wide = wide;
    const size_t SELr = run.sel(), SSTATEr = run.sstate(), SNEWTr = run.snewt();
    run.bounds.resize(P + 1);
    // inner bounds at even offsets: every sub-chunk but the last has an even length (the self-check sweeps on across a bound)
    // Blocked fold (scan_blocked.cuh): whole-series calls at 4 … 13 row tiles whose per-θ block table fits a quarter of the free HBM
    const int NTs = sblk_nt(R);
    const int64_t blk_lo = n_lo / BLK, blk_hi = std::min<int64_t>((N + BLK - 1) / BLK, (n_hi + BLK - 1) / BLK + 1);   // + the look-ahead block of the self-check
    const int64_t nblk_series = blk_hi - blk_lo;
    const size_t stab_bytes = sizeof(double) * (size_t)nblk_series * sblk_doubles(NTs) * (size_t)B;
    static const bool bfold_on = [] { const char* e = getenv("PIORAN_K3_BLOCKED_FOLD"); return !(e && !strcmp(e, "0")); }();
    // (a range in the middle of a series — the time axis split across devices — qualifies when it sits on the block grid)
    bool bfold = bfold_on && c->sweep_kernel != PIORAN_SWEEP_SCALAR && NTs >= 4 && NTs <= 13 && (n_lo % BLK) == 0 &&
                 (n_hi == N || (n_hi % BLK) == 0) && len / P >= 64;
    if (bfold && stab_bytes > c->stab.cap) {
        size_t free_b = 0, total_b = 0;
        CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
        if (stab_bytes > (free_b + c->stab.cap) / 4) bfold = false;
    }
    const int64_t bmask = bfold ? ~(int64_t)7 : ~(int64_t)1;     // chunk bounds on the table's block grid
    run.bfold = bfold; run.NTs = NTs;
    if (bfold) { SUB = 1; run.SUB = 1; }      // the blocked re-filter sweeps a whole chunk in 0.8 ms: no inner boundaries
    for (int k = 0; k <= P; k++) run.bounds[k] = k == P ? n_hi : n_lo + ((int64_t)((__int128)len * k / P) & bmask);

    int rc;
    if ((rc = upload_generic(c, B, Jt, N, a, b, cc, d, mu, nu, nullptr, nullptr, run.gi))) return rc;
    const size_t nch = (size_t)B * P;
    // workspace (doubles): elems | pref | gstate | cstate | parts (+1 dummy pair) | out | total | scratch | init | prev | sums
    const size_t n_el = nch * SELr, n_gs = (size_t)B * G1 * SSTATEr, n_cs = nch * SSTATEr, n_pt = 2 * (nch * SUB + 1);
    const size_t n_chk = 4 * (nch * SUB + 1);
    const size_t n_sel = nch * (SUB - 1) * SELr, n_sst = nch * (SUB - 1) * SSTATEr, n_gt = (size_t)B * G1 * SELr;
    const size_t n_tot = (size_t)B * SELr, n_scr = 2 * (size_t)B * SELr, n_init = (size_t)B * SSTATEr;
    const size_t n_prev = (size_t)std::max(0, max_prev) * B * SELr;
    const size_t n_tm = nch * SNEWTr, n_nel = nch * run.snel();
    if ((rc = c->misc.ensure(sizeof(double) * (3 * n_el + n_gs + 2 * n_cs + n_tm + 2 * n_nel + n_pt + B + n_tot + n_scr + n_init + n_prev + 3 * (size_t)B + n_sel + n_sst + 2 * n_gt + n_chk + B))))
        return rc;
    run.elems = c->misc.as<double>();
    run.pref = run.elems + n_el;
    run.gstate = run.pref + n_el;
    run.cstate = run.gstate + n_gs;
    run.parts = run.cstate + n_cs;
    run.out = run.parts + n_pt;
    run.total = run.out + B;
    run.scratch = run.total + n_tot;
    run.init = run.scratch + n_scr;
    run.prev = run.init + n_init;
    run.sums = run.prev + n_prev;
    run.subel = run.sums + 3 * (size_t)B;
    run.substate = run.subel + n_sel;
    run.tot0 = run.substate + n_sst;
    run.tot1 = run.tot0 + n_gt;
    run.chk = run.tot1 + n_gt;
    run.err = run.chk + n_chk;
    run.ksbuf = run.err + B;
    run.exits = run.ksbuf + n_el;
    run.tm = run.exits + n_cs;
    run.nel0 = run.tm + n_tm;
    run.nel1 = run.nel0 + n_nel;
    if ((rc = c->rows.ensure(sizeof(int) * (Jt + 1) + sizeof(int64_t) * (P + 2) + sizeof(int) * 2 * (size_t)std::max(R, 1)))) return rc;   // + the fold's row tables
    run.bounds_dev = c->rows.as<int64_t>();
    run.term_row_dev = reinterpret_cast<int*>(run.bounds_dev + P + 2);
    CUDA_TRY(cudaMemcpyAsync(run.bounds_dev, run.bounds.data(), sizeof(int64_t) * (P + 1), cudaMemcpyHostToDevice, c->stream));
    run.term_row_host = term_row;            // (run = ScanRun{} above dropped the previous one)
    CUDA_TRY(cudaMemcpyAsync(run.term_row_dev, run.term_row_host.data(), sizeof(int) * Jt, cudaMemcpyHostToDevice, c->stream));
    // no host synchronisation here: the sources live in `run`, and a copy from pageable memory is staged before the call returns

    ScanArgs sa{};
    sa.t = s->t; sa.y = s->y; sa.s2 = s->s2; sa.N = N; sa.P = P; sa.bounds = run.bounds_dev;
    sa.a = run.gi.a; sa.b = run.gi.b; sa.c = run.gi.c; sa.d = run.gi.d; sa.Jt = Jt; sa.term_row = run.term_row_dev;
    sa.mu = run.gi.mu; sa.nu = run.gi.nu; sa.elems = run.elems; sa.SUB = SUB; sa.subel = run.subel;
    if (bfold) {
        // per-θ block table (rows in logical order, the data row at R), then one CTA of NTs warps per chunk
        if ((rc = c->stab.ensure(stab_bytes))) return rc;
        std::vector<int> rmeta(2 * (size_t)std::max(R, 1));
        for (int m = 0; m < Jt; m++) {
            const int tr = term_row[m];
            if (tr < 0) { rmeta[-tr - 1] = m; rmeta[R + (-tr - 1)] = ROW_REAL; }
            else { rmeta[tr] = m; rmeta[R + tr] = ROW_COS; rmeta[tr + 1] = m; rmeta[R + tr + 1] = ROW_SIN; }
        }
        int* rmeta_dev = run.term_row_dev + Jt + 1;           // behind the chunk bounds and the term rows in c->rows
        CUDA_TRY(cudaMemcpyAsync(rmeta_dev, rmeta.data(), sizeof(int) * rmeta.size(), cudaMemcpyHostToDevice, c->stream));
        CUDA_TRY(cudaStreamSynchronize(c->stream));          // rmeta is a local
        const int64_t tstride = nblk_series * sblk_doubles(NTs);
        // the kernels index the table by the ABSOLUTE block number: hand them the base shifted by the range's first block
        run.stab = c->stab.as<double>() - (size_t)blk_lo * sblk_doubles(NTs); run.stab_stride = tstride;
        scan_block_table_kernel<<<dim3((unsigned)nblk_series, B), 128, 0, c->stream>>>(c->stab.as<double>(), tstride, s->t, s->y, s->s2, N, run.gi.a,
                                                                                     run.gi.b, run.gi.c, run.gi.d, Jt, rmeta_dev, rmeta_dev + R, R,
                                                                                     NTs, run.gi.mu, run.gi.nu, blk_lo);
        // the blocked fold writes the live rank only: everything else of the composites must read as zero
        CUDA_TRY(cudaMemsetAsync(run.elems, 0, sizeof(double) * n_el, c->stream));
        if (n_sel) CUDA_TRY(cudaMemsetAsync(run.subel, 0, sizeof(double) * n_sel, c->stream));
        const int LDSr = wide ? SRW : SR;
#define PIORAN_SFB_CASE(nt)                                                                                                          \
        case nt: {                                                                                                                   \
            CUDA_TRY(cudaFuncSetAttribute(scan_fold_blocked_kernel<nt>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sfb_smem_bytes<nt>()));     \
            scan_fold_blocked_kernel<nt><<<dim3(P, B), nt * 32, sfb_smem_bytes<nt>(), c->stream>>>(sa, run.stab, tstride, R, LDSr, (int)SELr); \
        } break;
        switch (NTs) {
            PIORAN_SFB_CASE(4) PIORAN_SFB_CASE(5) PIORAN_SFB_CASE(6) PIORAN_SFB_CASE(7) PIORAN_SFB_CASE(8) PIORAN_SFB_CASE(9)
            PIORAN_SFB_CASE(10) PIORAN_SFB_CASE(11) PIORAN_SFB_CASE(12) PIORAN_SFB_CASE(13)
        }
#undef PIORAN_SFB_CASE
        c->launches += 2;
        CUDA_TRY(cudaGetLastError());
    }
    if (wide) {
        // states handed to pass 3 are read over the full 96 rows: what the pass-2 kernels leave outside the live rank must be zero
        CUDA_TRY(cudaMemsetAsync(run.gstate, 0, sizeof(double) * (n_gs + n_cs), c->stream));
        if (n_sst) CUDA_TRY(cudaMemsetAsync(run.substate, 0, sizeof(double) * n_sst, c->stream));
        if (!bfold) {
            CUDA_TRY(cudaFuncSetAttribute(scanw_fold_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FOLDW_SMEM_BYTES));
            scanw_fold_kernel<<<dim3(P, B), FOLDW_THREADS, FOLDW_SMEM_BYTES, c->stream>>>(sa);
            c->launches++;
        }
        const int Rw = run.rr();
        const size_t smw = run.smem();
        CUDA_TRY(cudaFuncSetAttribute(scanw_ks_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smw));
        CUDA_TRY(cudaFuncSetAttribute(scanw_group_states_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smw));
        CUDA_TRY(cudaFuncSetAttribute(scanw_states_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smw));
        CUDA_TRY(cudaFuncSetAttribute(scanw_substates_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smw));
        double* src = run.elems;
        double* dst = run.pref;
        for (int dd = 1; dd < G2 && P > 1; dd *= 2) {
            scanw_ks_kernel<<<dim3(P, B), 256, smw, c->stream>>>(src, dst, P, G2, dd, Rw);
            c->launches++;
            double* const wrote = dst;
            dst = (src == run.elems) ? run.ksbuf : src;
            src = wrote;
        }
        run.pref = src;
        scanw_gather_kernel<<<dim3(G1, B), 256, 0, c->stream>>>(run.pref, run.tot0, P, G2, G1);
        c->launches++;
        src = run.tot0; dst = run.tot1;
        for (int dd = 1; dd < G1; dd *= 2) {
            scanw_ks_kernel<<<dim3(G1, B), 256, smw, c->stream>>>(src, dst, G1, G1, dd, Rw);
            c->launches++;
            std::swap(src, dst);
        }
        run.tp = src;
        CUDA_TRY(cudaGetLastError());
        run.valid = true;
        return 0;
    }
    if (!bfold) {
        scan_fold_kernel<<<dim3(P, B), 256, 0, c->stream>>>(sa);
        c->launches++;
    }
    CUDA_TRY(cudaFuncSetAttribute(scan_ks_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SCAN_SMEM_BYTES));
    CUDA_TRY(cudaFuncSetAttribute(scan_group_states_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SCAN_SMEM_BYTES));
    CUDA_TRY(cudaFuncSetAttribute(scan_states_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SCAN_SMEM_BYTES));
    CUDA_TRY(cudaFuncSetAttribute(scan_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SCAN_SMEM_BYTES));
    CUDA_TRY(cudaFuncSetAttribute(scan_substates_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SCAN_SMEM_BYTES));
    const int Rr = scan_live_rank(run.R);
    // (a) prefix composites inside the groups: Kogge–Stone over segments of G2 chunks, ping-pong between the two buffers
    {
        double* src = run.elems;
        double* dst = run.pref;
        for (int dd = 1; dd < G2 && P > 1; dd *= 2) {
            scan_ks_kernel<<<dim3(P, B), 256, SCAN_SMEM_BYTES, c->stream>>>(src, dst, P, G2, dd, Rr);
            c->launches++;
            double* const wrote = dst;
            dst = (src == run.elems) ? run.ksbuf : src;     // never back into the fold's output
            src = wrote;
        }
        run.pref = src;      // the buffer the last level wrote (the fold's own output when there is a single chunk per group)
    }
    // (b) running products of the group totals; the last one is the composite of the whole range
    {
        scan_gather_kernel<<<dim3(G1, B), 256, 0, c->stream>>>(run.pref, run.tot0, P, G2, G1);
        c->launches++;
        double* src = run.tot0;
        double* dst = run.tot1;
        for (int dd = 1; dd < G1; dd *= 2) {
            scan_ks_kernel<<<dim3(G1, B), 256, SCAN_SMEM_BYTES, c->stream>>>(src, dst, G1, G1, dd, Rr);
            c->launches++;
            std::swap(src, dst);
        }
        run.tp = src;
    }
    if (want_total) {
        for (int i = 0; i < B; i++)
            CUDA_TRY(cudaMemcpyAsync(run.total + (size_t)i * SEL, run.tp + ((size_t)i * G1 + G1 - 1) * SEL, sizeof(double) * SEL,
                                     cudaMemcpyDeviceToDevice, c->stream));
    }
    CUDA_TRY(cudaGetLastError());
    run.valid = true;
    return 0;
}

// Pass 3 from the per-θ block table (scan_blocked.cuh): one CTA of four warps per work item.
static int launch_scan_sweep_blocked(pioran_ctx* c, const ScanRun& run, const WorkItem* work, int nitems) {
    const int LDSr = run.wide ? SRW : SR;
#define PIORAN_SSB_CASE(nt)                                                                                                       \
    case nt: {                                                                                                                    \
        CUDA_TRY(cudaFuncSetAttribute(scan_sweep_blocked_kernel<nt>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ssb_smem_bytes<nt>()));    \
        scan_sweep_blocked_kernel<nt><<<nitems, SSB_W * 32, ssb_smem_bytes<nt>(), c->stream>>>(work, run.stab, run.stab_stride, run.R, LDSr);    \
    } break;
    switch (run.NTs) {
        PIORAN_SSB_CASE(4) PIORAN_SSB_CASE(5) PIORAN_SSB_CASE(6) PIORAN_SSB_CASE(7) PIORAN_SSB_CASE(8) PIORAN_SSB_CASE(9)
        PIORAN_SSB_CASE(10) PIORAN_SSB_CASE(11) PIORAN_SSB_CASE(12) PIORAN_SSB_CASE(13)
        default: return fail(PIORAN_EUNSUPPORTED, "no blocked re-filter for %d row tiles", run.NTs);
    }
#undef PIORAN_SSB_CASE
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// Pass 3 at ranks 65 … 96: one CTA per work item (scan_wide.cuh).
static int launch_wide_chunk(pioran_ctx* c, const BatchArgs& args, int nitems) {
    const int TS = std::max(5, (args.R + 15) / 16);
    if (TS == 5) celerite_wide_chunk_kernel<5><<<nitems, WIDE_THREADS, 0, c->stream>>>(args);
    else celerite_wide_chunk_kernel<6><<<nitems, WIDE_THREADS, 0, c->stream>>>(args);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

// Phase 2: states entering every chunk (from `init_dev`, or from the start of the series when it is null), re-filter of
// every chunk, partial sums in run.parts.
static int scan_phase2(pioran_ctx* c, Series* s, ScanRun& run, const double* init_dev, int warm_subs = 0, bool states_ready = false) {
    const int B = run.B, P = run.P, NW = CHUNK_NW, SUB = run.SUB;
    const size_t nch = (size_t)B * P, nsub = nch * SUB;
    const size_t nitems = (nsub + NW - 1) / NW * NW;
    std::vector<WorkItem>& items = run.items_host;
    items.assign(nitems, WorkItem{});
    const int PS = P * SUB;     // sub-chunks per parameter vector, g = ch·SUB + j
    auto bound = [&](int g) { return g >= PS ? run.bounds[P] : scan_sub_bound(run.bounds[g / SUB], run.bounds[g / SUB + 1], g % SUB, SUB); };
    auto state_at = [&](int th, int g) -> const double* {       // the state entering sub-chunk g of parameter vector th
        const size_t q = (size_t)th * P + g / SUB;
        const int j = g % SUB;
        if (j == 0) return (g == 0 && !init_dev) ? nullptr : run.cstate + q * run.sstate();
        return run.substate + (q * (SUB - 1) + (j - 1)) * run.sstate();
    };
    for (size_t k = 0; k < nitems; k++) {
        const size_t e = std::min(k, nsub - 1);
        const int th = (int)(e / PS), g = (int)(e % PS);
        WorkItem& w = items[k];
        w.table = nullptr; w.t = s->t; w.y = s->y; w.s2 = s->s2; w.N = run.N;
        w.theta_begin = th; w.par_begin = th; w.count = 1; w.out_begin = 0;
        // refinement pass: start warm_subs sub-chunks earlier (at most at the start of the range) and discard the run-up
        const int gs = std::max(0, g - warm_subs);
        w.n_begin = bound(gs);
        w.n_warm = bound(g) - bound(gs);
        w.n_end = bound(g + 1);
        w.init = state_at(th, gs);
        w.part = k < nsub ? run.parts + 2 * e : run.parts + 2 * nsub;   // padding warps write to the dummy pair
        w.chk = k < nsub ? run.chk + 4 * e : run.chk + 4 * nsub;
        // self-check: re-sweep the first steps of the NEXT sub-chunk from this sweep's own state (n_ext), and sum the first
        // steps of this one separately (n_head) for the previous work item's comparison
        // (a range in the middle of a series also checks its hand-over: its first sub-chunk sums its head for the rank before,
        // its last one sweeps on into the next rank's range — pioran_celerite_scan_range_check)
        const bool first = g == 0, last = g == PS - 1;
        w.n_head = (first && !init_dev) ? 0 : scan_check_steps(bound(g + 1) - bound(g));
        // (after a range of odd length the look-ahead would break the even/odd alternation of the steps: no look-ahead then,
        // and the caller's comparison reads "not verified" — parallel.scan_bounds keeps the inner bounds even)
        if (last) w.n_ext = (run.n_hi < run.N && ((run.n_hi - run.n_lo) & 1) == 0) ? scan_check_steps(run.N - run.n_hi) : 0;
        else w.n_ext = scan_check_steps(bound(g + 2) - bound(g + 1));
    }
    run.check_scale = std::max(1.0, (double)(run.n_hi - run.n_lo) / ((double)P * SUB * SCAN_CHECK_STEPS));
    int rc;
    c->work_key.clear();
    if ((rc = c->work.ensure(sizeof(WorkItem) * nitems))) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->work.p, items.data(), sizeof(WorkItem) * nitems, cudaMemcpyHostToDevice, c->stream));
    if (run.wide) {
        const int Rw = run.rr();
        const size_t smw = run.smem();
        if (!states_ready && P > 1) {
            scanw_group_states_kernel<<<dim3(run.G1, B), 256, smw, c->stream>>>(run.tp, run.gstate, run.G1, Rw);
            scanw_states_kernel<<<dim3(P, B), 256, smw, c->stream>>>(run.pref, run.gstate, run.cstate, P, run.G2, run.G1, Rw);
            c->launches += 2;
        }
        if (!states_ready && SUB > 1) {
            scanw_substates_kernel<<<dim3(P * (SUB - 1), B), 256, smw, c->stream>>>(run.subel, run.cstate, run.substate, P, SUB, Rw);
            c->launches++;
        }
        CUDA_TRY(cudaGetLastError());
        BatchArgs wargs{};
        wargs.work = c->work.as<WorkItem>();
        wargs.a = run.gi.a; wargs.b = run.gi.b; wargs.c = run.gi.c; wargs.d = run.gi.d;
        wargs.Jt = run.Jt; wargs.term_row = run.term_row_dev; wargs.R = run.R;
        wargs.mu = run.gi.mu; wargs.nu = run.gi.nu; wargs.pstride = 1;
        wargs.out = run.out;
        return run.bfold ? launch_scan_sweep_blocked(c, run, c->work.as<WorkItem>(), (int)nsub) : launch_wide_chunk(c, wargs, (int)nsub);
    }
    if (!states_ready && (P > 1 || init_dev)) {
        scan_group_states_kernel<<<dim3(run.G1, B), 256, SCAN_SMEM_BYTES, c->stream>>>(run.tp, run.gstate, run.G1, init_dev, scan_live_rank(run.R));
        scan_states_kernel<<<dim3(P, B), 256, SCAN_SMEM_BYTES, c->stream>>>(run.pref, run.gstate, run.cstate, P, run.G2, run.G1,
                                                                             init_dev ? 1 : 0, scan_live_rank(run.R));
        c->launches += 2;
    }
    if (!states_ready && SUB > 1) {
        scan_substates_kernel<<<dim3(P * (SUB - 1), B), 256, SCAN_SMEM_BYTES, c->stream>>>(
            run.subel, run.cstate, run.substate, P, SUB, init_dev ? 1 : 0, scan_live_rank(run.R));
        c->launches++;
    }
    CUDA_TRY(cudaGetLastError());
    BatchArgs args{};
    args.work = c->work.as<WorkItem>();
    args.a = run.gi.a; args.b = run.gi.b; args.c = run.gi.c; args.d = run.gi.d;
    args.Jt = run.Jt; args.term_row = run.term_row_dev; args.R = run.R;
    args.mu = run.gi.mu; args.nu = run.gi.nu; args.pstride = 1;
    args.out = run.out;
    if (run.bfold) return launch_scan_sweep_blocked(c, run, c->work.as<WorkItem>(), (int)nsub);
    return dispatch_chunked(c, run.BS, args, (int)(nitems / NW));
}

// Pass 3 chunk by chunk (Newton refinement, scan.cuh): SUB launches; launch j sweeps sub-chunk j of EVERY chunk from the state
// the previous launch left behind (j = 0: the chunk state S̃_k) and stores the state it arrives at — in the inner-boundary slot
// the next launch starts from, or (last sub-chunk) in run.exits.  The inner states are then those of the exact recursion
// started from S̃_k, so only the chunk boundaries carry a self-check.
static int scan_seq_pass(pioran_ctx* c, Series* s, ScanRun& run) {
    const int B = run.B, P = run.P, NW = CHUNK_NW, SUB = run.SUB;
    const size_t nch = (size_t)B * P;
    const size_t npl = (nch + NW - 1) / NW * NW;       // work items per launch
    const int PS = P * SUB;
    std::vector<WorkItem>& items = run.items_host;
    items.assign(npl * SUB, WorkItem{});
    auto bound = [&](int g) { return g >= PS ? run.bounds[P] : scan_sub_bound(run.bounds[g / SUB], run.bounds[g / SUB + 1], g % SUB, SUB); };
    for (int j = 0; j < SUB; j++)
        for (size_t k = 0; k < npl; k++) {
            const bool real = k < nch;
            const size_t e = std::min(k, nch - 1);
            const int th = (int)(e / P), ch = (int)(e % P), g = ch * SUB + j;
            WorkItem& w = items[(size_t)j * npl + k];
            w.table = nullptr; w.t = s->t; w.y = s->y; w.s2 = s->s2; w.N = run.N;
            w.theta_begin = th; w.par_begin = th; w.count = 1; w.out_begin = 0;
            w.n_begin = bound(g); w.n_end = bound(g + 1); w.n_warm = 0;
            if (j == 0) w.init = ch == 0 ? nullptr : run.cstate + e * run.sstate();
            else w.init = run.substate + (e * (SUB - 1) + (j - 1)) * run.sstate();
            const size_t slot = real ? (size_t)th * PS + g : nch * SUB;       // padding warps write to the dummy slots
            w.part = run.parts + 2 * slot;
            w.chk = run.chk + 4 * slot;
            w.n_head = (j == 0 && ch > 0) ? scan_check_steps(bound(g + 1) - bound(g)) : 0;
            w.n_ext = (j == SUB - 1 && ch < P - 1) ? scan_check_steps(bound(g + 2) - bound(g + 1)) : 0;
            w.exit = nullptr;
            if (real && j < SUB - 1) w.exit = run.substate + (e * (SUB - 1) + j) * run.sstate();
            else if (real && ch < P - 1) w.exit = run.exits + e * run.sstate();
        }
    run.check_scale = std::max(1.0, (double)(run.n_hi - run.n_lo) / ((double)P * SCAN_CHECK_STEPS));
    int rc;
    c->work_key.clear();
    if ((rc = c->work.ensure(sizeof(WorkItem) * items.size()))) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->work.p, items.data(), sizeof(WorkItem) * items.size(), cudaMemcpyHostToDevice, c->stream));
    BatchArgs args{};
    args.a = run.gi.a; args.b = run.gi.b; args.c = run.gi.c; args.d = run.gi.d;
    args.Jt = run.Jt; args.term_row = run.term_row_dev; args.R = run.R;
    args.mu = run.gi.mu; args.nu = run.gi.nu; args.pstride = 1;
    args.out = run.out;
    for (int j = 0; j < SUB; j++) {
        args.work = c->work.as<WorkItem>() + (size_t)j * npl;
        if ((rc = run.bfold ? launch_scan_sweep_blocked(c, run, args.work, (int)nch)
                  : run.wide ? launch_wide_chunk(c, args, (int)nch) : dispatch_chunked(c, run.BS, args, (int)(npl / NW)))) return rc;
    }
    return 0;
}

// One Newton step on the chunk states: (T_k | m_k) of every chunk from its composite and current state, then the linear
// recurrence of the corrections along the chunks (needs the exits of a scan_seq_pass over the current states).
static int scan_newton_step(pioran_ctx* c, ScanRun& run) {
    const int P = run.P, B = run.B;
    double* src = run.nel0;
    double* dst = run.nel1;
    if (run.wide) {
        const int Rw = run.rr();
        const size_t smw = run.smem();
        CUDA_TRY(cudaFuncSetAttribute(scanw_newton_T_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smw));
        CUDA_TRY(cudaFuncSetAttribute(scanw_newton_ks_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smw));
        scanw_newton_T_kernel<<<dim3(P, B), 256, smw, c->stream>>>(run.elems, run.cstate, run.tm, P, Rw);
        scanw_newton_prep_kernel<<<dim3(P, B), 256, 0, c->stream>>>(run.tm, run.exits, run.cstate, src, P);
        c->launches += 2;
        for (int d = 1; d < P - 1; d *= 2) {
            scanw_newton_ks_kernel<<<dim3(P, B), 256, smw, c->stream>>>(src, dst, P, d, Rw);
            c->launches++;
            std::swap(src, dst);
        }
        scanw_newton_apply_kernel<<<dim3(P, B), 256, 0, c->stream>>>(src, run.cstate, P);
        c->launches++;
        CUDA_TRY(cudaGetLastError());
        return 0;
    }
    const int Rr = scan_live_rank(run.R);
    CUDA_TRY(cudaFuncSetAttribute(scan_newton_T_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SCAN_SMEM_BYTES));
    CUDA_TRY(cudaFuncSetAttribute(scan_newton_ks_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SCAN_SMEM_BYTES));
    scan_newton_T_kernel<<<dim3(P, B), 256, SCAN_SMEM_BYTES, c->stream>>>(run.elems, run.cstate, run.tm, P, Rr);
    scan_newton_prep_kernel<<<dim3(P, B), 256, 0, c->stream>>>(run.tm, run.exits, run.cstate, src, P);
    c->launches += 2;
    for (int d = 1; d < P - 1; d *= 2) {
        scan_newton_ks_kernel<<<dim3(P, B), 256, SCAN_SMEM_BYTES, c->stream>>>(src, dst, P, d, Rr);
        c->launches++;
        std::swap(src, dst);
    }
    scan_newton_apply_kernel<<<dim3(P, B), 256, 0, c->stream>>>(src, run.cstate, P);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    return 0;
}

static int scan_logl_locked(pioran_ctx* c, Series* s, int series_id, int B, int Jt, const double* a, const double* b,
                            const double* cc, const double* d, const double* mu, const double* nu, double* logl_out) {
    ScanRun run;
    int rc;
    cudaEventRecord(c->ev_beg, c->stream);
    if ((rc = scan_phase1(c, s, series_id, B, Jt, a, b, cc, d, mu, nu, 0, s->N, false, 0, run))) return rc;
    // Self-check and refinement ladder (scan.cuh: scan_check_estimate, Newton refinement).  The composites lose accuracy where
    // the covariance is ill-conditioned (steep PSD slopes: the scan's value was seen 1e-8 … 1e-6 away from the sequential
    // sweep's).  When the estimate of a parameter vector exceeds the tolerance, the chunk states are corrected by Newton steps
    // whose residual is the exact recursion itself (chunk-by-chunk sweeps that return their exit states), each verified the same
    // way.  A parameter vector is accepted when its estimate meets the tolerance, or when the Newton iteration has converged and
    // stalls at a level the tolerance cannot resolve: what is left then is the rounding noise of an FP64 evaluation of THIS
    // covariance — two sweeps that reach a boundary by different routes differ by it, the sequential sweep included (its own
    // distance from an 80-bit evaluation on such rows is of the same size) — capped (scan_floor_cap).  What still fails
    // (breakdown of the composites on a barely positive definite covariance) goes to the sequential sweep.
    c->scan_last_est = 0.0; c->scan_last_fallback = 0; c->scan_last_refined = 0;
    c->scan_hist_est.assign(B, {}); c->scan_hist_val.assign(B, {});
    std::vector<double> est(B), val(B), prev_rel(B, 0.0), prev_val(B, 0.0);
    std::vector<char> accepted(B, 0);
    std::vector<int> redo;
    const int PS = run.P * run.SUB;
    for (int level = 0;; level++) {
        // level 0: all sub-chunks at once from the scan's states; level 1: chunk by chunk from the same chunk states (exits for
        // the first Newton step); level ≥ 2: chunk by chunk from the corrected states
        if (level == 0) { if ((rc = scan_phase2(c, s, run, nullptr))) return rc; }
        else {
            if (level == 1) CUDA_TRY(cudaMemsetAsync(run.exits, 0, sizeof(double) * (size_t)B * run.P * run.sstate(), c->stream));
            if (level >= 2 && (rc = scan_newton_step(c, run))) return rc;
            if ((rc = scan_seq_pass(c, s, run))) return rc;
        }
        scan_finish_kernel<<<(B + 127) / 128, 128, 0, c->stream>>>(run.parts, run.chk, run.check_scale, PS, B, s->N, run.out, run.err);
        c->launches++;
        cudaEventRecord(c->ev_end, c->stream);
        note_kernel(c, KF_SCAN_FINISH);
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaMemcpyAsync(val.data(), run.out, sizeof(double) * (size_t)B, cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(cudaMemcpyAsync(est.data(), run.err, sizeof(double) * (size_t)B, cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(cudaStreamSynchronize(c->stream));
        redo.clear();
        for (int i = 0; i < B; i++) {
            if (accepted[i]) continue;
            const double rel = est[i] / std::max(1.0, std::fabs(val[i]));
            c->scan_hist_est[i].push_back(rel); c->scan_hist_val[i].push_back(val[i]);
            bool ok = !(c->scan_tol > 0.0) || rel <= c->scan_tol;
            // converged Newton iteration at the rounding floor of this covariance (level ≥ 3: two Newton steps done): the
            // estimate no longer moves (within 4× of the previous pass) and the value changed by no more than the floor cap
            // between the last two Newton steps (the estimate itself is pessimistic: it extends the mismatch of 8 steps to the
            // whole chunk; the pass-to-pass change of the value is what the iteration can still resolve)
            const double moved = std::fabs(val[i] - prev_val[i]) / std::max(1.0, std::fabs(val[i]));
            if (!ok && level >= 3 && c->scan_floor_cap > 0.0 && rel > 0.25 * prev_rel[i] && rel < 4.0 * prev_rel[i] &&
                moved <= c->scan_floor_cap && rel <= 1e3 * c->scan_floor_cap)
                ok = true;
            prev_rel[i] = rel; prev_val[i] = val[i];
            if (ok || level == 0) logl_out[i] = val[i];
            if (ok) {
                accepted[i] = 1;
                if (level > 0) c->scan_last_refined++;
                if (!(rel <= c->scan_last_est)) c->scan_last_est = rel;     // NaN sticks
            } else {
                redo.push_back(i);
            }
        }
        if (redo.empty() || run.P < 2 || level >= 1 + SCAN_MAX_NEWTON) break;
    }
    {
        for (int i : redo) {
            const double rel = est[i] / std::max(1.0, std::fabs(val[i]));
            if (!(rel <= c->scan_last_est)) c->scan_last_est = rel;
        }
        if (!redo.empty()) {
            const size_t nr = redo.size();
            std::vector<double> ra(nr * Jt), rb(nr * Jt), rcc(nr * Jt), rd(nr * Jt), rmu(nr), rnu(nr), rout(nr);
            for (size_t k = 0; k < nr; k++) {
                const size_t i = (size_t)redo[k];
                std::copy(a + i * Jt, a + (i + 1) * Jt, ra.begin() + k * Jt);
                std::copy(b + i * Jt, b + (i + 1) * Jt, rb.begin() + k * Jt);
                std::copy(cc + i * Jt, cc + (i + 1) * Jt, rcc.begin() + k * Jt);
                std::copy(d + i * Jt, d + (i + 1) * Jt, rd.begin() + k * Jt);
                rmu[k] = mu ? mu[i] : 0.0; rnu[k] = nu ? nu[i] : 1.0;
            }
            ExplicitSet x;
            if ((rc = explicit_front(c, series_id, (int)nr, Jt, rb.data(), rd.data(), WIDE_MAX_RANK, LOGL_LIMIT, x)) ||
                (rc = generic_logl_locked(c, x, (int)nr, Jt, ra.data(), rb.data(), rcc.data(), rd.data(), rmu.data(), rnu.data(),
                                          nullptr, nullptr, rout.data())))
                return rc;
            for (size_t k = 0; k < nr; k++) logl_out[redo[k]] = rout[k];
            c->scan_last_fallback = (int)nr;
        }
    }
    return PIORAN_OK;
}

extern "C" int pioran_celerite_logl_scan(pioran_ctx* c, int series_id, int B, int Jt, const double* a, const double* b,
                                         const double* cc, const double* d, const double* mu, const double* nu,
                                         double* logl_out) try {
    if (is_group(c))
        return group_first(c, series_id, [&](pioran_ctx* ch, int id) { return pioran_celerite_logl_scan(ch, id, B, Jt, a, b, cc, d, mu, nu, logl_out); });
    if (!c || !a || !b || !cc || !d || !logl_out) return fail(PIORAN_EINVAL, "NULL argument");
    if (B < 1 || Jt < 1) return fail(PIORAN_EINVAL, "B and Jt must be >= 1");
    PIORAN_COMPUTE_LOCK(c);
    CUDA_TRY(cudaSetDevice(c->device));
    Series* s = get_series(c, series_id);
    if (!s) return fail(PIORAN_EINVAL, "unknown series id %d", series_id);
    return scan_logl_locked(c, s, series_id, B, Jt, a, b, cc, d, mu, nu, logl_out);
} catch (...) { return guard_fail(); }

// ---- time axis split across GPUs (SURVEY §8e): each rank folds its own step range, the ranks exchange one composite each,
// and every rank re-filters its range from the state the earlier ranges leave behind.
extern "C" int pioran_scan_composite_doubles(void) { return SEL; }

extern "C" int pioran_celerite_scan_range_begin(pioran_ctx* c, int series_id, int Jt, const double* a, const double* b,
                                                const double* cc, const double* d, const double* mu, const double* nu,
                                                int64_t n_lo, int64_t n_hi, int max_prev, double* composite_out) try {
    if (is_group(c))
        return group_first(c, series_id, [&](pioran_ctx* ch, int id) {
            return pioran_celerite_scan_range_begin(ch, id, Jt, a, b, cc, d, mu, nu, n_lo, n_hi, max_prev, composite_out);
        });
    if (!c || !a || !b || !cc || !d || !composite_out) return fail(PIORAN_EINVAL, "NULL argument");
    PIORAN_COMPUTE_LOCK(c);
    CUDA_TRY(cudaSetDevice(c->device));
    Series* s = get_series(c, series_id);
    if (!s) return fail(PIORAN_EINVAL, "unknown series id %d", series_id);
    if (Jt < 1 || n_lo < 0 || n_hi > s->N || n_hi - n_lo < 1 || max_prev < 0)
        return fail(PIORAN_EINVAL, "bad range [%lld, %lld) of a series of %lld steps", (long long)n_lo, (long long)n_hi, (long long)s->N);
    ScanRun& run = *scan_slot(c);
    int rc;
    cudaEventRecord(c->ev_beg, c->stream);
    if ((rc = scan_phase1(c, s, series_id, 1, Jt, a, b, cc, d, mu, nu, n_lo, n_hi, true, max_prev, run))) { run.valid = false; return rc; }
    run.epoch = c->epoch;
    CUDA_TRY(cudaMemcpyAsync(composite_out, run.total, sizeof(double) * SEL, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

extern "C" int pioran_celerite_scan_range_end(pioran_ctx* c, int nprev, const double* composites_prev, double* sums_out) try {
    if (is_group(c)) return pioran_celerite_scan_range_end(c->children[0], nprev, composites_prev, sums_out);
    if (!c || !sums_out || (nprev > 0 && !composites_prev)) return fail(PIORAN_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> lk(c->mu);
    CUDA_TRY(cudaSetDevice(c->device));
    ScanRun& run = *scan_slot(c);
    if (!run.valid) return fail(PIORAN_EINVAL, "no range in progress: call pioran_celerite_scan_range_begin first");
    if (run.epoch != c->epoch) {
        run.valid = false;
        return fail(PIORAN_EINVAL, "the range in progress was invalidated by another call on this context between "
                                   "pioran_celerite_scan_range_begin and _end (they share its workspaces)");
    }
    Series* s = get_series(c, run.series_id);
    if (!s) return fail(PIORAN_EINVAL, "the series of the range in progress was freed");
    if (nprev < 0 || (size_t)nprev * SEL > (size_t)(run.sums - run.prev))
        return fail(PIORAN_EINVAL, "nprev = %d exceeds the max_prev announced to scan_range_begin", nprev);
    if ((nprev == 0) != (run.n_lo == 0))
        return fail(PIORAN_EINVAL, "a range starting at step %lld needs %s earlier composites", (long long)run.n_lo, run.n_lo == 0 ? "no" : "the");
    int rc;
    const double* init = nullptr;
    if (nprev > 0) {
        CUDA_TRY(cudaMemcpyAsync(run.prev, composites_prev, sizeof(double) * (size_t)nprev * SEL, cudaMemcpyHostToDevice, c->stream));
        scan_chain_kernel<<<dim3(1, 1), 256, SCAN_SMEM_BYTES, c->stream>>>(run.prev, nprev, 1, run.init, scan_live_rank(run.R));
        c->launches++;
        init = run.init;
    }
    if ((rc = scan_phase2(c, s, run, init))) return rc;
    scan_partial_kernel<<<1, 32, 0, c->stream>>>(run.parts, run.chk, run.check_scale, run.P * run.SUB, 1, run.sums);
    c->launches++;
    cudaEventRecord(c->ev_end, c->stream);
    note_kernel(c, KF_SCAN_PARTIAL);
    CUDA_TRY(cudaGetLastError());
    double sums3[3], chk_first[4], chk_last[4];
    const size_t nsub = (size_t)run.P * run.SUB;
    CUDA_TRY(cudaMemcpyAsync(sums3, run.sums, sizeof(double) * 3, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(chk_first, run.chk, sizeof(double) * 4, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(chk_last, run.chk + 4 * (nsub - 1), sizeof(double) * 4, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    {
        const WorkItem& wf = run.items_host[0];
        const WorkItem& wl = run.items_host[nsub - 1];
        double* k = c->scan_range_chk;
        k[0] = sums3[2]; k[1] = chk_first[0]; k[2] = chk_first[1]; k[3] = chk_last[2]; k[4] = chk_last[3];
        k[5] = wf.n_head; k[6] = wl.n_ext; k[7] = run.check_scale;
    }
    sums_out[0] = sums3[0]; sums_out[1] = sums3[1];
    // this range's part of the self-check estimate, in log L units (the caller sums the ranks' parts and divides by |log L|;
    // the hand-over between ranges is not covered): pioran_ctx_last_scan_check
    c->scan_last_est = sums3[2]; c->scan_last_fallback = 0; c->scan_last_refined = 0;
    run.valid = false;
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

extern "C" int pioran_celerite_scan_range_check(pioran_ctx* c, double* out8) try {
    if (is_group(c)) return pioran_celerite_scan_range_check(c->children[0], out8);
    if (!c || !out8) return fail(PIORAN_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> lk(c->mu);
    std::copy(c->scan_range_chk, c->scan_range_chk + 8, out8);
    return PIORAN_OK;
} catch (...) { return guard_fail(); }

extern "C" int pioran_direct_logl(pioran_ctx* c, int series_id, int B, int Jt, const double* a, const double* b,
                                  const double* cc, const double* d, const double* mu, const double* nu,
                                  double* nll_out, int* info_out) try {
    if (!c || !a || !b || !cc || !d || !nll_out) return fail(PIORAN_EINVAL, "NULL argument");
    if (B < 1 || Jt < 1) return fail(PIORAN_EINVAL, "B and Jt must be >= 1");
    if (is_group(c))   // the parameter vectors are independent: contiguous slices, one per device
        return group_fanout(c, series_id, B, [&](pioran_ctx* ch, int id, int64_t, int beg, int nb) {
            const size_t o = (size_t)beg * Jt;
            return pioran_direct_logl(ch, id, nb, Jt, a + o, b + o, cc + o, d + o, at(mu, beg), at(nu, beg), nll_out + beg, at(info_out, beg));
        });
    PIORAN_COMPUTE_LOCK(c);
    CUDA_TRY(cudaSetDevice(c->device));
    Series* s = get_series(c, series_id);
    if (!s) return fail(PIORAN_EINVAL, "unknown series id %d", series_id);
    const int64_t N = s->N;
    const int nblk = (int)((N + 1 + DNB - 1) / DNB);        // +1: the augmented (y − μ)ᵀ row
    const int64_t ld = (int64_t)nblk * DNB;
    const int nfull = (int)(N / DNB);                       // blocks without padding or the augmented row
    const size_t tab_per = sizeof(double) * 4 * (size_t)Jt * DNB * (size_t)nfull;      // separable factors per block (dense_fill_tables_kernel)
    const size_t mat_per = sizeof(double) * (size_t)ld * (size_t)ld;
    const size_t per = mat_per + tab_per;
    size_t free_b = 0, total_b = 0;
    CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
    const size_t budget = std::min<size_t>(free_b / 2 + c->misc.cap, (size_t)32 << 30);
    if (per > budget)
        return fail(PIORAN_ENOMEM, "dense path needs %zu bytes per parameter vector at N = %lld (free: %zu); use the celerite entry",
                    per, (long long)N, free_b);
    const int chunk = (int)std::min<size_t>((size_t)B, budget / per);
    int rc;
    GenericInputs gi;
    if ((rc = upload_generic(c, B, Jt, N, a, b, cc, d, mu, nu, nullptr, nullptr, gi))) return rc;
    if ((rc = c->misc.ensure(per * (size_t)chunk))) return rc;
    if ((rc = c->out.ensure(sizeof(double) * 3 * (size_t)chunk + sizeof(int) * (size_t)chunk))) return rc;
    double* A = c->misc.as<double>();
    double* tab = A + (size_t)chunk * (size_t)ld * (size_t)ld;
    double* acc = c->out.as<double>();
    double* nll = acc + 2 * (size_t)chunk;
    int* info = reinterpret_cast<int*>(nll + chunk);
    const int ntri = nblk * (nblk + 1) / 2;
    // the separable fill keeps four Jt × 64 factor tables in shared memory (Jt ≤ 97); beyond that every entry is evaluated from
    // the reference's formula, which needs the coefficients only
    size_t fill_smem = sizeof(double) * dense_fill_smem_doubles(Jt);
    const bool fill_tables = fill_smem <= 227 * 1024;
    if (!fill_tables) fill_smem = sizeof(double) * (4 * (size_t)Jt + 2 * DNB);
    if (fill_smem > 227 * 1024) return fail(PIORAN_EUNSUPPORTED, "Jt = %d is too large for the dense path", Jt);
    CUDA_TRY(cudaFuncSetAttribute(dense_fill_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fill_smem));
    if (!c->side) {
        int prio_least = 0, prio_greatest = 0;
        CUDA_TRY(cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest));
        CUDA_TRY(cudaStreamCreateWithPriority(&c->side, cudaStreamNonBlocking, prio_least));
        CUDA_TRY(cudaStreamCreateWithPriority(&c->hi, cudaStreamNonBlocking, prio_greatest));
        CUDA_TRY(cudaEventCreateWithFlags(&c->ev_fact, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&c->ev_bulk, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&c->ev_fill, cudaEventDisableTiming));
        for (cudaEvent_t& e : c->ev_col) CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        CUDA_TRY(cudaFuncSetAttribute(dense_syrk_async_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DENSE_SYRK_ASYNC_SMEM));
    }
    // PIORAN_K4_FILL=direct: every covariance entry from the reference's formula (src/Celerite.jl:42-44) instead of the separable
    // factors — the accuracy cross-check of the fill (tests/tools/fuzz_dense.py)
    static const int fill_direct = [] { const char* e = getenv("PIORAN_K4_FILL"); return e && !strcmp(e, "direct") ? 1 : 0; }();
    cudaEventRecord(c->ev_beg, c->stream);
    for (int th0 = 0; th0 < B; th0 += chunk) {
        const int nb = std::min(chunk, B - th0);
        CUDA_TRY(cudaMemsetAsync(acc, 0, sizeof(double) * 3 * (size_t)chunk + sizeof(int) * (size_t)chunk, c->stream));
        if (nfull > 0 && fill_tables && !fill_direct) {
            dense_fill_tables_kernel<<<dim3(nfull, nb), 256, 0, c->stream>>>(tab, nfull, s->t, Jt, gi.a, gi.b, gi.c, gi.d, th0);
            c->launches++;
        }
        // the first group's block columns are filled first: its panel chain (nothing else could run beside it) then overlaps the
        // fill of the rest (PIORAN_K4_FILL_SPLIT=0: one launch)
        static const bool fill_split = [] { const char* e = getenv("PIORAN_K4_FILL_SPLIT"); return !(e && !strcmp(e, "0")); }();
        // PIORAN_K4_GROUP: panels per group of the factorisation below (1 … 8, default 4)
        static const int G = [] { const char* e = getenv("PIORAN_K4_GROUP"); const int g = e ? atoi(e) : 4; return g >= 1 && g <= 8 ? g : 4; }();
        const bool split = fill_split && nblk > 2 * G;
        const int fdir = fill_direct || !fill_tables;
        if (split) {
            const int mt = nblk - G;
            dense_fill_kernel<<<dim3(nblk * G, nb), 256, fill_smem, c->stream>>>(A, ld, N, s->t, s->y, s->s2, Jt, gi.a, gi.b, gi.c,
                                                                                 gi.d, gi.mu, gi.nu, th0, tab, nfull, fdir, 1, G);
            CUDA_TRY(cudaEventRecord(c->ev_join, c->stream));
            dense_fill_kernel<<<dim3(mt * (mt + 1) / 2, nb), 256, fill_smem, c->stream>>>(A, ld, N, s->t, s->y, s->s2, Jt, gi.a, gi.b, gi.c,
                                                                                         gi.d, gi.mu, gi.nu, th0, tab, nfull, fdir, 2, G);
            c->launches += 2;
        } else {
            dense_fill_kernel<<<dim3(ntri, nb), 256, fill_smem, c->stream>>>(A, ld, N, s->t, s->y, s->s2, Jt, gi.a, gi.b, gi.c,
                                                                             gi.d, gi.mu, gi.nu, th0, tab, nfull, fdir, 0, G);
            c->launches++;
            CUDA_TRY(cudaEventRecord(c->ev_join, c->stream));
        }
        CUDA_TRY(cudaEventRecord(c->ev_fill, c->stream));
        // Look-ahead over two streams (round 2): the panel chain (potrf, trsm and the narrow updates inside a group of panels and
        // onto the NEXT group's block columns) runs on a high-priority stream; the bulk of a group's trailing update (the blocks
        // behind the next group) runs on a low-priority side stream as soon as the group is factorised, beside the factorisation
        // of the next group.  The narrow updates onto the next group's columns wait for the previous bulk (they read-modify-write
        // tiles it wrote); consecutive bulks are ordered by their stream.
        cudaStream_t S1 = c->hi, S2 = c->side;
        static const bool syrk_async = [] { const char* e = getenv("PIORAN_K4_SYRK"); return !(e && !strcmp(e, "regs")); }();
        auto syrk = [&](dim3 grid, cudaStream_t st, int kb_, int kw_, int j0_, int narrow_) {
            if (syrk_async) dense_syrk_async_kernel<<<grid, 256, DENSE_SYRK_ASYNC_SMEM, st>>>(A, ld, kb_, kw_, j0_, narrow_);
            else dense_syrk_kernel<<<grid, 256, 0, st>>>(A, ld, kb_, kw_, j0_, narrow_);
            c->launches++;
        };
        bool bulk_pending = false;
        CUDA_TRY(cudaStreamWaitEvent(S1, c->ev_join, 0));      // the fill of the first group's columns (and everything before it) precedes the chain
        // PIORAN_K4_GROUP0: size of the FIRST group (default: G).  Nothing runs beside its chain, so a shorter first group hands
        // the side stream its first bulk earlier — measured: 8.92 (4) / 8.98 (3) / 9.02 (2) / 9.14 ms (1); the shorter bulk then
        // ends before the second group's chain does.
        static const int G0 = [] { const char* e = getenv("PIORAN_K4_GROUP0"); const int g = e ? atoi(e) : G; return g >= 1 && g <= G ? g : G; }();
        // Of the updates onto the next group's block columns only the FIRST column's is on the panel chain (the next potrf needs
        // it); the others go to the side stream ahead of the bulk, and the chain waits for column c's just before it updates
        // that column itself (PIORAN_K4_SIDE_NARROW=0: all of them on the chain).
        static const bool side_narrow = [] { const char* e = getenv("PIORAN_K4_SIDE_NARROW"); return !(e && !strcmp(e, "0")); }();
        bool col_pending[8] = {false, false, false, false, false, false, false, false};   // next-group column c updated on the side stream
        // PIORAN_K4_TRACE=1: time stamps of the group boundaries on both streams, printed to stderr (development aid)
        static const bool trace = [] { const char* e = getenv("PIORAN_K4_TRACE"); return e && !strcmp(e, "1"); }();
        std::vector<std::pair<std::string, cudaEvent_t>> marks;
        auto mark = [&](const char* what, int kb_, cudaStream_t st) {
            if (!trace) return;
            cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, st);
            marks.emplace_back(std::string(what) + " " + std::to_string(kb_), e);
        };
        mark("start (fill queued)", 0, c->stream);
        // Groups of G panels: inside a group every panel is applied to the next block column alone (narrow update with all the
        // group's panels so far), so that a trailing tile is read and written once per G panels.
        for (int kb = 0; kb < nblk;) {
            const int Gp = std::min(kb == 0 ? G0 : G, nblk - kb);
            bool done = false;
            for (int g = 0; g < Gp; g++) {
                const int k = kb + g;
                dense_potrf_kernel<<<dim3(1, nb), 256, 0, S1>>>(A, ld, N, k, acc, info);
                c->launches++;
                const int m = nblk - k - 1;         // block rows below panel k
                if (m == 0) { done = true; break; }
                dense_trsm_kernel<<<dim3(m, nb), DNB, 0, S1>>>(A, ld, k);
                c->launches++;
                if (g < Gp - 1) {                   // the group's panels so far onto block column k+1 (rows ≥ k+1)
                    if (col_pending[g + 1]) {       // … after the previous group's update of that column
                        CUDA_TRY(cudaStreamWaitEvent(S1, c->ev_col[g + 1], 0));
                        col_pending[g + 1] = false;
                    }
                    syrk(dim3(m, nb), S1, kb, g + 1, k + 1, 1);
                }
            }
            mark("chain of group done, kb =", kb, S1);
            const int rem = nblk - (kb + Gp);       // blocks behind the group
            if (done || rem <= 0) break;
            const int nextG = std::min(G, rem);
            const bool bulk = rem > nextG;
            const int nside = side_narrow ? nextG - 1 : 0;      // next-group columns 1 … nside on the side stream
            if (kb == 0 && split) {                 // everything behind the first group needs the rest of the fill
                CUDA_TRY(cudaStreamWaitEvent(S1, c->ev_fill, 0));
                CUDA_TRY(cudaStreamWaitEvent(S2, c->ev_fill, 0));
            }
            if (bulk || nside > 0) {
                CUDA_TRY(cudaEventRecord(c->ev_fact, S1));
                CUDA_TRY(cudaStreamWaitEvent(S2, c->ev_fact, 0));
            }
            for (int cidx = 1; cidx <= nside; cidx++) {          // (the side stream is in order: these follow the previous bulk)
                syrk(dim3(rem - cidx, nb), S2, kb, Gp, kb + Gp + cidx, 1);
                CUDA_TRY(cudaEventRecord(c->ev_col[cidx], S2));
                col_pending[cidx] = true;
            }
            if (bulk) {                             // all of the group's panels onto the blocks behind the NEXT group, on the side stream
                const int mb = rem - nextG;
                syrk(dim3(mb * (mb + 1) / 2, nb), S2, kb, Gp, kb + Gp + nextG, 0);
            }
            if (bulk_pending) CUDA_TRY(cudaStreamWaitEvent(S1, c->ev_bulk, 0));      // the previous bulk wrote the tiles updated next
            for (int cidx = 0; cidx < nextG; cidx++) {   // … and onto the next group's block columns (rows from the column's own block on)
                if (cidx >= 1 && cidx <= nside) continue;
                syrk(dim3(rem - cidx, nb), S1, kb, Gp, kb + Gp + cidx, 1);
            }
            if (bulk || nside > 0) CUDA_TRY(cudaEventRecord(c->ev_bulk, S2));
            if (bulk || nside > 0) mark("side stream (narrow + bulk) done, kb =", kb, S2);
            mark("first next-group column updated, kb =", kb, S1);
            bulk_pending = bulk || nside > 0;
            kb += Gp;
        }
        if (bulk_pending) CUDA_TRY(cudaStreamWaitEvent(S1, c->ev_bulk, 0));
        CUDA_TRY(cudaEventRecord(c->ev_join, S1));
        CUDA_TRY(cudaStreamWaitEvent(c->stream, c->ev_join, 0));
        dense_finish_kernel<<<(nb + 127) / 128, 128, 0, c->stream>>>(acc, info, N, nb, nll);
        c->launches++;
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaMemcpyAsync(nll_out + th0, nll, sizeof(double) * nb, cudaMemcpyDeviceToHost, c->stream));
        if (info_out) CUDA_TRY(cudaMemcpyAsync(info_out + th0, info, sizeof(int) * nb, cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(cudaStreamSynchronize(c->stream));   // the workspace is reused by the next chunk
        for (size_t i = 0; i < marks.size(); i++) {
            float ms = 0.f;
            cudaEventSynchronize(marks[i].second);
            cudaEventElapsedTime(&ms, marks[0].second, marks[i].second);
            fprintf(stderr, "[K4 trace] %8.3f ms  %s\n", ms, marks[i].first.c_str());
            if (i) cudaEventDestroy(marks[i].second);
        }
        if (!marks.empty()) cudaEventDestroy(marks[0].second);
    }
    cudaEventRecord(c->ev_end, c->stream);
    note_kernel(c, KF_DENSE_FINISH);
    return PIORAN_OK;
} catch (...) { return guard_fail(); }
