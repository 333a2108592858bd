// capi.cu — the extern "C" boundary declared in include/ezkl_b200.h: process-wide configuration, the devices of the process,
// per-(thread, device) contexts, the base-table registry with its replicas, host<->device staging, the device workers behind the
// multi-device host-pointer paths and the host-side tail (point normalisation).  No CPU fallback lives here: every compute
// entry point needs an initialised CUDA device and fails with an error code otherwise.
#include <atomic>
#include <condition_variable>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "../../include/ezkl_b200.h"
#include "../../include/ezkl_b200_parts.h"
#include "msm.cuh"
#include "ntt.cuh"
#include "poly.cuh"
#include "quotient.cuh"

namespace b200 {

// ---- configuration: the environment is read once, in b200_init --------------------------------------------------------------
static Config g_cfg;
const Config& config() { return g_cfg; }
static int env_int(const char* name, int dflt) { const char* e = getenv(name); return e ? atoi(e) : dflt; }
static void read_config() {
    Config c;
    if (const char* e = getenv("B200_WS_BUDGET_MB")) c.ws_budget_call = (size_t)atol(e) << 20;
    if (const char* e = getenv("B200_WS_TOTAL_MB")) c.ws_budget_total = (size_t)atol(e) << 20;
    c.ntt_v1 = env_int("B200_NTT_V", 2) == 1;
    c.ntt_logg = env_int("B200_NTT_LOGG", -1);
    c.ntt_threads = env_int("B200_NTT_THREADS", 0);
    c.ntt_nofull = getenv("B200_NTT_NOFULL") != nullptr;
    c.msm_reduce_m = env_int("B200_MSM_REDUCE_M", 0);
    c.msm_reduce2 = env_int("B200_MSM_REDUCE2", 0);
    c.msm_reduce_threads = env_int("B200_MSM_REDUCE_THREADS", 0);
    c.shard_min_logn = env_int("B200_SHARD_MIN_LOGN", 22);
    g_cfg = c;
}

// ---- process state ----------------------------------------------------------------------------------------------------------------
static constexpr int MAX_DEV = 8;
struct DeviceState { int id = -1; NttContext ntt; };
static DeviceState g_devs[MAX_DEV];
static std::atomic<int> g_ndev{0};
static std::atomic<bool> g_inited{false};
static std::atomic<int> g_active{0};            // entry points in flight (b200_shutdown waits for them)
static std::atomic<uint64_t> g_epoch{1};        // bumped by b200_shutdown: contexts of an older epoch are gone
static std::atomic<uint64_t> g_launches{0};
static std::mutex g_mu;                         // tables, plans, context registry

// One registered base vector: a window-precomputed table replica per device of the process.
struct BaseSet {
    size_t n = 0; int c = 0, W = 0;
    MsmTable* t[MAX_DEV] = {};
};
static std::unordered_map<uint64_t, BaseSet*> g_tables;
static uint64_t g_next_handle = 1;

// Per (calling thread, device) context: stream, scratch, staging.  The registry owns the objects so that b200_shutdown can
// release the device memory of threads that are still alive (or already gone).
struct Ctx {
    int slot = 0, dev = 0;
    cudaStream_t stream = nullptr;
    MsmWorkspace msm_ws;
    PolyWorkspace poly_ws;
    QuotientWorkspace quot_ws;
    StagingRing ring;
    DevBuf stage_a, stage_b, stage_c, small;
    // pinned bounce buffers for large pageable <-> device copies (two slots, pipelined against the DMA engine)
    uint8_t* bounce[2] = {nullptr, nullptr};
    cudaEvent_t bounce_ev[2] = {nullptr, nullptr};
    // the scratch above is per thread, not per stream: a call on another stream first waits for the previous call's work
    cudaEvent_t last_ev = nullptr;
    cudaStream_t last_stream = nullptr;
    bool has_last = false;
    void release() {
        cudaSetDevice(dev);
        DevBuf* bufs[] = {&msm_ws.counts, &msm_ws.offs, &msm_ws.ents, &msm_ws.subs, &msm_ws.sums, &msm_ws.misc, &poly_ws.scratch, &quot_ws.prog,
                          &stage_a, &stage_b, &stage_c, &small};
        for (DevBuf* b : bufs) b->release();
        ring.release(); poly_ws.ring.release(); quot_ws.ring.release();
        for (int i = 0; i < 2; ++i) { if (bounce[i]) cudaFreeHost(bounce[i]); if (bounce_ev[i]) cudaEventDestroy(bounce_ev[i]); bounce[i] = nullptr; bounce_ev[i] = nullptr; }
        if (last_ev) cudaEventDestroy(last_ev);
        if (stream) cudaStreamDestroy(stream);
        last_ev = nullptr; stream = nullptr;
    }
};
static std::vector<Ctx*> g_ctxs;
static std::atomic<int> g_nctx{0};

// restores the calling thread's current device on every exit of a scope that switches devices with cudaSetDevice
struct CurrentDevice {
    int prev = 0;
    CurrentDevice() { cudaGetDevice(&prev); }
    ~CurrentDevice() { cudaSetDevice(prev); }
};

// waits for the work that may still read a registered base vector, then frees every replica on its own device
static void free_bases(BaseSet* bs) {
    CurrentDevice keep;
    for (int s = 0; s < MAX_DEV; ++s) if (bs->t[s]) { cudaSetDevice(bs->t[s]->device); cudaDeviceSynchronize(); msm_table_free(bs->t[s]); delete bs->t[s]; }
    delete bs;
}

struct TlCtx {
    Ctx* c[MAX_DEV] = {};
    uint64_t epoch = 0;
    ~TlCtx() {                                   // a calling thread ends: give its device memory back
        if (epoch != g_epoch.load() || !g_inited.load()) return;
        std::lock_guard<std::mutex> lk(g_mu);
        if (epoch != g_epoch.load()) return;
        CurrentDevice keep;
        for (int s = 0; s < MAX_DEV; ++s) if (c[s]) {
            for (size_t i = 0; i < g_ctxs.size(); ++i) if (g_ctxs[i] == c[s]) { g_ctxs.erase(g_ctxs.begin() + i); break; }
            c[s]->release(); delete c[s]; g_nctx--;
        }
    }
};
static thread_local TlCtx tl;

struct CallGuard {
    bool ok;
    CallGuard() { g_active++; ok = g_inited.load(); if (!ok) set_error("b200: not initialised (call b200_init first)"); }
    ~CallGuard() { g_active--; }
};

static int get_ctx(Ctx** out, int slot = 0) {
    if (!g_inited.load()) { set_error("b200: not initialised (call b200_init first)"); return -3; }
    const uint64_t ep = g_epoch.load();
    if (tl.epoch != ep) { for (int s = 0; s < MAX_DEV; ++s) tl.c[s] = nullptr; tl.epoch = ep; }
    B200_CHECK(slot >= 0 && slot < g_ndev.load(), -1, "b200: device slot %d out of range", slot);
    if (!tl.c[slot]) {
        Ctx* c = new Ctx();
        c->slot = slot; c->dev = g_devs[slot].id;
        int cur = 0; cudaGetDevice(&cur);
        cudaError_t e = cudaSetDevice(c->dev);
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->last_ev, cudaEventDisableTiming);
        if (g_ndev.load() > 1) cudaSetDevice(cur);
        if (e != cudaSuccess) { set_error("b200: context creation on device %d failed: %s", c->dev, cudaGetErrorString(e)); delete c; return -2; }
        std::lock_guard<std::mutex> lk(g_mu);
        g_ctxs.push_back(c); g_nctx++;
        tl.c[slot] = c;
    }
    *out = tl.c[slot];
    return 0;
}
// which device of the process a device pointer lives on (single-device processes skip the query)
static int slot_of(const void* dptr) {
    const int nd = g_ndev.load();
    if (nd <= 1 || !dptr) return 0;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, dptr) != cudaSuccess) { cudaGetLastError(); return 0; }
    for (int s = 0; s < nd; ++s) if (g_devs[s].id == at.device) return s;
    return 0;
}
// makes the context's device current for the duration of an entry point (multi-device processes only; a single-device process
// keeps the caller's current device, which is the one b200_init selected)
struct DevGuard {
    int prev = -1;
    explicit DevGuard(const Ctx* c) { if (g_ndev.load() > 1) { cudaGetDevice(&prev); if (prev != c->dev) cudaSetDevice(c->dev); else prev = -1; } }
    ~DevGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
// stream of a call + ordering of the per-thread scratch across streams
struct StreamScope {
    Ctx* c; cudaStream_t st;
    StreamScope(Ctx* c_, void* user) : c(c_), st(user ? (cudaStream_t)user : c_->stream) {
        if (c->has_last && c->last_stream != st) cudaStreamWaitEvent(st, c->last_ev, 0);
    }
    ~StreamScope() { if (cudaEventRecord(c->last_ev, st) == cudaSuccess) { c->last_stream = st; c->has_last = true; } else cudaGetLastError(); }
};
#define B200_ENTER(c, dptr)                                                \
    CallGuard _cg; if (!_cg.ok) return -3;                                 \
    Ctx* c; if (int _rc = get_ctx(&c, slot_of(dptr))) return _rc;          \
    DevGuard _dg(c)

// device scratch a single call may take, for batch splitting
static size_t call_budget() {
    if (g_cfg.ws_budget_call) return g_cfg.ws_budget_call;
    const int nd = g_ndev.load() > 0 ? g_ndev.load() : 1;
    const int per_dev = (g_nctx.load() + nd - 1) / nd;          // calling threads holding scratch on one device
    const size_t per = g_cfg.ws_budget_total / (size_t)(per_dev > 0 ? per_dev : 1);
    const size_t lo = (size_t)256 << 20, hi = (size_t)12 << 30;
    return per < lo ? lo : (per > hi ? hi : per);
}
// host Fr values arrive with 8-byte alignment (Rust / C callers); Fr is alignas(16), so always copy bytewise
static inline Fr as_fr(const b200_fr* p) { Fr r; memcpy(&r, p, sizeof r); return r; }

// NTT pre / post scaling as the ABI passes it (mode 0 none, 1 constant c[0], 3 cycle c[i mod 3]); -1 on a bad mode or missing constants
static int decode_scales(int pre_mode, const b200_fr* pre, int post_mode, const b200_fr* post, NttScale* a, NttScale* b) {
    B200_CHECK((pre_mode == 0 || pre_mode == 1 || pre_mode == 3) && (post_mode == 0 || post_mode == 1 || post_mode == 3), -1, "ntt: scale mode must be 0, 1 or 3");
    B200_CHECK((pre_mode == 0 || pre) && (post_mode == 0 || post), -1, "ntt: scale constants missing");
    a->mode = pre_mode; b->mode = post_mode;
    for (int i = 0; i < pre_mode; ++i) a->c[i] = as_fr(pre + i);
    for (int i = 0; i < post_mode; ++i) b->c[i] = as_fr(post + i);
    return 0;
}
// coeff_to_extended's pre-scale: coefficient i times zeta^(i mod 3) (zeta is a cube root of unity)
static NttScale coset_scale(const Fr& zeta) {
    NttScale s;
    s.mode = 3; s.c[0] = fp_one<FrTag>(); s.c[1] = zeta; s.c[2] = zeta * zeta;
    return s;
}
// extended_to_coeff's post-scale: the inverse transform's divisor times zeta^-(i mod 3), where zeta^-1 = zeta^2
static NttScale coset_unscale(const Fr& zeta, const Fr& divisor) {
    NttScale s;
    s.mode = 3; s.c[0] = divisor; s.c[1] = divisor * (zeta * zeta); s.c[2] = divisor * zeta;
    return s;
}

// ---- large host <-> device copies of PAGEABLE caller memory (what a Rust Vec<Fr> is) ------------------------------------------------
// cudaMemcpyAsync from pageable memory runs at 6-7 GB/s on this box (one driver thread copying into its own staging buffer).  Here the
// copy is cut into 16 MiB chunks that four host threads move into a pinned bounce buffer while the DMA engine drains the other one, so
// the PCIe link (Gen5 x16) is fed at memcpy-pool speed.  Small copies keep the plain path.
static constexpr size_t BOUNCE_BYTES = (size_t)16 << 20;
struct HostSeg { uint8_t* p; size_t bytes; };          // one caller buffer (a column); a list of them maps onto ONE contiguous device range
// copies bytes [lo, hi) of the virtual concatenation of `segs` between the caller's buffers and `flat` (the pinned slot, offset 0 = byte lo0)
static void seg_copy_range(const HostSeg* segs, size_t nsegs, size_t lo0, size_t lo, size_t hi, uint8_t* flat, bool to_flat) {
    size_t pos = 0;
    for (size_t i = 0; i < nsegs && pos < hi; ++i) {
        const size_t s0 = pos, s1 = pos + segs[i].bytes;
        pos = s1;
        if (s1 <= lo) continue;
        const size_t a = lo > s0 ? lo : s0, b = hi < s1 ? hi : s1;
        if (to_flat) memcpy(flat + (a - lo0), segs[i].p + (a - s0), b - a);
        else memcpy(segs[i].p + (a - s0), flat + (a - lo0), b - a);
    }
}
static void seg_copy_parallel(const HostSeg* segs, size_t nsegs, size_t lo, size_t hi, uint8_t* flat, bool to_flat) {
    const int T = 4;
    const size_t bytes = hi - lo;
    if (bytes < ((size_t)2 << 20)) { seg_copy_range(segs, nsegs, lo, lo, hi, flat, to_flat); return; }
    const size_t part = ((bytes / T) + 4095) & ~(size_t)4095;
    std::thread th[T - 1];
    for (int i = 1; i < T; ++i) {
        const size_t a = lo + part * i, b = a + part < hi ? a + part : hi;
        if (a < b) th[i - 1] = std::thread([=] { seg_copy_range(segs, nsegs, lo, a, b, flat, to_flat); });
    }
    seg_copy_range(segs, nsegs, lo, lo, lo + part < hi ? lo + part : hi, flat, to_flat);
    for (int i = 1; i < T; ++i) if (th[i - 1].joinable()) th[i - 1].join();
}
static int bounce_ready(Ctx* c) {
    if (c->bounce[0]) return 0;
    for (int i = 0; i < 2; ++i) {
        B200_CUDA(cudaMallocHost((void**)&c->bounce[i], BOUNCE_BYTES));
        B200_CUDA(cudaEventCreateWithFlags(&c->bounce_ev[i], cudaEventDisableTiming));
    }
    return 0;
}
// caller buffers -> contiguous device range.  When the call returns every SOURCE has been read; the device copies are ordered on `st`.
static int h2d_segments(Ctx* c, void* d_dst, const HostSeg* segs, size_t nsegs, cudaStream_t st) {
    size_t total = 0;
    for (size_t i = 0; i < nsegs; ++i) total += segs[i].bytes;
    if (total < ((size_t)8 << 20)) {
        size_t off = 0;
        for (size_t i = 0; i < nsegs; ++i) { B200_CUDA(cudaMemcpyAsync((uint8_t*)d_dst + off, segs[i].p, segs[i].bytes, cudaMemcpyHostToDevice, st)); off += segs[i].bytes; }
        return 0;
    }
    if (int rc = bounce_ready(c)) return rc;
    int slot = 0;
    for (size_t off = 0; off < total; off += BOUNCE_BYTES, slot ^= 1) {
        const size_t nb = total - off < BOUNCE_BYTES ? total - off : BOUNCE_BYTES;
        B200_CUDA(cudaEventSynchronize(c->bounce_ev[slot]));                       // the DMA that last read this slot is done
        seg_copy_parallel(segs, nsegs, off, off + nb, c->bounce[slot], true);
        B200_CUDA(cudaMemcpyAsync((uint8_t*)d_dst + off, c->bounce[slot], nb, cudaMemcpyHostToDevice, st));
        B200_CUDA(cudaEventRecord(c->bounce_ev[slot], st));
    }
    return 0;
}
// contiguous device range -> caller buffers.  Synchronous for the host: when the call returns the destinations hold the data.
static int d2h_segments(Ctx* c, const void* d_src, const HostSeg* segs, size_t nsegs, cudaStream_t st) {
    size_t total = 0;
    for (size_t i = 0; i < nsegs; ++i) total += segs[i].bytes;
    if (total < ((size_t)8 << 20)) {
        size_t off = 0;
        for (size_t i = 0; i < nsegs; ++i) { B200_CUDA(cudaMemcpyAsync(segs[i].p, (const uint8_t*)d_src + off, segs[i].bytes, cudaMemcpyDeviceToHost, st)); off += segs[i].bytes; }
        B200_CUDA(cudaStreamSynchronize(st));
        return 0;
    }
    if (int rc = bounce_ready(c)) return rc;
    const size_t nchunks = (total + BOUNCE_BYTES - 1) / BOUNCE_BYTES;
    for (size_t i = 0; i <= nchunks; ++i) {                                        // chunk i's DMA overlaps chunk i-1's host copy
        if (i < nchunks) {
            const size_t off = i * BOUNCE_BYTES, nb = total - off < BOUNCE_BYTES ? total - off : BOUNCE_BYTES;
            B200_CUDA(cudaMemcpyAsync(c->bounce[i & 1], (const uint8_t*)d_src + off, nb, cudaMemcpyDeviceToHost, st));
            B200_CUDA(cudaEventRecord(c->bounce_ev[i & 1], st));
        }
        if (i > 0) {
            const size_t off = (i - 1) * BOUNCE_BYTES, nb = total - off < BOUNCE_BYTES ? total - off : BOUNCE_BYTES;
            B200_CUDA(cudaEventSynchronize(c->bounce_ev[(i - 1) & 1]));
            seg_copy_parallel(segs, nsegs, off, off + nb, c->bounce[(i - 1) & 1], false);
        }
    }
    return 0;
}
// every stride-th element of one caller buffer (count elements of `elem` bytes) -> contiguous device range, through the same pinned
// bounce buffers and pipeline as h2d_segments (a coset part of an extended column).  When the call returns every source element has been read.
static void gather_range(const uint8_t* src, size_t i0, size_t i1, size_t elem, size_t stride_bytes, uint8_t* flat) {
    for (size_t i = i0; i < i1; ++i) memcpy(flat + i * elem, src + i * stride_bytes, elem);
}
static int h2d_strided(Ctx* c, void* d_dst, const uint8_t* src, size_t count, size_t elem, size_t stride, cudaStream_t st) {
    if (int rc = bounce_ready(c)) return rc;
    const size_t per = BOUNCE_BYTES / elem, stride_bytes = stride * elem;
    int slot = 0;
    for (size_t i0 = 0; i0 < count; i0 += per, slot ^= 1) {
        const size_t m = count - i0 < per ? count - i0 : per;
        B200_CUDA(cudaEventSynchronize(c->bounce_ev[slot]));                       // the DMA that last read this slot is done
        const uint8_t* s0 = src + i0 * stride_bytes;
        uint8_t* flat = c->bounce[slot];
        const int T = 4;
        if (m * elem < ((size_t)2 << 20)) gather_range(s0, 0, m, elem, stride_bytes, flat);
        else {
            std::thread th[T - 1];
            const size_t q = (m + T - 1) / T;
            for (int t = 1; t < T; ++t) {
                const size_t a = q * t, b = a + q < m ? a + q : m;
                if (a < b) th[t - 1] = std::thread([=] { gather_range(s0, a, b, elem, stride_bytes, flat); });
            }
            gather_range(s0, 0, q < m ? q : m, elem, stride_bytes, flat);
            for (int t = 1; t < T; ++t) if (th[t - 1].joinable()) th[t - 1].join();
        }
        B200_CUDA(cudaMemcpyAsync((uint8_t*)d_dst + i0 * elem, flat, m * elem, cudaMemcpyHostToDevice, st));
        B200_CUDA(cudaEventRecord(c->bounce_ev[slot], st));
    }
    return 0;
}
static int h2d_one(Ctx* c, void* d_dst, const void* h_src, size_t bytes, cudaStream_t st) { HostSeg s{(uint8_t*)const_cast<void*>(h_src), bytes}; return h2d_segments(c, d_dst, &s, 1, st); }
static int d2h_one(Ctx* c, void* h_dst, const void* d_src, size_t bytes, cudaStream_t st) { HostSeg s{(uint8_t*)h_dst, bytes}; return d2h_segments(c, d_src, &s, 1, st); }

// XYZZ (host) -> normalised Jacobian, one shared inversion (Montgomery's trick over zz*zzz)
static void normalize_host(const G1Xyzz* pts, size_t n, b200_g1_jac* out) {
    std::vector<Fq> prod(n), pref(n);
    Fq acc = fp_one<FqTag>();
    for (size_t i = 0; i < n; ++i) {
        pref[i] = acc;
        if (!g1_is_identity(pts[i])) { prod[i] = pts[i].zz * pts[i].zzz; acc = acc * prod[i]; }
    }
    Fq inv = fp_inv(acc);
    for (size_t i = n; i-- > 0;) {
        G1Jac j;
        if (g1_is_identity(pts[i])) {
            j.x = fp_zero<FqTag>(); j.y = fp_one<FqTag>(); j.z = fp_zero<FqTag>();
        } else {
            Fq t = inv * pref[i];            // 1 / (zz * zzz)
            inv = inv * prod[i];
            Fq zz_inv = t * pts[i].zzz, zzz_inv = t * pts[i].zz;
            j.x = pts[i].x * zz_inv; j.y = pts[i].y * zzz_inv; j.z = fp_one<FqTag>();
        }
        memcpy(&out[i], &j, sizeof j);
    }
}

// ---- profiling (CUDA events on the launching stream) ------------------------------------------------------------
static std::atomic<bool> g_prof{false};
struct ProfRec { int cls; cudaEvent_t e0, e1; };
static std::mutex g_prof_mu;
static std::vector<ProfRec> g_prof_recs;
static thread_local std::vector<ProfRec> tl_prof_open;
bool prof_enabled() { return g_prof.load(std::memory_order_relaxed); }
void prof_mark(int cls, cudaStream_t st, bool begin) {
    if (begin) {
        ProfRec r; r.cls = cls;
        cudaEventCreate(&r.e0); cudaEventCreate(&r.e1);
        cudaEventRecord(r.e0, st);
        tl_prof_open.push_back(r);
    } else {
        for (size_t i = tl_prof_open.size(); i-- > 0;) {
            if (tl_prof_open[i].cls == cls) {
                ProfRec r = tl_prof_open[i];
                tl_prof_open.erase(tl_prof_open.begin() + i);
                cudaEventRecord(r.e1, st);
                std::lock_guard<std::mutex> lk(g_prof_mu);
                g_prof_recs.push_back(r);
                break;
            }
        }
    }
}

static BaseSet* find_bases(uint64_t h) {
    std::lock_guard<std::mutex> lk(g_mu);
    auto it = g_tables.find(h);
    return it == g_tables.end() ? nullptr : it->second;
}

static NttPlan* warm_plan(int slot, uint32_t log_n, const Fr& omega, cudaStream_t st) {
    std::lock_guard<std::mutex> lk(g_mu);
    NttContext& nc = g_devs[slot].ntt;
    size_t before = nc.plans.size();
    NttPlan* p = nc.get(log_n, omega, st);
    if (p && nc.plans.size() != before) cudaStreamSynchronize(st);   // tables complete before other threads use them
    return p;
}

static int ntt_call(Ctx* c, const Fr* src, size_t src_stride, size_t n_in, Fr* tmp, Fr* dst, size_t dst_stride, uint32_t log_n,
                    const Fr& omega, const NttScale& pre, const NttScale& post, int batch, cudaStream_t st) {
    if (log_n < 1 || log_n > 28) { set_error("ntt: log_n = %u out of range [1, 28]", log_n); return -1; }
    NttPlan* plan = warm_plan(c->slot, log_n, omega, st);         // looked up / built under g_mu; the vector of plans is never touched unlocked
    if (!plan) return -2;
    int rc = ntt_run(plan, src, src_stride, n_in, tmp, (size_t)1 << log_n, dst, dst_stride, log_n, omega, pre, post, batch, st);
    if (!rc) g_launches += (uint64_t)ntt_launches_per_run(log_n);
    return rc;
}

// ---- device workers: one host thread per extra device, so that the host-pointer entry points of a multi-device process drive
//      every PCIe link and every GPU at once (a single thread staging pageable memory serialises on its own copies) ------------
struct Job { std::function<int()> fn; int rc = 0; std::string err; bool done = false; };
struct Worker {
    std::thread th; std::mutex mu; std::condition_variable cv; std::deque<Job*> q; bool stop = false;
};
static Worker* g_workers[MAX_DEV] = {};
static std::mutex g_multi_mu;                    // multi-device host-pointer operations take every device: one at a time
static std::mutex g_done_mu;
static std::condition_variable g_done_cv;
static void worker_main(Worker* w, int dev) {
    cudaSetDevice(dev);
    for (;;) {
        Job* j;
        {
            std::unique_lock<std::mutex> lk(w->mu);
            w->cv.wait(lk, [&] { return w->stop || !w->q.empty(); });
            if (w->q.empty()) return;
            j = w->q.front(); w->q.pop_front();
        }
        j->rc = j->fn();
        if (j->rc) j->err = get_error();
        { std::lock_guard<std::mutex> lk(g_done_mu); j->done = true; }
        g_done_cv.notify_all();
    }
}
// fn(slot) for every slot < nslots: slot 0 on the calling thread, the others on their device workers; first failure wins
static int run_on_slots(int nslots, const std::function<int(int)>& fn) {
    std::vector<Job> jobs(nslots);
    for (int s = 1; s < nslots; ++s) {
        jobs[s].fn = [&fn, s] { return fn(s); };
        std::lock_guard<std::mutex> lk(g_workers[s]->mu);
        g_workers[s]->q.push_back(&jobs[s]);
        g_workers[s]->cv.notify_one();
    }
    int rc = fn(0);
    std::string err = rc ? get_error() : "";
    {
        std::unique_lock<std::mutex> lk(g_done_mu);
        g_done_cv.wait(lk, [&] { for (int s = 1; s < nslots; ++s) if (!jobs[s].done) return false; return true; });
    }
    for (int s = 1; s < nslots && !rc; ++s) if (jobs[s].rc) { rc = jobs[s].rc; err = jobs[s].err; }
    if (rc) set_error("%s", err.c_str());
    return rc;
}

// ---- MSM building blocks ------------------------------------------------------------------------------------------------------
// device-resident columns on the context's device -> XYZZ partial sums on that device (sub-batches bounded by the scratch budget)
static int msm_dev_on(Ctx* c, const BaseSet* bs, const Fr* sc, size_t n, size_t stride, size_t batch, size_t base_off, G1Xyzz* out, cudaStream_t st) {
    const MsmTable* t = bs->t[c->slot];
    B200_CHECK(t, -1, "msm: the bases have no replica on device slot %d", c->slot);
    const size_t per_col = msm_workspace_per_column(*t, n);
    size_t sub = call_budget() / (per_col ? per_col : 1);
    if (sub < 1) sub = 1;
    if (sub > 4096) sub = 4096;
    for (size_t b0 = 0; b0 < batch; b0 += sub) {
        const size_t nb = batch - b0 < sub ? batch - b0 : sub;
        if (int rc = msm_run(*t, sc + b0 * stride, n, stride, (int)nb, out + b0, c->msm_ws, st, base_off)) return rc;
        g_launches += (uint64_t)msm_launches_per_run();
    }
    return 0;
}
// host columns cols[j][base_off .. base_off + n) for j < count -> XYZZ partial sums on the host, staged in sub-batches
static int msm_host_on(Ctx* c, const BaseSet* bs, const b200_fr* const* cols, size_t count, size_t n, size_t base_off, G1Xyzz* h_out) {
    if (count == 0) return 0;
    if (n == 0) { memset(h_out, 0, sizeof(G1Xyzz) * count); return 0; }
    DevGuard dg(c);
    size_t sub = call_budget() / (sizeof(Fr) * n * 2);
    if (sub < 1) sub = 1;
    if (sub > count) sub = count;
    if (c->stage_a.ensure(sizeof(Fr) * n * sub) || c->small.ensure(sizeof(G1Xyzz) * count)) return -2;
    StreamScope ss(c, nullptr);
    for (size_t b0 = 0; b0 < count; b0 += sub) {
        const size_t nb = count - b0 < sub ? count - b0 : sub;
        std::vector<HostSeg> segs(nb);
        for (size_t b = 0; b < nb; ++b) {
            B200_CHECK(cols[b0 + b], -1, "msm: scalars[%zu] is null", b0 + b);
            segs[b] = HostSeg{(uint8_t*)const_cast<b200_fr*>(cols[b0 + b] + base_off), sizeof(Fr) * n};
        }
        if (int rc = h2d_segments(c, c->stage_a.p, segs.data(), nb, ss.st)) return rc;
        if (int rc = msm_dev_on(c, bs, c->stage_a.as<Fr>(), n, n, nb, base_off, c->small.as<G1Xyzz>() + b0, ss.st)) return rc;
        if (b0 + nb < count) B200_CUDA(cudaStreamSynchronize(ss.st));      // the staging buffer is reused by the next sub-batch
    }
    return d2h_one(c, h_out, c->small.p, sizeof(G1Xyzz) * count, ss.st);
}
static void slice_bounds(size_t n, int g, int world, size_t* lo, size_t* hi) {
    const size_t base = n / world, rem = n % world;
    *lo = (size_t)g * base + ((size_t)g < rem ? (size_t)g : rem);
    *hi = *lo + base + ((size_t)g < rem ? 1 : 0);
}

}  // namespace b200

using namespace b200;

#pragma GCC visibility push(default)
extern "C" {

int b200_version(void) { return 200; }
const char* b200_last_error(void) { return get_error(); }
uint64_t b200_launch_count(void) { return g_launches.load(); }
int b200_device_count(void) { return g_inited.load() ? g_ndev.load() : 0; }

static int init_devices(const int* ids, int n) {
    if (g_inited.load()) {               // idempotent for the same device set; a different set needs b200_shutdown first
        bool same = n == g_ndev.load();
        for (int s = 0; same && s < n; ++s) same = ids[s] < 0 || ids[s] == g_devs[s].id;
        B200_CHECK(same, -1, "b200_init: already initialised with another device set (call b200_shutdown first)");
        return 0;
    }
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) { set_error("b200_init: no CUDA device (%s)", cudaGetErrorString(e)); return -2; }
    read_config();
    int first = 0;
    for (int s = 0; s < n; ++s) {
        int device = ids[s];
        if (device < 0) { B200_CUDA(cudaGetDevice(&device)); }
        B200_CHECK(device < count, -1, "b200_init: device %d >= device count %d", device, count);
        cudaDeviceProp prop;
        B200_CUDA(cudaGetDeviceProperties(&prop, device));
        B200_CHECK(prop.major == 10, -2, "b200_init: device %d is sm_%d%d; this library carries sm_100a code only", device, prop.major, prop.minor);
        B200_CUDA(cudaSetDevice(device));
        B200_CUDA(cudaFree(0));
        g_devs[s].id = device;
        if (s == 0) first = device;
    }
    for (int s = 0; s < n && n > 1; ++s) {          // NVLink peer mappings: every device may load from / store to every other
        B200_CUDA(cudaSetDevice(g_devs[s].id));
        for (int q = 0; q < n; ++q) if (q != s) {
            cudaError_t pe = cudaDeviceEnablePeerAccess(g_devs[q].id, 0);
            if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) { set_error("b200_init: no peer access %d -> %d (%s)", g_devs[s].id, g_devs[q].id, cudaGetErrorString(pe)); return -2; }
            cudaGetLastError();
        }
    }
    B200_CUDA(cudaSetDevice(first));
    g_ndev.store(n);
    for (int s = 1; s < n; ++s) {
        g_workers[s] = new Worker();
        g_workers[s]->th = std::thread(worker_main, g_workers[s], g_devs[s].id);
    }
    g_inited.store(true);
    return 0;
}
int b200_init(int device) { return init_devices(&device, 1); }
int b200_init_multi(int n_devices) {
    B200_CHECK(n_devices == 1 || n_devices == 2 || n_devices == 4 || n_devices == 8, -1, "b200_init_multi: n_devices = %d, want 1, 2, 4 or 8", n_devices);
    int ids[MAX_DEV];
    for (int i = 0; i < n_devices; ++i) ids[i] = i;
    return init_devices(ids, n_devices);
}

void b200_shutdown(void) {
    if (!g_inited.exchange(false)) return;                    // new entry points now fail with -3
    while (g_active.load() > 0) std::this_thread::yield();    // calls in flight on other threads finish first
    for (int s = 1; s < MAX_DEV; ++s) if (g_workers[s]) {
        { std::lock_guard<std::mutex> lk(g_workers[s]->mu); g_workers[s]->stop = true; }
        g_workers[s]->cv.notify_all();
        g_workers[s]->th.join();
        delete g_workers[s]; g_workers[s] = nullptr;
    }
    std::lock_guard<std::mutex> lk(g_mu);
    CurrentDevice keep;
    for (auto& kv : g_tables) free_bases(kv.second);
    g_tables.clear();
    for (Ctx* c : g_ctxs) { c->release(); delete c; }          // streams and scratch of every calling thread, alive or not
    g_ctxs.clear(); g_nctx.store(0);
    g_epoch++;
    for (int s = 0; s < g_ndev.load(); ++s) { cudaSetDevice(g_devs[s].id); g_devs[s].ntt.release(); g_devs[s].id = -1; }
    g_ndev.store(0);
}

// ---- profiling -------------------------------------------------------------------------------------------------
int b200_profile_enable(int on) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    for (auto& r : g_prof_recs) { cudaEventDestroy(r.e0); cudaEventDestroy(r.e1); }
    g_prof_recs.clear();
    g_prof.store(on != 0);
    return 0;
}
int b200_profile_read(int cls, double* total_ms, uint64_t* count) {
    B200_CHECK(cls >= 0 && cls < PROF_NCLASS && total_ms && count, -1, "profile_read: bad argument");
    {
        CurrentDevice keep;
        for (int s = 0; s < g_ndev.load(); ++s) { B200_CUDA(cudaSetDevice(g_devs[s].id)); B200_CUDA(cudaDeviceSynchronize()); }
    }
    std::lock_guard<std::mutex> lk(g_prof_mu);
    double ms = 0; uint64_t n = 0;
    for (auto& r : g_prof_recs) if (r.cls == cls) { float t = 0; if (cudaEventElapsedTime(&t, r.e0, r.e1) == cudaSuccess) { ms += t; ++n; } else cudaGetLastError(); }
    *total_ms = ms; *count = n;
    return 0;
}

// ---- memory helpers ---------------------------------------------------------------------------------------
int b200_dev_alloc(void** d_ptr, size_t bytes) { B200_ENTER(c, nullptr); B200_CUDA(cudaMalloc(d_ptr, bytes)); return 0; }
int b200_dev_alloc_on(int slot, void** d_ptr, size_t bytes) {
    CallGuard cg; if (!cg.ok) return -3;
    Ctx* c; if (int rc = get_ctx(&c, slot)) return rc;
    DevGuard dg(c);
    B200_CUDA(cudaMalloc(d_ptr, bytes));
    return 0;
}
int b200_dev_free(void* d_ptr) { B200_CUDA(cudaFree(d_ptr)); return 0; }
int b200_dev_upload(void* d_dst, const void* h_src, size_t bytes) {
    B200_ENTER(c, d_dst);
    B200_CUDA(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, c->stream));
    B200_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
}
int b200_dev_upload_async(void* d_dst, const void* h_src, size_t bytes, void* stream) {
    B200_ENTER(c, d_dst);
    B200_CHECK(d_dst && h_src, -1, "dev_upload_async: null pointer");
    B200_CUDA(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, stream ? (cudaStream_t)stream : c->stream));     // truly asynchronous only from pinned memory
    return 0;
}
int b200_dev_download(void* h_dst, const void* d_src, size_t bytes) {
    B200_ENTER(c, d_src);
    B200_CUDA(cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, c->stream));
    B200_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
}
int b200_host_alloc(void** h_ptr, size_t bytes) { B200_CUDA(cudaMallocHost(h_ptr, bytes)); return 0; }
int b200_host_free(void* h_ptr) { B200_CUDA(cudaFreeHost(h_ptr)); return 0; }
int b200_sync(void) { B200_ENTER(c, nullptr); B200_CUDA(cudaStreamSynchronize(c->stream)); return 0; }
// the calling thread's library stream on every device of the process
int b200_sync_all(void) {
    CallGuard cg; if (!cg.ok) return -3;
    for (int s = 0; s < g_ndev.load(); ++s) { Ctx* c; if (int rc = get_ctx(&c, s)) return rc; B200_CUDA(cudaStreamSynchronize(c->stream)); }
    return 0;
}

// ---- bases ---------------------------------------------------------------------------------------------------
// device base vector on the context's device -> handle of its window table, built there and replicated to the other devices
static int bases_register_on(Ctx* c, const G1Affine* d_bases, size_t n, int window_bits, uint64_t* handle, cudaStream_t st) {
    B200_CHECK(d_bases && handle && n > 0, -1, "bases_register: null argument or n == 0");
    B200_CHECK(window_bits == 0 || (window_bits >= 4 && window_bits <= 24), -1, "bases_register: window_bits %d not in {0, 4..24}", window_bits);
    BaseSet* bs = new BaseSet();
    auto fail = [&](int rc) { free_bases(bs); return rc; };
    MsmTable* t = new MsmTable();
    bs->t[c->slot] = t;
    if (int rc = msm_table_build(t, d_bases, n, window_bits, st)) return fail(rc);
    g_launches += (uint64_t)(t->W - 1);
    bs->n = n; bs->c = t->c; bs->W = t->W;
    // replicas: the finished table crosses NVLink once per extra device (cheaper than rebuilding: one inversion per point and level)
    for (int s = 0; s < g_ndev.load(); ++s) if (s != c->slot) {
        MsmTable* r = new MsmTable();
        *r = *t; r->d_table = nullptr; r->device = g_devs[s].id;
        bs->t[s] = r;
        cudaError_t e;
        {
            CurrentDevice keep;
            cudaSetDevice(r->device);
            e = cudaMalloc(&r->d_table, sizeof(G1Affine) * n * t->W);
        }
        if (e != cudaSuccess) { set_error("bases_register: replica on device %d: %s", r->device, cudaGetErrorString(e)); return fail(-2); }
        e = cudaMemcpyPeerAsync(r->d_table, r->device, t->d_table, t->device, sizeof(G1Affine) * n * t->W, st);
        if (e != cudaSuccess) { set_error("bases_register: peer copy: %s", cudaGetErrorString(e)); return fail(-2); }
    }
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { set_error("bases_register: %s", cudaGetErrorString(e)); return fail(-2); }
    std::lock_guard<std::mutex> lk(g_mu);
    *handle = g_next_handle++;
    g_tables[*handle] = bs;
    return 0;
}
int b200_bases_register_dev(const void* d_bases, size_t n, int window_bits, uint64_t* handle) {
    B200_ENTER(c, d_bases);
    StreamScope ss(c, nullptr);
    return bases_register_on(c, reinterpret_cast<const G1Affine*>(d_bases), n, window_bits, handle, ss.st);
}
int b200_bases_register(const b200_g1_affine* bases, size_t n, int window_bits, uint64_t* handle) {
    B200_ENTER(c, nullptr);
    B200_CHECK(bases && handle && n > 0, -1, "bases_register: null argument or n == 0");
    if (c->stage_a.ensure(sizeof(G1Affine) * n)) return -2;
    StreamScope ss(c, nullptr);
    if (int rc = h2d_one(c, c->stage_a.p, bases, sizeof(G1Affine) * n, ss.st)) return rc;
    return bases_register_on(c, c->stage_a.as<G1Affine>(), n, window_bits, handle, ss.st);
}
int b200_bases_release(uint64_t handle) {
    CallGuard cg; if (!cg.ok) return -3;
    BaseSet* bs = nullptr;
    {
        std::lock_guard<std::mutex> lk(g_mu);
        auto it = g_tables.find(handle);
        B200_CHECK(it != g_tables.end(), -1, "bases_release: unknown handle %llu", (unsigned long long)handle);
        bs = it->second;
        g_tables.erase(it);
    }
    free_bases(bs);
    return 0;
}
int b200_bases_info(uint64_t handle, size_t* n, int* window_bits, int* windows) {
    BaseSet* t = find_bases(handle);
    B200_CHECK(t, -1, "bases_info: unknown handle %llu", (unsigned long long)handle);
    if (n) *n = t->n;
    if (window_bits) *window_bits = t->c;
    if (windows) *windows = t->W;
    return 0;
}

// ---- MSM -----------------------------------------------------------------------------------------------------
int b200_msm_batch_dev(uint64_t bases, const void* d_scalars, size_t n, size_t stride, size_t batch, void* d_out_xyzz, void* stream) {
    B200_ENTER(c, d_scalars);
    BaseSet* t = find_bases(bases);
    B200_CHECK(t, -1, "msm: unknown bases handle %llu", (unsigned long long)bases);
    B200_CHECK(d_scalars && d_out_xyzz, -1, "msm: null pointer");
    B200_CHECK(n <= t->n, -1, "msm: %zu scalars per column, %zu bases registered", n, t->n);
    B200_CHECK(batch <= 1 || stride >= n, -1, "msm: column stride %zu < column length %zu", stride, n);
    if (batch == 0) return 0;
    StreamScope ss(c, stream);
    return msm_dev_on(c, t, reinterpret_cast<const Fr*>(d_scalars), n, stride, batch, 0, reinterpret_cast<G1Xyzz*>(d_out_xyzz), ss.st);
}
int b200_msm_batch(uint64_t bases, const b200_fr* const* scalars, size_t n, size_t batch, b200_g1_jac* out) {
    B200_ENTER(c, nullptr);
    B200_CHECK(scalars && out, -1, "msm: null pointer");
    if (batch == 0) return 0;
    BaseSet* t = find_bases(bases);
    B200_CHECK(t, -1, "msm: unknown bases handle %llu", (unsigned long long)bases);
    B200_CHECK(n <= t->n, -1, "msm: %zu scalars but only %zu bases registered", n, t->n);
    for (size_t b = 0; b < batch; ++b) B200_CHECK(scalars[b] || n == 0, -1, "msm: scalars[%zu] is null", b);
    std::vector<G1Xyzz> h(batch);
    const int nd = g_ndev.load();
    if (nd == 1 || n * batch < ((size_t)1 << 16)) {
        if (int rc = msm_host_on(c, t, scalars, batch, n, 0, h.data())) return rc;
    } else if (batch >= (size_t)nd) {
        // columns dealt round-robin over the devices: no exchange at all, every device stages and commits its own columns
        std::lock_guard<std::mutex> lk(g_multi_mu);
        std::vector<std::vector<const b200_fr*>> mine(nd);
        for (size_t b = 0; b < batch; ++b) mine[b % nd].push_back(scalars[b]);
        std::vector<std::vector<G1Xyzz>> part(nd);
        int rc = run_on_slots(nd, [&](int s) -> int {
            Ctx* cs; if (int r = get_ctx(&cs, s)) return r;
            part[s].resize(mine[s].size());
            return msm_host_on(cs, t, mine[s].data(), mine[s].size(), n, 0, part[s].data());
        });
        if (rc) return rc;
        for (size_t b = 0; b < batch; ++b) h[b] = part[b % nd][b / nd];
    } else {
        // fewer columns than devices: split the (scalar, base) pairs of every column into one contiguous range per device
        // (each against its table replica), then add the per-device partial sums in device order
        std::lock_guard<std::mutex> lk(g_multi_mu);
        std::vector<std::vector<G1Xyzz>> part(nd, std::vector<G1Xyzz>(batch));
        int rc = run_on_slots(nd, [&](int s) -> int {
            Ctx* cs; if (int r = get_ctx(&cs, s)) return r;
            size_t lo, hi; slice_bounds(n, s, nd, &lo, &hi);
            return msm_host_on(cs, t, scalars, batch, hi - lo, lo, part[s].data());
        });
        if (rc) return rc;
        for (size_t b = 0; b < batch; ++b) { G1Xyzz acc = part[0][b]; for (int s = 1; s < nd; ++s) acc = g1_add(acc, part[s][b]); h[b] = acc; }
    }
    normalize_host(h.data(), batch, out);
    return 0;
}
int b200_msm(uint64_t bases, const b200_fr* scalars, size_t n, b200_g1_jac* out) {
    const b200_fr* cols[1] = {scalars};
    return b200_msm_batch(bases, cols, n, 1, out);
}
// out[g] = sum of points[g * count .. (g + 1) * count)
static int g1_sum_on(const G1Xyzz* pts, size_t groups, size_t count, G1Xyzz* out, cudaStream_t st) {
    B200_CHECK(pts && out, -1, "g1_sum: null pointer");
    int rc = g1_sum_run(pts, groups, count, out, st);
    if (!rc) g_launches += 1;
    return rc;
}
// base-split MSM on device-resident slices (north star: bases split across the GPUs, partial sums reduced over NVLink)
int b200_msm_sharded_dev(uint64_t bases, const void* const* d_scalar_slices, size_t n, size_t batch, b200_g1_jac* out) {
    CallGuard cg; if (!cg.ok) return -3;
    const int nd = g_ndev.load();
    B200_CHECK(d_scalar_slices && out, -1, "msm_sharded: null pointer");
    BaseSet* t = find_bases(bases);
    B200_CHECK(t, -1, "msm: unknown bases handle %llu", (unsigned long long)bases);
    B200_CHECK(n <= t->n && batch >= 1 && batch <= 4096, -1, "msm_sharded: bad sizes");
    Ctx* cs[MAX_DEV];
    for (int s = 0; s < nd; ++s) if (int rc = get_ctx(&cs[s], s)) return rc;
    CurrentDevice keep;
    // gather buffer on device 0: [column][device] XYZZ partials
    if (cs[0]->small.ensure(sizeof(G1Xyzz) * batch * (nd + 2))) return -2;
    G1Xyzz* gather = cs[0]->small.as<G1Xyzz>();
    for (int s = 0; s < nd; ++s) {
        B200_CHECK(d_scalar_slices[s], -1, "msm_sharded: slice %d is null", s);
        size_t lo, hi; slice_bounds(n, s, nd, &lo, &hi);
        B200_CUDA(cudaSetDevice(cs[s]->dev));
        StreamScope ss(cs[s], nullptr);
        G1Xyzz* part = gather + batch * nd;           // device 0: a staging row behind the gather matrix
        if (s != 0) { if (cs[s]->small.ensure(sizeof(G1Xyzz) * batch)) return -2; part = cs[s]->small.as<G1Xyzz>(); }
        if (int rc = msm_dev_on(cs[s], t, reinterpret_cast<const Fr*>(d_scalar_slices[s]), hi - lo, hi - lo, batch, lo, part, ss.st)) return rc;
        // partial sums travel to device 0 over NVLink: column b of device s lands at gather[b * nd + s]
        B200_CUDA(cudaMemcpy2DAsync(gather + s, sizeof(G1Xyzz) * nd, part, sizeof(G1Xyzz), sizeof(G1Xyzz), batch, cudaMemcpyDefault, ss.st));
    }
    for (int s = 1; s < nd; ++s) { B200_CUDA(cudaSetDevice(cs[s]->dev)); B200_CUDA(cudaStreamSynchronize(cs[s]->stream)); }
    B200_CUDA(cudaSetDevice(cs[0]->dev));
    std::vector<G1Xyzz> h(batch);
    {
        StreamScope ss(cs[0], nullptr);
        G1Xyzz* sums = gather + batch * (nd + 1);
        if (int rc = g1_sum_on(gather, batch, nd, sums, ss.st)) return rc;
        B200_CUDA(cudaMemcpyAsync(h.data(), sums, sizeof(G1Xyzz) * batch, cudaMemcpyDeviceToHost, ss.st));
        B200_CUDA(cudaStreamSynchronize(ss.st));
    }
    normalize_host(h.data(), batch, out);
    return 0;
}
int b200_g1_sum_dev(const void* d_points_xyzz, size_t groups, size_t count, void* d_out_xyzz, void* stream) {
    B200_ENTER(c, d_points_xyzz);
    StreamScope ss(c, stream);
    return g1_sum_on(reinterpret_cast<const G1Xyzz*>(d_points_xyzz), groups, count, reinterpret_cast<G1Xyzz*>(d_out_xyzz), ss.st);
}
static int g1_fft_on(Ctx* c, const G1Affine* in, uint32_t log_n, const b200_fr* omega, const b200_fr* scale, G1Affine* out, cudaStream_t st) {
    B200_CHECK(in && omega && out, -1, "g1_fft: null pointer");
    const Fr w = as_fr(omega);
    Fr sc = fp_one<FrTag>();
    if (scale) sc = as_fr(scale);
    int rc = g1_fft_run(in, log_n, w, scale ? &sc : nullptr, out, c->msm_ws.misc, st);
    if (!rc) g_launches += (uint64_t)g1_fft_launches(log_n);
    return rc;
}
int b200_g1_fft_dev(const void* d_in_affine, uint32_t log_n, const b200_fr* omega, const b200_fr* scale, void* d_out_affine, void* stream) {
    B200_ENTER(c, d_in_affine);
    StreamScope ss(c, stream);
    return g1_fft_on(c, reinterpret_cast<const G1Affine*>(d_in_affine), log_n, omega, scale, reinterpret_cast<G1Affine*>(d_out_affine), ss.st);
}
int b200_g1_fft(const b200_g1_affine* in, uint32_t log_n, const b200_fr* omega, const b200_fr* scale, b200_g1_affine* out) {
    B200_ENTER(c, nullptr);
    B200_CHECK(in && omega && out && log_n <= 26, -1, "g1_fft: bad argument");
    const size_t bytes = sizeof(G1Affine) << log_n;
    if (c->stage_a.ensure(bytes) || c->stage_b.ensure(bytes)) return -2;
    StreamScope ss(c, nullptr);
    if (int rc = h2d_one(c, c->stage_a.p, in, bytes, ss.st)) return rc;
    if (int rc = g1_fft_on(c, c->stage_a.as<G1Affine>(), log_n, omega, scale, c->stage_b.as<G1Affine>(), ss.st)) return rc;
    return d2h_one(c, out, c->stage_b.p, bytes, ss.st);
}
int b200_g1_fixed_base_mul_dev(const void* d_scalars, size_t n, const b200_g1_affine* base, void* d_out_affine, void* stream) {
    B200_ENTER(c, d_scalars);
    B200_CHECK(d_scalars && base && d_out_affine, -1, "g1_fixed_base_mul: null pointer");
    G1Affine b; memcpy(&b, base, sizeof b);
    StreamScope ss(c, stream);
    int rc = g1_fixed_base_mul_run(reinterpret_cast<const Fr*>(d_scalars), n, b, reinterpret_cast<G1Affine*>(d_out_affine), ss.st);
    if (!rc && n) g_launches += 1;
    return rc;
}
int b200_g1_generate_dev(uint64_t seed, size_t n, void* d_out_affine, void* stream) {
    B200_ENTER(c, d_out_affine);
    B200_CHECK(d_out_affine, -1, "g1_generate: null pointer");
    StreamScope ss(c, stream);
    int rc = g1_generate_run(seed, n, reinterpret_cast<G1Affine*>(d_out_affine), ss.st);
    if (!rc && n) g_launches += 1;
    return rc;
}
int b200_g1_normalize(const b200_g1_xyzz* points, size_t n, b200_g1_jac* out) {
    B200_CHECK(points && out, -1, "g1_normalize: null pointer");
    if (n == 0) return 0;
    std::vector<G1Xyzz> tmp(n);
    memcpy(tmp.data(), points, sizeof(G1Xyzz) * n);
    normalize_host(tmp.data(), n, out);
    return 0;
}

// ---- NTT -----------------------------------------------------------------------------------------------------
int b200_ntt_dev(const void* d_src, size_t src_stride, size_t n_in, void* d_tmp, void* d_dst, size_t dst_stride, uint32_t log_n,
                 const b200_fr* omega, int pre_mode, const b200_fr* pre, int post_mode, const b200_fr* post, size_t batch, void* stream) {
    B200_ENTER(c, d_src);
    B200_CHECK(d_src && d_tmp && d_dst && omega, -1, "ntt: null pointer");
    NttScale a, b;
    if (int rc = decode_scales(pre_mode, pre, post_mode, post, &a, &b)) return rc;
    if (batch == 0) return 0;
    StreamScope ss(c, stream);
    return ntt_call(c, reinterpret_cast<const Fr*>(d_src), src_stride, n_in, reinterpret_cast<Fr*>(d_tmp), reinterpret_cast<Fr*>(d_dst), dst_stride,
                    log_n, as_fr(omega), a, b, (int)batch, ss.st);
}

// one transform of 2^log_n elements split across the devices of the process in contiguous natural-order slices (slice g of
// 2^log_n / n_devices elements on device g).  Enqueued on the calling thread's library stream of every device; b200_sync_all
// (or any later call on those streams) orders after it.  The exchanges of the six-step scheme are peer loads / stores inside
// the butterfly kernels (ntt.cu: ntt_run_sharded).
static int ntt_sharded_on(Ctx* const* cs, int nd, const Fr* const* src, Fr* const* tmp, Fr* const* dst, uint32_t log_n, uint64_t n_in, const Fr& omega,
                          const NttScale& pre, const NttScale& post) {
    NttPlan* plans[MAX_DEV]; int ids[MAX_DEV]; cudaStream_t st[MAX_DEV]; cudaEvent_t ev[MAX_DEV];
    {
        CurrentDevice keep;
        for (int s = 0; s < nd; ++s) {
            cudaSetDevice(cs[s]->dev);
            plans[s] = warm_plan(s, log_n, omega, cs[s]->stream);
            if (!plans[s]) return -2;
            ids[s] = cs[s]->dev; st[s] = cs[s]->stream; ev[s] = cs[s]->last_ev;
            if (cs[s]->has_last && cs[s]->last_stream != st[s]) cudaStreamWaitEvent(st[s], cs[s]->last_ev, 0);
        }
    }
    int rc = ntt_run_sharded(plans, nd, ids, src, tmp, dst, log_n, omega, pre, post, n_in, st, ev);
    for (int s = 0; s < nd && !rc; ++s) { cs[s]->last_stream = st[s]; cs[s]->has_last = true; }       // ev[s] was recorded after the last pass
    if (!rc) g_launches += (uint64_t)ntt_launches_per_run(log_n) * nd;
    return rc;
}
int b200_ntt_sharded_dev(const void* const* d_src_slices, void* const* d_tmp_slices, void* const* d_dst_slices, uint32_t log_n, size_t n_in, const b200_fr* omega,
                         int pre_mode, const b200_fr* pre, int post_mode, const b200_fr* post) {
    CallGuard cg; if (!cg.ok) return -3;
    const int nd = g_ndev.load();
    B200_CHECK(nd >= 2, -1, "ntt_sharded: needs a multi-device process (b200_init_multi)");
    B200_CHECK(d_src_slices && d_tmp_slices && d_dst_slices && omega, -1, "ntt_sharded: null pointer");
    NttScale a, b;
    if (int rc = decode_scales(pre_mode, pre, post_mode, post, &a, &b)) return rc;
    Ctx* cs[MAX_DEV];
    for (int s = 0; s < nd; ++s) {
        if (int rc = get_ctx(&cs[s], s)) return rc;
        B200_CHECK(d_src_slices[s] && d_tmp_slices[s] && d_dst_slices[s], -1, "ntt_sharded: slice %d is null", s);
    }
    return ntt_sharded_on(cs, nd, reinterpret_cast<const Fr* const*>(d_src_slices), reinterpret_cast<Fr* const*>(d_tmp_slices), reinterpret_cast<Fr* const*>(d_dst_slices),
                          log_n, n_in, as_fr(omega), a, b);
}

// host path on ONE device: polynomials src[p] (n_in each) -> dst[p] (2^log_n each), staged in sub-batches
static int ntt_host_on(Ctx* c, const b200_fr* const* src, b200_fr* const* dst, size_t batch, size_t n_in, uint32_t log_n, const Fr& omega,
                       const NttScale& pre, const NttScale& post) {
    if (batch == 0) return 0;
    DevGuard dg(c);
    const size_t N = (size_t)1 << log_n;
    size_t sub = call_budget() / (sizeof(Fr) * N * 3);
    if (sub < 1) sub = 1;
    if (sub > batch) sub = batch;
    if (c->stage_a.ensure(sizeof(Fr) * n_in * sub) || c->stage_b.ensure(sizeof(Fr) * N * sub) || c->stage_c.ensure(sizeof(Fr) * N * sub)) return -2;
    StreamScope ss(c, nullptr);
    for (size_t b0 = 0; b0 < batch; b0 += sub) {
        const size_t nb = batch - b0 < sub ? batch - b0 : sub;
        std::vector<HostSeg> up(nb), down(nb);
        for (size_t p = 0; p < nb; ++p) {
            B200_CHECK(src[b0 + p] && dst[b0 + p], -1, "ntt: polynomial %zu is null", b0 + p);
            up[p] = HostSeg{(uint8_t*)const_cast<b200_fr*>(src[b0 + p]), sizeof(Fr) * n_in};
            down[p] = HostSeg{(uint8_t*)dst[b0 + p], sizeof(Fr) * N};
        }
        if (int rc = h2d_segments(c, c->stage_a.p, up.data(), nb, ss.st)) return rc;
        if (int rc = ntt_call(c, c->stage_a.as<Fr>(), n_in, n_in, c->stage_b.as<Fr>(), c->stage_c.as<Fr>(), N, log_n, omega, pre, post, (int)nb, ss.st)) return rc;
        if (int rc = d2h_segments(c, c->stage_c.p, down.data(), nb, ss.st)) return rc;
    }
    return 0;
}
// shared host path: on a multi-device process a batch is dealt over the devices; a single large transform is sharded.
// n_in_or_null: input elements per polynomial, NULL = 2^log_n
static int ntt_host(const b200_fr* const* src, b200_fr* const* dst, size_t batch, const size_t* n_in_or_null, uint32_t log_n, const Fr& omega,
                    const NttScale& pre, const NttScale& post) {
    B200_ENTER(c, nullptr);
    B200_CHECK(log_n >= 1 && log_n <= 28, -1, "ntt: log_n = %u out of range [1, 28]", log_n);
    const size_t N = (size_t)1 << log_n, n_in = n_in_or_null ? *n_in_or_null : N;
    B200_CHECK(n_in <= N, -1, "ntt: %zu input elements > 2^%u", n_in, log_n);
    if (batch == 0) return 0;
    const int nd = g_ndev.load();
    if (nd > 1 && batch >= 2 && N * batch >= ((size_t)1 << 18)) {
        std::lock_guard<std::mutex> lk(g_multi_mu);
        std::vector<std::vector<const b200_fr*>> s_in(nd);
        std::vector<std::vector<b200_fr*>> s_out(nd);
        for (size_t p = 0; p < batch; ++p) { s_in[p % nd].push_back(src[p]); s_out[p % nd].push_back(dst[p]); }
        return run_on_slots(nd, [&](int s) -> int {
            Ctx* cs; if (int r = get_ctx(&cs, s)) return r;
            return ntt_host_on(cs, s_in[s].data(), s_out[s].data(), s_in[s].size(), n_in, log_n, omega, pre, post);
        });
    }
    if (nd > 1 && batch == 1 && (int)log_n >= g_cfg.shard_min_logn) {
        // one large transform: every device uploads its contiguous slice over its own PCIe link, the passes exchange over NVLink
        std::lock_guard<std::mutex> lk(g_multi_mu);
        B200_CHECK(src[0] && dst[0], -1, "ntt: polynomial 0 is null");
        const size_t slice = N / nd;
        Fr* sl_src[MAX_DEV]; Fr* sl_tmp[MAX_DEV]; Fr* sl_dst[MAX_DEV]; Ctx* wcs[MAX_DEV];
        int rc = run_on_slots(nd, [&](int s) -> int {
            Ctx* cs; if (int r = get_ctx(&cs, s)) return r;
            DevGuard dg(cs);
            if (cs->stage_a.ensure(sizeof(Fr) * slice) || cs->stage_b.ensure(sizeof(Fr) * slice)) return -2;
            wcs[s] = cs; sl_src[s] = cs->stage_a.as<Fr>(); sl_tmp[s] = cs->stage_b.as<Fr>(); sl_dst[s] = cs->stage_a.as<Fr>();
            const size_t lo = slice * s, hi = lo + slice < n_in ? lo + slice : n_in;
            if (hi > lo) B200_CUDA(cudaMemcpyAsync(sl_src[s], src[0] + lo, sizeof(Fr) * (hi - lo), cudaMemcpyHostToDevice, cs->stream));
            B200_CUDA(cudaStreamSynchronize(cs->stream));
            return 0;
        });
        if (rc) return rc;
        // the passes are enqueued on the worker contexts' streams from this thread (the workers are idle under g_multi_mu)
        if ((rc = ntt_sharded_on(wcs, nd, sl_src, sl_tmp, sl_dst, log_n, n_in, omega, pre, post))) return rc;
        return run_on_slots(nd, [&](int s) -> int {
            Ctx* cs = wcs[s];
            DevGuard dg(cs);
            B200_CUDA(cudaMemcpyAsync(dst[0] + slice * s, sl_dst[s], sizeof(Fr) * slice, cudaMemcpyDeviceToHost, cs->stream));
            B200_CUDA(cudaStreamSynchronize(cs->stream));
            return 0;
        });
    }
    return ntt_host_on(c, src, dst, batch, n_in, log_n, omega, pre, post);
}
int b200_fft_batch(b200_fr* const* a, size_t batch, uint32_t log_n, const b200_fr* omega) {
    B200_CHECK(a && omega, -1, "fft: null pointer");
    NttScale none;
    return ntt_host(a, a, batch, nullptr, log_n, as_fr(omega), none, none);
}
int b200_fft(b200_fr* a, uint32_t log_n, const b200_fr* omega) { b200_fr* p[1] = {a}; return b200_fft_batch(p, 1, log_n, omega); }
int b200_ifft_batch(b200_fr* const* a, size_t batch, uint32_t log_n, const b200_fr* omega_inv, const b200_fr* divisor) {
    B200_CHECK(a && omega_inv && divisor, -1, "ifft: null pointer");
    NttScale none, post;
    post.mode = 1; post.c[0] = as_fr(divisor);
    return ntt_host(a, a, batch, nullptr, log_n, as_fr(omega_inv), none, post);
}
int b200_ifft(b200_fr* a, uint32_t log_n, const b200_fr* omega_inv, const b200_fr* divisor) {
    b200_fr* p[1] = {a};
    return b200_ifft_batch(p, 1, log_n, omega_inv, divisor);
}
int b200_coeff_to_extended_batch(const b200_fr* const* coeffs, size_t batch, size_t n_coeffs, uint32_t ext_k, const b200_fr* ext_omega, const b200_fr* zeta, b200_fr* const* out) {
    B200_CHECK(coeffs && out && ext_omega && zeta, -1, "coeff_to_extended: null pointer");
    NttScale none;
    return ntt_host(coeffs, out, batch, &n_coeffs, ext_k, as_fr(ext_omega), coset_scale(as_fr(zeta)), none);
}
int b200_coeff_to_extended(const b200_fr* coeffs, size_t n_coeffs, uint32_t ext_k, const b200_fr* ext_omega, const b200_fr* zeta, b200_fr* out) {
    const b200_fr* s[1] = {coeffs}; b200_fr* d[1] = {out};
    return b200_coeff_to_extended_batch(s, 1, n_coeffs, ext_k, ext_omega, zeta, d);
}
int b200_extended_to_coeff(b200_fr* a, uint32_t ext_k, const b200_fr* ext_omega_inv, const b200_fr* ext_ifft_divisor, const b200_fr* zeta) {
    B200_CHECK(a && ext_omega_inv && ext_ifft_divisor && zeta, -1, "extended_to_coeff: null pointer");
    NttScale none;
    b200_fr* p[1] = {a};
    return ntt_host(p, p, 1, nullptr, ext_k, as_fr(ext_omega_inv), none, coset_unscale(as_fr(zeta), as_fr(ext_ifft_divisor)));
}

// ---- polynomial ops --------------------------------------------------------------------------------------------
static int poly_op_on(int op, const Fr* a, const Fr* b, const b200_fr* s, Fr* out, size_t n, cudaStream_t st) {
    B200_CHECK(op >= 0 && op <= 4, -1, "poly_op: unknown op %d", op);
    B200_CHECK(a && out && (op == POLY_SCALE || b) && (op < POLY_SCALE || s), -1, "poly_op: missing operand for op %d", op);
    Fr sv = fp_zero<FrTag>();
    if (s) sv = as_fr(s);
    int rc = poly_binary(op, a, b, s ? &sv : nullptr, out, n, st);
    if (!rc && n) g_launches += 1;
    return rc;
}
int b200_poly_op_dev(int op, const void* d_a, const void* d_b, const b200_fr* s, void* d_out, size_t n, void* stream) {
    B200_ENTER(c, d_a);
    StreamScope ss(c, stream);
    return poly_op_on(op, reinterpret_cast<const Fr*>(d_a), reinterpret_cast<const Fr*>(d_b), s, reinterpret_cast<Fr*>(d_out), n, ss.st);
}
int b200_poly_op(int op, const b200_fr* a, const b200_fr* b, const b200_fr* s, b200_fr* out, size_t n) {
    B200_ENTER(c, nullptr);
    B200_CHECK(a && out, -1, "poly_op: null pointer");
    if (n == 0) return 0;
    const bool need_b = op != POLY_SCALE;
    B200_CHECK(!need_b || b, -1, "poly_op: missing operand b");
    if (c->stage_a.ensure(sizeof(Fr) * n) || (need_b && c->stage_b.ensure(sizeof(Fr) * n))) return -2;
    StreamScope ss(c, nullptr);
    if (int rc = h2d_one(c, c->stage_a.p, a, sizeof(Fr) * n, ss.st)) return rc;
    if (need_b) { if (int rc = h2d_one(c, c->stage_b.p, b, sizeof(Fr) * n, ss.st)) return rc; }
    if (int rc = poly_op_on(op, c->stage_a.as<Fr>(), need_b ? c->stage_b.as<Fr>() : nullptr, s, c->stage_a.as<Fr>(), n, ss.st)) return rc;
    return d2h_one(c, out, c->stage_a.p, sizeof(Fr) * n, ss.st);
}
// d_polys: host array of device addresses
static int lincomb_on(Ctx* c, const Fr* const* d_polys, const b200_fr* scalars, size_t count, size_t n, Fr* out, cudaStream_t st) {
    B200_CHECK(out && (count == 0 || (d_polys && scalars)), -1, "poly_lincomb: null pointer");
    std::vector<Fr> sv(count);
    if (count) memcpy(sv.data(), scalars, sizeof(Fr) * count);
    int rc = poly_lincomb(d_polys, sv.data(), count, out, n, c->poly_ws, st);
    if (!rc && n) g_launches += 1;
    return rc;
}
int b200_poly_lincomb_dev(const void* const* d_polys, const b200_fr* scalars, size_t count, size_t n, void* d_out, void* stream) {
    B200_ENTER(c, d_out);
    StreamScope ss(c, stream);
    return lincomb_on(c, reinterpret_cast<const Fr* const*>(d_polys), scalars, count, n, reinterpret_cast<Fr*>(d_out), ss.st);
}
int b200_poly_lincomb(const b200_fr* const* polys, const b200_fr* scalars, size_t count, size_t n, b200_fr* out) {
    B200_ENTER(c, nullptr);
    B200_CHECK(out && (count == 0 || (polys && scalars)), -1, "poly_lincomb: null pointer");
    if (n == 0) return 0;
    if (c->stage_a.ensure(sizeof(Fr) * n * (count ? count : 1)) || c->stage_b.ensure(sizeof(Fr) * n)) return -2;
    std::vector<const Fr*> ptrs(count);
    std::vector<HostSeg> up(count);
    for (size_t j = 0; j < count; ++j) {
        B200_CHECK(polys[j], -1, "poly_lincomb: polys[%zu] is null", j);
        ptrs[j] = c->stage_a.as<Fr>() + j * n;
        up[j] = HostSeg{(uint8_t*)const_cast<b200_fr*>(polys[j]), sizeof(Fr) * n};
    }
    StreamScope ss(c, nullptr);
    if (int rc = h2d_segments(c, c->stage_a.p, up.data(), count, ss.st)) return rc;
    if (int rc = lincomb_on(c, ptrs.data(), scalars, count, n, c->stage_b.as<Fr>(), ss.st)) return rc;
    return d2h_one(c, out, c->stage_b.p, sizeof(Fr) * n, ss.st);
}
static int scale_cycle_on(Ctx* c, Fr* a, size_t n, const b200_fr* consts, uint32_t period, cudaStream_t st) {
    B200_CHECK(a && consts && period > 0 && period <= 1024, -1, "poly_scale_cycle: bad argument");
    const Fr* d_consts = reinterpret_cast<const Fr*>(c->ring.push(consts, sizeof(Fr) * period, st));
    if (!d_consts) {
        if (c->small.ensure(sizeof(Fr) * period)) return -2;
        if (int rc = h2d_one(c, c->small.p, consts, sizeof(Fr) * period, st)) return rc;
        d_consts = c->small.as<Fr>();
    }
    int rc = poly_scale_cycle(a, d_consts, period, a, n, st);
    if (!rc && n) g_launches += 1;
    return rc;
}
int b200_poly_scale_cycle_dev(void* d_a, size_t n, const b200_fr* consts, uint32_t period, void* stream) {
    B200_ENTER(c, d_a);
    StreamScope ss(c, stream);
    return scale_cycle_on(c, reinterpret_cast<Fr*>(d_a), n, consts, period, ss.st);
}
int b200_poly_scale_cycle(b200_fr* a, size_t n, const b200_fr* consts, uint32_t period) {
    B200_ENTER(c, nullptr);
    B200_CHECK(a && consts, -1, "poly_scale_cycle: null pointer");
    if (n == 0) return 0;
    if (c->stage_a.ensure(sizeof(Fr) * n)) return -2;
    StreamScope ss(c, nullptr);
    if (int rc = h2d_one(c, c->stage_a.p, a, sizeof(Fr) * n, ss.st)) return rc;
    if (int rc = scale_cycle_on(c, c->stage_a.as<Fr>(), n, consts, period, ss.st)) return rc;
    return d2h_one(c, a, c->stage_a.p, sizeof(Fr) * n, ss.st);
}
static int poly_eval_on(Ctx* c, const Fr* polys, size_t stride, size_t n, const b200_fr* x, size_t batch, Fr* out, cudaStream_t st) {
    B200_CHECK(polys && x && out, -1, "poly_eval: null pointer");
    if (batch == 0) return 0;
    std::vector<Fr> xv(batch);
    memcpy(xv.data(), x, sizeof(Fr) * batch);
    int rc = poly_eval(polys, stride, n, xv.data(), out, (int)batch, c->poly_ws, st);
    if (!rc && n) g_launches += 2;
    return rc;
}
int b200_poly_eval_batch_dev(const void* d_polys, size_t stride, size_t n, const b200_fr* x, size_t batch, void* d_out, void* stream) {
    B200_ENTER(c, d_polys);
    StreamScope ss(c, stream);
    return poly_eval_on(c, reinterpret_cast<const Fr*>(d_polys), stride, n, x, batch, reinterpret_cast<Fr*>(d_out), ss.st);
}
int b200_poly_eval_batch(const b200_fr* const* polys, size_t n, const b200_fr* x, size_t batch, b200_fr* out) {
    B200_ENTER(c, nullptr);
    B200_CHECK(polys && x && out, -1, "poly_eval: null pointer");
    if (batch == 0) return 0;
    if (c->stage_a.ensure(sizeof(Fr) * (n ? n : 1) * batch) || c->small.ensure(sizeof(Fr) * batch)) return -2;
    std::vector<HostSeg> up(batch);
    for (size_t p = 0; p < batch; ++p) {
        B200_CHECK(n == 0 || polys[p], -1, "poly_eval: polys[%zu] is null", p);
        up[p] = HostSeg{(uint8_t*)const_cast<b200_fr*>(polys[p]), sizeof(Fr) * n};
    }
    StreamScope ss(c, nullptr);
    if (n) { if (int rc = h2d_segments(c, c->stage_a.p, up.data(), batch, ss.st)) return rc; }
    if (int rc = poly_eval_on(c, c->stage_a.as<Fr>(), n, n, x, batch, c->small.as<Fr>(), ss.st)) return rc;
    return d2h_one(c, out, c->small.p, sizeof(Fr) * batch, ss.st);
}
int b200_poly_eval(const b200_fr* coeffs, size_t n, const b200_fr* x, b200_fr* out) {
    const b200_fr* p[1] = {coeffs};
    return b200_poly_eval_batch(p, n, x, 1, out);
}
static int batch_invert_on(Ctx* c, Fr* a, size_t n, cudaStream_t st) {
    B200_CHECK(a, -1, "batch_invert: null pointer");
    int rc = poly_batch_invert(a, n, c->poly_ws, st);
    if (!rc && n) g_launches += 1;
    return rc;
}
int b200_batch_invert_dev(void* d_a, size_t n, void* stream) {
    B200_ENTER(c, d_a);
    StreamScope ss(c, stream);
    return batch_invert_on(c, reinterpret_cast<Fr*>(d_a), n, ss.st);
}
int b200_batch_invert(b200_fr* a, size_t n) {
    B200_ENTER(c, nullptr);
    B200_CHECK(a, -1, "batch_invert: null pointer");
    if (n == 0) return 0;
    if (c->stage_a.ensure(sizeof(Fr) * n)) return -2;
    StreamScope ss(c, nullptr);
    if (int rc = h2d_one(c, c->stage_a.p, a, sizeof(Fr) * n, ss.st)) return rc;
    if (int rc = batch_invert_on(c, c->stage_a.as<Fr>(), n, ss.st)) return rc;
    return d2h_one(c, a, c->stage_a.p, sizeof(Fr) * n, ss.st);
}
// `batch` columns: column p at a + p * a_stride, its running product / sum at out + p * out_stride, starting from inits[p]
static int prefix_scan_on(Ctx* c, int product, const Fr* a, size_t a_stride, size_t n, size_t batch, const b200_fr* inits, Fr* out, size_t out_stride,
                          cudaStream_t st) {
    B200_CHECK(a && inits && out, -1, "prefix_scan: null pointer");
    B200_CHECK(batch <= 1 || (a_stride >= n && out_stride >= n), -1, "prefix_scan: column stride smaller than the column");
    if (batch == 0) return 0;
    std::vector<Fr> iv(batch);
    memcpy(iv.data(), inits, sizeof(Fr) * batch);
    int rc = poly_prefix_scan(product != 0, a, a_stride, n, iv.data(), out, out_stride, (int)batch, c->poly_ws, st);
    if (!rc && n) g_launches += 3;
    return rc;
}
int b200_prefix_scan_dev(int product, const void* d_a, size_t n, const b200_fr* init, void* d_out, void* stream) {
    B200_ENTER(c, d_a);
    StreamScope ss(c, stream);
    return prefix_scan_on(c, product, reinterpret_cast<const Fr*>(d_a), n, n, 1, init, reinterpret_cast<Fr*>(d_out), n, ss.st);
}
int b200_prefix_scan_batch_dev(int product, const void* d_a, size_t a_stride, size_t n, size_t batch, const b200_fr* inits, void* d_out, size_t out_stride, void* stream) {
    B200_ENTER(c, d_a);
    StreamScope ss(c, stream);
    return prefix_scan_on(c, product, reinterpret_cast<const Fr*>(d_a), a_stride, n, batch, inits, reinterpret_cast<Fr*>(d_out), out_stride, ss.st);
}
int b200_prefix_scan(int product, const b200_fr* a, size_t n, const b200_fr* init, b200_fr* out) {
    B200_ENTER(c, nullptr);
    B200_CHECK(a && init && out, -1, "prefix_scan: null pointer");
    if (n == 0) return 0;
    if (c->stage_a.ensure(sizeof(Fr) * n) || c->stage_b.ensure(sizeof(Fr) * n)) return -2;
    StreamScope ss(c, nullptr);
    if (int rc = h2d_one(c, c->stage_a.p, a, sizeof(Fr) * n, ss.st)) return rc;
    if (int rc = prefix_scan_on(c, product, c->stage_a.as<Fr>(), n, n, 1, init, c->stage_b.as<Fr>(), n, ss.st)) return rc;
    return d2h_one(c, out, c->stage_b.p, sizeof(Fr) * n, ss.st);
}
static int kate_division_on(Ctx* c, const Fr* a, size_t n, const b200_fr* b, Fr* q, cudaStream_t st) {
    B200_CHECK(a && b && q, -1, "kate_division: null pointer");
    const Fr bv = as_fr(b);
    int rc = poly_kate_division(a, n, &bv, q, c->poly_ws, st);
    if (!rc && n > 1) g_launches += 3;
    return rc;
}
int b200_kate_division_dev(const void* d_a, size_t n, const b200_fr* b, void* d_q, void* stream) {
    B200_ENTER(c, d_a);
    StreamScope ss(c, stream);
    return kate_division_on(c, reinterpret_cast<const Fr*>(d_a), n, b, reinterpret_cast<Fr*>(d_q), ss.st);
}
int b200_kate_division(const b200_fr* a, size_t n, const b200_fr* b, b200_fr* q) {
    B200_ENTER(c, nullptr);
    B200_CHECK(a && b && q, -1, "kate_division: null pointer");
    B200_CHECK(n >= 1, -1, "kate_division: empty polynomial");
    if (n == 1) return 0;
    if (c->stage_a.ensure(sizeof(Fr) * n) || c->stage_b.ensure(sizeof(Fr) * n)) return -2;
    StreamScope ss(c, nullptr);
    if (int rc = h2d_one(c, c->stage_a.p, a, sizeof(Fr) * n, ss.st)) return rc;
    if (int rc = kate_division_on(c, c->stage_a.as<Fr>(), n, b, c->stage_b.as<Fr>(), ss.st)) return rc;
    return d2h_one(c, q, c->stage_b.p, sizeof(Fr) * (n - 1), ss.st);
}

// ---- mv-lookup multiplicities --------------------------------------------------------------------------------------------------
// d_inputs: host array of device addresses
static int lookup_on(Ctx* c, const Fr* table, size_t n_table, const void* const* d_inputs, size_t n_inputs, size_t n_rows, Fr* m, uint64_t* missing,
                     cudaStream_t st) {
    B200_CHECK(table && m && d_inputs && n_inputs >= 1, -1, "lookup_multiplicities: null pointer");
    const void* d_ptrs = c->ring.push(d_inputs, sizeof(void*) * n_inputs, st);
    if (!d_ptrs) {
        if (c->small.ensure(sizeof(void*) * n_inputs)) return -2;
        if (int rc = h2d_one(c, c->small.p, d_inputs, sizeof(void*) * n_inputs, st)) return rc;
        B200_CUDA(cudaStreamSynchronize(st));
        d_ptrs = c->small.p;
    }
    unsigned long long* d_missing = nullptr;
    if (int rc = lookup_multiplicities_run(table, n_table, reinterpret_cast<const Fr* const*>(d_ptrs), n_inputs, n_rows, m, c->msm_ws.misc, &d_missing, st)) return rc;
    g_launches += 3;
    if (missing) {
        unsigned long long h = 0;
        if (int rc = d2h_one(c, &h, d_missing, sizeof h, st)) return rc;
        *missing = h;
    }
    return 0;
}
int b200_lookup_multiplicities_dev(const void* d_table, size_t n_table, const void* const* d_inputs, size_t n_inputs, size_t n_rows, void* d_m, uint64_t* missing, void* stream) {
    B200_ENTER(c, d_table);
    StreamScope ss(c, stream);
    return lookup_on(c, reinterpret_cast<const Fr*>(d_table), n_table, d_inputs, n_inputs, n_rows, reinterpret_cast<Fr*>(d_m), missing, ss.st);
}
int b200_lookup_multiplicities(const b200_fr* table, size_t n_table, const b200_fr* const* inputs, size_t n_inputs, size_t n_rows, b200_fr* m, uint64_t* missing) {
    B200_ENTER(c, nullptr);
    B200_CHECK(table && inputs && m && n_inputs >= 1, -1, "lookup_multiplicities: null pointer");
    if (c->stage_a.ensure(sizeof(Fr) * (n_table + n_inputs * (n_rows ? n_rows : 1))) || c->stage_b.ensure(sizeof(Fr) * n_table)) return -2;
    // the table, then every input column, back to back in stage_a
    std::vector<HostSeg> up{HostSeg{(uint8_t*)const_cast<b200_fr*>(table), sizeof(Fr) * n_table}};
    std::vector<const void*> ptrs(n_inputs);
    for (size_t j = 0; j < n_inputs; ++j) {
        B200_CHECK(inputs[j] || n_rows == 0, -1, "lookup_multiplicities: inputs[%zu] is null", j);
        ptrs[j] = c->stage_a.as<Fr>() + n_table + j * n_rows;
        if (n_rows) up.push_back(HostSeg{(uint8_t*)const_cast<b200_fr*>(inputs[j]), sizeof(Fr) * n_rows});
    }
    StreamScope ss(c, nullptr);
    if (int rc = h2d_segments(c, c->stage_a.p, up.data(), up.size(), ss.st)) return rc;
    if (int rc = lookup_on(c, c->stage_a.as<Fr>(), n_table, ptrs.data(), n_inputs, n_rows, c->stage_b.as<Fr>(), missing, ss.st)) return rc;
    return d2h_one(c, m, c->stage_b.p, sizeof(Fr) * n_table, ss.st);
}

// ---- quotient numerator (evaluate_h) ------------------------------------------------------------------------------
static_assert(sizeof(b200_instr) == sizeof(QInstr) && sizeof(b200_col_ref) == sizeof(QLoad), "ABI structs must match the kernel's");
// columns: host array of device addresses
static int quotient_eval_on(Ctx* c, const Fr* const* columns, size_t n_columns, uint32_t k, uint32_t ext_k, const b200_col_ref* loads, size_t n_loads,
                            const b200_fr* constants, size_t n_constants, const b200_instr* program, size_t n_instr, Fr* out, cudaStream_t st) {
    B200_CHECK(out && (n_columns == 0 || columns) && (n_loads == 0 || loads) && (n_constants == 0 || constants) && (n_instr == 0 || program), -1, "quotient_eval: null pointer");
    B200_CHECK(ext_k >= k && ext_k <= 28, -1, "quotient_eval: need k <= ext_k <= 28");
    const uint64_t N = 1ull << ext_k, scale = 1ull << (ext_k - k);
    std::vector<QLoad> ql(n_loads);
    for (size_t i = 0; i < n_loads; ++i) {
        ql[i].column = loads[i].column;
        const int64_t off = (int64_t)loads[i].rotation * (int64_t)scale;           // Rotation(r) on the extended domain = r * 2^(ext_k - k)
        ql[i].offset = (uint32_t)(((off % (int64_t)N) + (int64_t)N) % (int64_t)N);
    }
    int rc = quotient_eval_run(columns, n_columns, ext_k, ql.data(), n_loads, reinterpret_cast<const Fr*>(constants), n_constants,
                               reinterpret_cast<const QInstr*>(program), n_instr, out, c->quot_ws, st);
    if (!rc) g_launches += 1;
    return rc;
}
int b200_quotient_eval_dev(const void* const* d_columns, size_t n_columns, uint32_t k, uint32_t ext_k, const b200_col_ref* loads, size_t n_loads,
                           const b200_fr* constants, size_t n_constants, const b200_instr* program, size_t n_instr, void* d_out, void* stream) {
    B200_ENTER(c, d_out);
    StreamScope ss(c, stream);
    return quotient_eval_on(c, reinterpret_cast<const Fr* const*>(d_columns), n_columns, k, ext_k, loads, n_loads, constants, n_constants, program, n_instr,
                            reinterpret_cast<Fr*>(d_out), ss.st);
}
int b200_quotient_eval(const b200_fr* const* columns, size_t n_columns, uint32_t k, uint32_t ext_k, const b200_col_ref* loads, size_t n_loads,
                       const b200_fr* constants, size_t n_constants, const b200_instr* program, size_t n_instr, b200_fr* out) {
    B200_ENTER(c, nullptr);
    B200_CHECK(out && (n_columns == 0 || columns), -1, "quotient_eval: null pointer");
    B200_CHECK(ext_k >= 1 && ext_k <= 28, -1, "quotient_eval: ext_k out of range");
    const size_t N = (size_t)1 << ext_k;
    if (c->stage_a.ensure(sizeof(Fr) * N * (n_columns ? n_columns : 1)) || c->stage_b.ensure(sizeof(Fr) * N)) return -2;
    std::vector<const Fr*> ptrs(n_columns);
    std::vector<HostSeg> up(n_columns);
    for (size_t i = 0; i < n_columns; ++i) {
        B200_CHECK(columns[i], -1, "quotient_eval: column %zu is null", i);
        ptrs[i] = c->stage_a.as<Fr>() + i * N;
        up[i] = HostSeg{(uint8_t*)const_cast<b200_fr*>(columns[i]), sizeof(Fr) * N};
    }
    StreamScope ss(c, nullptr);
    if (int rc = h2d_segments(c, c->stage_a.p, up.data(), n_columns, ss.st)) return rc;
    if (int rc = quotient_eval_on(c, ptrs.data(), n_columns, k, ext_k, loads, n_loads, constants, n_constants, program, n_instr, c->stage_b.as<Fr>(), ss.st)) return rc;
    return d2h_one(c, out, c->stage_b.p, sizeof(Fr) * N, ss.st);
}

// evaluate_h at its natural boundary: the CPU evaluator receives coefficient-form polynomials and builds their cosets itself
// (UPSTREAM plonk/evaluation.rs: `advice_polys.iter().map(|a| domain.coeff_to_extended(a))`), and vanishing/prover.rs then divides by
// the vanishing polynomial and converts back.  One call does the same on the device, so a coefficient column crosses PCIe once
// (n elements) instead of its coset twice (2^ext_k down, 2^ext_k up).
int b200_evaluate_h(const b200_fr* const* polys, const size_t* lengths, size_t n_columns, uint32_t k, uint32_t ext_k, const b200_fr* ext_omega, const b200_fr* zeta,
                    const b200_col_ref* loads, size_t n_loads, const b200_fr* constants, size_t n_constants, const b200_instr* program, size_t n_instr,
                    const b200_fr* t_evaluations, uint32_t t_period, const b200_fr* ext_omega_inv, const b200_fr* ext_ifft_divisor, b200_fr* out) {
    B200_ENTER(c, nullptr);
    B200_CHECK(out && ext_omega && zeta && (n_columns == 0 || (polys && lengths)), -1, "evaluate_h: null pointer");
    B200_CHECK(ext_k >= k && ext_k >= 1 && ext_k <= 28, -1, "evaluate_h: need k <= ext_k <= 28");
    B200_CHECK(!t_evaluations || (t_period >= 1 && t_period <= 1024 && ext_omega_inv && ext_ifft_divisor), -1, "evaluate_h: finishing needs t_evaluations, its period and the inverse-transform constants");
    const size_t N = (size_t)1 << ext_k;
    size_t n_coeff_cols = 0, max_len = 0;
    for (size_t i = 0; i < n_columns; ++i) {
        B200_CHECK(polys[i] && lengths[i] >= 1 && lengths[i] <= N, -1, "evaluate_h: column %zu is null or longer than 2^ext_k", i);
        if (lengths[i] < N) { ++n_coeff_cols; if (lengths[i] > max_len) max_len = lengths[i]; }
    }
    // device layout: stage_c = every column on the extended domain, stage_a = coefficient staging (one sub-batch), stage_b = NTT scratch / output
    if (c->stage_c.ensure(sizeof(Fr) * N * (n_columns ? n_columns : 1))) return -2;
    size_t sub = n_coeff_cols ? call_budget() / (sizeof(Fr) * (N + max_len)) : 1;
    if (sub < 1) sub = 1;
    if (sub > n_coeff_cols) sub = n_coeff_cols ? n_coeff_cols : 1;
    if (c->stage_a.ensure(sizeof(Fr) * (max_len ? max_len : 1) * sub) || c->stage_b.ensure(sizeof(Fr) * N * sub)) return -2;
    StreamScope ss(c, nullptr);
    Fr* ext = c->stage_c.as<Fr>();
    const NttScale pre = coset_scale(as_fr(zeta));
    NttScale none;
    std::vector<size_t> group;           // coefficient columns of equal length are transformed together
    auto flush = [&](size_t len) -> int {
        if (group.empty()) return 0;
        std::vector<HostSeg> up(group.size());
        for (size_t p = 0; p < group.size(); ++p) up[p] = HostSeg{(uint8_t*)const_cast<b200_fr*>(polys[group[p]]), sizeof(Fr) * len};
        if (int rc = h2d_segments(c, c->stage_a.p, up.data(), up.size(), ss.st)) return rc;
        // transform into scratch-free destinations: each polynomial lands in its own column of `ext` (dst stride = distance between them is
        // irregular, so one launch per run of consecutive column indices)
        size_t p0 = 0;
        while (p0 < group.size()) {
            size_t p1 = p0 + 1;
            while (p1 < group.size() && group[p1] == group[p1 - 1] + 1) ++p1;
            if (int rc = ntt_call(c, c->stage_a.as<Fr>() + p0 * len, len, len, c->stage_b.as<Fr>(), ext + group[p0] * N, N, ext_k, as_fr(ext_omega), pre, none, (int)(p1 - p0), ss.st)) return rc;
            p0 = p1;
        }
        B200_CUDA(cudaStreamSynchronize(ss.st));          // the coefficient staging buffer is reused by the next group
        group.clear();
        return 0;
    };
    size_t cur_len = 0;
    for (size_t i = 0; i < n_columns; ++i) {
        if (lengths[i] == N) { if (int rc = h2d_one(c, ext + i * N, polys[i], sizeof(Fr) * N, ss.st)) return rc; continue; }
        if (!group.empty() && (lengths[i] != cur_len || group.size() == sub)) { if (int rc = flush(cur_len)) return rc; }
        cur_len = lengths[i];
        group.push_back(i);
    }
    if (int rc = flush(cur_len)) return rc;
    std::vector<const Fr*> ptrs(n_columns);
    for (size_t i = 0; i < n_columns; ++i) ptrs[i] = ext + i * N;
    Fr* h = c->stage_b.as<Fr>();
    if (int rc = quotient_eval_on(c, ptrs.data(), n_columns, k, ext_k, loads, n_loads, constants, n_constants, program, n_instr, h, ss.st)) return rc;
    if (t_evaluations) {
        if (int rc = scale_cycle_on(c, h, N, t_evaluations, t_period, ss.st)) return rc;
        const NttScale post = coset_unscale(as_fr(zeta), as_fr(ext_ifft_divisor));
        if (int rc = ntt_call(c, h, N, N, ext, h, N, ext_k, as_fr(ext_omega_inv), none, post, 1, ss.st)) return rc;      // `ext` is free again: scratch
    }
    return d2h_one(c, out, h, sizeof(Fr) * N, ss.st);
}

// ---- the extended domain one coset part at a time (include/ezkl_b200_parts.h) ---------------------------------------------------------
// Power tables of the parts' pre-scales c_r^i (c_r = zeta * ext_omega^r, i < 2^k) for r in [part0, part0 + nparts), built on the host and
// staged into c->small; part_scale(r - part0) selects one.
static int stage_part_tables(Ctx* c, uint32_t k, uint32_t part0, uint32_t nparts, const Fr& ext_omega, const Fr& zeta, cudaStream_t st) {
    const size_t len = geo_table_len(k);
    std::vector<Fr> h(len * nparts);
    Fr cr = zeta * fp_pow_u64(ext_omega, part0);
    for (uint32_t j = 0; j < nparts; ++j) { geo_table_fill(cr, k, h.data() + len * j); cr = cr * ext_omega; }
    if (c->small.ensure(sizeof(Fr) * h.size())) return -2;
    return h2d_one(c, c->small.p, h.data(), sizeof(Fr) * h.size(), st);
}
static NttScale part_scale(Ctx* c, uint32_t k, uint32_t j) {
    NttScale s;
    s.mode = NTT_SCALE_GEOMETRIC;
    s.lo_bits = geo_lo_bits(k);
    s.lo = c->small.as<Fr>() + geo_table_len(k) * j;
    s.hi = s.lo + ((size_t)1 << s.lo_bits);
    return s;
}
static int part_args_check(uint32_t k, uint32_t ext_k, uint32_t part, size_t n_coeffs) {
    B200_CHECK(k >= 1 && ext_k >= k && ext_k <= 28, -1, "coeff_to_extended_part: need 1 <= k <= ext_k <= 28");
    B200_CHECK(part < (1u << (ext_k - k)), -1, "coeff_to_extended_part: part %u >= 2^(ext_k - k)", part);
    B200_CHECK(n_coeffs <= ((size_t)1 << k), -1, "coeff_to_extended_part: %zu coefficients > 2^k", n_coeffs);
    return 0;
}
int b200_coeff_to_extended_part_dev(const void* d_coeffs, size_t src_stride, size_t n_coeffs, void* d_tmp, void* d_out, size_t dst_stride, uint32_t k,
                                    uint32_t ext_k, uint32_t part, const b200_fr* ext_omega, const b200_fr* zeta, size_t batch, void* stream) {
    B200_ENTER(c, d_coeffs);
    B200_CHECK(d_coeffs && d_tmp && d_out && ext_omega && zeta, -1, "coeff_to_extended_part: null pointer");
    if (int rc = part_args_check(k, ext_k, part, n_coeffs)) return rc;
    B200_CHECK(batch <= 65535, -1, "coeff_to_extended_part: batch %zu out of range", batch);
    if (batch == 0) return 0;
    StreamScope ss(c, stream);
    const Fr w = as_fr(ext_omega);
    if (int rc = stage_part_tables(c, k, part, 1, w, as_fr(zeta), ss.st)) return rc;
    NttScale none;
    return ntt_call(c, reinterpret_cast<const Fr*>(d_coeffs), src_stride, n_coeffs, reinterpret_cast<Fr*>(d_tmp), reinterpret_cast<Fr*>(d_out), dst_stride, k,
                    fp_pow_u64(w, 1ull << (ext_k - k)), part_scale(c, k, 0), none, (int)batch, ss.st);
}
int b200_coeff_to_extended_part_batch(const b200_fr* const* coeffs, size_t batch, size_t n_coeffs, uint32_t k, uint32_t ext_k, uint32_t part,
                                      const b200_fr* ext_omega, const b200_fr* zeta, b200_fr* const* out) {
    B200_ENTER(c, nullptr);
    B200_CHECK(coeffs && out && ext_omega && zeta, -1, "coeff_to_extended_part: null pointer");
    if (int rc = part_args_check(k, ext_k, part, n_coeffs)) return rc;
    if (batch == 0) return 0;
    const size_t n = (size_t)1 << k, n_in = n_coeffs ? n_coeffs : 1;
    size_t sub = call_budget() / (sizeof(Fr) * n * 3);
    if (sub < 1) sub = 1;
    if (sub > batch) sub = batch;
    if (sub > 65535) sub = 65535;
    if (c->stage_a.ensure(sizeof(Fr) * n_in * sub) || c->stage_b.ensure(sizeof(Fr) * n * sub) || c->stage_c.ensure(sizeof(Fr) * n * sub)) return -2;
    StreamScope ss(c, nullptr);
    const Fr w = as_fr(ext_omega);
    if (int rc = stage_part_tables(c, k, part, 1, w, as_fr(zeta), ss.st)) return rc;
    const Fr wn = fp_pow_u64(w, 1ull << (ext_k - k));
    NttScale none;
    for (size_t b0 = 0; b0 < batch; b0 += sub) {
        const size_t nb = batch - b0 < sub ? batch - b0 : sub;
        std::vector<HostSeg> up(nb), down(nb);
        for (size_t p = 0; p < nb; ++p) {
            B200_CHECK((coeffs[b0 + p] || n_coeffs == 0) && out[b0 + p], -1, "coeff_to_extended_part: polynomial %zu is null", b0 + p);
            up[p] = HostSeg{(uint8_t*)const_cast<b200_fr*>(coeffs[b0 + p]), sizeof(Fr) * n_coeffs};
            down[p] = HostSeg{(uint8_t*)out[b0 + p], sizeof(Fr) * n};
        }
        if (n_coeffs) { if (int rc = h2d_segments(c, c->stage_a.p, up.data(), nb, ss.st)) return rc; }
        if (int rc = ntt_call(c, c->stage_a.as<Fr>(), n_in, n_coeffs, c->stage_b.as<Fr>(), c->stage_c.as<Fr>(), n, k, wn, part_scale(c, k, 0), none, (int)nb, ss.st)) return rc;
        if (int rc = d2h_segments(c, c->stage_c.p, down.data(), nb, ss.st)) return rc;
    }
    return 0;
}

// argument checks shared by both evaluate_h_parts entries; counts the coefficient and extended columns
static int parts_args_check(const size_t* lengths, size_t n_columns, uint32_t k, uint32_t ext_k, const b200_fr* t_evaluations, uint32_t t_period,
                            const b200_fr* ext_omega_inv, const b200_fr* ext_ifft_divisor, size_t* n_coeff, size_t* n_ext, size_t* coeff_elems) {
    B200_CHECK(k >= 1 && ext_k >= k && ext_k <= 28, -1, "evaluate_h_parts: need 1 <= k <= ext_k <= 28");
    const uint32_t d = 1u << (ext_k - k);
    B200_CHECK(!t_evaluations || (t_period >= 1 && t_period <= 1024 && d % t_period == 0 && ext_omega_inv && ext_ifft_divisor), -1,
               "evaluate_h_parts: finishing needs t_evaluations, a period dividing 2^(ext_k - k) and the inverse-transform constants");
    const size_t n = (size_t)1 << k, N = (size_t)1 << ext_k;
    *n_coeff = *n_ext = *coeff_elems = 0;
    for (size_t i = 0; i < n_columns; ++i) {
        if (lengths[i] == N) ++*n_ext;
        else {
            B200_CHECK(lengths[i] >= 1 && lengths[i] <= n, -1, "evaluate_h_parts: column %zu has %zu elements: neither <= 2^k (coefficients) nor 2^ext_k (extended)", i, lengths[i]);
            ++*n_coeff; *coeff_elems += lengths[i];
        }
    }
    return 0;
}
// The d parts of one evaluate_h.  Column i is a coefficient column (coeff[i], device, lengths[i] <= 2^k), or an extended column read either in
// place (ext_dev[i], device, 2^ext_k elements, stride d per part) or gathered from the host per part (ext_host[i]).  parts: device buffer of
// (n_coeff + n_ext_host) * 2^k elements; scratch: 2^ext_k elements; out: 2^ext_k elements.  Tables of the pre-scales are in c->small.
static int evaluate_h_parts_on(Ctx* c, const Fr* const* coeff, const Fr* const* ext_dev, const b200_fr* const* ext_host, const size_t* lengths, size_t n_columns,
                               uint32_t k, uint32_t ext_k, const Fr& ext_omega, const Fr& zeta, const b200_col_ref* loads, size_t n_loads,
                               const b200_fr* constants, size_t n_constants, const b200_instr* program, size_t n_instr, const b200_fr* t_evaluations,
                               uint32_t t_period, const b200_fr* ext_omega_inv, const b200_fr* ext_ifft_divisor, Fr* parts, Fr* scratch, Fr* out, cudaStream_t st) {
    const uint32_t log_d = ext_k - k, d = 1u << log_d;
    const size_t n = (size_t)1 << k, N = (size_t)1 << ext_k;
    const Fr wn = fp_pow_u64(ext_omega, d);
    if (int rc = stage_part_tables(c, k, 0, d, ext_omega, zeta, st)) return rc;
    // every column's buffer inside a part: coefficient columns, then host-gathered extended columns, in column order
    std::vector<size_t> slot(n_columns, 0);
    size_t ns = 0;
    for (size_t i = 0; i < n_columns; ++i) if (lengths[i] != N) slot[i] = ns++;
    for (size_t i = 0; i < n_columns; ++i) if (lengths[i] == N && ext_host) slot[i] = ns++;
    // runs of coefficient columns transformed in one launch: equal length, sources at one stride, consecutive slots, at most d columns
    // (the transform scratch holds d parts)
    struct Run { size_t first, last, count, stride; };
    std::vector<Run> runs;
    for (size_t i = 0; i < n_columns; ++i) {
        if (lengths[i] == N) continue;
        if (!runs.empty()) {
            Run& r = runs.back();
            const uintptr_t a = (uintptr_t)coeff[r.last], b = (uintptr_t)coeff[i];
            const size_t gap = b > a ? (size_t)(b - a) / sizeof(Fr) : 0;
            if (lengths[i] == lengths[r.first] && b > a && (b - a) % sizeof(Fr) == 0 && gap >= lengths[i] && (r.count == 1 || gap == r.stride) && r.count < d) {
                r.stride = gap; r.last = i; ++r.count; continue;
            }
        }
        runs.push_back(Run{i, i, 1, lengths[i]});
    }
    // per-part program: the caller's, then (finishing) one multiplication of the row result by the part's vanishing factor
    std::vector<QInstr> prog(n_instr);
    if (n_instr) memcpy(prog.data(), program, sizeof(QInstr) * n_instr);
    std::vector<Fr> consts(n_constants);
    if (n_constants) memcpy(consts.data(), constants, sizeof(Fr) * n_constants);
    const bool fuse = t_evaluations && n_instr;
    if (fuse) {
        QInstr m;
        m.op_dst = QOP_MUL | Q_NOSTORE; m.a = (uint32_t)QSRC_PREV << 30; m.b = ((uint32_t)QSRC_CONST << 30) | (uint32_t)n_constants; m.c = 0;
        prog.push_back(m);
        consts.push_back(fp_zero<FrTag>());
    }
    std::vector<QLoad> ql(n_loads);
    for (size_t i = 0; i < n_loads; ++i) {
        ql[i].column = loads[i].column;
        ql[i].offset = (uint32_t)((((int64_t)loads[i].rotation % (int64_t)n) + (int64_t)n) % (int64_t)n);     // Rotation(rot) inside a part
    }
    std::vector<const Fr*> ptrs(n_columns);
    std::vector<uint32_t> shift(n_columns);
    NttScale none;
    for (uint32_t r = 0; r < d; ++r) {
        const NttScale pre = part_scale(c, k, r);
        for (const Run& run : runs) {
            if (int rc = ntt_call(c, coeff[run.first], run.stride, lengths[run.first], scratch, parts + slot[run.first] * n, n, k, wn, pre, none, (int)run.count, st)) return rc;
        }
        for (size_t i = 0; i < n_columns; ++i) {
            if (lengths[i] != N) { ptrs[i] = parts + slot[i] * n; shift[i] = 0; }
            else if (ext_host) {
                B200_CHECK(ext_host[i], -1, "evaluate_h_parts: column %zu is null", i);
                if (int rc = h2d_strided(c, parts + slot[i] * n, reinterpret_cast<const uint8_t*>(ext_host[i] + r), n, sizeof(Fr), d, st)) return rc;
                ptrs[i] = parts + slot[i] * n; shift[i] = 0;
            } else { ptrs[i] = ext_dev[i] + r; shift[i] = log_d; }
        }
        if (fuse) consts.back() = as_fr(t_evaluations + (r % t_period));
        if (int rc = quotient_eval_part_run(ptrs.data(), shift.data(), n_columns, k, log_d, ql.data(), n_loads, consts.data(), consts.size(), prog.data(), prog.size(),
                                            out + r, c->quot_ws, st)) return rc;
        g_launches += 1;
    }
    if (t_evaluations) {
        const NttScale post = coset_unscale(zeta, as_fr(ext_ifft_divisor));
        if (int rc = ntt_call(c, out, N, N, scratch, out, N, ext_k, as_fr(ext_omega_inv), none, post, 1, st)) return rc;
    }
    return 0;
}
int b200_evaluate_h_parts_dev(const void* const* d_polys, const size_t* lengths, size_t n_columns, uint32_t k, uint32_t ext_k, const b200_fr* ext_omega,
                              const b200_fr* zeta, const b200_col_ref* loads, size_t n_loads, const b200_fr* constants, size_t n_constants,
                              const b200_instr* program, size_t n_instr, const b200_fr* t_evaluations, uint32_t t_period, const b200_fr* ext_omega_inv,
                              const b200_fr* ext_ifft_divisor, void* d_out, void* stream) {
    B200_ENTER(c, d_out);
    B200_CHECK(d_out && ext_omega && zeta && (n_columns == 0 || (d_polys && lengths)) && (n_loads == 0 || loads) && (n_constants == 0 || constants) &&
               (n_instr == 0 || program), -1, "evaluate_h_parts: null pointer");
    size_t n_coeff, n_ext, coeff_elems;
    if (int rc = parts_args_check(lengths, n_columns, k, ext_k, t_evaluations, t_period, ext_omega_inv, ext_ifft_divisor, &n_coeff, &n_ext, &coeff_elems)) return rc;
    std::vector<const Fr*> cols(n_columns);
    for (size_t i = 0; i < n_columns; ++i) { B200_CHECK(d_polys[i], -1, "evaluate_h_parts: column %zu is null", i); cols[i] = reinterpret_cast<const Fr*>(d_polys[i]); }
    const size_t n = (size_t)1 << k, N = (size_t)1 << ext_k;
    if (c->stage_c.ensure(sizeof(Fr) * n * (n_coeff ? n_coeff : 1)) || c->stage_b.ensure(sizeof(Fr) * N)) return -2;
    StreamScope ss(c, stream);
    return evaluate_h_parts_on(c, cols.data(), cols.data(), nullptr, lengths, n_columns, k, ext_k, as_fr(ext_omega), as_fr(zeta), loads, n_loads, constants, n_constants,
                               program, n_instr, t_evaluations, t_period, ext_omega_inv, ext_ifft_divisor, c->stage_c.as<Fr>(), c->stage_b.as<Fr>(),
                               reinterpret_cast<Fr*>(d_out), ss.st);
}
int b200_evaluate_h_parts(const b200_fr* const* polys, const size_t* lengths, size_t n_columns, uint32_t k, uint32_t ext_k, const b200_fr* ext_omega,
                          const b200_fr* zeta, const b200_col_ref* loads, size_t n_loads, const b200_fr* constants, size_t n_constants,
                          const b200_instr* program, size_t n_instr, const b200_fr* t_evaluations, uint32_t t_period, const b200_fr* ext_omega_inv,
                          const b200_fr* ext_ifft_divisor, b200_fr* out) {
    B200_ENTER(c, nullptr);
    B200_CHECK(out && ext_omega && zeta && (n_columns == 0 || (polys && lengths)) && (n_loads == 0 || loads) && (n_constants == 0 || constants) &&
               (n_instr == 0 || program), -1, "evaluate_h_parts: null pointer");
    size_t n_coeff, n_ext, coeff_elems;
    if (int rc = parts_args_check(lengths, n_columns, k, ext_k, t_evaluations, t_period, ext_omega_inv, ext_ifft_divisor, &n_coeff, &n_ext, &coeff_elems)) return rc;
    for (size_t i = 0; i < n_columns; ++i) B200_CHECK(polys[i], -1, "evaluate_h_parts: column %zu is null", i);
    const size_t n = (size_t)1 << k, N = (size_t)1 << ext_k;
    // device layout: stage_a = resident coefficients (packed in column order), stage_c = one part of every column, stage_b = [output | scratch]
    if (c->stage_a.ensure(sizeof(Fr) * (coeff_elems ? coeff_elems : 1)) || c->stage_c.ensure(sizeof(Fr) * n * (n_coeff + n_ext ? n_coeff + n_ext : 1)) ||
        c->stage_b.ensure(sizeof(Fr) * N * 2)) return -2;
    std::vector<const Fr*> cols(n_columns, nullptr);
    std::vector<HostSeg> up;
    size_t off = 0;
    for (size_t i = 0; i < n_columns; ++i) {
        if (lengths[i] == N) continue;
        cols[i] = c->stage_a.as<Fr>() + off;
        up.push_back(HostSeg{(uint8_t*)const_cast<b200_fr*>(polys[i]), sizeof(Fr) * lengths[i]});
        off += lengths[i];
    }
    StreamScope ss(c, nullptr);
    if (!up.empty()) { if (int rc = h2d_segments(c, c->stage_a.p, up.data(), up.size(), ss.st)) return rc; }
    Fr* h = c->stage_b.as<Fr>();
    if (int rc = evaluate_h_parts_on(c, cols.data(), nullptr, polys, lengths, n_columns, k, ext_k, as_fr(ext_omega), as_fr(zeta), loads, n_loads, constants, n_constants,
                                     program, n_instr, t_evaluations, t_period, ext_omega_inv, ext_ifft_divisor, c->stage_c.as<Fr>(), h + N, h, ss.st)) return rc;
    return d2h_one(c, out, h, sizeof(Fr) * N, ss.st);
}

}  // extern "C"
#pragma GCC visibility pop
