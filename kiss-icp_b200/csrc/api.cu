// Host side of the C-ABI (include/kiss_icp_b200.h). Thin: argument checks, H2D/D2H copies,
// capacity management of the HBM voxel table, and ONE cooperative launch per call.
// There is no CPU fallback anywhere in this file: without a CUDA device every compute entry
// point returns KB_ERR_NO_DEVICE.
#include <cuda_runtime.h>

#include <algorithm>
#include <array>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <numeric>
#include <string>
#include <vector>

#include "../../include/kiss_icp_b200.h"
#include "../../include/kiss_icp_b200_debug.h"
#include "kernels.cuh"

using namespace kb;

namespace {

thread_local std::string tl_err;
thread_local int tl_device = 0;
thread_local cudaStream_t tl_user_stream = nullptr;
thread_local int tl_grid_blocks = 0;

int fail(int status, const char *fmt, ...) {
    char buf[4096];  // (room for the per-CTA phase marks of the hang reports)
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    tl_err = buf;
    return status;
}

#define CK(call)                                                                              \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess) return fail(KB_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); \
    } while (0)
#define RET(call)              \
    do {                       \
        int s_ = (call);       \
        if (s_ != KB_OK) return s_; \
    } while (0)

int device_count() {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

bool device_is_stuck(int device);
template <class T>
struct DBuf {
    T *p = nullptr;
    size_t n = 0;
    int ensure(size_t count) {
        if (count <= n) return KB_OK;
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
        // grow with 25% headroom: scan sizes jitter from frame to frame and a cudaFree/cudaMalloc
        // pair per new maximum would put milliseconds of allocator time on the hot path
        const size_t want = std::max<size_t>(count + count / 4, 1024);
        CK(cudaMalloc(&p, want * sizeof(T)));
        n = want;
        return KB_OK;
    }
    ~DBuf() {
        if (p && !device_is_stuck(-1)) cudaFree(p);  // (-1: any device)
    }
};

// KB_TRACE_STALLS=<ms>: report host-side API calls of the frame paths that block longer than <ms> (diagnostic)
struct StallTrace {
    const char *what;
    std::chrono::steady_clock::time_point t0;
    static double limit_ms() {
        static const double v = [] {
            const char *e = std::getenv("KB_TRACE_STALLS");
            return e ? std::atof(e) : 0.0;
        }();
        return v;
    }
    explicit StallTrace(const char *w) : what(w) {
        if (limit_ms() > 0.0) t0 = std::chrono::steady_clock::now();
    }
    ~StallTrace() {
        if (limit_ms() > 0.0) {
            const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
            if (ms > limit_ms()) std::fprintf(stderr, "[kb stall] %s took %.1f ms\n", what, ms);
        }
    }
};

size_t pow2_at_least(size_t v) {
    size_t p = 1;
    while (p < v) p <<= 1;
    return p;
}

int watchdog_check_fwd(int device);
int watchdog_init_fwd(int device);
void device_stuck_fwd(int device);
std::string phase_marks_fwd(int device);

// execution context: device, stream, persistent-grid size and the cross-CTA scratch
struct Exec {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int grid = 0;
    Scratch sc{};  // all pointers null, profiling off
    TeamScratch team{};  // ll / out (qrec belongs to the caller's workspace)
    size_t icp_smem = 96 * 1024;  // dynamic shared memory of the ICP kernels: candidate coordinates of the team's source points (KB_ICP_SMEM_KB)
    int icp_team_q = TQ_PER_CTA;  // source points per CTA of the ICP team (KB_ICP_TEAM_Q; 0 = whole-grid ICP loop)
    unsigned tag_seq = 0;  // launch sequence number of the tagged ICP protocol
    unsigned long long launches = 0;
    bool bar_dirty = true;  // the barrier words may be non-zero (a kernel without Grid::finish() ran last)
    std::vector<const void *> smem_opted;  // kernels opted in to > 48 KB of dynamic shared memory on THIS context's device
    unsigned next_tag_base() { return (++tag_seq) << 13; }  // 8192 epochs per launch

    int init() {
        if (device_count() <= 0) return fail(KB_ERR_NO_DEVICE, "no CUDA device visible (this library has no CPU fallback)");
        device = tl_device;
        CK(cudaSetDevice(device));
        RET(watchdog_init_fwd(device));
        if (tl_user_stream) {
            stream = tl_user_stream;
        } else {
            CK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
            own_stream = true;
        }
        int sms = 0, coop = 0;
        CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
        CK(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device));
        if (!coop) return fail(KB_ERR_CUDA, "device does not support cooperative launch");
        grid = tl_grid_blocks > 0 ? std::min(tl_grid_blocks, sms) : sms;
        grid = std::min(grid, 256);  // the two-level gather tree of the ICP loop handles up to 16 x 16 CTAs
        CK(cudaMalloc(&sc.bar, BAR_WORDS * sizeof(unsigned)));
        CK(cudaMemsetAsync(sc.bar, 0, BAR_WORDS * sizeof(unsigned), stream));
        CK(cudaMalloc(&sc.blk_d, sizeof(double) * 2 * grid * NPART));
        CK(cudaMalloc(&sc.blk_i, sizeof(int) * 2 * grid));
        CK(cudaMalloc(&sc.ll_part, sizeof(uint4) * NPART * grid));
        CK(cudaMalloc(&sc.ll_res, sizeof(uint4) * LL_RES));
        CK(cudaMalloc(&sc.ll_group, sizeof(uint4) * NPART * 16));
        CK(cudaMemsetAsync(sc.ll_group, 0, sizeof(uint4) * NPART * 16, stream));
        CK(cudaMemsetAsync(sc.ll_part, 0, sizeof(uint4) * NPART * grid, stream));
        CK(cudaMemsetAsync(sc.ll_res, 0, sizeof(uint4) * LL_RES, stream));
        CK(cudaMalloc(&team.ll, sizeof(uint4) * 2 * NPART * TEAM_MAX * TEAM_MAX));  // 11 MB: one copy of the partials per reader
        CK(cudaMemsetAsync(team.ll, 0, sizeof(uint4) * 2 * NPART * TEAM_MAX * TEAM_MAX, stream));
        CK(cudaMalloc(&team.out, sizeof(double) * 16));
        if (const char *e = std::getenv("KB_ICP_TEAM_Q")) icp_team_q = std::max(0, std::min(std::atoi(e), TQ_MAX));
        if (const char *e = std::getenv("KB_ICP_SMEM_KB")) icp_smem = static_cast<size_t>(std::max(60, std::min(std::atoi(e), 180))) * 1024;
        team.smem_bytes = static_cast<int>(icp_smem);
        team.radius_frac = 0.2;
        if (const char *e = std::getenv("KB_ICP_RADIUS")) team.radius_frac = std::max(0.01, std::min(std::atof(e), 0.45));
        CK(cudaMalloc(&sc.dbg, sizeof(unsigned long long) * (64 + 4 * grid)));
        CK(cudaMemsetAsync(sc.dbg, 0, sizeof(unsigned long long) * (64 + 4 * grid), stream));
        return KB_OK;
    }
    ~Exec() {
        if (device_is_stuck(device)) return;
        if (sc.bar) cudaFree(sc.bar);
        if (sc.blk_d) cudaFree(sc.blk_d);
        if (sc.blk_i) cudaFree(sc.blk_i);
        if (sc.ll_part) cudaFree(sc.ll_part);
        if (sc.ll_res) cudaFree(sc.ll_res);
        if (sc.ll_group) cudaFree(sc.ll_group);
        if (sc.dbg) cudaFree(sc.dbg);
        if (team.ll) cudaFree(team.ll);
        if (team.out) cudaFree(team.out);
        if (own_stream && stream) cudaStreamDestroy(stream);
    }
    template <class P>
    int coop(void (*kern)(P), const P &p, size_t smem = 0, bool self_reset = false) {
        CK(cudaSetDevice(device));
        if (smem > 48 * 1024) {  // opt in to large dynamic shared memory once per kernel AND device (the attribute is per device)
            const void *k = reinterpret_cast<const void *>(kern);
            if (std::find(smem_opted.begin(), smem_opted.end(), k) == smem_opted.end()) {
                CK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
                smem_opted.push_back(k);
            }
        }
        if (!self_reset || bar_dirty)  // kernels that end with Grid::finish() leave the barrier words zeroed themselves
            CK(cudaMemsetAsync(sc.bar, 0, BAR_WORDS * sizeof(unsigned), stream));
        bar_dirty = !self_reset;
        void *args[] = {const_cast<P *>(&p)};
        CK(cudaLaunchCooperativeKernel(reinterpret_cast<const void *>(kern), dim3(grid), dim3(BLOCK), args, smem, stream));
        ++launches;
        return KB_OK;
    }
    template <class A, class B>
    int coop(void (*kern)(A, B), const A &a, const B &b) {
        CK(cudaSetDevice(device));
        CK(cudaMemsetAsync(sc.bar, 0, BAR_WORDS * sizeof(unsigned), stream));
        bar_dirty = true;
        void *args[] = {const_cast<A *>(&a), const_cast<B *>(&b)};
        CK(cudaLaunchCooperativeKernel(reinterpret_cast<const void *>(kern), dim3(grid), dim3(BLOCK), args, 0, stream));
        ++launches;
        return KB_OK;
    }
    // wait for the stream with a deadline (KB_SYNC_TIMEOUT_S, default 30 s; 0 = wait forever): a launch that never
    // ends is reported as KB_ERR_CUDA instead of hanging the caller (the device watchdog should have fired long before)
    int sync() {
        RET(wait_deadline([&] { return cudaStreamQuery(stream); }, "stream"));
        return watchdog_check_fwd(device);
    }
    template <class Q>
    int wait_deadline(Q query, const char *what) {
        static const double limit_s = [] {
            const char *e = std::getenv("KB_SYNC_TIMEOUT_S");
            return e ? std::atof(e) : 30.0;
        }();
        const auto t0 = std::chrono::steady_clock::now();
        for (unsigned spins = 0;; ++spins) {
            const cudaError_t e = query();
            if (e == cudaSuccess) return KB_OK;
            if (e != cudaErrorNotReady) return fail(KB_ERR_CUDA, "%s wait failed: %s", what, cudaGetErrorString(e));
            if ((spins & 0x3ff) == 0x3ff && limit_s > 0.0 &&
                std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() > limit_s) {
                const int wd = watchdog_check_fwd(device);
                device_stuck_fwd(device);
                if (wd != KB_OK) return wd;
                return fail(KB_ERR_CUDA, "the device did not finish the %s within %.0f s (launch %llu): giving up; %s", what, limit_s, launches,
                            phase_marks_fwd(device).c_str());
            }
        }
    }
};

// the device watchdog's report (device_ops.cuh): mapped host words per device, checked after every synchronisation
struct WatchdogHost {
    unsigned *host = nullptr;  // [0] flag [1] code [2] block [3] thread [4] a [5] b
};
WatchdogHost g_wd[64];
int watchdog_init(int device) {
    static std::mutex mu;
    std::lock_guard<std::mutex> lock(mu);
    if (device < 0 || device >= 64 || g_wd[device].host) return KB_OK;
    unsigned *h = nullptr, *d = nullptr;
    CK(cudaHostAlloc(&h, 8 * sizeof(unsigned), cudaHostAllocMapped));
    std::memset(h, 0, 8 * sizeof(unsigned));
    CK(cudaHostGetDevicePointer(&d, h, 0));
    CK(cudaMemcpyToSymbol(g_kb_wd_host, &d, sizeof(d)));
    // give up after 2^24 polls (of the order of 10 s, below the host's 30 s deadline). 2^22 (a second or two) fired once in
    // ~40 full-file test runs at the FIRST grid barrier of a launch; whether that was a stall or a deadlock is not known.
    unsigned init[8] = {0, 0, 0, 0, 0, 0, 0, 24};
    if (const char *e = std::getenv("KB_WATCHDOG_SHIFT")) init[7] = static_cast<unsigned>(std::max(10, std::min(std::atoi(e), 31)));
    CK(cudaMemcpyToSymbol(g_kb_wd, init, sizeof(init)));
    g_wd[device].host = h;
    return KB_OK;
}
// after a synchronisation: did a spin loop of the last launches give up?
int watchdog_check(int device) {
    unsigned *h = (device >= 0 && device < 64) ? g_wd[device].host : nullptr;
    if (!h || !*reinterpret_cast<volatile unsigned *>(h)) return KB_OK;
    const unsigned code = h[1], block = h[2], thread = h[3], a = h[4], b = h[5];
    h[0] = 0;
    unsigned zero = 0;
    cudaMemcpyToSymbol(g_kb_wd, &zero, sizeof(zero));  // re-arm
    static const char *names[] = {"?", "grid barrier", "ICP gather", "ICP result record", "ICP team gather"};
    // where every CTA of the last k_register_frame was (the launch has ended: a plain copy)
    std::string marks;
    unsigned m[256];
    if (cudaMemcpyFromSymbol(m, g_kb_marks, sizeof(m)) == cudaSuccess) {
        marks = "; phase marks per CTA:";
        char buf[16];
        for (int i = 0; i < 160; ++i) {
            std::snprintf(buf, sizeof(buf), " %x", m[i]);
            marks += buf;
        }
    }
    cudaGetLastError();
    return fail(KB_ERR_CUDA, "device watchdog: a kernel gave up waiting at the %s (block %u, thread %u, a=%u, b=%u; grid barrier: a = target, b = counter); "
                             "the results of that launch are invalid%s",
                names[code < sizeof(names) / sizeof(names[0]) ? code : 0], block, thread, a, b, marks.c_str());
}

bool g_stuck[64];
void device_stuck_fwd(int device) {
    if (device >= 0 && device < 64) g_stuck[device] = true;
}
// a launch on this device never ended: cudaFree & co. would block forever, so the destructors leak instead
bool device_is_stuck(int device) {
    if (device < 0) {
        for (bool b : g_stuck)
            if (b) return true;
        return false;
    }
    return device < 64 && g_stuck[device];
}
std::string phase_marks_fwd(int device) {
    // the compute stream is stuck: read the marks on a stream of their own (bounded wait, the copy engine is free)
    unsigned marks[256];
    cudaStream_t side = nullptr;
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&side, cudaStreamNonBlocking) != cudaSuccess) return "";
    std::string out;
    if (cudaMemcpyFromSymbolAsync(marks, g_kb_marks, sizeof(marks), 0, cudaMemcpyDeviceToHost, side) == cudaSuccess) {
        const auto t0 = std::chrono::steady_clock::now();
        cudaError_t q;
        while ((q = cudaStreamQuery(side)) == cudaErrorNotReady &&
               std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() < 5.0) {
        }
        if (q == cudaSuccess) {
            out = "phase marks per CTA:";
            char buf[16];
            for (int i = 0; i < 160; ++i) {
                std::snprintf(buf, sizeof(buf), " %x", marks[i]);
                out += buf;
            }
        } else {
            out = "(phase marks unreadable)";
        }
    }
    return out;  // (the side stream is leaked with the rest of the stuck context)
}
int watchdog_check_fwd(int device) { return watchdog_check(device); }
int watchdog_init_fwd(int device) { return watchdog_init(device); }

int make_exec(std::shared_ptr<Exec> *out) {
    auto e = std::make_shared<Exec>();
    RET(e->init());
    *out = e;
    return KB_OK;
}

// per-call workspace sized by the largest cloud seen
struct Work {
    DBuf<double> in, ts, tmp, pre, ds1, src, work, tp;
    DBuf<double> pre_b, ds1_b, src_b;  // second front-end set (Workspace::fr[1])
    DBuf<QList> qrec;                  // per source point: candidate lists of the ICP team
    DBuf<int> next, touched, ds_chunk, ds_order, ds2_chunk, ds2_order, cnt;
    DBuf<int4> ds_slots, ds2_slots;
    DBuf<int2> ds_sim, ds2_sim;
    int ensure(size_t n) {
        n = std::max<size_t>(n, 1);
        RET(in.ensure(3 * n));
        RET(ts.ensure(n));
        RET(tmp.ensure(3 * n));
        RET(pre.ensure(3 * n));
        RET(ds1.ensure(3 * n));
        RET(src.ensure(3 * n));
        RET(work.ensure(3 * n));
        RET(tp.ensure(3 * n));
        RET(next.ensure(n));
        RET(touched.ensure(n));
        const size_t b = pow2_at_least(2 * n);
        RET(ds_slots.ensure(b));
        RET(ds_chunk.ensure(DS_MAX_CHUNKS));
        RET(ds_order.ensure(b));
        RET(ds_sim.ensure(b));
        RET(ds2_slots.ensure(b));
        RET(ds2_chunk.ensure(DS_MAX_CHUNKS));
        RET(ds2_order.ensure(b));
        RET(ds2_sim.ensure(b));
        RET(cnt.ensure(8));
        return KB_OK;
    }
    // the buffers only a pipeline needs: the second front-end set; the candidate lists of the ICP team
    int ensure_pipeline(size_t n) {
        n = std::max<size_t>(n, 1);
        RET(pre_b.ensure(3 * n));
        RET(ds1_b.ensure(3 * n));
        RET(src_b.ensure(3 * n));
        return qrec.ensure(n);
    }
    DsScratch ds_view() { return DsScratch{ds_slots.p, ds_chunk.p, ds_order.p, ds_sim.p}; }
    DsScratch ds2_view() { return DsScratch{ds2_slots.p, ds2_chunk.p, ds2_order.p, ds2_sim.p}; }
    Workspace view() {
        Workspace w;
        w.tmp = tmp.p;
        w.fr[0] = Front{pre.p, ds1.p, src.p, cnt.p};
        w.fr[1] = Front{pre_b.p, ds1_b.p, src_b.p, cnt.p + 4};
        w.work = work.p;
        w.tp = tp.p;
        w.next = next.p;
        w.touched = touched.p;
        w.ds = ds_view();
        w.ds2 = ds2_view();
        return w;
    }
};

bool to_se3(const double M[16], SE3 *T) { return se3_from_matrix(M, T); }

}  // namespace

// =============================================================================================
struct kb_map {
    std::shared_ptr<Exec> ex;
    double voxel_size, max_distance;
    unsigned cap;
    size_t capacity = 0;
    int4 *slots = nullptr;
    double *points = nullptr;
    int *head = nullptr;
    int *pcount = nullptr;
    int *pending = nullptr;
    int *counters = nullptr;
    int h_counters[C_NCOUNTERS] = {0};
    Work ws;
    DBuf<double> q_in, q_outp, q_outd;
    DBuf<unsigned long long> q_cand;
    bool borrowed = false;

    MapView view() const {
        MapView m;
        m.slots = slots;
        m.points = points;
        m.head = head;
        m.pcount = pcount;
        m.pending = pending;
        m.counters = counters;
        m.mask = static_cast<unsigned>(capacity - 1);
        m.cap = static_cast<int>(cap);
        m.voxel_size = voxel_size;
        m.max_distance = max_distance;
        m.map_resolution = std::sqrt(voxel_size * voxel_size / cap);
        m.vdiv = make_voxel_div(voxel_size);
        return m;
    }
    // the table a rebuild moves the map into. Rebuilds are periodic in steady state (tombstones of voxels that left
    // max_distance accumulate until load 0.5) and mostly keep the size, so the previous table is kept as a spare
    // and the two ping-pong: cudaMalloc/cudaFree of a few hundred MB took 10-300 ms on the hot path.
    struct Table {
        size_t capacity = 0;
        int4 *slots = nullptr;
        double *points = nullptr;
        int *head = nullptr, *pcount = nullptr, *pending = nullptr, *counters = nullptr;
    };
    Table spare;
    static void free_table(Table &t) {
        if (t.slots) cudaFree(t.slots);
        if (t.points) cudaFree(t.points);
        if (t.head) cudaFree(t.head);
        if (t.pcount) cudaFree(t.pcount);
        if (t.pending) cudaFree(t.pending);
        if (t.counters) cudaFree(t.counters);
        t = Table{};
    }
    Table current() const { return Table{capacity, slots, points, head, pcount, pending, counters}; }
    void adopt(const Table &t) {
        capacity = t.capacity;
        slots = t.slots;
        points = t.points;
        head = t.head;
        pcount = t.pcount;
        pending = t.pending;
        counters = t.counters;
    }
    ~kb_map() {
        if (ex && device_is_stuck(ex->device)) return;
        if (ex) cudaSetDevice(ex->device);
        Table t = current();
        free_table(t);
        free_table(spare);
    }
    // an empty table of cap_slots slots: the spare if it has that size, else a fresh allocation
    int take_table(size_t cap_slots, Table *out) {
        Table t;
        if (spare.capacity == cap_slots) {
            t = spare;
            spare = Table{};
        } else {
            free_table(spare);
            t.capacity = cap_slots;
            auto bail = [&](cudaError_t e) {
                free_table(t);
                return fail(KB_ERR_CUDA, "voxel table allocation (%zu slots): %s", cap_slots, cudaGetErrorString(e));
            };
            cudaError_t e;
            if ((e = cudaMalloc(&t.slots, cap_slots * sizeof(int4))) != cudaSuccess) return bail(e);
            if ((e = cudaMalloc(&t.points, cap_slots * cap * 3 * sizeof(double))) != cudaSuccess) return bail(e);
            if ((e = cudaMalloc(&t.head, cap_slots * sizeof(int))) != cudaSuccess) return bail(e);
            if ((e = cudaMalloc(&t.pcount, cap_slots * sizeof(int))) != cudaSuccess) return bail(e);
            if ((e = cudaMalloc(&t.pending, cap_slots * PEND * sizeof(int))) != cudaSuccess) return bail(e);
            if ((e = cudaMalloc(&t.counters, sizeof(int) * C_NCOUNTERS)) != cudaSuccess) return bail(e);
        }
        k_map_fill<<<std::min<size_t>(4096, (cap_slots + 255) / 256), 256, 0, ex->stream>>>(t.slots, t.head, t.pcount, cap_slots);
        ++ex->launches;
        CK(cudaGetLastError());
        CK(cudaMemsetAsync(t.counters, 0, sizeof(int) * C_NCOUNTERS, ex->stream));
        *out = t;
        return KB_OK;
    }
    // make room for `extra` more voxels at load factor <= 0.5 (tombstones count as load)
    bool would_grow(size_t extra) const {  // ensure_capacity(extra) would rebuild the table (needs an idle stream)
        const size_t live = static_cast<size_t>(h_counters[C_LIVE]), tomb = static_cast<size_t>(h_counters[C_TOMB]);
        return !capacity || (live + tomb + extra) * 2 > capacity;
    }
    int ensure_capacity(size_t extra, size_t force_want = 0) {
        CK(cudaSetDevice(ex->device));
        const size_t live = static_cast<size_t>(h_counters[C_LIVE]), tomb = static_cast<size_t>(h_counters[C_TOMB]);
        if (!force_want && capacity && (live + tomb + extra) * 2 <= capacity) return KB_OK;
        // grow/rebuild target: load factor <= 1/3 right after the rebuild (tombstones then accumulate up to 1/2)
        static const size_t cap_factor = [] {
            const char *e = std::getenv("KB_MAP_CAP_FACTOR");  // tuning aid: slots per expected voxel after a rebuild
            return (e && std::atoi(e) >= 2) ? static_cast<size_t>(std::atoi(e)) : size_t(3);
        }();
        // never shrink on the hot path: the spare table has the current size, a smaller one would mean cudaMalloc
        const size_t want = force_want ? force_want
                                       : std::max<size_t>({pow2_at_least(cap_factor * (live + extra)), size_t(1) << 14, capacity});
        if (want > (size_t(1) << 31)) return fail(KB_ERR_INVALID_ARG, "voxel table would exceed 2^31 slots");
        StallTrace trace("voxel table rebuild");
        Table nt;
        RET(take_table(want, &nt));
        if (capacity && live) {
            MapView from = view();
            MapView to = from;
            to.slots = nt.slots;
            to.points = nt.points;
            to.head = nt.head;
            to.pcount = nt.pcount;
            to.pending = nt.pending;
            to.counters = nt.counters;
            to.mask = static_cast<unsigned>(want - 1);
            k_map_rehash<<<std::min<size_t>(2048, (capacity * 32 + 255) / 256), 256, 0, ex->stream>>>(from, to);
            ++ex->launches;
            CK(cudaGetLastError());
            CK(cudaMemcpyAsync(h_counters, nt.counters, sizeof(int) * C_NCOUNTERS, cudaMemcpyDeviceToHost, ex->stream));
            RET(ex->sync());
        } else {
            std::memset(h_counters, 0, sizeof(h_counters));
        }
        Table old = current();
        adopt(nt);
        free_table(spare);  // (empty unless take_table allocated)
        spare = old;        // stays allocated: the next same-size rebuild moves back into it
        return KB_OK;
    }
    // allocate the table AND its spare for `slots` slots now (pipeline creation), so that neither growth nor the
    // periodic tombstone rebuild has to call cudaMalloc while frames are being registered
    int reserve(size_t slots) {
        slots = pow2_at_least(slots);
        if (slots > capacity) RET(ensure_capacity(0, slots));
        if (spare.capacity != capacity) {
            Table t;
            RET(take_table(capacity, &t));  // frees a spare of another size
            spare = t;
        }
        return KB_OK;
    }
    int pull_counters() {
        CK(cudaMemcpyAsync(h_counters, counters, sizeof(int) * C_NCOUNTERS, cudaMemcpyDeviceToHost, ex->stream));
        RET(ex->sync());
        if (h_counters[C_STATUS] & ST_TABLE_FULL) return fail(KB_ERR_CUDA, "voxel table overflow (internal capacity bug)");
        return KB_OK;
    }
    // d_pts already on the device
    int update_dev(const double *d_pts, size_t n, bool has_pose, const SE3 &pose, bool do_add, bool do_remove,
                   const V3 &origin) {
        RET(ensure_capacity(do_add ? n : 0));
        MapUpdParams P;
        P.m = view();
        P.sc = ex->sc;
        P.pts = d_pts;
        P.n = static_cast<int>(n);
        P.has_pose = has_pose;
        P.pose = pose;
        P.do_add = do_add && n > 0;
        P.do_remove = do_remove;
        P.origin = origin;
        P.tp = ws.tp.p;
        P.next = ws.next.p;
        P.touched = ws.touched.p;
        RET(ex->coop(k_map_update, P));
        return KB_OK;
    }
    static constexpr size_t kChunk = size_t(1) << 18;
    int update_host(const double *xyz, size_t n, bool has_pose, const SE3 &pose, bool do_add, bool do_remove,
                    const V3 &origin) {
        CK(cudaSetDevice(ex->device));
        if (do_add) {
            for (size_t off = 0; off < n; off += kChunk) {
                const size_t c = std::min(kChunk, n - off);
                RET(ws.in.ensure(3 * c));
                RET(ws.tp.ensure(3 * c));
                RET(ws.next.ensure(c));
                RET(ws.touched.ensure(c));
                CK(cudaMemcpyAsync(ws.in.p, xyz + 3 * off, c * 24, cudaMemcpyHostToDevice, ex->stream));
                RET(update_dev(ws.in.p, c, has_pose, pose, true, false, origin));
                RET(pull_counters());
            }
        }
        if (do_remove) {
            RET(update_dev(nullptr, 0, false, pose, false, true, origin));
            RET(pull_counters());
        }
        return KB_OK;
    }
};

struct kb_registration {
    int max_iter;
    double conv;
    int threads;
    Work ws;
    DBuf<double> out;  // pose[16] + sys[NACC]
    DBuf<int> iout;    // iters, ncorr
    int last_iters = 0;
};

struct kb_preprocessor {
    std::shared_ptr<Exec> ex;
    double max_range, min_range;
    int deskew, threads;
    Work ws;
};

struct kb_threshold {
    double min_motion_th, max_range, model_sse;
    int num_samples;
};

struct kb_pipeline {
    std::shared_ptr<Exec> ex;
    kb_config cfg;
    kb_map *map = nullptr;
    Work ws;
    PipeState *d_state = nullptr;
    FrameResult *d_res = nullptr;
    FrameResult *h_res = nullptr;  // pinned
    FrameResult last{};
    bool has_last = false;
    long long next_id = 0;  // id of the next frame to register (Workspace::fr[id & 1] holds its front end)
    long long last_id = 0;  // id of the frame `last` describes
    Work vox_ws;            // scratch of kb_pipeline_voxelize (must not clobber the clouds of the last frame)
    unsigned long long grow_retries = 0;
    std::vector<kb_frame_stats> history;
    std::vector<std::array<double, 20>> history_stamps;  // the frames' %globaltimer stamps, ns modulo 2^40 (profiling on)
    size_t history_cap = 0;
    // frame queue of kb_pipeline_register_frames: frame k+1 is copied in while frame k is registered
    static constexpr int Q_DEPTH = 4;  // frame k registering, k+1 being prefetched by the same launch, k+2 / k+3 copying
    struct Slot {
        DBuf<double> in, ts;  // device copy of one queued frame
        void *pin_xyz = nullptr, *pin_ts = nullptr;  // pinned staging, used only when the caller's memory is pageable
        size_t pin_xyz_bytes = 0, pin_ts_bytes = 0;
        cudaEvent_t copied = nullptr, done = nullptr, read = nullptr;
    };
    Slot q[Q_DEPTH];
    cudaStream_t copy_stream = nullptr, res_stream = nullptr;
    FrameResult *q_res = nullptr;      // [Q_DEPTH] pinned host copies of the frame results
    FrameResult *q_res_dev = nullptr;  // [Q_DEPTH] device side: where the kernels write them
    ~kb_pipeline() {
        if (ex && device_is_stuck(ex->device)) {
            map = nullptr;  // (leaked on purpose)
            return;
        }
        if (ex) cudaSetDevice(ex->device);
        for (Slot &s : q) {
            if (s.pin_xyz) cudaFreeHost(s.pin_xyz);
            if (s.pin_ts) cudaFreeHost(s.pin_ts);
            if (s.copied) cudaEventDestroy(s.copied);
            if (s.done) cudaEventDestroy(s.done);
            if (s.read) cudaEventDestroy(s.read);
        }
        if (copy_stream) cudaStreamDestroy(copy_stream);
        if (res_stream) cudaStreamDestroy(res_stream);
        if (q_res_dev) cudaFree(q_res_dev);
        if (q_res) cudaFreeHost(q_res);
        delete map;
        if (d_state) cudaFree(d_state);
        if (d_res) cudaFree(d_res);
        if (h_res) cudaFreeHost(h_res);
    }
};

namespace {
struct DefaultCtx {
    std::shared_ptr<Exec> ex;
    Work ws;
};
thread_local std::unique_ptr<DefaultCtx> tl_ctx;
int default_ctx(DefaultCtx **out) {
    if (!tl_ctx || tl_ctx->ex->device != tl_device || (tl_user_stream && tl_ctx->ex->stream != tl_user_stream)) {
        auto c = std::make_unique<DefaultCtx>();
        RET(make_exec(&c->ex));
        tl_ctx = std::move(c);
    }
    *out = tl_ctx.get();
    return KB_OK;
}

int run_downsample(Exec &ex, Work &ws, const double *d_in, size_t n, double v1, double *d_out, int *d_n1, double v2,
                   double *d_out2, int *d_n2) {
    DsParams P;
    P.sc = ex.sc;
    P.in = d_in;
    P.n = static_cast<int>(n);
    P.voxel_size = v1;
    P.ds = ws.ds_view();
    P.out = d_out;
    P.out_n = d_n1;
    P.voxel_size2 = v2;
    P.out2 = d_out2;
    P.out_n2 = d_n2;
    return ex.coop(k_downsample, P);
}
}  // namespace

extern "C" {

const char *kb_last_error(void) { return tl_err.c_str(); }
const char *kb_version(void) { return "kiss_icp_b200 0.1 (sm_100a)"; }
int kb_device_count(void) { return device_count(); }
int kb_set_device(int device) {
    if (device < 0 || device >= device_count()) return fail(KB_ERR_INVALID_ARG, "device %d out of range", device);
    tl_device = device;
    return KB_OK;
}
int kb_set_stream(void *cuda_stream) {
    tl_user_stream = static_cast<cudaStream_t>(cuda_stream);
    return KB_OK;
}
int kb_set_grid_blocks(int blocks) {
    if (blocks < 0) return fail(KB_ERR_INVALID_ARG, "blocks < 0");
    tl_grid_blocks = blocks;
    return KB_OK;
}

// ------------------------------------------------------------------------------- VoxelHashMap
static int map_create_impl(double voxel_size, double max_distance, unsigned cap, std::shared_ptr<Exec> ex, kb_map **out) {
    if (!out) return fail(KB_ERR_INVALID_ARG, "out == NULL");
    if (!(voxel_size > 0.0)) return fail(KB_ERR_INVALID_ARG, "voxel_size must be > 0");
    if (cap < 1 || cap > 1023) return fail(KB_ERR_INVALID_ARG, "max_points_per_voxel must be in [1, 1023]");
    auto m = std::make_unique<kb_map>();
    if (ex)
        m->ex = ex;
    else
        RET(make_exec(&m->ex));
    m->voxel_size = voxel_size;
    m->max_distance = max_distance;
    m->cap = cap;
    RET(m->ensure_capacity(0));
    RET(m->ex->sync());
    *out = m.release();
    return KB_OK;
}
int kb_map_create(double voxel_size, double max_distance, unsigned max_points_per_voxel, kb_map **out) {
    return map_create_impl(voxel_size, max_distance, max_points_per_voxel, nullptr, out);
}
int kb_map_destroy(kb_map *map) {
    if (map && !map->borrowed) delete map;
    return KB_OK;
}
int kb_map_clear(kb_map *map) {
    if (!map) return fail(KB_ERR_INVALID_ARG, "map == NULL");
    CK(cudaSetDevice(map->ex->device));
    k_map_fill<<<std::min<size_t>(4096, (map->capacity + 255) / 256), 256, 0, map->ex->stream>>>(map->slots, map->head,
                                                                                             map->pcount, map->capacity);
    ++map->ex->launches;
    CK(cudaMemsetAsync(map->counters, 0, sizeof(int) * C_NCOUNTERS, map->ex->stream));
    std::memset(map->h_counters, 0, sizeof(map->h_counters));
    return map->ex->sync();
}
int kb_map_empty(const kb_map *map, int *out_is_empty) {
    if (!map || !out_is_empty) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    *out_is_empty = map->h_counters[C_LIVE] == 0 ? 1 : 0;
    return KB_OK;
}
int kb_map_update_origin(kb_map *map, const double *xyz, size_t n, const double origin[3]) {
    if (!map || (!xyz && n) || !origin) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    return map->update_host(xyz, n, false, se3_identity(), true, true, V3{origin[0], origin[1], origin[2]});
}
int kb_map_update_pose(kb_map *map, const double *xyz, size_t n, const double pose[16]) {
    if (!map || (!xyz && n) || !pose) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    SE3 T;
    if (!to_se3(pose, &T)) return fail(KB_ERR_NOT_SE3, "pose is not in SE(3)");
    return map->update_host(xyz, n, true, T, true, true, T.t);
}
int kb_map_add_points(kb_map *map, const double *xyz, size_t n) {
    if (!map || (!xyz && n)) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    return map->update_host(xyz, n, false, se3_identity(), true, false, V3{0, 0, 0});
}
int kb_map_remove_far(kb_map *map, const double origin[3]) {
    if (!map || !origin) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    return map->update_host(nullptr, 0, false, se3_identity(), false, true, V3{origin[0], origin[1], origin[2]});
}
int kb_map_compact(kb_map *map) {
    if (!map) return fail(KB_ERR_INVALID_ARG, "map == NULL");
    const size_t live = static_cast<size_t>(map->h_counters[C_LIVE]);
    const size_t want = std::max<size_t>(pow2_at_least(2 * live + 2), size_t(1) << 14);
    if (want >= map->capacity && map->h_counters[C_TOMB] == 0) return KB_OK;
    RET(map->ensure_capacity(0, want));
    return map->ex->sync();
}
int kb_map_num_points(const kb_map *map, size_t *out) {
    if (!map || !out) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    *out = static_cast<size_t>(map->h_counters[C_POINTS]);
    return KB_OK;
}
int kb_map_num_voxels(const kb_map *map, size_t *out) {
    if (!map || !out) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    *out = static_cast<size_t>(map->h_counters[C_LIVE]);
    return KB_OK;
}
int kb_map_params(const kb_map *map, double *voxel_size, double *max_distance, unsigned *max_points_per_voxel) {
    if (!map) return fail(KB_ERR_INVALID_ARG, "map == NULL");
    if (voxel_size) *voxel_size = map->voxel_size;
    if (max_distance) *max_distance = map->max_distance;
    if (max_points_per_voxel) *max_points_per_voxel = map->cap;
    return KB_OK;
}

int kb_map_dump(const kb_map *cmap, int *voxels, int *counts, double *points, size_t voxel_capacity,
                size_t point_capacity, size_t *n_voxels, size_t *n_points) {
    kb_map *map = const_cast<kb_map *>(cmap);
    if (!map || !n_voxels || !n_points) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    CK(cudaSetDevice(map->ex->device));
    const size_t nv = static_cast<size_t>(map->h_counters[C_LIVE]), np = static_cast<size_t>(map->h_counters[C_POINTS]);
    *n_voxels = nv;
    *n_points = np;
    if (!voxels && !counts && !points) return KB_OK;
    if (voxel_capacity < nv || point_capacity < np) return fail(KB_ERR_CAPACITY, "dump buffers too small");
    if (nv == 0) return KB_OK;
    DBuf<int4> d_vox;
    DBuf<double> d_pts;
    DBuf<int> d_tot;
    RET(d_vox.ensure(nv));
    RET(d_pts.ensure(3 * np));
    RET(d_tot.ensure(2));
    ExportParams P;
    P.m = map->view();
    P.sc = map->ex->sc;
    P.vox_out = d_vox.p;
    P.pts_out = d_pts.p;
    P.totals = d_tot.p;
    RET(map->ex->coop(k_map_export, P));
    std::vector<int4> hv(nv);
    std::vector<double> hp(3 * np);
    int tot[2];
    CK(cudaMemcpyAsync(hv.data(), d_vox.p, nv * sizeof(int4), cudaMemcpyDeviceToHost, map->ex->stream));
    CK(cudaMemcpyAsync(hp.data(), d_pts.p, 3 * np * sizeof(double), cudaMemcpyDeviceToHost, map->ex->stream));
    CK(cudaMemcpyAsync(tot, d_tot.p, sizeof(tot), cudaMemcpyDeviceToHost, map->ex->stream));
    RET(map->ex->sync());
    if (static_cast<size_t>(tot[0]) != nv || static_cast<size_t>(tot[1]) != np)
        return fail(KB_ERR_CUDA, "map export count mismatch (%d/%zu voxels, %d/%zu points)", tot[0], nv, tot[1], np);
    // canonical voxel order: ascending (x, y, z)
    std::vector<size_t> start(nv);
    size_t acc = 0;
    for (size_t i = 0; i < nv; ++i) {
        start[i] = acc;
        acc += static_cast<size_t>(hv[i].w);
    }
    std::vector<size_t> order(nv);
    std::iota(order.begin(), order.end(), size_t(0));
    std::sort(order.begin(), order.end(), [&](size_t a, size_t b) {
        if (hv[a].x != hv[b].x) return hv[a].x < hv[b].x;
        if (hv[a].y != hv[b].y) return hv[a].y < hv[b].y;
        return hv[a].z < hv[b].z;
    });
    size_t o = 0;
    for (size_t r = 0; r < nv; ++r) {
        const size_t i = order[r];
        if (voxels) {
            voxels[3 * r] = hv[i].x;
            voxels[3 * r + 1] = hv[i].y;
            voxels[3 * r + 2] = hv[i].z;
        }
        if (counts) counts[r] = hv[i].w;
        if (points) std::memcpy(points + 3 * o, hp.data() + 3 * start[i], sizeof(double) * 3 * hv[i].w);
        o += static_cast<size_t>(hv[i].w);
    }
    return KB_OK;
}
int kb_map_pointcloud(const kb_map *map, double *out_xyz, size_t capacity, size_t *n_out) {
    if (!map || !n_out) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    const size_t np = static_cast<size_t>(map->h_counters[C_POINTS]);
    *n_out = np;
    if (!out_xyz || capacity == 0) return KB_OK;
    if (capacity < np) return fail(KB_ERR_CAPACITY, "pointcloud buffer too small");
    size_t nv, npp;
    return kb_map_dump(map, nullptr, nullptr, out_xyz, static_cast<size_t>(map->h_counters[C_LIVE]), capacity, &nv, &npp);
}

static int nn_launch(kb_map *map, const double *d_q, size_t n, double *d_p, double *d_d, unsigned long long *d_cand) {
    if (n == 0) return KB_OK;
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, map->ex->device);
    const int threads = 256;
    const size_t want = (n * 32 + threads - 1) / threads;
    const unsigned blocks = static_cast<unsigned>(std::min<size_t>(want, static_cast<size_t>(sms) * 4));  // 4 CTAs/SM, grid-stride
    if (d_cand)
        k_nn_query<true><<<blocks, threads, 0, map->ex->stream>>>(map->view(), d_q, n, d_p, d_d, d_cand);
    else
        k_nn_query<false><<<blocks, threads, 0, map->ex->stream>>>(map->view(), d_q, n, d_p, d_d, nullptr);
    ++map->ex->launches;
    CK(cudaGetLastError());
    return KB_OK;
}
int kb_map_closest_neighbors_dev(const kb_map *cmap, const double *d_queries, size_t n, double *d_out_points,
                                 double *d_out_dist) {
    kb_map *map = const_cast<kb_map *>(cmap);
    if (!map || (n && (!d_queries || !d_out_points || !d_out_dist))) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    CK(cudaSetDevice(map->ex->device));
    return nn_launch(map, d_queries, n, d_out_points, d_out_dist, nullptr);  // asynchronous on the map's stream
}
int kb_map_closest_neighbors(const kb_map *cmap, const double *queries, size_t n, double *out_points, double *out_dist) {
    kb_map *map = const_cast<kb_map *>(cmap);
    if (!map || (n && (!queries || !out_points || !out_dist))) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    CK(cudaSetDevice(map->ex->device));
    const size_t chunk = size_t(1) << 22;
    for (size_t off = 0; off < n; off += chunk) {
        const size_t c = std::min(chunk, n - off);
        RET(map->q_in.ensure(3 * c));
        RET(map->q_outp.ensure(3 * c));
        RET(map->q_outd.ensure(c));
        CK(cudaMemcpyAsync(map->q_in.p, queries + 3 * off, c * 24, cudaMemcpyHostToDevice, map->ex->stream));
        RET(nn_launch(map, map->q_in.p, c, map->q_outp.p, map->q_outd.p, nullptr));
        CK(cudaMemcpyAsync(out_points + 3 * off, map->q_outp.p, c * 24, cudaMemcpyDeviceToHost, map->ex->stream));
        CK(cudaMemcpyAsync(out_dist + off, map->q_outd.p, c * 8, cudaMemcpyDeviceToHost, map->ex->stream));
        RET(map->ex->sync());
    }
    return KB_OK;
}
int kb_map_query_bytes_dev(const kb_map *cmap, const double *d_queries, size_t n, double *bytes) {
    kb_map *map = const_cast<kb_map *>(cmap);
    if (!map || !bytes || (n && !d_queries)) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    CK(cudaSetDevice(map->ex->device));
    RET(map->q_outp.ensure(3 * n));
    RET(map->q_outd.ensure(n));
    RET(map->q_cand.ensure(1));
    CK(cudaMemsetAsync(map->q_cand.p, 0, sizeof(unsigned long long), map->ex->stream));
    RET(nn_launch(map, d_queries, n, map->q_outp.p, map->q_outd.p, map->q_cand.p));
    unsigned long long cand = 0;
    CK(cudaMemcpyAsync(&cand, map->q_cand.p, sizeof(cand), cudaMemcpyDeviceToHost, map->ex->stream));
    RET(map->ex->sync());
    // SURVEY.md 8(d): 24 (query) + 27*16 (slot probes) + 24*candidates + 32 (result) per query
    *bytes = static_cast<double>(n) * (24.0 + 27.0 * 16.0 + 32.0) + 24.0 * static_cast<double>(cand);
    return KB_OK;
}
int kb_map_sync(const kb_map *map) {
    if (!map) return fail(KB_ERR_INVALID_ARG, "map == NULL");
    return map->ex->sync();
}

// ------------------------------------------------------------------------------- Registration
int kb_registration_create(int max_num_iterations, double convergence_criterion, int max_num_threads,
                           kb_registration **out) {
    if (!out) return fail(KB_ERR_INVALID_ARG, "out == NULL");
    if (device_count() <= 0) return fail(KB_ERR_NO_DEVICE, "no CUDA device visible (this library has no CPU fallback)");
    if (max_num_iterations > 8000) return fail(KB_ERR_INVALID_ARG, "max_num_iterations > 8000 is not supported");
    auto r = new kb_registration();
    r->max_iter = max_num_iterations;
    r->conv = convergence_criterion;
    r->threads = max_num_threads;
    *out = r;
    return KB_OK;
}
int kb_registration_destroy(kb_registration *reg) {
    delete reg;
    return KB_OK;
}
static int registration_run(kb_registration *reg, const double *xyz, size_t n, kb_map *map, const SE3 &guess,
                            double max_dist, double kscale, bool system_only) {
    Exec &ex = *map->ex;
    CK(cudaSetDevice(ex.device));
    RET(reg->ws.src.ensure(3 * std::max<size_t>(n, 1)));
    RET(reg->ws.work.ensure(3 * std::max<size_t>(n, 1)));
    RET(reg->out.ensure(16 + NACC));
    RET(reg->iout.ensure(2));
    RET(reg->ws.qrec.ensure(std::max<size_t>(n, 1)));
    if (n) CK(cudaMemcpyAsync(reg->ws.src.p, xyz, n * 24, cudaMemcpyHostToDevice, ex.stream));
    IcpParams P;
    P.m = map->view();
    P.sc = ex.sc;
    P.src = reg->ws.src.p;
    P.work = reg->ws.work.p;
    P.n = static_cast<int>(n);
    P.guess = guess;
    P.max_dist = max_dist;
    P.kscale = kscale;
    P.max_iter = reg->max_iter;
    P.conv = reg->conv;
    P.out_pose = reg->out.p;
    P.out_iters = reg->iout.p;
    P.system_only = system_only ? 1 : 0;
    P.out_sys = reg->out.p + 16;
    P.out_ncorr = reg->iout.p + 1;
    P.tag_base = ex.next_tag_base();
    P.team = ex.team;
    P.team.qrec = reg->ws.qrec.p;
    P.icp_team_q = ex.icp_team_q;
    return ex.coop(k_icp, P, system_only ? 0 : std::max<size_t>(QC_BYTES, ex.icp_smem));
}
int kb_registration_align_points_to_map(kb_registration *reg, const double *xyz, size_t n, const kb_map *cmap,
                                        const double initial_guess[16], double max_correspondence_distance,
                                        double kernel_scale, double out_pose[16]) {
    kb_map *map = const_cast<kb_map *>(cmap);
    if (!reg || !map || (!xyz && n) || !initial_guess || !out_pose) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    SE3 g;
    if (!to_se3(initial_guess, &g)) return fail(KB_ERR_NOT_SE3, "initial_guess is not in SE(3)");
    RET(registration_run(reg, xyz, n, map, g, max_correspondence_distance, kernel_scale, false));
    int it = 0;
    CK(cudaMemcpyAsync(out_pose, reg->out.p, 16 * sizeof(double), cudaMemcpyDeviceToHost, map->ex->stream));
    CK(cudaMemcpyAsync(&it, reg->iout.p, sizeof(int), cudaMemcpyDeviceToHost, map->ex->stream));
    RET(map->ex->sync());
    reg->last_iters = it;
    return KB_OK;
}
int kb_registration_last_iterations(const kb_registration *reg, int *out) {
    if (!reg || !out) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    *out = reg->last_iters;
    return KB_OK;
}
int kb_registration_build_system(kb_registration *reg, const double *xyz, size_t n, const kb_map *cmap,
                                 double max_correspondence_distance, double kernel_scale, double JTJ[36], double JTr[6],
                                 int *n_correspondences) {
    kb_map *map = const_cast<kb_map *>(cmap);
    if (!reg || !map || (!xyz && n) || !JTJ || !JTr) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    RET(registration_run(reg, xyz, n, map, se3_identity(), max_correspondence_distance, kernel_scale, true));
    double sys[NACC];
    int nc = 0;
    CK(cudaMemcpyAsync(sys, reg->out.p + 16, sizeof(sys), cudaMemcpyDeviceToHost, map->ex->stream));
    CK(cudaMemcpyAsync(&nc, reg->iout.p + 1, sizeof(int), cudaMemcpyDeviceToHost, map->ex->stream));
    RET(map->ex->sync());
    // same expansion as the device (icp_expand), host side
    for (int i = 0; i < 36; ++i) JTJ[i] = 0.0;
    JTJ[0] = JTJ[7] = JTJ[14] = sys[0];
    JTJ[6 * 3 + 1] = -sys[3];
    JTJ[6 * 3 + 2] = sys[2];
    JTJ[6 * 4 + 0] = sys[3];
    JTJ[6 * 4 + 2] = -sys[1];
    JTJ[6 * 5 + 0] = -sys[2];
    JTJ[6 * 5 + 1] = sys[1];
    JTJ[6 * 3 + 3] = sys[4];
    JTJ[6 * 4 + 3] = sys[5];
    JTJ[6 * 4 + 4] = sys[6];
    JTJ[6 * 5 + 3] = sys[7];
    JTJ[6 * 5 + 4] = sys[8];
    JTJ[6 * 5 + 5] = sys[9];
    for (int i = 0; i < 6; ++i)
        for (int j = i + 1; j < 6; ++j) JTJ[6 * i + j] = JTJ[6 * j + i];
    for (int i = 0; i < 6; ++i) JTr[i] = sys[10 + i];
    if (n_correspondences) *n_correspondences = nc;
    return KB_OK;
}

// ------------------------------------------------------------------------------- Preprocessor
int kb_preprocessor_create(double max_range, double min_range, int deskew, int max_num_threads, kb_preprocessor **out) {
    if (!out) return fail(KB_ERR_INVALID_ARG, "out == NULL");
    auto p = std::make_unique<kb_preprocessor>();
    RET(make_exec(&p->ex));
    p->max_range = max_range;
    p->min_range = min_range;
    p->deskew = deskew;
    p->threads = max_num_threads;
    *out = p.release();
    return KB_OK;
}
int kb_preprocessor_destroy(kb_preprocessor *pre) {
    delete pre;
    return KB_OK;
}
int kb_preprocessor_preprocess(kb_preprocessor *pre, const double *xyz, size_t n, const double *timestamps,
                               size_t n_timestamps, const double relative_motion[16], double *out_xyz, size_t capacity,
                               size_t *n_out) {
    if (!pre || (!xyz && n) || (!timestamps && n_timestamps) || !relative_motion || !n_out)
        return fail(KB_ERR_INVALID_ARG, "NULL argument");
    SE3 T;
    if (!to_se3(relative_motion, &T)) return fail(KB_ERR_NOT_SE3, "relative_motion is not in SE(3)");
    const bool do_deskew = pre->deskew && n_timestamps > 0;
    if (do_deskew && n_timestamps < n)
        return fail(KB_ERR_OUT_OF_RANGE, "timestamps (%zu) shorter than frame (%zu): the reference throws std::out_of_range",
                    n_timestamps, n);
    Exec &ex = *pre->ex;
    CK(cudaSetDevice(ex.device));
    RET(pre->ws.ensure(std::max(n, n_timestamps)));
    if (n) CK(cudaMemcpyAsync(pre->ws.in.p, xyz, n * 24, cudaMemcpyHostToDevice, ex.stream));
    if (do_deskew) CK(cudaMemcpyAsync(pre->ws.ts.p, timestamps, n_timestamps * 8, cudaMemcpyHostToDevice, ex.stream));
    PreParams P;
    P.sc = ex.sc;
    P.in = pre->ws.in.p;
    P.ts = pre->ws.ts.p;
    P.n = static_cast<int>(n);
    P.n_ts = do_deskew ? static_cast<int>(n_timestamps) : 0;
    P.deskew = pre->deskew;
    P.motion = T;
    P.max_range = pre->max_range;
    P.min_range = pre->min_range;
    P.tmp = pre->ws.tmp.p;
    P.out = pre->ws.pre.p;
    P.out_n = pre->ws.cnt.p;
    RET(ex.coop(k_preprocess, P));
    int kept = 0;
    CK(cudaMemcpyAsync(&kept, pre->ws.cnt.p, sizeof(int), cudaMemcpyDeviceToHost, ex.stream));
    RET(ex.sync());
    *n_out = static_cast<size_t>(kept);
    if (!out_xyz) return KB_OK;
    if (capacity < static_cast<size_t>(kept)) return fail(KB_ERR_CAPACITY, "output buffer too small");
    if (kept) CK(cudaMemcpyAsync(out_xyz, pre->ws.pre.p, static_cast<size_t>(kept) * 24, cudaMemcpyDeviceToHost, ex.stream));
    return ex.sync();
}

// ------------------------------------------------------------------------------- AdaptiveThreshold
int kb_threshold_create(double initial_threshold, double min_motion_threshold, double max_range, kb_threshold **out) {
    if (!out) return fail(KB_ERR_INVALID_ARG, "out == NULL");
    auto t = new kb_threshold();
    t->min_motion_th = min_motion_threshold;
    t->max_range = max_range;
    t->model_sse = initial_threshold * initial_threshold;  // Threshold.cpp:35
    t->num_samples = 1;
    *out = t;
    return KB_OK;
}
int kb_threshold_destroy(kb_threshold *th) {
    delete th;
    return KB_OK;
}
int kb_threshold_compute(const kb_threshold *th, double *out_sigma) {
    if (!th || !out_sigma) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    *out_sigma = std::sqrt(th->model_sse / th->num_samples);  // Threshold.hpp:38
    return KB_OK;
}
int kb_threshold_update_model_deviation(kb_threshold *th, const double model_deviation[16]) {
    if (!th || !model_deviation) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    SE3 T;
    if (!to_se3(model_deviation, &T)) return fail(KB_ERR_NOT_SE3, "model_deviation is not in SE(3)");
    // scalar bookkeeping (Threshold.cpp:38-49); inside RegisterFrame the same update runs on the device
    const double theta = angle_axis_angle(q_to_matrix(T.q));
    const double delta_rot = 2.0 * th->max_range * std::sin(theta / 2.0);
    const double delta_trans = norm(T.t);
    const double model_error = delta_trans + delta_rot;
    if (model_error > th->min_motion_th) {
        th->model_sse += model_error * model_error;
        th->num_samples++;
    }
    return KB_OK;
}

// ------------------------------------------------------------------------------- VoxelDownsample
int kb_voxel_down_sample(const double *xyz, size_t n, double voxel_size, double *out_xyz, size_t capacity, size_t *n_out) {
    if ((!xyz && n) || !n_out) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    if (n >= (size_t(1) << 30)) return fail(KB_ERR_INVALID_ARG, "frame too large");
    DefaultCtx *c;
    RET(default_ctx(&c));
    Exec &ex = *c->ex;
    CK(cudaSetDevice(ex.device));
    RET(c->ws.ensure(n));
    if (n) CK(cudaMemcpyAsync(c->ws.in.p, xyz, n * 24, cudaMemcpyHostToDevice, ex.stream));
    RET(run_downsample(ex, c->ws, c->ws.in.p, n, voxel_size, c->ws.ds1.p, c->ws.cnt.p, 0.0, nullptr, nullptr));
    int m = 0;
    CK(cudaMemcpyAsync(&m, c->ws.cnt.p, sizeof(int), cudaMemcpyDeviceToHost, ex.stream));
    RET(ex.sync());
    *n_out = static_cast<size_t>(m);
    if (!out_xyz) return KB_OK;
    if (capacity < static_cast<size_t>(m)) return fail(KB_ERR_CAPACITY, "output buffer too small");
    if (m) CK(cudaMemcpyAsync(out_xyz, c->ws.ds1.p, static_cast<size_t>(m) * 24, cudaMemcpyDeviceToHost, ex.stream));
    return ex.sync();
}

static int correct_kitti_launch(Exec &ex, const double *d_in, double *d_out, size_t n) {
    if (!n) return KB_OK;
    const double angle = (0.205 * M_PI) / 180.0;  // VERTICAL_ANGLE_OFFSET, kiss_icp_pybind.cpp:130
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ex.device);
    const unsigned blocks = static_cast<unsigned>(std::min<size_t>((n + 255) / 256, static_cast<size_t>(sms) * 8));
    k_correct_kitti<<<blocks, 256, 0, ex.stream>>>(d_in, d_out, n, std::sin(angle), std::cos(angle));
    ++ex.launches;
    CK(cudaGetLastError());
    return KB_OK;
}
int kb_correct_kitti_scan(const double *xyz, size_t n, double *out_xyz) {
    if (n && (!xyz || !out_xyz)) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    if (n >= (size_t(1) << 30)) return fail(KB_ERR_INVALID_ARG, "frame too large");
    DefaultCtx *c;
    RET(default_ctx(&c));
    Exec &ex = *c->ex;
    CK(cudaSetDevice(ex.device));
    RET(c->ws.in.ensure(3 * std::max<size_t>(n, 1)));
    RET(c->ws.tmp.ensure(3 * std::max<size_t>(n, 1)));
    if (n) CK(cudaMemcpyAsync(c->ws.in.p, xyz, n * 24, cudaMemcpyHostToDevice, ex.stream));
    RET(correct_kitti_launch(ex, c->ws.in.p, c->ws.tmp.p, n));
    if (n) CK(cudaMemcpyAsync(out_xyz, c->ws.tmp.p, n * 24, cudaMemcpyDeviceToHost, ex.stream));
    return ex.sync();
}
int kb_correct_kitti_scan_dev(const double *d_xyz, size_t n, double *d_out_xyz) {
    if (n && (!d_xyz || !d_out_xyz)) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    DefaultCtx *c;
    RET(default_ctx(&c));
    CK(cudaSetDevice(c->ex->device));
    return correct_kitti_launch(*c->ex, d_xyz, d_out_xyz, n);  // asynchronous on the calling thread's stream
}

// ------------------------------------------------------------------------------- KissICP pipeline
void kb_config_default(kb_config *cfg) {
    if (!cfg) return;
    cfg->voxel_size = 1.0;
    cfg->max_range = 100.0;
    cfg->min_range = 0.0;
    cfg->max_points_per_voxel = 20;
    cfg->min_motion_th = 0.1;
    cfg->initial_threshold = 2.0;
    cfg->max_num_iterations = 500;
    cfg->convergence_criterion = 0.0001;
    cfg->max_num_threads = 0;
    cfg->deskew = 1;
}

static int pipeline_push_state(kb_pipeline *p, const SE3 &pose, const SE3 &delta, double sse, int ns) {
    PipeState s;
    s.last_pose = pose;
    s.last_delta = delta;
    s.model_sse = sse;
    s.num_samples = ns;
    s.vetoed = 0;
    s.front_id = -1;
    CK(cudaMemcpyAsync(p->d_state, &s, sizeof(s), cudaMemcpyHostToDevice, p->ex->stream));
    return p->ex->sync();
}

int kb_pipeline_create(const kb_config *cfg, kb_pipeline **out) {
    if (!cfg || !out) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    if (cfg->max_num_iterations > 8000) return fail(KB_ERR_INVALID_ARG, "max_num_iterations > 8000 is not supported");
    auto p = std::make_unique<kb_pipeline>();
    RET(make_exec(&p->ex));
    p->cfg = *cfg;
    RET(map_create_impl(cfg->voxel_size, cfg->max_range, static_cast<unsigned>(cfg->max_points_per_voxel), p->ex, &p->map));
    p->map->borrowed = true;
    {
        // size the local map for the sensor: occupied voxels within max_range are surface-like, ~10 pi r^2 for
        // r = max_range / voxel_size (KITTI: ~300k at 100 m / 1 m), at load factor 1/3; capped at 2^20 slots
        // (0.66 GB per table at 20 points per voxel) - beyond that the table grows on demand
        const double r = cfg->max_range / cfg->voxel_size;
        const double est = std::min(3.0 * 10.0 * 3.14159265358979 * r * r, double(size_t(1) << 20));
        size_t slots = std::max<size_t>(static_cast<size_t>(est), size_t(1) << 14);
        if (const char *e = std::getenv("KB_MAP_RESERVE_SLOTS")) slots = static_cast<size_t>(std::atoll(e));  // 0: none
        if (slots) {
            // out of device memory (many pipelines on one GPU): reserve less; the minimal table of map_create_impl grows on demand
            size_t want = std::min<size_t>(slots, size_t(1) << 31);
            int st;
            while ((st = p->map->reserve(want)) != KB_OK && want > (size_t(1) << 14)) {
                cudaGetLastError();
                want >>= 2;
            }
            if (st != KB_OK) cudaGetLastError();
        }
    }
    CK(cudaMalloc(&p->d_state, sizeof(PipeState)));
    CK(cudaMalloc(&p->d_res, sizeof(FrameResult)));
    CK(cudaMemsetAsync(p->d_res, 0, sizeof(FrameResult), p->ex->stream));  // (fields a launch does not write are read back too)
    CK(cudaHostAlloc(&p->h_res, sizeof(FrameResult), cudaHostAllocDefault));
    std::memset(&p->last, 0, sizeof(p->last));
    se3_to_matrix(se3_identity(), p->last.pose);
    se3_to_matrix(se3_identity(), p->last.delta);
    p->last.model_sse = cfg->initial_threshold * cfg->initial_threshold;
    p->last.num_samples = 1;
    RET(pipeline_push_state(p.get(), se3_identity(), se3_identity(), p->last.model_sse, 1));
    *out = p.release();
    return KB_OK;
}
int kb_pipeline_destroy(kb_pipeline *p) {
    if (p) {
        p->map->borrowed = false;
        kb_map *m = p->map;
        p->map = nullptr;
        cudaSetDevice(p->ex->device);
        delete m;
        delete p;
    }
    return KB_OK;
}

// expected new voxels: at most one per downsampled point; the 0.5-voxel downsample keeps ~1/9 of a scan, so
// size for max(n/4, 2x the last frame's count) and let the kernel veto the frame if that was too optimistic
static size_t pipeline_extra(const kb_pipeline *p, size_t n) {
    const size_t extra = std::max<size_t>(n / 4, 2 * static_cast<size_t>(p->has_last ? p->last.n_ds : 0) + 1024);
    return std::min(extra, n);
}

// enqueue one RegisterFrame on the pipeline's stream; the result goes to `res` (device-visible memory)
// `next_xyz` (may be null): the frame after this one, already on the device, no timestamps -> its front end is prefetched
static int pipeline_launch(kb_pipeline *p, long long id, const double *d_xyz, size_t n, const double *d_ts, size_t n_ts,
                           bool in_f32, FrameResult *res, const double *next_xyz = nullptr, size_t next_n = 0) {
    Exec &ex = *p->ex;
    FrameParams P;
    P.m = p->map->view();
    P.sc = ex.sc;
    P.team = ex.team;
    P.team.qrec = p->ws.qrec.p;
    P.icp_team_q = ex.icp_team_q;
    P.id = id;
    P.next_in = next_xyz;
    P.next_n = static_cast<int>(next_n);
    P.next_in_f32 = in_f32 ? 1 : 0;
    P.ws = p->ws.view();
    P.st = p->d_state;
    P.res = res;
    P.in = d_xyz;
    P.ts = d_ts;
    P.n = static_cast<int>(n);
    P.n_ts = static_cast<int>(n_ts);
    P.deskew = p->cfg.deskew;
    P.max_range = p->cfg.max_range;
    P.min_range = p->cfg.min_range;
    P.voxel_size = p->cfg.voxel_size;
    P.max_iter = p->cfg.max_num_iterations;
    P.conv = p->cfg.convergence_criterion;
    P.min_motion_th = p->cfg.min_motion_th;
    P.tag_base = ex.next_tag_base();
    P.in_f32 = in_f32 ? 1 : 0;
    return ex.coop(k_register_frame, P, std::max<size_t>(QC_BYTES, ex.icp_smem), true);
}

// take over the result of a frame that ran (not vetoed): host mirror of the counters, history
static int pipeline_absorb(kb_pipeline *p, const FrameResult &r, size_t n, long long id) {
    p->last = r;
    p->last_id = id;
    p->has_last = true;
    p->map->h_counters[C_LIVE] = p->last.map_live;
    p->map->h_counters[C_TOMB] = p->last.map_tomb;
    p->map->h_counters[C_POINTS] = p->last.map_points;
    p->map->h_counters[C_STATUS] = p->last.map_status;
    if (p->history.size() < p->history_cap) {
        kb_frame_stats st;
        std::memcpy(st.pose, p->last.pose, sizeof(st.pose));
        for (int i = 0; i < 6; ++i)
            st.phase_us[i] = (static_cast<double>(p->last.t_ns[i + 1]) - static_cast<double>(p->last.t_ns[i])) * 1e-3;
        st.icp_queries = p->last.icp_queries;
        st.icp_candidates = p->last.icp_candidates;
        st.iterations = p->last.iterations;
        st.n_points_in = static_cast<int>(n);
        st.n_preprocessed = p->last.n_pre;
        st.n_downsampled = p->last.n_ds;
        st.n_source = p->last.n_src;
        st.map_points = p->last.map_points;
        st.map_voxels = p->last.map_live;
        st.team = p->last.team;
        p->history.push_back(st);
        std::array<double, 20> ts;
        for (int i = 0; i < 20; ++i) ts[i] = static_cast<double>(p->last.t_ns[i] & ((1ull << 40) - 1));
        p->history_stamps.push_back(ts);
    }
    if (p->last.map_status & ST_TABLE_FULL) return fail(KB_ERR_CUDA, "voxel table overflow (internal capacity bug)");
    return KB_OK;
}

// a vetoed frame modified nothing: grow the table for its now known voxel count and let frames run again
static int pipeline_after_veto(kb_pipeline *p, const FrameResult &r, size_t n) {
    ++p->grow_retries;
    p->map->h_counters[C_STATUS] = 0;
    CK(cudaMemsetAsync(&p->d_state->vetoed, 0, sizeof(int), p->ex->stream));
    return p->map->ensure_capacity(std::max<size_t>(static_cast<size_t>(r.n_ds), pipeline_extra(p, n)) + 1);
}

// blocking RegisterFrame on device-resident input
static int pipeline_run(kb_pipeline *p, const double *d_xyz, size_t n, const double *d_ts, size_t n_ts, bool in_f32 = false) {
    Exec &ex = *p->ex;
    RET(p->map->ensure_capacity(pipeline_extra(p, n)));
    const long long id = p->next_id++;
    for (int attempt = 0; attempt < 3; ++attempt) {
        {
            StallTrace t("blocking: launch");
            RET(pipeline_launch(p, id, d_xyz, n, d_ts, n_ts, in_f32, p->d_res));
        }
        {
            StallTrace t("blocking: result D2H enqueue");
            CK(cudaMemcpyAsync(p->h_res, p->d_res, sizeof(FrameResult), cudaMemcpyDeviceToHost, ex.stream));
        }
        {
            StallTrace t("blocking: stream sync");
            RET(ex.sync());
        }
        if (!(p->h_res->map_status & ST_NEED_GROW)) return pipeline_absorb(p, *p->h_res, n, id);
        RET(pipeline_after_veto(p, *p->h_res, n));
    }
    return fail(KB_ERR_CUDA, "voxel table could not be grown (internal capacity bug)");
}

static int pipeline_check(kb_pipeline *p, const void *xyz, size_t n, const void *ts, size_t n_ts, bool *use_ts) {
    if (!p || (!xyz && n) || (!ts && n_ts)) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    if (n >= (size_t(1) << 30)) return fail(KB_ERR_INVALID_ARG, "frame too large");
    *use_ts = p->cfg.deskew && n_ts > 0;
    if (*use_ts && n_ts < n)
        return fail(KB_ERR_OUT_OF_RANGE, "timestamps (%zu) shorter than frame (%zu): the reference throws std::out_of_range",
                    n_ts, n);
    return KB_OK;
}

int kb_pipeline_register_frame(kb_pipeline *p, const double *xyz, size_t n, const double *timestamps, size_t n_timestamps) {
    bool use_ts;
    RET(pipeline_check(p, xyz, n, timestamps, n_timestamps, &use_ts));
    Exec &ex = *p->ex;
    CK(cudaSetDevice(ex.device));
    RET(p->ws.ensure(std::max(n, use_ts ? n_timestamps : 0)));
    RET(p->ws.ensure_pipeline(std::max(n, use_ts ? n_timestamps : 0)));
    {
        StallTrace t("blocking: H2D enqueue");
        if (n) CK(cudaMemcpyAsync(p->ws.in.p, xyz, n * 24, cudaMemcpyHostToDevice, ex.stream));
        if (use_ts) CK(cudaMemcpyAsync(p->ws.ts.p, timestamps, n_timestamps * 8, cudaMemcpyHostToDevice, ex.stream));
    }
    return pipeline_run(p, p->ws.in.p, n, p->ws.ts.p, use_ts ? n_timestamps : 0);
}
int kb_pipeline_register_frame_f32(kb_pipeline *p, const float *xyz, size_t n, const double *timestamps, size_t n_timestamps) {
    bool use_ts;
    RET(pipeline_check(p, xyz, n, timestamps, n_timestamps, &use_ts));
    Exec &ex = *p->ex;
    CK(cudaSetDevice(ex.device));
    RET(p->ws.ensure(std::max(n, use_ts ? n_timestamps : 0)));
    RET(p->ws.ensure_pipeline(std::max(n, use_ts ? n_timestamps : 0)));
    if (n) CK(cudaMemcpyAsync(p->ws.in.p, xyz, n * 12, cudaMemcpyHostToDevice, ex.stream));  // half the bytes of the f64 path
    if (use_ts) CK(cudaMemcpyAsync(p->ws.ts.p, timestamps, n_timestamps * 8, cudaMemcpyHostToDevice, ex.stream));
    return pipeline_run(p, p->ws.in.p, n, p->ws.ts.p, use_ts ? n_timestamps : 0, true);
}
int kb_pipeline_register_frame_dev(kb_pipeline *p, const double *d_xyz, size_t n, const double *d_timestamps,
                                   size_t n_timestamps) {
    bool use_ts;
    RET(pipeline_check(p, d_xyz, n, d_timestamps, n_timestamps, &use_ts));
    CK(cudaSetDevice(p->ex->device));
    RET(p->ws.ensure(std::max(n, use_ts ? n_timestamps : 0)));
    RET(p->ws.ensure_pipeline(std::max(n, use_ts ? n_timestamps : 0)));
    return pipeline_run(p, d_xyz, n, d_timestamps, use_ts ? n_timestamps : 0);
}
// ---- queued registration of a whole sequence ------------------------------------------------------------------
static int queue_init(kb_pipeline *p, size_t max_n, bool any_ts, bool device_input) {
    if (!p->copy_stream) {
        CK(cudaStreamCreateWithFlags(&p->copy_stream, cudaStreamNonBlocking));
        for (auto &s : p->q) {
            CK(cudaEventCreateWithFlags(&s.copied, cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&s.read, cudaEventDisableTiming));
        }
        CK(cudaStreamCreateWithFlags(&p->res_stream, cudaStreamNonBlocking));
        CK(cudaHostAlloc(&p->q_res, sizeof(FrameResult) * kb_pipeline::Q_DEPTH, cudaHostAllocDefault));
        CK(cudaMalloc(&p->q_res_dev, sizeof(FrameResult) * kb_pipeline::Q_DEPTH));
        CK(cudaMemsetAsync(p->q_res_dev, 0, sizeof(FrameResult) * kb_pipeline::Q_DEPTH, p->ex->stream));
    }
    if (!device_input)
        for (auto &s : p->q) {
            RET(s.in.ensure(3 * std::max<size_t>(max_n, 1)));
            if (any_ts) RET(s.ts.ensure(std::max<size_t>(max_n, 1)));
        }
    return KB_OK;
}

static bool is_pinned(const void *ptr) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

// host -> device on the copy stream; pageable sources go through this slot's pinned staging buffer so that the copy
// is truly asynchronous (the memcpy into it overlaps the frame being registered)
static int queue_upload(kb_pipeline *p, void *dst, const void *src, size_t bytes, void **pin, size_t *pin_bytes) {
    if (!bytes) return KB_OK;
    if (!is_pinned(src)) {
        if (*pin_bytes < bytes) {
            if (*pin) cudaFreeHost(*pin);
            *pin = nullptr;
            *pin_bytes = 0;
            CK(cudaHostAlloc(pin, bytes + bytes / 4, cudaHostAllocDefault));
            *pin_bytes = bytes + bytes / 4;
        }
        std::memcpy(*pin, src, bytes);
        src = *pin;
    }
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, p->copy_stream));
    return KB_OK;
}

int kb_pipeline_register_frames(kb_pipeline *p, const void *const *xyz, const size_t *n, const double *const *timestamps,
                                const size_t *n_timestamps, size_t count, int layout, double *poses_out) {
    if (!p || (count && (!xyz || !n))) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    if (layout != KB_FRAMES_HOST_F64 && layout != KB_FRAMES_HOST_F32 && layout != KB_FRAMES_DEVICE_F64)
        return fail(KB_ERR_INVALID_ARG, "unknown frame layout %d", layout);
    constexpr size_t D = kb_pipeline::Q_DEPTH;
    Exec &ex = *p->ex;
    CK(cudaSetDevice(ex.device));
    const bool dev_in = layout == KB_FRAMES_DEVICE_F64, f32 = layout == KB_FRAMES_HOST_F32;
    // like a loop over RegisterFrame, an invalid frame stops the sequence AFTER the frames before it were registered
    size_t valid = 0, max_n = 0;
    bool any_ts = false;
    int bad_status = KB_OK;
    std::string bad_msg;
    std::vector<char> use_ts(count, 0);
    for (; valid < count; ++valid) {
        bool u = false;
        const size_t nt = (timestamps && n_timestamps) ? n_timestamps[valid] : 0;
        bad_status = pipeline_check(p, xyz[valid], n[valid], (timestamps && nt) ? timestamps[valid] : nullptr, nt, &u);
        if (bad_status != KB_OK) {
            bad_msg = tl_err;
            break;
        }
        use_ts[valid] = u;
        any_ts |= u;
        max_n = std::max(max_n, std::max(n[valid], u ? nt : size_t(0)));
    }
    RET(ex.sync());
    RET(p->ws.ensure(max_n));
    RET(p->ws.ensure_pipeline(max_n));
    RET(queue_init(p, max_n, any_ts, dev_in));

    // Pipeline: frame k is registered by launch k, whose idle CTAs also compute the front end of frame k + 1 when that
    // frame has no timestamps (nothing of it depends on frame k's pose then); so frame k + 1 must be on the device when
    // launch k starts: uploads run one frame ahead of the launches, Q_DEPTH - 1 launches may be in flight.
    size_t next_submit = 0, next_absorb = 0, next_upload = 0;
    int attempts = 0;
    const long long id0 = p->next_id;
    auto upload = [&](size_t u) -> int {  // host layouts: frame u -> slot u % D on the copy stream
        auto &s = p->q[u % D];
        StallTrace t("queue: H2D enqueue");
        RET(queue_upload(p, s.in.p, xyz[u], n[u] * (f32 ? 12 : 24), &s.pin_xyz, &s.pin_xyz_bytes));
        if (use_ts[u]) RET(queue_upload(p, s.ts.p, timestamps[u], n_timestamps[u] * 8, &s.pin_ts, &s.pin_ts_bytes));
        CK(cudaEventRecord(s.copied, p->copy_stream));
        return KB_OK;
    };
    auto run = [&]() -> int {
    while (next_absorb < valid) {
        const size_t inflight = next_submit - next_absorb;
        bool submit = next_submit < valid && inflight + 1 < D;
        if (submit && inflight > 0 && p->map->would_grow(pipeline_extra(p, n[next_submit]))) submit = false;  // drain first
        if (submit) {
            const size_t k = next_submit, nk = n[k], ntk = use_ts[k] ? n_timestamps[k] : 0;
            auto &s = p->q[k % D];
            RET(p->map->ensure_capacity(pipeline_extra(p, nk)));  // rebuilds only with nothing in flight
            const bool prefetch = k + 1 < valid && !use_ts[k + 1] && n[k + 1] > 0;
            const double *d_xyz, *d_ts = nullptr, *d_next = nullptr;
            if (dev_in) {
                d_xyz = static_cast<const double *>(xyz[k]);
                if (ntk) d_ts = timestamps[k];
                if (prefetch) d_next = static_cast<const double *>(xyz[k + 1]);
            } else {
                for (; next_upload <= k + (prefetch ? 1 : 0); ++next_upload) RET(upload(next_upload));
                CK(cudaStreamWaitEvent(ex.stream, s.copied, 0));
                if (prefetch) CK(cudaStreamWaitEvent(ex.stream, p->q[(k + 1) % D].copied, 0));
                d_xyz = s.in.p;
                d_ts = s.ts.p;
                if (prefetch) d_next = p->q[(k + 1) % D].in.p;
            }
            {
                StallTrace t("queue: launch");
                RET(pipeline_launch(p, id0 + static_cast<long long>(k), d_xyz, nk, d_ts, ntk, f32, p->q_res_dev + k % D, d_next,
                                    prefetch ? n[k + 1] : 0));
                CK(cudaEventRecord(s.done, ex.stream));
                // result read-back on its own stream: neither the next kernel nor the next H2D waits for it (letting
                // the kernel write to mapped host memory instead was measured ~1% slower)
                CK(cudaStreamWaitEvent(p->res_stream, s.done, 0));
                CK(cudaMemcpyAsync(p->q_res + k % D, p->q_res_dev + k % D, sizeof(FrameResult), cudaMemcpyDeviceToHost,
                                   p->res_stream));
                CK(cudaEventRecord(s.read, p->res_stream));
            }
            ++next_submit;
            continue;
        }
        const size_t k = next_absorb;
        {
            StallTrace t("queue: wait for oldest frame");
            cudaEvent_t ev = p->q[k % D].read;  // also frees this slot's buffers for frame k + D
            RET(ex.wait_deadline([&] { return cudaEventQuery(ev); }, "queued frame"));
        }
        const FrameResult r = p->q_res[k % D];
        if (r.map_status & ST_NEED_GROW) {  // frames queued behind it were skipped on the device: replay from k
            if (++attempts >= 3) return fail(KB_ERR_CUDA, "voxel table could not be grown (internal capacity bug)");
            RET(ex.sync());
            CK(cudaStreamSynchronize(p->res_stream));
            RET(pipeline_after_veto(p, r, n[k]));
            next_submit = k;
            next_upload = k;
            continue;
        }
        attempts = 0;
        RET(watchdog_check(ex.device));
        p->next_id = id0 + static_cast<long long>(k) + 1;
        const int st = pipeline_absorb(p, r, n[k], id0 + static_cast<long long>(k));
        if (st != KB_OK) {
            ex.sync();
            return st;
        }
        if (poses_out) std::memcpy(poses_out + 16 * k, r.pose, sizeof(double) * 16);
        ++next_absorb;
    }
    return KB_OK;
    };
    const int st = run();
    if (st != KB_OK) {
        // an error in the middle of the queue: launches may still be in flight and finished frames not absorbed. Let them
        // finish and absorb what completed, so that the host mirrors (pose, counters, last clouds) match the device.
        const std::string msg = tl_err;
        if (!device_is_stuck(ex.device) && cudaStreamSynchronize(p->copy_stream) == cudaSuccess && ex.sync() == KB_OK &&
            cudaStreamSynchronize(p->res_stream) == cudaSuccess) {
            for (; next_absorb < next_submit; ++next_absorb) {
                const size_t k = next_absorb;
                const FrameResult r = p->q_res[k % D];
                if (r.map_status & ST_NEED_GROW) {
                    pipeline_after_veto(p, r, n[k]);  // clears the sticky veto; the frames behind it were skipped
                    break;
                }
                if (r.map_status & ST_SKIPPED) break;
                p->next_id = id0 + static_cast<long long>(k) + 1;
                if (pipeline_absorb(p, r, n[k], id0 + static_cast<long long>(k)) != KB_OK) break;
                if (poses_out) std::memcpy(poses_out + 16 * k, r.pose, sizeof(double) * 16);
            }
        }
        cudaGetLastError();
        tl_err = msg;
        return st;
    }
    if (bad_status != KB_OK) {
        tl_err = bad_msg;
        return bad_status;
    }
    return KB_OK;
}

int kb_pipeline_grow_retries(const kb_pipeline *p, unsigned long long *out) {
    if (!p || !out) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    *out = p->grow_retries;
    return KB_OK;
}
int kb_pipeline_last_cloud_sizes(const kb_pipeline *p, size_t *n_preprocessed, size_t *n_source) {
    if (!p) return fail(KB_ERR_INVALID_ARG, "p == NULL");
    if (n_preprocessed) *n_preprocessed = p->has_last ? static_cast<size_t>(p->last.n_pre) : 0;
    if (n_source) *n_source = p->has_last ? static_cast<size_t>(p->last.n_src) : 0;
    return KB_OK;
}
int kb_pipeline_last_clouds(const kb_pipeline *cp, double *preprocessed_xyz, size_t cap_preprocessed, double *source_xyz,
                            size_t cap_source) {
    kb_pipeline *p = const_cast<kb_pipeline *>(cp);
    if (!p) return fail(KB_ERR_INVALID_ARG, "p == NULL");
    if (!p->has_last) return KB_OK;
    CK(cudaSetDevice(p->ex->device));
    const size_t npre = static_cast<size_t>(p->last.n_pre), nsrc = static_cast<size_t>(p->last.n_src);
    if (preprocessed_xyz) {
        if (cap_preprocessed < npre) return fail(KB_ERR_CAPACITY, "preprocessed buffer too small");
        if (npre) CK(cudaMemcpyAsync(preprocessed_xyz, (p->last_id & 1) ? p->ws.pre_b.p : p->ws.pre.p, npre * 24, cudaMemcpyDeviceToHost, p->ex->stream));
    }
    if (source_xyz) {
        if (cap_source < nsrc) return fail(KB_ERR_CAPACITY, "source buffer too small");
        if (nsrc) CK(cudaMemcpyAsync(source_xyz, (p->last_id & 1) ? p->ws.src_b.p : p->ws.src.p, nsrc * 24, cudaMemcpyDeviceToHost, p->ex->stream));
    }
    return p->ex->sync();
}
int kb_pipeline_voxelize(kb_pipeline *p, const double *xyz, size_t n, double *source_xyz, size_t cap_source,
                         size_t *n_source, double *downsample_xyz, size_t cap_downsample, size_t *n_downsample) {
    if (!p || (!xyz && n) || !n_source || !n_downsample) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    Exec &ex = *p->ex;
    CK(cudaSetDevice(ex.device));
    RET(p->vox_ws.ensure(n));
    if (n) CK(cudaMemcpyAsync(p->vox_ws.in.p, xyz, n * 24, cudaMemcpyHostToDevice, ex.stream));
    RET(run_downsample(ex, p->vox_ws, p->vox_ws.in.p, n, p->cfg.voxel_size * 0.5, p->vox_ws.ds1.p, p->vox_ws.cnt.p + 1,
                       p->cfg.voxel_size * 1.5, p->vox_ws.src.p, p->vox_ws.cnt.p + 2));
    int c[2] = {0, 0};
    CK(cudaMemcpyAsync(c, p->vox_ws.cnt.p + 1, sizeof(c), cudaMemcpyDeviceToHost, ex.stream));
    RET(ex.sync());
    *n_downsample = static_cast<size_t>(c[0]);
    *n_source = static_cast<size_t>(c[1]);
    if (source_xyz) {
        if (cap_source < *n_source) return fail(KB_ERR_CAPACITY, "source buffer too small");
        if (*n_source) CK(cudaMemcpyAsync(source_xyz, p->vox_ws.src.p, *n_source * 24, cudaMemcpyDeviceToHost, ex.stream));
    }
    if (downsample_xyz) {
        if (cap_downsample < *n_downsample) return fail(KB_ERR_CAPACITY, "downsample buffer too small");
        if (*n_downsample)
            CK(cudaMemcpyAsync(downsample_xyz, p->vox_ws.ds1.p, *n_downsample * 24, cudaMemcpyDeviceToHost, ex.stream));
    }
    return ex.sync();
}
int kb_pipeline_pose(const kb_pipeline *p, double out[16]) {
    if (!p || !out) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    std::memcpy(out, p->last.pose, sizeof(double) * 16);
    return KB_OK;
}
int kb_pipeline_delta(const kb_pipeline *p, double out[16]) {
    if (!p || !out) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    std::memcpy(out, p->last.delta, sizeof(double) * 16);
    return KB_OK;
}
static int pipeline_set(kb_pipeline *p, const double pose[16], const double delta[16]) {
    SE3 a, b;
    if (!to_se3(pose, &a) || !to_se3(delta, &b)) return fail(KB_ERR_NOT_SE3, "matrix is not in SE(3)");
    CK(cudaSetDevice(p->ex->device));
    RET(pipeline_push_state(p, a, b, p->last.model_sse, p->last.num_samples));
    std::memcpy(p->last.pose, pose, sizeof(double) * 16);
    std::memcpy(p->last.delta, delta, sizeof(double) * 16);
    return KB_OK;
}
int kb_pipeline_set_pose(kb_pipeline *p, const double pose[16]) {
    if (!p || !pose) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    return pipeline_set(p, pose, p->last.delta);
}
int kb_pipeline_set_delta(kb_pipeline *p, const double delta[16]) {
    if (!p || !delta) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    return pipeline_set(p, p->last.pose, delta);
}
kb_map *kb_pipeline_voxel_map(kb_pipeline *p) { return p ? p->map : nullptr; }
int kb_pipeline_last_sigma(const kb_pipeline *p, double *out) {
    if (!p || !out) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    *out = p->last.sigma;
    return KB_OK;
}
int kb_pipeline_debug_stamps(const kb_pipeline *p, double *ns, int n) {
    if (!p || !ns) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    const int total = 64 + 4 * p->ex->grid;
    std::vector<unsigned long long> t(total);
    CK(cudaSetDevice(p->ex->device));
    CK(cudaMemcpyAsync(t.data(), p->ex->sc.dbg, sizeof(unsigned long long) * total, cudaMemcpyDeviceToHost, p->ex->stream));
    RET(p->ex->sync());
    for (int i = 0; i < n && i < total; ++i) ns[i] = static_cast<double>(static_cast<long long>(t[i] - t[0]));
    return KB_OK;
}
int kb_debug_ldlt6(const double A[36], const double b[6], double x_loop[6], double x_unrolled[6]) {
    // host evaluation of the two LDLT implementations the device uses (same source, __host__ __device__)
    if (!A || !b || !x_loop || !x_unrolled) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    ldlt6_solve(A, b, x_loop);
    ldlt6_solve_reg(A, b, x_unrolled);
    return KB_OK;
}
int kb_debug_icp_solve(const double A[36], const double b[6], double x_exact[6], double x_fast[6], double T_exact[16],
                       double T_fast[16]) {
    // host evaluation of the exact and the latency-optimised solve/exp/compose the ICP loop uses
    if (!A || !b || !x_exact || !x_fast || !T_exact || !T_fast) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    ldlt6_solve_reg(A, b, x_exact);
    ldlt6_solve_fast(A, b, x_fast);
    const SE3 base = se3_exp(b);
    se3_to_matrix(se3_mul(se3_exp(x_exact), base), T_exact);
    se3_to_matrix(se3_mul_fast(se3_exp_fast(x_fast), base), T_fast);
    return KB_OK;
}
int kb_debug_icp_schur(const double acc[16], double x_schur[6], double x_ldlt[6], int *used_schur) {
    // host evaluation: the structured Schur solve vs the pivoted LDL^T on the same 16 accumulators
    if (!acc || !x_schur || !x_ldlt || !used_schur) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    double JTJ[36], JTr[6], rhs[6];
    for (int i = 0; i < 36; ++i) JTJ[i] = 0.0;
    JTJ[0] = JTJ[7] = JTJ[14] = acc[0];
    JTJ[6 * 3 + 1] = -acc[3]; JTJ[6 * 3 + 2] = acc[2]; JTJ[6 * 4 + 0] = acc[3]; JTJ[6 * 4 + 2] = -acc[1];
    JTJ[6 * 5 + 0] = -acc[2]; JTJ[6 * 5 + 1] = acc[1];
    JTJ[6 * 3 + 3] = acc[4]; JTJ[6 * 4 + 3] = acc[5]; JTJ[6 * 4 + 4] = acc[6];
    JTJ[6 * 5 + 3] = acc[7]; JTJ[6 * 5 + 4] = acc[8]; JTJ[6 * 5 + 5] = acc[9];
    for (int i = 0; i < 6; ++i)
        for (int j = i + 1; j < 6; ++j) JTJ[6 * i + j] = JTJ[6 * j + i];
    for (int i = 0; i < 6; ++i) { JTr[i] = acc[10 + i]; rhs[i] = -JTr[i]; }
    ldlt6_solve_reg(JTJ, rhs, x_ldlt);
    *used_schur = icp_solve_schur(acc, x_schur) ? 1 : 0;
    if (!*used_schur) for (int i = 0; i < 6; ++i) x_schur[i] = x_ldlt[i];
    return KB_OK;
}
int kb_debug_barrier_ns(int iters, double *ns_per_barrier) {
    if (!ns_per_barrier || iters < 1) return fail(KB_ERR_INVALID_ARG, "bad argument");
    DefaultCtx *c;
    RET(default_ctx(&c));
    RET(c->ex->coop(k_barrier_bench, c->ex->sc, iters));
    unsigned long long t[2];
    CK(cudaMemcpyAsync(t, c->ex->sc.dbg + 8, sizeof(t), cudaMemcpyDeviceToHost, c->ex->stream));
    RET(c->ex->sync());
    *ns_per_barrier = static_cast<double>(t[1] - t[0]) / iters;
    return KB_OK;
}
int kb_pipeline_last_ds_profile(const kb_pipeline *p, double us[10]) {
    if (!p || !us) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    const unsigned long long *t = p->last.t_ns;
    // ds1: clear, dedupe, count, prefix+rank, replay+emit ; ds2: same
    const unsigned long long a[6] = {t[1], t[12], t[13], t[14], t[15], t[2]};
    const unsigned long long b[6] = {t[2], t[16], t[17], t[18], t[19], t[3]};
    for (int i = 0; i < 5; ++i) {
        us[i] = (static_cast<double>(a[i + 1]) - static_cast<double>(a[i])) * 1e-3;
        us[5 + i] = (static_cast<double>(b[i + 1]) - static_cast<double>(b[i])) * 1e-3;
    }
    return KB_OK;
}
int kb_pipeline_last_map_profile(const kb_pipeline *p, double us[3]) {
    if (!p || !us) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    const double t4 = static_cast<double>(p->last.t_ns[4]), a = static_cast<double>(p->last.t_ns[8]);
    const double b = static_cast<double>(p->last.t_ns[9]), t5 = static_cast<double>(p->last.t_ns[5]);
    us[0] = (a - t4) * 1e-3;  // transform + find-or-claim + pending lists
    us[1] = (b - a) * 1e-3;   // per-voxel ordered insertion
    us[2] = (t5 - b) * 1e-3;  // eviction scan
    return KB_OK;
}
int kb_pipeline_last_cache_stats(const kb_pipeline *p, double out[3]) {
    if (!p || !out) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    for (int i = 0; i < 3; ++i) out[i] = p->last.cache_stats[i];
    return KB_OK;
}
int kb_pipeline_last_icp_work(const kb_pipeline *p, double *queries, double *candidates) {
    if (!p) return fail(KB_ERR_INVALID_ARG, "p == NULL");
    if (queries) *queries = p->last.icp_queries;
    if (candidates) *candidates = p->last.icp_candidates;
    return KB_OK;
}
int kb_pipeline_threshold(const kb_pipeline *p, double *out_sigma) {
    if (!p || !out_sigma) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    *out_sigma = std::sqrt(p->last.model_sse / p->last.num_samples);  // ComputeThreshold(), Threshold.hpp:38
    return KB_OK;
}
int kb_pipeline_last_iterations(const kb_pipeline *p, int *out) {
    if (!p || !out) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    *out = p->last.iterations;
    return KB_OK;
}
int kb_pipeline_last_profile(const kb_pipeline *p, double *us, int n) {
    if (!p || !us) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    for (int i = 0; i < n && i < 6; ++i) us[i] = (static_cast<double>(p->last.t_ns[i + 1]) - static_cast<double>(p->last.t_ns[i])) * 1e-3;
    return KB_OK;
}
int kb_any_device_stuck(void) { return device_is_stuck(-1) ? 1 : 0; }
int kb_pipeline_set_profiling(kb_pipeline *p, int enabled) {
    if (!p) return fail(KB_ERR_INVALID_ARG, "p == NULL");
    p->ex->sc.profile = enabled;  // 1: all stamps (incl. one per ICP iteration, ~1 us each); 2: phase boundaries only
    std::memset(p->last.t_ns, 0, sizeof(p->last.t_ns));
    return KB_OK;
}
int kb_pipeline_set_history(kb_pipeline *p, size_t capacity) {
    if (!p) return fail(KB_ERR_INVALID_ARG, "p == NULL");
    p->history.clear();
    p->history_stamps.clear();
    p->history.reserve(capacity);
    p->history_cap = capacity;
    return KB_OK;
}
int kb_pipeline_get_history(const kb_pipeline *p, kb_frame_stats *out, size_t capacity, size_t *n_out) {
    if (!p || !n_out) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    *n_out = p->history.size();
    if (!out) return KB_OK;
    if (capacity < p->history.size()) return fail(KB_ERR_CAPACITY, "history buffer too small");
    std::memcpy(out, p->history.data(), p->history.size() * sizeof(kb_frame_stats));
    return KB_OK;
}
int kb_pipeline_history_stamps(const kb_pipeline *p, double *out, size_t capacity, size_t *n_out) {
    if (!p || !n_out) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    *n_out = p->history_stamps.size();
    if (!out) return KB_OK;
    if (capacity < p->history_stamps.size()) return fail(KB_ERR_CAPACITY, "stamp buffer too small");
    for (size_t i = 0; i < p->history_stamps.size(); ++i) std::memcpy(out + 20 * i, p->history_stamps[i].data(), 20 * sizeof(double));
    return KB_OK;
}
int kb_pipeline_launch_count(const kb_pipeline *p, unsigned long long *out) {
    if (!p || !out) return fail(KB_ERR_INVALID_ARG, "NULL argument");
    *out = p->ex->launches;
    return KB_OK;
}

}  // extern "C"
