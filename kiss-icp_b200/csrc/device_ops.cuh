// Device-side building blocks of the registration hot path (sm_100a).
//
// Execution model: every op below is written for a PERSISTENT COOPERATIVE GRID — one CTA per
// SM (or fewer), all CTAs co-resident, phases separated by a hand-rolled grid barrier (one
// L2 atomic + acquire spin, ~1 us) instead of kernel boundaries. A whole
// KissICP::RegisterFrame is therefore ONE launch (k_register_frame in kernels.cu); the same
// ops are also wrapped as stand-alone kernels for the module-level API.
//
// Data layout in HBM
//   VoxelHashMap  -> open-addressed table of 16-byte slots {x,y,z,w} (one 128-bit load per
//                    probe). w = point count (>=0), KB_EMPTY or KB_TOMB. The slot index IS the
//                    index of the voxel's point block: points[slot][cap][3] FP64 (AoS, 24 B /
//                    point, insertion order) — no indirection, no allocator; 180 GB of HBM
//                    makes the sparse block array affordable and the L2 only ever sees the
//                    touched sectors.
//   clouds        -> dense double[n][3], exactly the host layout of std::vector<Eigen::Vector3d>.
#pragma once

#include <cuda_runtime.h>

#include <cfloat>
#include <climits>
#include <cstdint>

#include "se3.cuh"

namespace kb {

constexpr int KB_EMPTY = -1;
constexpr int KB_TOMB = -2;
constexpr unsigned FULL = 0xffffffffu;
constexpr int BLOCK = 512;  // threads per CTA of every cooperative kernel
constexpr int NWARPS = BLOCK / 32;
constexpr int NACC = 16;  // unique accumulators of the 6x6 normal equations (see icp_accumulate)
constexpr int NPART = NACC + 5;  // per-CTA partial: accumulators, #correspondences, #candidate points, cache hits/fills/overflows
constexpr int DS_MAX_CHUNKS = 4096;  // downsample: 32-bucket chunks up to 131072 buckets (a 65k-point scan), coarser beyond
constexpr int BAR_ARRIVE = 32, BAR_TEAM = 64, BAR_TICKET = 96, BAR_WORDS = 128;  // word offsets inside Scratch::bar (one 128-byte line each)
constexpr int LL_RES = 16;        // est(7) + done flag, final pose(7), spare      // est(7) t_icp(7) final(7) conv cand_total query_total ...

enum Counter { C_LIVE = 0, C_TOMB = 1, C_POINTS = 2, C_STATUS = 3, C_TOUCHED = 4, C_NCOUNTERS = 8 };
enum StatusBit { ST_TABLE_FULL = 1, ST_NEED_GROW = 2, ST_SKIPPED = 4 };

// core/VoxelUtils.hpp:33-37 — FP64 DIVISION then floor then int cast (bit-exact with the CPU).
// A DDIV costs ~131 cycles on B200; when voxel_size is an exact power of two (1.0, 0.5, 2.0 ...:
// the reference defaults) x / v == x * (1/v) EXACTLY, so the division is replaced by a multiply.
struct VoxelDiv {
    double v, inv;
    bool pow2;
};
__host__ __device__ __forceinline__ VoxelDiv make_voxel_div(double voxel_size) {
    VoxelDiv d;
    d.v = voxel_size;
    unsigned long long bits;
    memcpy(&bits, &voxel_size, 8);
    const unsigned long long expo = (bits >> 52) & 0x7ffULL;
    // normal power of two whose reciprocal is also a normal power of two
    d.pow2 = (bits & 0x000fffffffffffffULL) == 0 && expo > 2 && expo < 2044 && voxel_size > 0.0;
    d.inv = d.pow2 ? 1.0 / voxel_size : 0.0;
    return d;
}

struct MapView {
    int4 *slots;      // [capacity]
    double *points;   // [capacity][cap][3]
    int *head;        // [capacity] overflow list head of the pending-insert set (-1 when idle)
    int *pcount;      // [capacity] size of the pending-insert set (0 when idle)
    int *pending;     // [capacity][32] input indices of the pending-insert set
    int *counters;    // [C_NCOUNTERS]
    unsigned mask;    // capacity - 1 (capacity is a power of two)
    int cap;          // max_points_per_voxel
    double voxel_size;
    double max_distance;
    double map_resolution;  // sqrt(voxel_size^2 / max_points_per_voxel)  VoxelHashMap.cpp:98
    VoxelDiv vdiv;          // voxel_size as a divisor (exact multiply when it is a power of two)
};

// cross-CTA scratch, sized by the grid
struct Scratch {
    unsigned *bar;  // [0] grid barrier counter, [BAR_ARRIVE] CTAs that left the kernel (Grid::finish), [BAR_TEAM] barrier counter of the front-end team: one 128-B
                    // line each (arrival atomics must not fight the epoch pollers); zeroed before each launch
    double *blk_d;  // [2][NPART][grid] doubles (ping-pong by ICP iteration parity; value-major so the reduce is coalesced)
    uint4 *ll_part;   // [NPART][grid] epoch-tagged partial systems, one 16-B chunk per value and CTA
    uint4 *ll_res;    // [LL_RES] epoch-tagged result record published by the coordinator
    uint4 *ll_group;  // [NPART][16] epoch-tagged group partials (second level of the gather tree)
    int *blk_i;     // [grid] ints
    unsigned long long *dbg;  // [64 + 4*grid] timestamps (profiling aid)
    int profile;              // 0: no in-kernel timestamps at all (%globaltimer reads cost ~1 us each on the critical path)
};

// ------------------------------------------------------------------------------------------
// grid barrier (all CTAs co-resident: cooperative launch)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned ld_relaxed_u32(const unsigned *p) {
    unsigned v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned *p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define KB_DBG(sc, i) \
    if (blockIdx.x == 0 && (threadIdx.x & 31) == 0) (sc).dbg[i] = globaltimer_ns()
// per-CTA timeline of the profiled ICP iteration: dbg[64 + 4*cta + k]
#define KB_CYC(sc, i) \
    if (blockIdx.x == 0 && threadIdx.x == 0) (sc).dbg[16 + (i)] = static_cast<unsigned long long>(clock64())
#define KB_DBG_CTA(sc, k) \
    if (threadIdx.x == 0) (sc).dbg[64 + 4 * blockIdx.x + (k)] = globaltimer_ns()

// ------------------------------------------------------------------------------------------
// epoch-tagged 16-byte chunks (the NCCL "LL" idea): a double travels as {lo32, tag, hi32, tag};
// each 8-byte half is a naturally atomic scalar write that validates itself, so a reader that
// sees both tags equal to the tag it waits for has the value — no flag, no fence, no second
// dependent load. Tags = launch sequence number * 8192 + iteration epoch.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void ll_store(uint4 *p, double v, unsigned tag) {
    const unsigned long long b = static_cast<unsigned long long>(__double_as_longlong(v));
    asm volatile("st.relaxed.gpu.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(static_cast<unsigned>(b)), "r"(tag),
                 "r"(static_cast<unsigned>(b >> 32)), "r"(tag)
                 : "memory");
}
__device__ __forceinline__ bool ll_load(const uint4 *p, unsigned tag, double *v) {
    unsigned a, b, c, d;
    // strong (relaxed.gpu) load: always served by the home L2 slice. A weak ld.global.cg is 2x cheaper per
    // polling round but was measured to see the new value ~1.2 us later (B200 has two L2 partitions).
    asm volatile("ld.relaxed.gpu.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "l"(p) : "memory");
    *v = __longlong_as_double(static_cast<long long>((static_cast<unsigned long long>(c) << 32) | a));
    return b == tag && d == tag;
}

__device__ __forceinline__ void fence_acq_rel_gpu() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }

// ------------------------------------------------------------------------------------------
// watchdog of the spin loops: the kernels below wait for each other with hand-rolled barriers and tagged polls. A
// protocol bug (or a CTA that died) would otherwise spin forever and take the GPU with it. Every spin loop counts
// its polls; after 2^g_kb_wd[7] of them (2^24: of the order of 10 s) the loop gives up, raises g_kb_wd[0] — which every other spin
// loop checks every 1024 polls and then leaves too — and reports where it was stuck to a word of mapped host
// memory. The launch then finishes with garbage and the host turns the flag into KB_ERR_CUDA.
// ------------------------------------------------------------------------------------------
__device__ unsigned g_kb_wd[8];          // [0] abort flag, [7] log2 of the poll limit (host-set)
__device__ unsigned *g_kb_wd_host;       // mapped host memory: [0] flag, [1] code, [2] block, [3] thread, [4] a, [5] b
// phase marks: thread 0 of every CTA drops a code into a device word at the phase boundaries of k_register_frame (one
// fire-and-forget store each). When a launch never ends, the host reads the words on a side stream and reports where
// every CTA was: the diagnostic for hangs that are not in a watched spin loop.
__device__ unsigned g_kb_marks[256];
__device__ __forceinline__ void kb_mark(unsigned code) {
    if (threadIdx.x == 0) *reinterpret_cast<volatile unsigned *>(&g_kb_marks[blockIdx.x & 255]) = code;
}
enum WatchdogCode { WD_GRID_BARRIER = 1, WD_ICP_GATHER16 = 2, WD_ICP_RESULT = 3, WD_TEAM_GATHER = 4 };

__device__ __noinline__ bool kb_spin_giveup(unsigned spins, int code, unsigned a, unsigned b) {
    if (*reinterpret_cast<volatile unsigned *>(&g_kb_wd[0]) != 0u) return true;  // somebody gave up: everybody leaves
    if ((spins >> g_kb_wd[7]) == 0u) return false;
    if (atomicCAS(&g_kb_wd[0], 0u, 1u) == 0u && g_kb_wd_host != nullptr) {
        volatile unsigned *h = g_kb_wd_host;
        h[1] = static_cast<unsigned>(code);
        h[2] = blockIdx.x;
        h[3] = threadIdx.x;
        h[4] = a;
        h[5] = b;
        __threadfence_system();
        h[0] = 1u;
    }
    return true;
}
// call once per poll; true = stop waiting
__device__ __forceinline__ bool kb_spin_check(unsigned &spins, int code, unsigned a, unsigned b) {
    return ((++spins & 0x3ffu) == 0u) && kb_spin_giveup(spins, code, a, b);
}

// A Grid is the set of CTAs that take part in a barrier: the whole launch (init) or a TEAM of consecutive
// CTAs (init_team) with its own counter word — k_register_frame splits the launch into an ICP team and a
// front-end team that work on different scans at the same time. rank/size replace blockIdx.x/gridDim.x in
// every op that may run on a team.
struct Grid {
    unsigned *bar;
    unsigned target;
    int rank, size;
    __device__ __forceinline__ void init(unsigned *b) {
        bar = b;
        target = 0;
        rank = static_cast<int>(blockIdx.x);
        size = static_cast<int>(gridDim.x);
    }
    // CTAs [first, first + count) of the launch; `word` = this team's counter (its own 128-byte line)
    __device__ __forceinline__ void init_team(unsigned *word, int first, int count) {
        bar = word;
        target = 0;
        rank = static_cast<int>(blockIdx.x) - first;
        size = count;
    }
    __device__ __forceinline__ void sync() {
        __syncthreads();
        if (threadIdx.x == 0) {
            target += static_cast<unsigned>(size);
            unsigned old;  // release our writes / acquire everybody else's
            asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], 1;" : "=r"(old) : "l"(bar) : "memory");
            unsigned spins = 0;
            unsigned seen;
            while ((seen = ld_relaxed_u32(bar)) < target) {
                // (report: the target and what the counter held - how many CTAs are missing)
                if (kb_spin_check(spins, WD_GRID_BARRIER, target, seen)) break;
            }
            __threadfence();  // acquire side; a gpu-scope fence also drops this SM's L1 lines (plain loads follow)
        }
        __syncthreads();
    }
    // every CTA, once, after its last sync(): the last one to leave re-arms the barrier for the next launch, which
    // saves the host a memset node in front of every launch (kernels launched with Exec::coop(..., self_reset))
    // (full-grid object only; also re-arms the team counter word)
    __device__ __forceinline__ void finish() {
        if (threadIdx.x == 0 && atomicAdd(bar + BAR_ARRIVE, 1u) == gridDim.x - 1) {
            atomicExch(bar + BAR_ARRIVE, 0u);
            atomicExch(bar + BAR_TEAM, 0u);
            atomicExch(bar + BAR_TICKET, 0u);
            atomicExch(bar, 0u);
        }
    }
};

// ------------------------------------------------------------------------------------------
// voxel arithmetic
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ int3 point_to_voxel(double x, double y, double z, const VoxelDiv &d) {
    if (d.pow2)
        return make_int3(static_cast<int>(floor(x * d.inv)), static_cast<int>(floor(y * d.inv)),
                         static_cast<int>(floor(z * d.inv)));
    return make_int3(static_cast<int>(floor(x / d.v)), static_cast<int>(floor(y / d.v)), static_cast<int>(floor(z / d.v)));
}
__device__ __forceinline__ int3 point_to_voxel(double x, double y, double z, double voxel_size) {
    return point_to_voxel(x, y, z, make_voxel_div(voxel_size));
}
// std::hash<Voxel> core/VoxelUtils.hpp:45-51 — needed ONLY to reproduce VoxelDownsample's
// output order (robin_map bucket order); the HBM map uses mix_hash below.
__device__ __forceinline__ unsigned ref_hash(int x, int y, int z) {
    return (static_cast<unsigned>(x) * 73856093u) ^ (static_cast<unsigned>(y) * 19349669u) ^
           (static_cast<unsigned>(z) * 83492791u);
}
// well-mixed hash for the open-addressed map (short probe chains)
__device__ __forceinline__ unsigned mix_hash(int x, int y, int z) {
    unsigned h = static_cast<unsigned>(x) * 0x9E3779B1u;
    h = (h ^ (h >> 15)) + static_cast<unsigned>(y) * 0x85EBCA77u;
    h = (h ^ (h >> 13)) + static_cast<unsigned>(z) * 0xC2B2AE3Du;
    h ^= h >> 16;
    h *= 0x7FEB352Du;
    h ^= h >> 15;
    h *= 0x846CA68Bu;
    h ^= h >> 16;
    return h;
}

__device__ __forceinline__ int4 cas_slot(int4 *addr, int4 expected, int4 desired) {
    unsigned __int128 e, d;
    memcpy(&e, &expected, 16);
    memcpy(&d, &desired, 16);
    unsigned __int128 old = atomicCAS(reinterpret_cast<unsigned __int128 *>(addr), e, d);
    int4 o;
    memcpy(&o, &old, 16);
    return o;
}

// the collision chain of voxel (x,y,z) from bucket h, whose slot s is already loaded: slot index of the voxel or -1;
// *cnt = its point count (untouched on a miss)
__device__ __forceinline__ int map_find_from(const MapView &m, int x, int y, int z, unsigned h, int4 s, int *cnt) {
    for (unsigned probes = 0; probes <= m.mask; ++probes) {
        if (s.w == KB_EMPTY) return -1;
        if (s.w != KB_TOMB && s.x == x && s.y == y && s.z == z) {
            *cnt = s.w;
            return static_cast<int>(h);
        }
        h = (h + 1) & m.mask;
        s = m.slots[h];
    }
    return -1;
}

// lookup: slot index of voxel (x,y,z) or -1; *cnt = its point count
__device__ __forceinline__ int map_find(const MapView &m, int x, int y, int z, int *cnt) {
    const unsigned h = mix_hash(x, y, z) & m.mask;
    return map_find_from(m, x, y, z, h, m.slots[h], cnt);
}

// find-or-claim for AddPoints. New voxels are claimed with w = 0 by one 128-bit CAS; tombstones
// are never reused while inserts race (they are dropped by the host-triggered rehash).
__device__ __forceinline__ int map_find_or_claim(const MapView &m, int x, int y, int z) {
    unsigned h = mix_hash(x, y, z) & m.mask;
    const int4 empty = make_int4(-1, -1, -1, KB_EMPTY);
    for (unsigned probes = 0; probes <= m.mask; ++probes) {
        int4 s = m.slots[h];
        if (s.w == KB_EMPTY) {
            s = cas_slot(&m.slots[h], empty, make_int4(x, y, z, 0));
            if (s.w == KB_EMPTY) {
                atomicAdd(&m.counters[C_LIVE], 1);
                return static_cast<int>(h);
            }
        }
        if (s.w != KB_TOMB && s.x == x && s.y == y && s.z == z) return static_cast<int>(h);
        h = (h + 1) & m.mask;
    }
    atomicOr(&m.counters[C_STATUS], ST_TABLE_FULL);
    return -1;
}

// ------------------------------------------------------------------------------------------
// block-level helpers
// ------------------------------------------------------------------------------------------
// exclusive rank of `flag` among the CTA's threads (thread order) + CTA total
__device__ __forceinline__ int block_rank(int flag, int *total, int *s_warp /*[NWARPS+1]*/) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned b = __ballot_sync(FULL, flag);
    const int rank = __popc(b & ((1u << lane) - 1u));
    __syncthreads();  // protect s_warp reuse
    if (lane == 0) s_warp[warp] = __popc(b);
    __syncthreads();
    int before = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < NWARPS; ++w) {
        const int c = s_warp[w];
        if (w < warp) before += c;
        tot += c;
    }
    *total = tot;
    return before + rank;
}

__device__ __forceinline__ int block_sum(int v, int *s_warp) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = v;
    __syncthreads();
    int tot = 0;
#pragma unroll
    for (int w = 0; w < NWARPS; ++w) tot += s_warp[w];
    return tot;
}

// offset of this CTA (sum of blk_i[0..b-1]) and grand total, read after a grid barrier
__device__ __forceinline__ void grid_offsets(const Grid &g, const int *blk_i, int *offset, int *total, int *s_two) {
    __syncthreads();
    if (threadIdx.x < 32) {
        int before = 0, tot = 0;
        for (int i = threadIdx.x; i < g.size; i += 32) {
            const int c = __ldcg(&blk_i[i]);
            tot += c;
            if (i < g.rank) before += c;
        }
        for (int o = 16; o > 0; o >>= 1) {
            before += __shfl_xor_sync(FULL, before, o);
            tot += __shfl_xor_sync(FULL, tot, o);
        }
        if (threadIdx.x == 0) {
            s_two[0] = before;
            s_two[1] = tot;
        }
    }
    __syncthreads();
    *offset = s_two[0];
    *total = s_two[1];
}

__device__ __forceinline__ void chunk_of(const Grid &g, long long n, long long *lo, long long *hi) {
    *lo = n * static_cast<unsigned>(g.rank) / static_cast<unsigned>(g.size);
    *hi = n * (static_cast<unsigned>(g.rank) + 1) / static_cast<unsigned>(g.size);
}

// ------------------------------------------------------------------------------------------
// op_preprocess — Preprocessor::Preprocess (core/Preprocessing.cpp:55-95)
//   deskew (constant velocity, referenced to the END of the scan) + strict range crop +
//   order-preserving compaction. Two passes around one grid barrier.
// ------------------------------------------------------------------------------------------
// per-warp staging of one query's neighbourhood: which voxel owns the j-th candidate point
constexpr int NN_FLAT_CAP = 32;  // fast path for max_points_per_voxel <= 32
struct WarpNN {
    unsigned char owner[27 * NN_FLAT_CAP];
    int slot[27];
    int start[27];
};

// Per-warp cache of the candidates that can still become a query's nearest neighbour (dynamic
// shared memory, QC_SLOTS queries per warp). Exactness argument: let p_f be the query position
// when the cache was filled, d* its nearest-neighbour distance then, and S the candidates with
// |c - p_f| <= d* + 2R. While the query has moved by delta <= R, its true nearest neighbour c'
// satisfies |c' - p| <= |c* - p| <= d* + delta, hence |c' - p_f| <= d* + 2 delta <= d* + 2R, so
// c' is in S; every candidate outside S is strictly farther than the minimum, so ties (resolved
// by the stored reference sequence numbers) are unaffected. The cache is also tied to the
// query's VOXEL: GetClosestNeighbor only looks at the 27 voxels around the current voxel, so a
// query that crosses a voxel face sees a different candidate set and must be re-probed —
// UNLESS d* + 3R < voxel_size: then every point within d* + 2R of p_f (the whole of S and any
// would-be closer point) is less than one voxel away from both p_f and p, i.e. inside the
// 27-voxel neighbourhood of either position, and the voxel does not matter. The map is immutable during
// AlignPointsToMap and ICP steps shrink geometrically, so after the first iterations a query
// costs no global memory traffic at all: ~30-cycle LDS instead of ~300-cycle L2 round trips,
// and ~10-40 candidates instead of the 135-300 of the full 27-voxel neighbourhood.
constexpr int QC_MAX = 64;   // cached candidates per query
constexpr int QC_SLOTS = 2;  // cached queries per warp
struct QCache {
    int vx, vy, vz;  // voxel of the query at fill time (the reference searches the 27 voxels around it)
    int pad;
    double pf[3];  // query position at fill time
    double p[3];   // current query position, carried across iterations
    int total;     // cached candidates, -1 = invalid
    int full;      // candidates of the full neighbourhood (bookkeeping of algorithmic bytes)
    int any_voxel; // 1: valid in whatever voxel the query is (d* + 3R < voxel_size, see below)
    int pad2;
    double pts[QC_MAX][3];
    int seq[QC_MAX];  // reference order of each cached candidate (tie-breaking)
};
constexpr size_t QC_BYTES = sizeof(QCache) * QC_SLOTS * NWARPS;

struct alignas(16) QListRaw {
    unsigned char bytes[32 + 24 + 4 * QC_MAX + 8];
};
struct Shared {
    int warp_i[NWARPS + 1];
    int two[2];
    alignas(16) int chunk_pref[DS_MAX_CHUNKS];  // exclusive prefix of the downsample chunk counts; op_icp_team: 2048 doubles of reduction scratch
    double warp_d[NWARPS][NPART];
    double warp_c[NWARPS];
    double red[NPART];
    WarpNN wnn[NWARPS];
    double sys[NACC];
    double omega[6];
    double mm[2];
    SE3 pending;
    SE3 t_icp;
    SE3 result;  // op_icp output (valid in every CTA)
    int iters;   // op_icp output
    double cand;     // candidate points examined by the last icp_pass (all CTAs)
    double cand_total, query_total;  // summed over the iterations of op_icp
    double cache_stats[3];           // NN-cache hits / fills / overflows summed over the iterations
    int flag;
    int is_last;
    int refill_n[2], refill_over[2];  // op_icp_team: source points whose candidate list went stale (by iteration parity)
    int refill_q[192];
    QListRaw rlist[NWARPS];      // op_icp_team: candidate list of a re-search, before it is staged (QList, icp_team.cuh)
};

// `in` is double[n][3], or float[n][3] when in_f32 (KITTI .bin / PointCloud2 payloads are float32; the reference
// widens them on the host — python/kiss_icp/datasets/kitti.py:66, ros/src/Utils.hpp:198-208 — here the H2D copy
// is half the size and the exact float->double widening happens on the device)
__device__ __forceinline__ V3 pre_load(const double *in, long long i, bool in_f32) {
    if (in_f32) {
        const float *f = reinterpret_cast<const float *>(in);
        return V3{static_cast<double>(f[3 * i]), static_cast<double>(f[3 * i + 1]), static_cast<double>(f[3 * i + 2])};
    }
    return V3{in[3 * i], in[3 * i + 1], in[3 * i + 2]};
}

__device__ __noinline__ void op_preprocess(Grid &g, const Scratch &sc, Shared &sh, const double *in, int n, const double *ts,
                              int n_ts, bool deskew, const SE3 &motion, double max_range, double min_range,
                              double *tmp, double *out, int *out_n, bool in_f32 = false) {
    const bool do_deskew = deskew && n_ts > 0;
    if (do_deskew) {
        // std::minmax_element over ALL stamps (Preprocessing.cpp:62-64)
        double mn = DBL_MAX, mx = -DBL_MAX;
        for (int i = static_cast<unsigned>(g.rank) * BLOCK + threadIdx.x; i < n_ts; i += static_cast<unsigned>(g.size) * BLOCK) {
            const double t = ts[i];
            mn = fmin(mn, t);
            mx = fmax(mx, t);
        }
        for (int o = 16; o > 0; o >>= 1) {
            mn = fmin(mn, __shfl_xor_sync(FULL, mn, o));
            mx = fmax(mx, __shfl_xor_sync(FULL, mx, o));
        }
        if ((threadIdx.x & 31) == 0) {
            sh.warp_d[threadIdx.x >> 5][0] = mn;
            sh.warp_d[threadIdx.x >> 5][1] = mx;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < NWARPS; ++w) {
                mn = fmin(mn, sh.warp_d[w][0]);
                mx = fmax(mx, sh.warp_d[w][1]);
            }
            sc.blk_d[2 * static_cast<unsigned>(g.rank)] = mn;
            sc.blk_d[2 * static_cast<unsigned>(g.rank) + 1] = mx;
        }
        g.sync();
        if (threadIdx.x == 0) {
            double a = DBL_MAX, b = -DBL_MAX;
            for (unsigned i = 0; i < static_cast<unsigned>(g.size); ++i) {
                a = fmin(a, __ldcg(&sc.blk_d[2 * i]));
                b = fmax(b, __ldcg(&sc.blk_d[2 * i + 1]));
            }
            sh.mm[0] = a;
            sh.mm[1] = b;
            se3_log(motion, sh.omega);  // relative_motion.log()  (:68)
        }
        __syncthreads();
    }
    long long lo, hi;
    chunk_of(g, n, &lo, &hi);
    // pass 1: deskew into tmp, count survivors of the crop
    int kept = 0;
    for (long long base = lo; base < hi; base += BLOCK) {
        const long long i = base + threadIdx.x;
        if (i < hi) {
            V3 p = pre_load(in, i, in_f32);
            if (do_deskew) {
                const double stamp = (ts[i] - sh.mm[0]) / (sh.mm[1] - sh.mm[0]);
                double a[6];
#pragma unroll
                for (int k = 0; k < 6; ++k) a[k] = (stamp - 1.0) * sh.omega[k];
                p = se3_act(se3_exp(a), p);
                tmp[3 * i] = p.x;
                tmp[3 * i + 1] = p.y;
                tmp[3 * i + 2] = p.z;
            }
            const double r = norm(p);
            kept += (r < max_range && r > min_range) ? 1 : 0;
        }
    }
    const int blk_kept = block_sum(kept, sh.warp_i);
    if (threadIdx.x == 0) sc.blk_i[static_cast<unsigned>(g.rank)] = blk_kept;
    g.sync();
    int offset, total;
    grid_offsets(g, sc.blk_i, &offset, &total, sh.two);
    if (static_cast<unsigned>(g.rank) == 0 && threadIdx.x == 0) *out_n = total;
    // pass 2: ordered compaction
    const double *src = do_deskew ? tmp : in;
    const bool src_f32 = in_f32 && !do_deskew;
    int run = offset;
    for (long long base = lo; base < hi; base += BLOCK) {
        const long long i = base + threadIdx.x;
        V3 p{0, 0, 0};
        int keep = 0;
        if (i < hi) {
            p = pre_load(src, i, src_f32);
            const double r = norm(p);
            keep = (r < max_range && r > min_range) ? 1 : 0;
        }
        int tile_total;
        const int rank = block_rank(keep, &tile_total, sh.warp_i);
        if (keep) {
            const long long o = run + rank;
            out[3 * o] = p.x;
            out[3 * o + 1] = p.y;
            out[3 * o + 2] = p.z;
        }
        run += tile_total;
    }
}

// ------------------------------------------------------------------------------------------
// op_downsample — VoxelDownsample (core/VoxelUtils.cpp:7-21)
//   keeps the first point (input order) of every voxel and emits them in the ITERATION ORDER
//   of the reference's tsl::robin_map: bucket_count = pow2 >= 2n (reserve(n), max load 0.5,
//   never rehashes while filling), home = std::hash<Voxel> & (B-1), robin-hood linear probing.
//   Facts used: (1) the SET of occupied buckets of robin-hood hashing equals that of plain
//   linear probing and does not depend on insertion order; (2) two entries in different
//   maximal occupied runs of the final table never interacted (the empty bucket between them
//   was always empty); (3) inside a run the layout DOES depend on history (a displaced entry
//   leapfrogs residents of equal probe distance), so each run is replayed exactly.
//   Phases: [clear] | dedupe: linear probing from the reference's home bucket with a 128-bit CAS +
//   atomicMin(first index), counting claimed buckets per chunk | one warp per chunk: exclusive
//   chunk prefix, singleton runs emitted per lane, longer runs replayed IN REGISTERS (lane =
//   bucket of the run, robin-hood swap chain via ballots) and emitted at their bucket's rank.
//   Two grid barriers per call (one when the caller pre-cleared the scratch tables).
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned robin_bucket_count(int n) {
    if (n <= 0) return 0;
    // reserve(n): size_t(ceil(float(n) / 0.5f)) rounded up to a power of two
    const float c = ceilf(static_cast<float>(n) / 0.5f);
    unsigned long long want = static_cast<unsigned long long>(c);
    unsigned long long p = 1;
    while (p < want) p <<= 1;
    return static_cast<unsigned>(p);
}

struct DsScratch {
    int4 *slots;     // [B] {voxel, first index}
    int *chunk_cnt;  // [DS_MAX_CHUNKS] claimed buckets per chunk of the table
    int *order;      // [B] general path only: run-local insertion order
    int2 *sim;       // [B] general path only: replayed layout {first index (-1 empty), home offset in run}
};

// chunk geometry: at most DS_MAX_CHUNKS chunks of at least 32 buckets (one warp-wide group): small tables
// still spread over hundreds of warps and the per-chunk counters see little atomic contention
__device__ __forceinline__ unsigned ds_chunk_shift(unsigned B) {
    unsigned sh = 5;
    while ((B >> sh) > static_cast<unsigned>(DS_MAX_CHUNKS)) ++sh;
    return sh;
}

// clear the scratch for a table of n inputs (grid-stride; the caller provides the barrier)
__device__ __forceinline__ void ds_clear(const Grid &g, const DsScratch &ds, int n_upper) {
    const unsigned B = robin_bucket_count(n_upper);
    const int4 empty = make_int4(-1, -1, -1, KB_EMPTY);
    for (unsigned i = static_cast<unsigned>(g.rank) * BLOCK + threadIdx.x; i < B; i += static_cast<unsigned>(g.size) * BLOCK) ds.slots[i] = empty;
    for (unsigned i = static_cast<unsigned>(g.rank) * BLOCK + threadIdx.x; i < static_cast<unsigned>(DS_MAX_CHUNKS); i += static_cast<unsigned>(g.size) * BLOCK)
        ds.chunk_cnt[i] = 0;
}

// general (slow, rare) replay of one run longer than a warp: lane 0, global scratch
__device__ __noinline__ void ds_replay_long_run(const DsScratch &ds, unsigned s, unsigned L, unsigned mask) {
    // insertion order by first index: order[s + rank]
    for (unsigned k = 0; k < L; ++k) {
        const int my = ds.slots[(s + k) & mask].w;
        unsigned rank = 0;
        for (unsigned j = 0; j < L; ++j) rank += (ds.slots[(s + j) & mask].w < my) ? 1u : 0u;
        ds.order[(s + rank) & mask] = static_cast<int>((s + k) & mask);
        ds.sim[(s + k) & mask] = make_int2(-1, 0);
    }
    for (unsigned k = 0; k < L; ++k) {
        const int4 e = ds.slots[ds.order[(s + k) & mask]];
        int ci = e.w;
        int ch = static_cast<int>(((ref_hash(e.x, e.y, e.z) & mask) - s) & mask);
        int r = ch;
        while (true) {  // insert_impl search: stop at the first bucket whose resident is "richer"
            const int2 t = ds.sim[(s + r) & mask];
            if (t.x < 0 || (r - ch) > (r - t.y)) break;
            ++r;
        }
        while (true) {  // insert_value: robin-hood swap chain until an empty bucket
            const int2 t = ds.sim[(s + r) & mask];
            if (t.x < 0) break;
            if ((r - ch) > (r - t.y)) {
                ds.sim[(s + r) & mask] = make_int2(ci, ch);
                ci = t.x;
                ch = t.y;
            }
            ++r;
        }
        ds.sim[(s + r) & mask] = make_int2(ci, ch);
    }
}

__device__ __noinline__ void op_downsample(Grid &g, const Scratch &sc, Shared &sh, const double *in, int n, double voxel_size,
                              const DsScratch &ds_in, double *out, int *out_n, unsigned long long *stamps = nullptr,
                              bool precleared = false) {
    (void)sc;
    const DsScratch ds = ds_in;
    const unsigned B = robin_bucket_count(n);
    if (B == 0) {
        if (static_cast<unsigned>(g.rank) == 0 && threadIdx.x == 0) *out_n = 0;
        return;  // uniform across the grid
    }
    const unsigned mask = B - 1;
    int4 *ds_slots = ds.slots;
    const int4 empty = make_int4(-1, -1, -1, KB_EMPTY);
    const unsigned csh = ds_chunk_shift(B);
    const unsigned CH = 1u << csh;
    const unsigned nchunks = (B + CH - 1) >> csh;
    if (!precleared) {
        ds_clear(g, ds, n);
        g.sync();
    }
    if (stamps && static_cast<unsigned>(g.rank) == 0 && threadIdx.x == 0) stamps[0] = globaltimer_ns();
    // (a) dedupe: first input index per voxel; claimed buckets are counted per chunk
    const VoxelDiv vd = make_voxel_div(voxel_size);
    for (int i = static_cast<unsigned>(g.rank) * BLOCK + threadIdx.x; i < n; i += static_cast<unsigned>(g.size) * BLOCK) {
        const int3 v = point_to_voxel(in[3 * i], in[3 * i + 1], in[3 * i + 2], vd);
        unsigned h = ref_hash(v.x, v.y, v.z) & mask;
        while (true) {
            int4 s = ds_slots[h];
            if (s.w == KB_EMPTY) s = cas_slot(&ds_slots[h], empty, make_int4(v.x, v.y, v.z, i));
            if (s.w == KB_EMPTY) {  // claimed with our index
                atomicAdd(&ds.chunk_cnt[h >> csh], 1);
                break;
            }
            if (s.x == v.x && s.y == v.y && s.z == v.z) {
                atomicMin(&ds_slots[h].w, i);
                break;
            }
            h = (h + 1) & mask;
        }
    }
    g.sync();
    if (stamps && static_cast<unsigned>(g.rank) == 0 && threadIdx.x == 0) stamps[1] = stamps[2] = stamps[3] = globaltimer_ns();
    // (b) exclusive prefix of the chunk counts (every CTA, in shared memory): DS_MAX_CHUNKS / BLOCK chunks per thread
    {
        constexpr int PER = DS_MAX_CHUNKS / BLOCK;
        const int t = threadIdx.x;
        int cv[PER];
        int v = 0;
#pragma unroll
        for (int k = 0; k < PER; ++k) {
            cv[k] = (PER * t + k < static_cast<int>(nchunks)) ? __ldcg(&ds.chunk_cnt[PER * t + k]) : 0;
            v += cv[k];
        }
        const int mine = v;
        const int lane = t & 31, warp = t >> 5;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int u = __shfl_up_sync(FULL, v, o);
            if (lane >= o) v += u;
        }
        __syncthreads();
        if (lane == 31) sh.warp_i[warp] = v;
        __syncthreads();
        int before = 0, total = 0;
#pragma unroll
        for (int w = 0; w < NWARPS; ++w) {
            const int c = sh.warp_i[w];
            if (w < warp) before += c;
            total += c;
        }
        int excl = before + v - mine;
#pragma unroll
        for (int k = 0; k < PER; ++k) {
            sh.chunk_pref[PER * t + k] = excl;
            excl += cv[k];
        }
        if (static_cast<unsigned>(g.rank) == 0 && t == 0) *out_n = total;
        __syncthreads();
    }
    // (c) one warp per chunk: singleton runs per lane, longer runs replayed in registers
    const int lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u;
    for (unsigned c = static_cast<unsigned>(g.rank) + static_cast<unsigned>(g.size) * (threadIdx.x >> 5); c < nchunks; c += static_cast<unsigned>(g.size) * NWARPS) {
        const unsigned cbase = c << csh;
        const unsigned cend = min(cbase + CH, B);
        int before = sh.chunk_pref[c];  // occupied buckets before the current group
        unsigned prev_occ = (ds_slots[(cbase - 1) & mask].w != KB_EMPTY) ? 1u : 0u;  // bucket before the group
        for (unsigned gb = cbase; gb < cend; gb += 32) {
            const unsigned b = gb + lane;
            const int4 e = (b < cend) ? ds_slots[b] : empty;
            const unsigned occ = __ballot_sync(FULL, e.w != KB_EMPTY);
            const unsigned left = (occ << 1) | prev_occ;                     // bit l: bucket l-1 occupied
            const unsigned nvalid = min(32u, cend - gb);                     // < 32 only for tables smaller than a warp
            const unsigned next_occ_bit = (ds_slots[(gb + nvalid) & mask].w != KB_EMPTY) ? 1u : 0u;  // wraps at the table end
            const unsigned right = (occ >> 1) | (next_occ_bit << (nvalid - 1));  // bit l: bucket l+1 occupied
            const unsigned starts = occ & ~left;                             // run starts in this group
            const unsigned single = starts & ~right;                         // runs of length 1
            if ((single >> lane) & 1u) {
                const long long o = before + __popc(occ & lt);
                const long long src = e.w;
                out[3 * o] = in[3 * src];
                out[3 * o + 1] = in[3 * src + 1];
                out[3 * o + 2] = in[3 * src + 2];
            }
            unsigned multi = starts & ~single;
            while (multi) {
                const int sb = __ffs(multi) - 1;
                multi &= multi - 1;
                const unsigned s = gb + sb;                                  // first bucket of the run
                const int o_run = before + __popc(occ & ((1u << sb) - 1u));  // its rank among occupied buckets
                // run length (may leave the group / chunk / wrap around the table end)
                unsigned L = 0;
                while (true) {
                    const unsigned o2 = __ballot_sync(FULL, ds_slots[(s + L + lane) & mask].w != KB_EMPTY);
                    if (o2 != FULL) {
                        L += __ffs(~o2) - 1;
                        break;
                    }
                    L += 32;
                }
                if (L <= 32) {
                    // lane k <-> entry found in bucket s+k; replay the inserts in first-index order
                    const int4 f = (static_cast<unsigned>(lane) < L) ? ds_slots[(s + lane) & mask] : empty;
                    const int idx = (static_cast<unsigned>(lane) < L) ? f.w : INT_MAX;
                    const int home = static_cast<int>(((ref_hash(f.x, f.y, f.z) & mask) - s) & mask);
                    int rank = 0;
                    for (unsigned j = 0; j < L; ++j) rank += (__shfl_sync(FULL, idx, j) < idx) ? 1 : 0;
                    int sim_idx = -1, sim_home = 0;  // lane r = bucket s+r of the replayed table
                    for (unsigned t = 0; t < L; ++t) {
                        const unsigned who = __ballot_sync(FULL, static_cast<unsigned>(lane) < L && rank == static_cast<int>(t));
                        const int srcl = __ffs(who) - 1;
                        int ci = __shfl_sync(FULL, idx, srcl), ch = __shfl_sync(FULL, home, srcl);
                        int from = ch;  // insert_impl + insert_value: next bucket >= from that is empty or "richer"
                        while (true) {
                            const unsigned cand = __ballot_sync(FULL, lane >= from && (sim_idx < 0 || sim_home > ch));
                            const int p = __ffs(cand) - 1;
                            const int di = __shfl_sync(FULL, sim_idx, p), dh = __shfl_sync(FULL, sim_home, p);
                            if (lane == p) {
                                sim_idx = ci;
                                sim_home = ch;
                            }
                            if (di < 0) break;  // landed in an empty bucket
                            ci = di;            // displaced resident carries on
                            ch = dh;
                            from = p + 1;
                        }
                    }
                    if (static_cast<unsigned>(lane) < L) {
                        const unsigned bk = s + lane;
                        const long long o = (bk >= B) ? static_cast<long long>(bk - B) : static_cast<long long>(o_run) + lane;
                        const long long src = sim_idx;
                        out[3 * o] = in[3 * src];
                        out[3 * o + 1] = in[3 * src + 1];
                        out[3 * o + 2] = in[3 * src + 2];
                    }
                } else {
                    if (lane == 0) ds_replay_long_run(ds, s, L, mask);
                    __syncwarp();
                    for (unsigned r = lane; r < L; r += 32) {
                        const unsigned bk = s + r;
                        const long long o = (bk >= B) ? static_cast<long long>(bk - B) : static_cast<long long>(o_run) + r;
                        const long long src = ds.sim[bk & mask].x;
                        out[3 * o] = in[3 * src];
                        out[3 * o + 1] = in[3 * src + 1];
                        out[3 * o + 2] = in[3 * src + 2];
                    }
                }
            }
            before += __popc(occ);
            prev_occ = occ >> 31;
        }
    }
}

// ------------------------------------------------------------------------------------------
// nn_search_warp — VoxelHashMap::GetClosestNeighbor (core/VoxelHashMap.cpp:46-70)
//   one warp per query: lanes 0..26 probe the 27 neighbour voxels (one 128-bit slot load
//   each, in the reference's voxel_shifts order), then the warp walks the occupied voxels,
//   lane i taking point i of the block. Ties resolve like the reference (first voxel in
//   shift order, first point in the voxel): lexicographic (distance, sequence) minimum.
//   distance = sqrt((dx*dx + dy*dy) + dz*dz) exactly as Eigen's (neighbor - query).norm().
// ------------------------------------------------------------------------------------------
__constant__ int c_shifts[27][3] = {
    {0, 0, 0},   {1, 0, 0},   {-1, 0, 0},  {0, 1, 0},   {0, -1, 0},  {0, 0, 1},   {0, 0, -1},
    {1, 1, 0},   {1, -1, 0},  {-1, 1, 0},  {-1, -1, 0}, {1, 0, 1},   {1, 0, -1},  {-1, 0, 1},
    {-1, 0, -1}, {0, 1, 1},   {0, 1, -1},  {0, -1, 1},  {0, -1, -1}, {1, 1, 1},   {1, 1, -1},
    {1, -1, 1},  {1, -1, -1}, {-1, 1, 1},  {-1, 1, -1}, {-1, -1, 1}, {-1, -1, -1}};

struct NNResult {
    double d;  // DBL_MAX on a miss
    V3 p;      // (0,0,0) on a miss
    int candidates;
};

__device__ __forceinline__ void nn_reduce(double &best, int &bseq, V3 &bp) {
    // lexicographic (distance, sequence) minimum across the warp. Distances are non-negative
    // doubles, so their bit patterns order like unsigned integers: three REDUX.MIN steps
    // (high word, low word, sequence) replace a 5-round 64-bit shuffle tree.
    const unsigned long long bits = static_cast<unsigned long long>(__double_as_longlong(best));
    const unsigned hi = static_cast<unsigned>(bits >> 32), lo = static_cast<unsigned>(bits);
    const unsigned mhi = __reduce_min_sync(FULL, hi);
    const unsigned mlo = __reduce_min_sync(FULL, hi == mhi ? lo : 0xffffffffu);
    const bool tie = (hi == mhi) && (lo == mlo);
    const unsigned mseq = __reduce_min_sync(FULL, tie ? static_cast<unsigned>(bseq) : 0xffffffffu);
    const unsigned who = __ballot_sync(FULL, tie && static_cast<unsigned>(bseq) == mseq);
    const int src = who ? (__ffs(who) - 1) : 0;
    bp.x = __shfl_sync(FULL, bp.x, src);
    bp.y = __shfl_sync(FULL, bp.y, src);
    bp.z = __shfl_sync(FULL, bp.z, src);
    best = __shfl_sync(FULL, best, src);
    bseq = __shfl_sync(FULL, bseq, src);
}

// 2^-50: d2 > b2 * (1 + NN_TIE_REL) implies sqrt(d2) > sqrt(b2) after rounding. Within that bound two distinct
// squares may round to the same root, and the reference's comparison of rounded roots has to be made.
constexpr double NN_TIE_REL = 8.8817841970012523e-16;

// candidate update with the reference's comparison (first strict minimum of the sqrt'ed norm),
// computing the ~92-cycle DSQRT only when the squared distance could still win
__device__ __forceinline__ void nn_consider(const V3 &c, const V3 &q, int seq, double &best, double &best_d2, int &bseq,
                                            V3 &bp) {
    const V3 df = c - q;
    const double d2 = sqnorm(df);
    if (d2 <= best_d2 * (1.0 + NN_TIE_REL)) {
        const double d = sqrt(d2);
        if (d < best) {
            best = d;
            best_d2 = d2;
            bseq = seq;
            bp = c;
        }
    }
}

// nearest neighbour among the candidates cached in shared memory (same order, same comparison)
__device__ __forceinline__ NNResult nn_search_cached(const QCache &qc, const V3 &q, int lane) {
    double best = DBL_MAX, best_d2 = DBL_MAX;
    int bseq = INT_MAX;
    V3 bp{0, 0, 0};
    const int total = qc.total;
    for (int k = lane; k < total; k += 32)
        nn_consider(V3{qc.pts[k][0], qc.pts[k][1], qc.pts[k][2]}, q, qc.seq[k], best, best_d2, bseq, bp);
    nn_reduce(best, bseq, bp);
    return NNResult{best, bp, qc.full};
}

// ONE square root per query instead of one per lane and candidate: the minimum is taken on squared
// distances (sqrt is monotone), which can only differ from the reference's comparison of rounded
// sqrt values if some other candidate's squared distance lies within NN_TIE_REL above the minimum
// (two distinct squares rounding to the same root). Every lane also tracks its second smallest
// square, nn_reduce_near detects that near tie, and the caller then redoes the search with
// nn_consider (in practice: never).
struct NNMin {
    double b2 = DBL_MAX;  // smallest square of this lane (after nn_reduce_near: of the warp)
    double s2 = DBL_MAX;  // second smallest distinct square of this lane
    int bseq = INT_MAX;   // sequence number (reference order) of the smallest
    V3 bp{0, 0, 0};       // its point
    __device__ __forceinline__ void add(double d2, int seq, const V3 &c) {
        if (d2 < b2) {
            s2 = b2;
            b2 = d2;
            bseq = seq;
            bp = c;
        } else if (d2 > b2 && d2 < s2) {
            s2 = d2;
        }
    }
};

// warp minimum of the lanes' accumulators (exact ties: smallest sequence number); true when another square of any
// lane lies within NN_TIE_REL above it, i.e. the rounded roots have to be compared instead
__device__ __forceinline__ bool nn_reduce_near(NNMin &a) {
    const double mine = a.b2;
    nn_reduce(a.b2, a.bseq, a.bp);
    const double lim = a.b2 * (1.0 + NN_TIE_REL);
    const bool near = (mine > a.b2 && mine <= lim) || (a.s2 <= lim);
    return __any_sync(FULL, near);
}

// nn_search_cached with one square root per query
__device__ __forceinline__ NNResult nn_search_cached_fast(const QCache &qc, const V3 &q, int lane) {
    NNMin a;
    const int total = qc.total;
    for (int k = lane; k < total; k += 32) {
        const V3 c{qc.pts[k][0], qc.pts[k][1], qc.pts[k][2]};
        a.add(sqnorm(c - q), qc.seq[k], c);
    }
    if (nn_reduce_near(a)) return nn_search_cached(qc, q, lane);
    return NNResult{sqrt(a.b2), a.bp, qc.full};
}

// 24-byte point record -> one 16-byte + one 8-byte load (records are 8-byte aligned, every other one 16-byte)
__device__ __forceinline__ V3 ld_point24(const double *rec) {
    const char *pp = reinterpret_cast<const char *>(rec);
    const bool even = ((reinterpret_cast<size_t>(pp) & 15) == 0);
    const double2 wide = *reinterpret_cast<const double2 *>(pp + (even ? 0 : 8));
    const double lone = *reinterpret_cast<const double *>(pp + (even ? 16 : 0));
    return even ? V3{wide.x, wide.y, lone} : V3{lone, wide.x, wide.y};
}

// lanes 0..26: point count and slot of neighbour voxel `lane` of voxel v (voxel_shifts order);
// {0, -1} for an absent voxel and on lanes 27..31
struct NNVoxel {
    int cnt, slot;
};
__device__ __forceinline__ NNVoxel nn_probe27(const MapView &m, const int3 &v, int lane) {
    NNVoxel r{0, -1};
    if (lane < 27) r.slot = map_find(m, v.x + c_shifts[lane][0], v.y + c_shifts[lane][1], v.z + c_shifts[lane][2], &r.cnt);
    return r;
}

// general path (max_points_per_voxel > NN_FLAT_CAP): the warp walks the occupied voxels one after the other, lane i
// taking point i of the block; sequence number = voxel * 1024 + point
__device__ __forceinline__ NNResult nn_walk_voxels(const MapView &m, const V3 &q, int lane, int cnt, int slot) {
    const int cap = m.cap;
    double best = DBL_MAX, best_d2 = DBL_MAX;
    int bseq = INT_MAX;
    V3 bp{0, 0, 0};
    unsigned occ = __ballot_sync(FULL, cnt > 0);
    int total = 0;
    while (occ) {
        const int vi = __ffs(occ) - 1;
        occ &= occ - 1;
        const int c = __shfl_sync(FULL, cnt, vi);
        const int s = __shfl_sync(FULL, slot, vi);
        total += c;
        const double *blk = m.points + static_cast<size_t>(s) * cap * 3;
        for (int k = lane; k < c; k += 32)
            nn_consider(V3{blk[3 * k], blk[3 * k + 1], blk[3 * k + 2]}, q, vi * 1024 + k, best, best_d2, bseq, bp);
    }
    nn_reduce(best, bseq, bp);
    return NNResult{best, bp, total};
}

// flatten the probed neighbourhood (cnt / slot of lanes 0..26, cap <= NN_FLAT_CAP) into `w`: candidate j (reference
// order: voxel_shifts order, then insertion order) is point j - w.start[v] of the block w.slot[v], v = w.owner[j].
// Returns the number of candidates.
__device__ __forceinline__ int nn_flatten(WarpNN &w, int lane, int cnt, int slot) {
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(FULL, incl, o);
        if (lane >= o) incl += t;
    }
    const int start = incl - cnt;
    const int total = __shfl_sync(FULL, incl, 31);
    __syncwarp();
    if (lane < 27) {
        w.slot[lane] = slot;
        w.start[lane] = start;
        for (int k = 0; k < cnt; ++k) w.owner[start + k] = static_cast<unsigned char>(lane);
    }
    __syncwarp();
    return total;
}

// squared radius of the candidate lists: the candidates within d* + 2R of the query (QCache's exactness argument)
__device__ __forceinline__ double nn_keep_thr2(double d, double cache_radius) {
    const double thr = d + 2.0 * cache_radius;
    return thr * thr * (1.0 + 1e-12);
}

// one step of an ordered warp compaction: the lanes with `keep` take positions count, count + 1, ... in lane order
// (returned), and count grows by their number
__device__ __forceinline__ int warp_compact(bool keep, int lane, int &count) {
    const unsigned mask = __ballot_sync(FULL, keep);
    const int pos = count + __popc(mask & ((1u << lane) - 1u));
    count += __popc(mask);
    return pos;
}

// FLAT GATHER over the flattened neighbourhood: candidate j goes to lane j % 32, so all loads of a round are
// independent — one L2 round trip instead of one per occupied voxel. One sqrt per query (NNMin); on a near tie
// the search is redone comparing rounded roots exactly like the reference.
__device__ __forceinline__ NNResult nn_flat_search_staged(const MapView &m, const V3 &q, int lane, WarpNN &w, int total) {
    const int cap = m.cap;
    NNMin a;
    constexpr int U = 2;
    for (int base = 0; base < total; base += 32 * U) {
        V3 c[U];
        bool ok[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int j = base + u * 32 + lane;
            ok[u] = j < total;
            if (ok[u]) {
                const int vi = w.owner[j];
                c[u] = ld_point24(m.points + (static_cast<size_t>(w.slot[vi]) * cap + (j - w.start[vi])) * 3);
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
            if (ok[u]) a.add(sqnorm(c[u] - q), base + u * 32 + lane, c[u]);
    }
    if (!nn_reduce_near(a)) return NNResult{total > 0 ? sqrt(a.b2) : DBL_MAX, a.bp, total};
    double best = DBL_MAX, best_d2 = DBL_MAX;
    int bseq = INT_MAX;
    V3 bp{0, 0, 0};
    for (int j = lane; j < total; j += 32) {
        const int vi = w.owner[j];
        const double *pp = m.points + (static_cast<size_t>(w.slot[vi]) * cap + (j - w.start[vi])) * 3;
        nn_consider(V3{pp[0], pp[1], pp[2]}, q, j, best, best_d2, bseq, bp);
    }
    nn_reduce(best, bseq, bp);
    return NNResult{best, bp, total};
}

__device__ __forceinline__ NNResult nn_flat_search(const MapView &m, const V3 &q, int lane, WarpNN &w, int cnt, int slot) {
    return nn_flat_search_staged(m, q, lane, w, nn_flatten(w, lane, cnt, slot));
}

__device__ __forceinline__ NNResult nn_search_warp(const MapView &m, const V3 &q, int lane, WarpNN &w,
                                                   QCache *fill = nullptr, double cache_radius = 0.0) {
    const int3 v = point_to_voxel(q.x, q.y, q.z, m.vdiv);
    const NNVoxel nv = nn_probe27(m, v, lane);
    const int cap = m.cap;
    if (cap > NN_FLAT_CAP) {
        const NNResult r = nn_walk_voxels(m, q, lane, nv.cnt, nv.slot);
        if (fill != nullptr && lane == 0) fill->total = -1;
        return r;
    }
    const NNResult r = nn_flat_search(m, q, lane, w, nv.cnt, nv.slot);
    const double best = r.d;
    const int total = r.candidates;
    if (fill != nullptr) {
        // second pass (L1-hot): keep the candidates within d* + 2R of the query, in reference order
        int count = -1;
        if (best < DBL_MAX) {
            const double thr2 = nn_keep_thr2(best, cache_radius);
            count = 0;
            constexpr int U2 = 4;
            for (int base = 0; base < total; base += 32 * U2) {
#pragma unroll
                for (int u = 0; u < U2; ++u) {
                    const int j = base + u * 32 + lane;
                    bool keep = false;
                    V3 c{0, 0, 0};
                    if (j < total) {
                        const int vi = w.owner[j];
                        c = ld_point24(m.points + (static_cast<size_t>(w.slot[vi]) * cap + (j - w.start[vi])) * 3);
                        keep = sqnorm(c - q) <= thr2;
                    }
                    const int pos = warp_compact(keep, lane, count);
                    if (keep && pos < QC_MAX) {
                        fill->pts[pos][0] = c.x;
                        fill->pts[pos][1] = c.y;
                        fill->pts[pos][2] = c.z;
                        fill->seq[pos] = j;
                    }
                }
            }
            if (count > QC_MAX) count = -1;
        }
        if (lane == 0) {
            fill->vx = v.x;
            fill->vy = v.y;
            fill->vz = v.z;
            fill->total = count;
            fill->full = total;
            fill->any_voxel = (best < DBL_MAX && best + 3.0 * cache_radius < m.voxel_size) ? 1 : 0;
            fill->pf[0] = q.x;
            fill->pf[1] = q.y;
            fill->pf[2] = q.z;
        }
        __syncwarp();
    }
    return r;
}

// ------------------------------------------------------------------------------------------
// icp_term — one correspondence of BuildLinearSystem (core/Registration.cpp:80-121)
//   J = [I | -hat(s)], w = k^2/(k + |r|^2)^2, JTJ += J^T w J, JTr += J^T w r. With N = -hat(s)
//   the 6x6 has only 16 distinct accumulators:
//     [0]      sum w                     (JTJ[0][0] = [1][1] = [2][2])
//     [1..3]   sum w*s.x, w*s.y, w*s.z   (the antisymmetric lower-left block)
//     [4..9]   lower triangle of N^T w N ((3,3),(4,3),(4,4),(5,3),(5,4),(5,5))
//     [10..15] JTr
//   Each product/sum is formed exactly as Eigen forms (J^T*w)*J entry by entry. Lane l (< 16)
//   of the warp owns accumulator l: the function returns that lane's term.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ double icp_term(int lane, const V3 &s, const V3 &t, double kscale) {
    const V3 r = s - t;
    const double r2 = sqnorm(r);
    const double w = (kscale * kscale) * fast_rcp((kscale + r2) * (kscale + r2));  // ~1 ulp from the reference's division
    const double xw = s.x * w, yw = s.y * w, zw = s.z * w;
    // all 16 terms are computed by every lane (a few dozen FP64 ops) and the lane's own one is
    // selected with predicated moves: a 16-way divergent switch would serialise 16 branches
    double t16[NACC];
    t16[0] = w;
    t16[1] = xw;
    t16[2] = yw;
    t16[3] = zw;
    t16[4] = zw * s.z + yw * s.y;    // (3,3)
    t16[5] = -(xw * s.y);            // (4,3)
    t16[6] = zw * s.z + xw * s.x;    // (4,4)
    t16[7] = -(xw * s.z);            // (5,3)
    t16[8] = -(yw * s.z);            // (5,4)
    t16[9] = yw * s.y + xw * s.x;    // (5,5)
    t16[10] = w * r.x;
    t16[11] = w * r.y;
    t16[12] = w * r.z;
    t16[13] = -(zw * r.y) + yw * r.z;
    t16[14] = zw * r.x - xw * r.z;
    t16[15] = -(yw * r.x) + xw * r.y;
    double v = 0.0;
#pragma unroll
    for (int i = 0; i < NACC; ++i) v = (lane == i) ? t16[i] : v;
    return v;
}

// expand the 16 accumulators to the (lower-triangle-complete) row-major 6x6 and rhs = -JTr
__device__ __forceinline__ void icp_expand(const double a[NACC], double JTJ[36], double JTr[6]) {
    for (int i = 0; i < 36; ++i) JTJ[i] = 0.0;
    JTJ[0] = JTJ[7] = JTJ[14] = a[0];
    // rows 3..5, cols 0..2 : entry (3+i, j) = N[j][i] * w,  N = [[0,z,-y],[-z,0,x],[y,-x,0]]
    JTJ[6 * 3 + 1] = -a[3];
    JTJ[6 * 3 + 2] = a[2];
    JTJ[6 * 4 + 0] = a[3];
    JTJ[6 * 4 + 2] = -a[1];
    JTJ[6 * 5 + 0] = -a[2];
    JTJ[6 * 5 + 1] = a[1];
    JTJ[6 * 3 + 3] = a[4];
    JTJ[6 * 4 + 3] = a[5];
    JTJ[6 * 4 + 4] = a[6];
    JTJ[6 * 5 + 3] = a[7];
    JTJ[6 * 5 + 4] = a[8];
    JTJ[6 * 5 + 5] = a[9];
    for (int i = 0; i < 6; ++i)
        for (int j = i + 1; j < 6; ++j) JTJ[6 * i + j] = JTJ[6 * j + i];
    for (int i = 0; i < 6; ++i) JTr[i] = a[10 + i];
}

// One DataAssociation + BuildLinearSystem pass of THIS CTA (Registration.cpp:60-121): `pending`
// is applied to every source point first (TransformPoints, :55-58), the moved point is written
// back to `work`, and the CTA's partial normal equations go to blk_d[parity][cta][NPART].
// Reduction order is fixed: query-strided per warp -> 16-warp shuffle tree -> CTAs in order.
__device__ __noinline__ void icp_queries(const Scratch &sc, Shared &sh, const MapView &m, const double *src, double *work, int n,
                            const SE3 &pending, double max_dist, double kscale, unsigned tag, bool dbg_on,
                            QCache *qcache, bool first) {
    // (copying sc / m / pending into locals was measured: -0.6 us on the query phase but slower overall, the
    // extra live registers spill in the search code)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (dbg_on) { KB_CYC(sc, 0); }
    if (dbg_on) { KB_DBG_CTA(sc, 3); }
    // query qi -> CTA qi % G, warp (qi / G) % NWARPS: every CTA gets n/G (+1) queries, so the FP64-issue-bound
    // query phase takes the same time on every SM
    const int gwarp = blockIdx.x + gridDim.x * warp, nwarps = gridDim.x * NWARPS;
    double acc = 0.0;  // lane l < 16 owns accumulator l
    int corr = 0;
    double cand = 0.0;
    int n_hit = 0, n_fill = 0, n_over = 0;
    int k = 0;
    for (int qi = gwarp; qi < n; qi += nwarps, ++k) {
        QCache *qc = (qcache != nullptr && k < QC_SLOTS) ? &qcache[warp * QC_SLOTS + k] : nullptr;
        V3 p;
        if (qc != nullptr && !first)
            p = V3{qc->p[0], qc->p[1], qc->p[2]};
        else
            p = V3{src[3 * qi], src[3 * qi + 1], src[3 * qi + 2]};
        p = se3_act(pending, p);
        NNResult r;
        if (qc != nullptr) {
            __syncwarp();
            if (lane == 0) {
                qc->p[0] = p.x;
                qc->p[1] = p.y;
                qc->p[2] = p.z;
                if (first) qc->total = -1;
            }
            __syncwarp();
            const double radius = 0.2 * m.voxel_size;
            const V3 moved = p - V3{qc->pf[0], qc->pf[1], qc->pf[2]};
            const int3 v = point_to_voxel(p.x, p.y, p.z, m.vdiv);
            if (qc->total >= 0 && sqnorm(moved) <= radius * radius &&
                (qc->any_voxel || (qc->vx == v.x && qc->vy == v.y && qc->vz == v.z)))
                r = nn_search_cached_fast(*qc, p, lane), ++n_hit;
            else {
                // (filled on the first iteration too: with a good constant-velocity prediction (steady driving) most
                // caches survive the first step, measured -4 us/scan)
                r = nn_search_warp(m, p, lane, sh.wnn[warp], qc, radius);
                ++n_fill;
                n_over += (qc->total < 0 && r.d < DBL_MAX) ? 1 : 0;
            }
        } else {
            if (lane == 0) {
                work[3 * qi] = p.x;
                work[3 * qi + 1] = p.y;
                work[3 * qi + 2] = p.z;
            }
            r = nn_search_warp(m, p, lane, sh.wnn[warp]);
        }
        cand += r.candidates;
        if (r.d < max_dist) {
            acc += icp_term(lane, p, r.p, kscale);
            ++corr;
        }
    }
    if (dbg_on && warp == 0) KB_DBG(sc, 1);
    if (lane < NACC) sh.warp_d[warp][lane] = acc;
    if (lane == NACC) sh.warp_d[warp][NACC] = static_cast<double>(corr);
    if (lane == NACC + 1) sh.warp_d[warp][NACC + 1] = cand;
    if (lane == NACC + 2) sh.warp_d[warp][NACC + 2] = static_cast<double>(n_hit);
    if (lane == NACC + 3) sh.warp_d[warp][NACC + 3] = static_cast<double>(n_fill);
    if (lane == NACC + 4) sh.warp_d[warp][NACC + 4] = static_cast<double>(n_over);
    __syncthreads();
    if (dbg_on) { KB_CYC(sc, 2); }
    // 16-warp tree per value: thread t -> value t/16, warp t%16 (NWARPS == 16)
    if (threadIdx.x < ((NPART * NWARPS + 31) / 32) * 32) {  // whole warps take part in the shuffles
        const int val = min(static_cast<int>(threadIdx.x) / NWARPS, NPART - 1);
        double v = sh.warp_d[threadIdx.x & (NWARPS - 1)][val];
#pragma unroll
        for (int o = NWARPS / 2; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
        if ((threadIdx.x & (NWARPS - 1)) == 0 && threadIdx.x < NPART * NWARPS)
            ll_store(&sc.ll_part[static_cast<size_t>(threadIdx.x / NWARPS) * gridDim.x + blockIdx.x], v, tag);
    }
    if (dbg_on) { KB_CYC(sc, 3); }
    if (dbg_on) { KB_DBG_CTA(sc, 0); }
    if (dbg_on && threadIdx.x == 0) sc.dbg[64 + 4 * blockIdx.x + 2] = static_cast<unsigned long long>(sh.warp_d[0][NACC + 3] + sh.warp_d[1][NACC + 3] + sh.warp_d[2][NACC + 3] + sh.warp_d[3][NACC + 3] + sh.warp_d[4][NACC + 3] + sh.warp_d[5][NACC + 3] + sh.warp_d[6][NACC + 3] + sh.warp_d[7][NACC + 3] + sh.warp_d[8][NACC + 3] + sh.warp_d[9][NACC + 3] + sh.warp_d[10][NACC + 3] + sh.warp_d[11][NACC + 3] + sh.warp_d[12][NACC + 3] + sh.warp_d[13][NACC + 3] + sh.warp_d[14][NACC + 3] + sh.warp_d[15][NACC + 3]);
}

// Two-level gather of the tagged partials (polling IS the rendezvous). The grid is cut into
// groups of GS = ceil(sqrt(G)) consecutive CTAs; the first CTA of a group (its leader) polls the
// <= 16 partials of its members — one 16-byte chunk per thread, so a gather is ONE load round —
// reduces them with a 16-lane shuffle tree (fixed order) and re-posts the group partial; CTA 0
// then gathers the <= 16 group partials the same way. Two short hops (~0.4 us each) instead of
// one CTA reading 148 x 21 chunks (~2 us).
__device__ __forceinline__ int icp_group_size() {
    int gs = 1;
    while (gs * gs < static_cast<int>(gridDim.x)) ++gs;
    return gs;
}

// thread t = (value e = t / 16, member m = t % 16); returns the sum over `count` chunks in lanes with m == 0
__device__ __forceinline__ double ll_gather16(const uint4 *base, int stride, int first, int count, unsigned tag) {
    const int e = threadIdx.x >> 4, m = threadIdx.x & 15;
    const bool active = e < NPART && m < count;
    double v = 0.0;
    bool ok = !active;
    unsigned spins = 0;
    while (!__all_sync(FULL, ok)) {
        if (!ok) ok = ll_load(&base[static_cast<size_t>(e) * stride + first + m], tag, &v);
        if (__any_sync(FULL, kb_spin_check(spins, WD_ICP_GATHER16, tag, static_cast<unsigned>(first)))) break;
    }
    if (!active) v = 0.0;
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

__device__ __forceinline__ void icp_gather(const Scratch &sc, Shared &sh, unsigned tag, int gs) {  // gs = icp_group_size(), hoisted out of the iteration
    const int G = static_cast<int>(gridDim.x);
    const int ngroups = (G + gs - 1) / gs;
    const int cta = static_cast<int>(blockIdx.x);
    const bool in_tree = threadIdx.x < ((NPART * 16 + 31) / 32) * 32;  // whole warps
    if (cta % gs == 0 && in_tree) {  // group leader
        const int gid = cta / gs, first = gid * gs;
        const double v = ll_gather16(sc.ll_part, G, first, min(gs, G - first), tag);
        if ((threadIdx.x & 15) == 0 && (threadIdx.x >> 4) < NPART) ll_store(&sc.ll_group[(threadIdx.x >> 4) * 16 + gid], v, tag);
    }
    if (cta == 0) {  // coordinator
        if (in_tree) {
            const double v = ll_gather16(sc.ll_group, 16, 0, ngroups, tag);
            if ((threadIdx.x & 15) == 0 && (threadIdx.x >> 4) < NPART) sh.red[threadIdx.x >> 4] = v;
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------
// op_icp — Registration::AlignPointsToMap (core/Registration.cpp:138-167), device resident.
//   Per iteration: every CTA runs its queries and posts its partial normal equations as
//   epoch-tagged chunks; CTA 0 (the fixed coordinator, so the large unrolled solve stays warm in
//   its instruction cache) gathers them in fixed CTA order, solves the 6x6, updates T_icp (kept
//   in its shared memory) and publishes {estimation, converged} as tagged chunks; all CTAs poll
//   that record. No flags, no fences, no host round trip: two L2 hops per iteration.
// ------------------------------------------------------------------------------------------
__device__ __noinline__ void op_icp(Grid &g, const Scratch &sc, Shared &sh, const MapView &m, const double *src, double *work,
                       int n, const SE3 &guess, double max_dist, double kscale, int max_iter, double conv,
                       QCache *qcache, unsigned tag_base) {
    (void)g;
    if (__ldcg(&m.counters[C_LIVE]) == 0 || max_iter <= 0) {  // voxel_map.Empty() -> initial_guess (:143)
        __syncthreads();
        if (threadIdx.x == 0) {
            sh.result = guess;
            sh.iters = 0;
            sh.cand_total = 0.0;
            sh.query_total = 0.0;
            sh.cache_stats[0] = sh.cache_stats[1] = sh.cache_stats[2] = 0.0;
        }
        __syncthreads();
        return;
    }
    if (threadIdx.x == 0) {
        sh.t_icp = se3_identity();
        sh.cand_total = 0.0;
        sh.cache_stats[0] = sh.cache_stats[1] = sh.cache_stats[2] = 0.0;
    }
    SE3 pending = guess;
    const int gs = icp_group_size();
    int j = 0;
    for (;; ++j) {
        if (sc.profile && blockIdx.x == 0 && threadIdx.x == 0 && j < 20) sc.dbg[41 + j] = globaltimer_ns();
        const bool dbg_on = sc.profile && (j == 4);
        const unsigned tag = tag_base + static_cast<unsigned>(j) + 1u;
        icp_queries(sc, sh, m, j == 0 ? src : work, work, n, pending, max_dist, kscale, tag, dbg_on, qcache, j == 0);
        if (dbg_on) { KB_CYC(sc, 4); }
        icp_gather(sc, sh, tag, gs);  // group leaders and the coordinator work, everybody else falls through
        if (blockIdx.x == 0) {
            if (threadIdx.x == 0) {
                if (dbg_on) { KB_CYC(sc, 5); }
                double sys[NACC];
#pragma unroll
                for (int i = 0; i < NACC; ++i) sys[i] = sh.red[i];
                double dx[6];
                if (dbg_on) { KB_CYC(sc, 6); }
                if (!icp_solve_schur(sys, dx)) {                  // :156 — structured 3x3 Schur solve; degenerate
                    double JTJ[36], JTr[6], rhs[6];               // systems take the pivoted LDL^T with Eigen's zero-pivot rule
                    icp_expand(sys, JTJ, JTr);
#pragma unroll
                    for (int i = 0; i < 6; ++i) rhs[i] = -JTr[i];
                    ldlt6_solve_fast(JTJ, rhs, dx);
                }
                if (dbg_on) { KB_CYC(sc, 7); }
                const SE3 est = se3_exp_fast(dx);                 // :157
                if (dbg_on) { KB_CYC(sc, 8); }
                const SE3 t_icp = se3_mul_fast(est, sh.t_icp);    // :161
                if (dbg_on) { KB_CYC(sc, 9); }
                double n2 = 0.0;
#pragma unroll
                for (int i = 0; i < 6; ++i) n2 += dx[i] * dx[i];
                const bool done = (sqrt(n2) < conv) || (j + 1 >= max_iter);  // :163 / :151
                ll_store(&sc.ll_res[0], est.q.x, tag);
                ll_store(&sc.ll_res[1], est.q.y, tag);
                ll_store(&sc.ll_res[2], est.q.z, tag);
                ll_store(&sc.ll_res[3], est.q.w, tag);
                ll_store(&sc.ll_res[4], est.t.x, tag);
                ll_store(&sc.ll_res[5], est.t.y, tag);
                ll_store(&sc.ll_res[6], est.t.z, tag);
                if (done) {
                    const SE3 fin = se3_mul(t_icp, guess);  // :166
                    ll_store(&sc.ll_res[8], fin.q.x, tag);
                    ll_store(&sc.ll_res[9], fin.q.y, tag);
                    ll_store(&sc.ll_res[10], fin.q.z, tag);
                    ll_store(&sc.ll_res[11], fin.q.w, tag);
                    ll_store(&sc.ll_res[12], fin.t.x, tag);
                    ll_store(&sc.ll_res[13], fin.t.y, tag);
                    ll_store(&sc.ll_res[14], fin.t.z, tag);
                }
                ll_store(&sc.ll_res[7], done ? 1.0 : 0.0, tag);
                if (dbg_on) { KB_CYC(sc, 10); }
                sh.t_icp = t_icp;
                sh.cand_total += sh.red[NACC + 1];
                for (int i = 0; i < 3; ++i) sh.cache_stats[i] += sh.red[NACC + 2 + i];
            }
        }
        if (threadIdx.x < 32) {
            // warp 0 of every CTA polls the tagged result record: lanes 0..7 = est(7) + done
            const int l = threadIdx.x;
            double v = 0.0;
            bool ok = l >= 8;
            unsigned spins = 0;
            while (!__all_sync(FULL, ok)) {
                if (!ok) ok = ll_load(&sc.ll_res[l], tag, &v);
                if (__any_sync(FULL, kb_spin_check(spins, WD_ICP_RESULT, tag, 0u))) break;
            }
            if (dbg_on) { KB_CYC(sc, 11); }
            const double dn = __shfl_sync(FULL, v, 7);
            if (dn != 0.0) {  // converged / out of iterations: the final pose rides in chunks 8..14
                ok = l >= 7;
                double f = 0.0;
                spins = 0;
                while (!__all_sync(FULL, ok)) {
                    if (!ok) ok = ll_load(&sc.ll_res[8 + l], tag, &f);
                    if (__any_sync(FULL, kb_spin_check(spins, WD_ICP_RESULT, tag, 1u))) break;
                }
                const double qx = __shfl_sync(FULL, f, 0), qy = __shfl_sync(FULL, f, 1), qz = __shfl_sync(FULL, f, 2);
                const double qw = __shfl_sync(FULL, f, 3), tx = __shfl_sync(FULL, f, 4), ty = __shfl_sync(FULL, f, 5);
                const double tz = __shfl_sync(FULL, f, 6);
                if (l == 0) sh.result = SE3{{qx, qy, qz, qw}, {tx, ty, tz}};
            }
            const double qx = __shfl_sync(FULL, v, 0), qy = __shfl_sync(FULL, v, 1), qz = __shfl_sync(FULL, v, 2);
            const double qw = __shfl_sync(FULL, v, 3), tx = __shfl_sync(FULL, v, 4), ty = __shfl_sync(FULL, v, 5);
            const double tz = __shfl_sync(FULL, v, 6);
            if (l == 0) {
                sh.pending = SE3{{qx, qy, qz, qw}, {tx, ty, tz}};
                sh.flag = dn != 0.0 ? 1 : 0;
                if (dbg_on) { KB_CYC(sc, 12); }
            }
        }
        __syncthreads();
        pending = sh.pending;
        if (sh.flag) break;
    }
    if (threadIdx.x == 0) {
        sh.iters = j + 1;
        sh.query_total = static_cast<double>(n) * (j + 1);
    }
    __syncthreads();
}

// ------------------------------------------------------------------------------------------
// op_map_update — VoxelHashMap::Update / AddPoints / RemovePointsFarFromLocation
//   (core/VoxelHashMap.cpp:83-132). AddPoints is sequential and order dependent in the
//   reference; voxels are independent of each other, so: phase A every new point finds or
//   claims its voxel and pushes itself on that voxel's pending list; phase B one thread per
//   touched voxel replays its pending points in ascending input index (= reference order)
//   with the reference's accept rule; phase C evicts by the first point of each voxel.
// ------------------------------------------------------------------------------------------
constexpr int PEND = 32;  // pending-insert indices kept per voxel in the coalesced array (more spill to a list)

__device__ __forceinline__ bool map_close(const V3 &e, const V3 &p, double res, double res2_lo, double res2_hi) {
    // (e - p).norm() < res  (VoxelHashMap.cpp:108): decided on the squared distance unless it is within a
    // few ulps of res^2, where the rounded sqrt is evaluated like the reference does
    const double d2 = sqnorm(e - p);
    return (d2 < res2_lo) || (d2 <= res2_hi && sqrt(d2) < res);
}

__device__ __noinline__ void op_map_add(Grid &g, Shared &sh, const MapView &m_in, const double *pts, int n, bool has_pose,
                           const SE3 &pose_in, double *tp, int *next, int *touched, unsigned long long *stamps = nullptr) {
    const MapView m = m_in;  // registers, not the caller's stack frame
    const SE3 pose = pose_in;
    // phase A: transform, find-or-claim the voxel, register the point on the voxel's pending set
    for (int i = blockIdx.x * BLOCK + threadIdx.x; i < n; i += gridDim.x * BLOCK) {
        V3 p{pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]};
        if (has_pose) p = se3_act(pose, p);  // VoxelHashMap.cpp:91-93
        tp[3 * i] = p.x;
        tp[3 * i + 1] = p.y;
        tp[3 * i + 2] = p.z;
        const int3 v = point_to_voxel(p.x, p.y, p.z, m.vdiv);
        const int s = map_find_or_claim(m, v.x, v.y, v.z);
        if (s < 0) continue;
        const int r = atomicAdd(&m.pcount[s], 1);
        if (r < PEND) {
            m.pending[static_cast<size_t>(s) * PEND + r] = i;
        } else {  // rare (only when one voxel receives > 32 points in one call): overflow list
            next[i] = atomicExch(&m.head[s], i);
        }
        if (r == 0) touched[atomicAdd(&m.counters[C_TOUCHED], 1)] = s;
    }
    g.sync();
    if (stamps && blockIdx.x == 0 && threadIdx.x == 0) stamps[0] = globaltimer_ns();
    // phase B: one WARP per touched voxel replays that voxel's new points in ascending input index
    // (= the reference's sequential order) with the reference's accept rule.
    const int n_touched = __ldcg(&m.counters[C_TOUCHED]);
    const int cap = m.cap;
    const double res = m.map_resolution;
    const double res2_lo = res * res * (1.0 - 1e-14), res2_hi = res * res * (1.0 + 1e-14);
    const int lane = threadIdx.x & 31;
    const int gw = blockIdx.x + gridDim.x * (threadIdx.x >> 5), nw = gridDim.x * NWARPS;
    for (int t = gw; t < n_touched; t += nw) {
        const int s = __ldcg(&touched[t]);
        const int L = m.pcount[s];
        int cnt = m.slots[s].w;
        double *vp = m.points + static_cast<size_t>(s) * cap * 3;
        int added = 0;
        if (L <= PEND && cap <= 32) {
            // fast path: lane r holds new point #r of the pending set, lane k holds existing point k
            const int idx = lane < L ? m.pending[static_cast<size_t>(s) * PEND + lane] : INT_MAX;
            V3 np{0, 0, 0};
            if (lane < L) np = V3{tp[3 * static_cast<size_t>(idx)], tp[3 * static_cast<size_t>(idx) + 1], tp[3 * static_cast<size_t>(idx) + 2]};
            V3 ex{0, 0, 0};
            if (lane < cnt) ex = V3{vp[3 * lane], vp[3 * lane + 1], vp[3 * lane + 2]};
            int rank = 0;  // position of my index in ascending order
            for (int j = 0; j < L; ++j) rank += (__shfl_sync(FULL, idx, j) < idx) ? 1 : 0;
            for (int r = 0; r < L && cnt < cap; ++r) {
                const unsigned who = __ballot_sync(FULL, lane < L && rank == r);
                const int src = __ffs(who) - 1;
                const V3 p{__shfl_sync(FULL, np.x, src), __shfl_sync(FULL, np.y, src), __shfl_sync(FULL, np.z, src)};
                const bool close = lane < cnt && map_close(ex, p, res, res2_lo, res2_hi);
                if (!__any_sync(FULL, close)) {
                    if (lane == cnt) {
                        ex = p;
                        vp[3 * cnt] = p.x;
                        vp[3 * cnt + 1] = p.y;
                        vp[3 * cnt + 2] = p.z;
                    }
                    ++cnt;
                    ++added;
                }
            }
        } else if (lane == 0) {
            // general path (huge pending sets or max_points_per_voxel > 32): serial replay, sources = array + list
            const int first = m.head[s];
            int last = -1;
            while (cnt < cap) {
                int pick = INT_MAX;
                for (int j = 0; j < min(L, PEND); ++j) {
                    const int v = m.pending[static_cast<size_t>(s) * PEND + j];
                    if (v > last && v < pick) pick = v;
                }
                for (int j = first; j != -1; j = next[j])
                    if (j > last && j < pick) pick = j;
                if (pick == INT_MAX) break;
                last = pick;
                const V3 p{tp[3 * static_cast<size_t>(pick)], tp[3 * static_cast<size_t>(pick) + 1], tp[3 * static_cast<size_t>(pick) + 2]};
                bool reject = false;
                for (int k = 0; k < cnt && !reject; ++k)
                    reject = map_close(V3{vp[3 * k], vp[3 * k + 1], vp[3 * k + 2]}, p, res, res2_lo, res2_hi);
                if (!reject) {
                    vp[3 * cnt] = p.x;
                    vp[3 * cnt + 1] = p.y;
                    vp[3 * cnt + 2] = p.z;
                    ++cnt;
                    ++added;
                }
            }
            m.head[s] = -1;
        }
        cnt = __shfl_sync(FULL, cnt, 0);
        added = __shfl_sync(FULL, added, 0);
        if (lane == 0) {
            m.slots[s].w = cnt;
            m.pcount[s] = 0;
            if (added) atomicAdd(&m.counters[C_POINTS], added);
        }
    }
    g.sync();
    if (stamps && blockIdx.x == 0 && threadIdx.x == 0) stamps[1] = globaltimer_ns();
    if (blockIdx.x == 0 && threadIdx.x == 0) m.counters[C_TOUCHED] = 0;
    (void)sh;
}

__device__ __noinline__ void op_map_remove_far(const MapView &m_in, const V3 &origin_in) {
    const MapView m = m_in;
    const V3 origin = origin_in;
    const double max_d2 = m.max_distance * m.max_distance;
    const size_t cap3 = static_cast<size_t>(m.cap) * 3;
    // The test is on voxel_points.front() (:125-126), which lives in the sparse point blocks (one 32-B sector per
    // voxel). That point lies inside its voxel, so the slot's key alone decides all voxels except the one-voxel
    // shell around the sphere: box corners farthest from / nearest to the origin bound the distance. The box is
    // widened by 1e-6 voxels so that rounding in PointToVoxel's division can never put the point outside it.
    const double v = m.voxel_size, slack = 1e-6 * v;
    const unsigned stride = gridDim.x * BLOCK;
    constexpr int EV_U = 4;  // independent slot loads in flight per thread (the scan is L2-latency-bound: 2 -> 4 measured)
    for (unsigned s0 = blockIdx.x * BLOCK + threadIdx.x; s0 <= m.mask; s0 += EV_U * stride) {
        int4 key[EV_U];
        bool in[EV_U];
#pragma unroll
        for (int u = 0; u < EV_U; ++u) {
            const unsigned s = s0 + u * stride;
            in[u] = s <= m.mask;
            key[u] = in[u] ? m.slots[s] : make_int4(0, 0, 0, -1);
        }
#pragma unroll
        for (int u = 0; u < EV_U; ++u) {
            const int w = key[u].w;
            if (!in[u] || w < 0) continue;
            const unsigned s = s0 + u * stride;
            const double lo[3] = {key[u].x * v - slack - origin.x, key[u].y * v - slack - origin.y, key[u].z * v - slack - origin.z};
            double far2 = 0.0, near2 = 0.0;
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                const double hi = lo[a] + v + 2.0 * slack;
                const double f = fmax(fabs(lo[a]), fabs(hi));
                const double n = (lo[a] > 0.0) ? lo[a] : ((hi < 0.0) ? -hi : 0.0);
                far2 += f * f;
                near2 += n * n;
            }
            bool remove;
            if (far2 < max_d2) {
                continue;  // the whole voxel is inside the sphere
            } else if (near2 >= max_d2) {
                remove = true;  // the whole voxel is outside
            } else {
                const double *vp = m.points + s * cap3;
                const V3 pt{vp[0], vp[1], vp[2]};
                remove = sqnorm(pt - origin) >= max_d2;
            }
            if (remove) {
                m.slots[s].w = KB_TOMB;
                atomicSub(&m.counters[C_LIVE], 1);
                atomicAdd(&m.counters[C_TOMB], 1);
                atomicSub(&m.counters[C_POINTS], w);
            }
        }
    }
}

}  // namespace kb
