// __global__ entry points. Cooperative (persistent-grid) kernels take one parameter struct by
// value; see device_ops.cuh for the ops and the data layout.
#pragma once

#include "device_ops.cuh"
#include "icp_team.cuh"

namespace kb {

// state of one kiss_icp::pipeline::KissICP instance, resident in HBM (KissICP.hpp:87-95)
struct PipeState {
    SE3 last_pose;
    SE3 last_delta;
    double model_sse;  // AdaptiveThreshold::model_sse_   Threshold.hpp:45
    int num_samples;   // AdaptiveThreshold::num_samples_ Threshold.hpp:46
    int vetoed;        // set by a frame that found the voxel table too small: frames already queued behind it
                       // must not run on the stale state, they return ST_SKIPPED until the host has grown the table
    long long front_id;  // id of the frame whose preprocessed / downsampled clouds are in Workspace::fr[id & 1]
                         // (written by the launch that prefetched them), -1: none
};

// what the host reads back after every RegisterFrame (one small D2H)
struct FrameResult {
    double pose[16];   // row-major new pose
    double delta[16];  // row-major last_delta
    double sigma;      // adaptive threshold used for this frame
    double model_sse;
    int num_samples;
    int iterations;
    int n_pre, n_ds, n_src;
    int map_live, map_tomb, map_points, map_status;
    int team;          // CTAs of the ICP team (0: the whole-grid loop ran)
    double icp_candidates;  // map points examined by all ICP iterations of this frame
    double icp_queries;     // GetClosestNeighbor calls (iterations x source points)
    double cache_stats[3];  // NN-cache hits / fills / overflows over all iterations
    unsigned long long t_ns[20];  // %globaltimer at phase boundaries (CTA 0): start, pre, ds1, ds2, icp, map, end
};

// output of the front end of one frame (Preprocess + Voxelize, KissICP.cpp:38,41): two sets, so that the next
// frame's front end can be computed while this frame is still being registered
struct Front {
    double *pre;  // [n][3] preprocessed frame
    double *ds1;  // [n][3] frame_downsample (0.5 v)
    double *src;  // [n][3] source (1.5 v)
    int *cnt;     // [4] n_pre, n_ds, n_src
};

struct Workspace {
    double *tmp;    // [n][3] deskewed points
    Front fr[2];    // by frame id parity
    double *work;   // [n][3] source in the map frame (ICP iterate of the whole-grid loop)
    double *tp;     // [n][3] points being inserted, map frame
    int *next;      // [n] pending-list links
    int *touched;   // [n] voxels touched by the current AddPoints
    DsScratch ds;    // [pow2 >= 2n] downsample scratch tables (0.5 v pass)
    DsScratch ds2;   // second set for the 1.5 v pass (both are cleared during preprocessing)
};

struct FrameParams {
    MapView m;
    Scratch sc;
    TeamScratch team;
    Workspace ws;
    PipeState *st;
    FrameResult *res;
    const double *in;
    const double *ts;
    int n, n_ts;
    int in_f32;  // the frame is float[n][3] instead of double[n][3]
    long long id;  // frame id (monotonic per pipeline; a frame replayed after a capacity veto keeps its id)
    // the frame after this one, when the caller already has it on the device (kb_pipeline_register_frames) and its
    // front end does not depend on this frame's result (no timestamps to deskew with): its preprocessing and
    // downsampling run on the CTAs the ICP team leaves idle. next_in == nullptr: none.
    const double *next_in;
    int next_n, next_in_f32;
    int deskew;
    double max_range, min_range, voxel_size;
    int max_iter;
    double conv, min_motion_th;
    int icp_team_q;  // source points per CTA of the ICP team; 0: whole-grid loop (op_icp)
    unsigned tag_base;
};

__device__ __forceinline__ void threshold_update(const SE3 &dev, double min_motion_th, double max_range,
                                                 double *sse, int *ns) {
    // AdaptiveThreshold::UpdateModelDeviation  core/Threshold.cpp:38-49
    const double theta = angle_axis_angle(q_to_matrix(dev.q));
    const double delta_rot = 2.0 * max_range * sin(theta / 2.0);
    const double delta_trans = norm(dev.t);
    const double model_error = delta_trans + delta_rot;
    if (model_error > min_motion_th) {
        *sse += model_error * model_error;
        *ns += 1;
    }
}

#define KB_STAMP(i) \
    if (P.sc.profile && blockIdx.x == 0 && threadIdx.x == 0) P.res->t_ns[i] = globaltimer_ns()

extern __shared__ __align__(16) unsigned char kb_dyn_smem[];  // QCache[NWARPS][QC_SLOTS] (op_icp) or the TeamSmem layout (op_icp_team)

// Preprocess + Voxelize of one frame on the CTAs of `g` (the whole launch, or the front-end team), KissICP.cpp:38,41,70-75.
// Three barriers of `g` inside; the caller provides the one behind it. No timestamps => `motion` is not used.
__device__ __noinline__ void op_front(Grid &g, const Scratch &sc, Shared &sh, const Workspace &ws, const Front &fr,
                                      const double *in, int n, const double *ts, int n_ts, bool deskew, const SE3 &motion,
                                      double max_range, double min_range, double voxel_size, bool in_f32,
                                      unsigned long long *t_ns /* stamps of the profiled launch or nullptr */) {
    // the downsample scratch tables of both passes are cleared here, under the preprocess barriers
    ds_clear(g, ws.ds, n);
    ds_clear(g, ws.ds2, n);
    op_preprocess(g, sc, sh, in, n, ts, n_ts, deskew, motion, max_range, min_range, ws.tmp, fr.pre, &fr.cnt[0], in_f32);
    g.sync();
    if (t_ns && g.rank == 0 && threadIdx.x == 0) t_ns[1] = globaltimer_ns();
    const int n_pre = __ldcg(&fr.cnt[0]);
    op_downsample(g, sc, sh, fr.pre, n_pre, voxel_size * 0.5, ws.ds, fr.ds1, &fr.cnt[1], t_ns ? &t_ns[12] : nullptr, true);
    g.sync();
    if (t_ns && g.rank == 0 && threadIdx.x == 0) t_ns[2] = globaltimer_ns();
    const int n_ds = __ldcg(&fr.cnt[1]);
    op_downsample(g, sc, sh, fr.ds1, n_ds, voxel_size * 1.5, ws.ds2, fr.src, &fr.cnt[2], t_ns ? &t_ns[16] : nullptr, true);
}

// ---- KissICP::RegisterFrame (pipeline/KissICP.cpp:35-68) as ONE persistent kernel ----------
//   [front end of this frame, unless a previous launch prefetched it]
//   capacity check | fill pass (all CTAs) | ICP iterations on the team  ||  front end of the NEXT frame on the rest
//   map update (all CTAs) | epilogue
__global__ void __launch_bounds__(BLOCK, 1) k_register_frame(const FrameParams P) {
    __shared__ Shared sh;
    Grid g;
    g.init(P.sc.bar);
    KB_STAMP(0);
    const SE3 last_pose = P.st->last_pose;
    const SE3 last_delta = P.st->last_delta;
    const double model_sse = P.st->model_sse;
    const int num_samples = P.st->num_samples;
    const long long front_id = P.st->front_id;
    if (P.st->vetoed) {  // written only by an EARLIER launch: uniform across the grid
        if (blockIdx.x == 0 && threadIdx.x == 0) P.res->map_status = ST_SKIPPED;
        g.finish();
        return;
    }
    const Front fr = P.ws.fr[P.id & 1];
    kb_mark(0x100u + (static_cast<unsigned>(P.id) & 0xffu) * 0x10000u);
    if (front_id != P.id) {  // uniform: written only by an earlier launch
        op_front(g, P.sc, sh, P.ws, fr, P.in, P.n, P.ts, P.n_ts, P.deskew != 0, last_delta, P.max_range, P.min_range,
                 P.voxel_size, P.in_f32 != 0, P.sc.profile ? P.res->t_ns : nullptr);
        g.sync();
    } else if (P.sc.profile && blockIdx.x == 0 && threadIdx.x == 0) {
        P.res->t_ns[1] = P.res->t_ns[2] = globaltimer_ns();  // front end prefetched by the previous launch
    }
    KB_STAMP(3);
    const int n_pre = __ldcg(&fr.cnt[0]), n_ds = __ldcg(&fr.cnt[1]), n_src = __ldcg(&fr.cnt[2]);
    // optimistic table capacity: the host sized the voxel table for the EXPECTED number of new voxels. If this
    // frame could push the load factor beyond 0.5, nothing has been modified yet: report and let the host grow
    // the table and replay the frame (rare; first frames of a sequence). The frame's front end stays valid.
    {
        const long long need = static_cast<long long>(__ldcg(&P.m.counters[C_LIVE])) + __ldcg(&P.m.counters[C_TOMB]) + n_ds;
        if (need * 2 > static_cast<long long>(P.m.mask) + 1) {
            if (blockIdx.x == 0 && threadIdx.x == 0) {
                P.res->map_status = ST_NEED_GROW;
                P.res->n_ds = n_ds;
                P.st->vetoed = 1;     // every CTA read it before the first grid barrier
                P.st->front_id = P.id;  // fr[id & 1] holds this frame's front end: the replay skips it
            }
            g.finish();
            return;  // uniform across the grid
        }
    }
    kb_mark(0x200u);
    // sigma, initial guess (KissICP.cpp:44,47)
    const double sigma = sqrt(model_sse / num_samples);
    const SE3 guess = se3_mul(last_pose, last_delta);
    // ICP (KissICP.cpp:50-54)
    const int G = static_cast<int>(gridDim.x);
    const bool icp_runs = __ldcg(&P.m.counters[C_LIVE]) != 0 && P.max_iter > 0;  // voxel_map.Empty() -> initial_guess
    int T = 0;
    if (icp_runs && P.icp_team_q > 0 && P.m.cap <= NN_FLAT_CAP && (static_cast<unsigned long long>(P.m.mask) + 1) * P.m.cap < (1ull << 31)) {
        T = icp_team_size(n_src, P.icp_team_q, G, P.team.smem_bytes);
    }
    if (T > 0) {
        if (P.sc.profile && blockIdx.x == 0 && threadIdx.x == 0) P.sc.dbg[30] = globaltimer_ns();
        icp_fill_pass(g, sh, P.m, fr.src, n_src, guess, P.team.qrec, P.team.radius_frac, P.sc.bar + BAR_TICKET);
        if (P.sc.profile && blockIdx.x == 0 && threadIdx.x == 0) P.sc.dbg[31] = globaltimer_ns();
        kb_mark(0x300u);
        g.sync();
        kb_mark(0x400u + static_cast<unsigned>(T));
        if (P.sc.profile && blockIdx.x == 0 && threadIdx.x == 0) P.sc.dbg[32] = P.res->t_ns[7] = globaltimer_ns();
        if (static_cast<int>(blockIdx.x) < T) {
            op_icp_team(P.team, P.sc, sh, P.m, n_src, guess, 3.0 * sigma, sigma, P.max_iter, P.conv,
                        kb_dyn_smem, T, P.tag_base);
            if (blockIdx.x == 0 && threadIdx.x == 0) {
                team_publish(P.team, sh);
                if (P.sc.profile) P.res->t_ns[10] = globaltimer_ns();  // iterations done (team member 0)
            }
        } else if (P.next_in != nullptr && 2 * (G - T) >= G) {
            // the CTAs the team does not need register nothing now: they run the next frame's front end
            Grid gf;
            gf.init_team(P.sc.bar + BAR_TEAM, T, G - T);
            const Front nf = P.ws.fr[(P.id + 1) & 1];
            op_front(gf, P.sc, sh, P.ws, nf, P.next_in, P.next_n, nullptr, 0, false, last_delta, P.max_range, P.min_range,
                     P.voxel_size, P.next_in_f32 != 0, nullptr);
            if (gf.rank == 0 && threadIdx.x == 0) {
                P.st->front_id = P.id + 1;  // visible to the next launch
                if (P.sc.profile) P.res->t_ns[11] = globaltimer_ns();  // (rank 0's own end: the other CTAs may still be emitting)
            }
        }
        kb_mark(0x500u);
        g.sync();
        kb_mark(0x600u);
        if (threadIdx.x == 0) team_collect(P.team, sh);
        __syncthreads();
    } else {
        op_icp(g, P.sc, sh, P.m, fr.src, P.ws.work, n_src, guess, 3.0 * sigma, sigma, P.max_iter, P.conv,
               reinterpret_cast<QCache *>(kb_dyn_smem), P.tag_base);
    }
    const SE3 new_pose = sh.result;
    const int iters = sh.iters;
    const double icp_cand = sh.cand_total, icp_q = sh.query_total;
    const double cs0 = sh.cache_stats[0], cs1 = sh.cache_stats[1], cs2 = sh.cache_stats[2];
    KB_STAMP(4);
    // Bookkeeping (KissICP.cpp:57-63: model deviation, threshold, delta, pose) is ~6 us of single-thread FP64
    // math; it only needs new_pose, so one thread of the LAST CTA does it now, hidden behind the map update's
    // first phase (that thread owns no insert work), instead of serially after the map update.
    // The pipeline state itself is stored after the last barrier: with a prefetched front end and no ICP (empty
    // map) there may be no barrier between the slowest CTA's read of the state and this point.
    const bool book = (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0);
    double sse = model_sse;
    int ns = num_samples;
    SE3 delta = last_delta;
    if (book) {
        const SE3 dev = se3_mul(se3_inverse(guess), new_pose);
        threshold_update(dev, P.min_motion_th, P.max_range, &sse, &ns);
        delta = se3_mul(se3_inverse(last_pose), new_pose);
        FrameResult *r = P.res;
        se3_to_matrix(new_pose, r->pose);
        se3_to_matrix(delta, r->delta);
        r->sigma = sigma;
        r->model_sse = sse;
        r->num_samples = ns;
        r->iterations = iters;
        r->icp_queries = icp_q;
        r->n_pre = n_pre;
        r->n_ds = n_ds;
        r->n_src = n_src;
        r->team = T;
        r->icp_candidates = icp_cand;
        r->cache_stats[0] = cs0;
        r->cache_stats[1] = cs1;
        r->cache_stats[2] = cs2;
    }
    // local_map_.Update(frame_downsample, new_pose) (KissICP.cpp:61)
    op_map_add(g, sh, P.m, fr.ds1, n_ds, true, new_pose, P.ws.tp, P.ws.next, P.ws.touched, P.sc.profile ? &P.res->t_ns[8] : nullptr);
    kb_mark(0x700u);
    op_map_remove_far(P.m, new_pose.t);
    kb_mark(0x800u);
    g.sync();
    kb_mark(0x900u);
    KB_STAMP(5);
    if (book) {
        P.st->model_sse = sse;
        P.st->num_samples = ns;
        P.st->last_delta = delta;
        P.st->last_pose = new_pose;
        FrameResult *r = P.res;
        r->map_live = P.m.counters[C_LIVE];
        r->map_tomb = P.m.counters[C_TOMB];
        r->map_points = P.m.counters[C_POINTS];
        r->map_status = P.m.counters[C_STATUS];
        if (P.sc.profile) r->t_ns[6] = globaltimer_ns();
    }
    g.finish();
}

// ---- _correct_kitti_scan (kiss_icp_pybind.cpp:127-138): one point per thread, 24 B in + 24 B out, HBM-bound ----
__global__ void __launch_bounds__(256) k_correct_kitti(const double *in, double *out, size_t n, double sn, double cs) {
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const V3 p = correct_kitti_point(V3{in[3 * i], in[3 * i + 1], in[3 * i + 2]}, sn, cs);
        out[3 * i] = p.x;
        out[3 * i + 1] = p.y;
        out[3 * i + 2] = p.z;
    }
}

// ---- stand-alone wrappers (module-level API) -------------------------------------------------
struct PreParams {
    Scratch sc;
    const double *in;
    const double *ts;
    int n, n_ts, deskew;
    SE3 motion;
    double max_range, min_range;
    double *tmp, *out;
    int *out_n;
};
__global__ void __launch_bounds__(BLOCK, 1) k_preprocess(const PreParams P) {
    __shared__ Shared sh;
    Grid g;
    g.init(P.sc.bar);
    op_preprocess(g, P.sc, sh, P.in, P.n, P.ts, P.n_ts, P.deskew != 0, P.motion, P.max_range, P.min_range, P.tmp,
                  P.out, P.out_n);
}

struct DsParams {
    Scratch sc;
    const double *in;
    int n;
    double voxel_size;
    DsScratch ds;
    double *out;
    int *out_n;
    // optional second stage (Voxelize): out2 = downsample(out, voxel_size2)
    double voxel_size2;
    double *out2;
    int *out_n2;
};
__global__ void __launch_bounds__(BLOCK, 1) k_downsample(const DsParams P) {
    __shared__ Shared sh;
    Grid g;
    g.init(P.sc.bar);
    op_downsample(g, P.sc, sh, P.in, P.n, P.voxel_size, P.ds, P.out, P.out_n);
    if (P.out2) {
        g.sync();
        const int n1 = __ldcg(P.out_n);
        op_downsample(g, P.sc, sh, P.out, n1, P.voxel_size2, P.ds, P.out2, P.out_n2);
    }
}

struct IcpParams {
    MapView m;
    Scratch sc;
    const double *src;
    double *work;
    int n;
    SE3 guess;
    double max_dist, kscale;
    int max_iter;
    double conv;
    double *out_pose;  // [16] row-major
    int *out_iters;
    // build-system-only mode (one pass, no solve): out_sys[NACC], out_ncorr
    int system_only;
    double *out_sys;
    int *out_ncorr;
    unsigned tag_base;
    TeamScratch team;
    int icp_team_q;  // source points per CTA of the ICP team; 0: whole-grid loop
};
__global__ void __launch_bounds__(BLOCK, 1) k_icp(const IcpParams P) {
    __shared__ Shared sh;
    Grid g;
    g.init(P.sc.bar);
    if (P.system_only) {
        icp_queries(P.sc, sh, P.m, P.src, P.work, P.n, se3_identity(), P.max_dist, P.kscale, P.tag_base + 1u, false,
                    nullptr, true);
        icp_gather(P.sc, sh, P.tag_base + 1u, icp_group_size());
        if (blockIdx.x == 0) {
            if (threadIdx.x == 0) {
                for (int i = 0; i < NACC; ++i) P.out_sys[i] = sh.red[i];
                *P.out_ncorr = static_cast<int>(sh.red[NACC]);
            }
        }
        return;
    }
    int T = 0;
    if (__ldcg(&P.m.counters[C_LIVE]) != 0 && P.max_iter > 0 && P.icp_team_q > 0 && P.m.cap <= NN_FLAT_CAP &&
        (static_cast<unsigned long long>(P.m.mask) + 1) * P.m.cap < (1ull << 31)) {
        T = icp_team_size(P.n, P.icp_team_q, static_cast<int>(gridDim.x), P.team.smem_bytes);
    }
    if (T > 0) {
        icp_fill_pass(g, sh, P.m, P.src, P.n, P.guess, P.team.qrec, P.team.radius_frac, P.sc.bar + BAR_TICKET);
        g.sync();
        if (static_cast<int>(blockIdx.x) >= T) return;
        op_icp_team(P.team, P.sc, sh, P.m, P.n, P.guess, P.max_dist, P.kscale, P.max_iter, P.conv,
                    kb_dyn_smem, T, P.tag_base);
    } else {
        op_icp(g, P.sc, sh, P.m, P.src, P.work, P.n, P.guess, P.max_dist, P.kscale, P.max_iter, P.conv,
               reinterpret_cast<QCache *>(kb_dyn_smem), P.tag_base);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        se3_to_matrix(sh.result, P.out_pose);
        *P.out_iters = sh.iters;
    }
}

struct MapUpdParams {
    MapView m;
    Scratch sc;
    const double *pts;
    int n;
    int has_pose;
    SE3 pose;
    int do_add, do_remove;
    V3 origin;
    double *tp;
    int *next;
    int *touched;
};
__global__ void __launch_bounds__(BLOCK, 1) k_map_update(const MapUpdParams P) {
    __shared__ Shared sh;
    Grid g;
    g.init(P.sc.bar);
    if (P.do_add) op_map_add(g, sh, P.m, P.pts, P.n, P.has_pose != 0, P.pose, P.tp, P.next, P.touched);
    if (P.do_remove) op_map_remove_far(P.m, P.origin);
}

// profiling aid: cost of the grid barrier itself
__global__ void __launch_bounds__(BLOCK, 1) k_barrier_bench(const Scratch sc, int iters) {
    Grid g;
    g.init(sc.bar);
    g.sync();
    if (blockIdx.x == 0 && threadIdx.x == 0) sc.dbg[8] = globaltimer_ns();
    for (int i = 0; i < iters; ++i) g.sync();
    if (blockIdx.x == 0 && threadIdx.x == 0) sc.dbg[9] = globaltimer_ns();
}

// table initialisation / clear
__global__ void k_map_fill(int4 *slots, int *head, int *pcount, size_t capacity) {
    const int4 empty = make_int4(-1, -1, -1, KB_EMPTY);
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < capacity;
         i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        slots[i] = empty;
        head[i] = -1;
        pcount[i] = 0;
    }
}

// rebuild into a larger / tombstone-free table: every live voxel moves with its block
__global__ void k_map_rehash(const MapView from, const MapView to) {
    const int lane = threadIdx.x & 31;
    const size_t gw = (blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x) >> 5;
    const size_t nw = (static_cast<size_t>(gridDim.x) * blockDim.x) >> 5;
    const size_t cap3 = static_cast<size_t>(from.cap) * 3;
    for (size_t s = gw; s <= from.mask; s += nw) {
        const int4 e = from.slots[s];
        if (e.w < 0) continue;
        int d = 0;
        if (lane == 0) d = map_find_or_claim(to, e.x, e.y, e.z);
        d = __shfl_sync(FULL, d, 0);
        if (d < 0) continue;
        const double *a = from.points + s * cap3;
        double *b = to.points + static_cast<size_t>(d) * cap3;
        for (int k = lane; k < e.w * 3; k += 32) b[k] = a[k];
        if (lane == 0) {
            to.slots[d].w = e.w;
            atomicAdd(&to.counters[C_POINTS], e.w);
        }
    }
}

// batched GetClosestNeighbor (VoxelHashMap.cpp:46-70): one warp per query, grid-stride.
// Bandwidth-bound at scale (BASELINE config 5): every query is three dependent DRAM round trips
// (query, 27 slot probes, candidate blocks), so the kernel is built for memory-level parallelism:
// <= 64 registers (4 CTAs of 256 threads = 32 warps per SM) and the NEXT query's point and first
// probe are issued before the current query's candidates are reduced.
struct NNProbe {
    V3 q;
    int3 v;
    unsigned h;  // first bucket of this lane's neighbour voxel
    int4 s;      // that bucket
};

__device__ __forceinline__ void nn_issue(const MapView &m, const double *__restrict__ q, size_t i, int lane, NNProbe &pr) {
    pr.q = V3{q[3 * i], q[3 * i + 1], q[3 * i + 2]};
    pr.v = point_to_voxel(pr.q.x, pr.q.y, pr.q.z, m.vdiv);
    if (lane < 27) {
        pr.h = mix_hash(pr.v.x + c_shifts[lane][0], pr.v.y + c_shifts[lane][1], pr.v.z + c_shifts[lane][2]) & m.mask;
        pr.s = m.slots[pr.h];
    }
}

// finish the probe started by nn_issue (collision chain), then gather + reduce exactly like nn_search_warp
__device__ __forceinline__ NNResult nn_finish(const MapView &m, const NNProbe &pr, int lane, WarpNN &w) {
    int cnt = 0, slot = -1;
    if (lane < 27)
        slot = map_find_from(m, pr.v.x + c_shifts[lane][0], pr.v.y + c_shifts[lane][1], pr.v.z + c_shifts[lane][2], pr.h,
                             pr.s, &cnt);
    if (m.cap <= NN_FLAT_CAP) return nn_flat_search(m, pr.q, lane, w, cnt, slot);
    return nn_walk_voxels(m, pr.q, lane, cnt, slot);
}

template <bool COUNT>
__global__ void __launch_bounds__(256, 4) k_nn_query(const MapView m, const double *__restrict__ q, size_t n,
                                                     double *__restrict__ out_p, double *__restrict__ out_d,
                                                     unsigned long long *cand_total) {
    __shared__ WarpNN wnn[8];  // blockDim.x == 256
    const int lane = threadIdx.x & 31;
    const size_t gw = (blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x) >> 5;
    const size_t nw = (static_cast<size_t>(gridDim.x) * blockDim.x) >> 5;
    unsigned long long cand = 0;
    NNProbe cur, nxt;
    if (gw < n) nn_issue(m, q, gw, lane, cur);
    for (size_t i = gw; i < n; i += nw) {
        const bool more = i + nw < n;
        if (more) nn_issue(m, q, i + nw, lane, nxt);  // next query's loads fly while this one is reduced
        const NNResult r = nn_finish(m, cur, lane, wnn[threadIdx.x >> 5]);
        if (lane == 0) {
            out_p[3 * i] = r.p.x;
            out_p[3 * i + 1] = r.p.y;
            out_p[3 * i + 2] = r.p.z;
            out_d[i] = r.d;
        }
        if (COUNT) cand += r.candidates;
        if (more) cur = nxt;
    }
    if (COUNT && lane == 0 && cand) atomicAdd(cand_total, cand);
}

// export of live voxels (checkpoint / Pointcloud / tests): ordered two-pass compaction by slot
struct ExportParams {
    MapView m;
    Scratch sc;
    int4 *vox_out;    // {x,y,z,count}
    double *pts_out;  // concatenated per-voxel points, slot order
    int *totals;      // [2] voxels, points
};
__global__ void __launch_bounds__(BLOCK, 1) k_map_export(const ExportParams P) {
    __shared__ Shared sh;
    __shared__ int s_scan[BLOCK];
    Grid g;
    g.init(P.sc.bar);
    long long lo, hi;
    chunk_of(g, static_cast<long long>(P.m.mask) + 1, &lo, &hi);
    int nv = 0, np = 0;
    for (long long i = lo + threadIdx.x; i < hi; i += BLOCK) {
        const int w = P.m.slots[i].w;
        if (w >= 0) {
            ++nv;
            np += w;
        }
    }
    const int bnv = block_sum(nv, sh.warp_i);
    const int bnp = block_sum(np, sh.warp_i);
    if (threadIdx.x == 0) {
        P.sc.blk_i[blockIdx.x] = bnv;
        P.sc.blk_i[gridDim.x + blockIdx.x] = bnp;
    }
    g.sync();
    int voff, vtot, poff, ptot;
    grid_offsets(g, P.sc.blk_i, &voff, &vtot, sh.two);
    grid_offsets(g, P.sc.blk_i + gridDim.x, &poff, &ptot, sh.two);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        P.totals[0] = vtot;
        P.totals[1] = ptot;
    }
    if (P.vox_out == nullptr) return;  // count-only call
    const size_t cap3 = static_cast<size_t>(P.m.cap) * 3;
    for (long long base = lo; base < hi; base += BLOCK) {
        const long long i = base + threadIdx.x;
        int4 e = make_int4(0, 0, 0, -1);
        if (i < hi) e = P.m.slots[i];
        const int live = e.w >= 0 ? 1 : 0;
        int tile_v;
        const int vrank = block_rank(live, &tile_v, sh.warp_i);
        // exclusive scan of point counts over the tile
        __syncthreads();
        s_scan[threadIdx.x] = live ? e.w : 0;
        __syncthreads();
        for (int o = 1; o < BLOCK; o <<= 1) {
            const int v = threadIdx.x >= o ? s_scan[threadIdx.x - o] : 0;
            __syncthreads();
            s_scan[threadIdx.x] += v;
            __syncthreads();
        }
        const int incl = s_scan[threadIdx.x];
        const int tile_p = s_scan[BLOCK - 1];
        if (live) {
            P.vox_out[voff + vrank] = e;
            const double *a = P.m.points + static_cast<size_t>(i) * cap3;
            double *b = P.pts_out + static_cast<size_t>(poff + incl - e.w) * 3;
            for (int k = 0; k < e.w * 3; ++k) b[k] = a[k];
        }
        voff += tile_v;
        poff += tile_p;
        __syncthreads();
    }
}

}  // namespace kb
