// Registration::AlignPointsToMap (core/Registration.cpp:138-167) on a TEAM of CTAs.
//
// Why: the loop is a dependent chain of ~18 iterations per scan. In op_icp (device_ops.cuh) every
// iteration crosses the whole 148-CTA grid three times (partials -> group leaders -> coordinator ->
// everybody, ~1.2 us per L2 hop) for ~1 us of useful work, and 15 of 16 warps of every SM wait. Here
//   * ONE pass over the map per scan (icp_fill_pass, every CTA of the launch, one warp per source point)
//     runs the 27-voxel search of GetClosestNeighbor (core/VoxelHashMap.cpp:46-70) and leaves, per point, the
//     short list of map points that can still become its nearest neighbour while it moves by <= R
//     (exactness argument: QCache in device_ops.cuh);
//   * the iterations then run on a small team (T = ceil(n / 80) CTAs, 31 for a KITTI scan): four lanes per source
//     point walk its list — candidate COORDINATES staged in shared memory, interleaved so that the walk is
//     bank-conflict free — and the T partial systems meet in ONE all-gather of epoch-tagged
//     16-byte chunks: every team CTA polls all T partials, adds them in the same fixed order and solves the
//     6x6 itself, so there is no coordinator, no broadcast hop and one L2 round trip per iteration;
//   * the rest of the launch (the other ~117 SMs) is free meanwhile: k_register_frame runs the NEXT scan's
//     preprocessing and voxel downsampling on it.
// A point whose list is no longer valid (moved > R, or left its voxel) is searched again by its whole warp
// inside the iteration (nn_search_list), exactly like the first time.
#pragma once

#include "device_ops.cuh"

namespace kb {

constexpr int TEAM_MAX = 96;    // CTAs of an ICP team (the gathered partials, 21 x TEAM_MAX doubles, fit the 16 KB reduction scratch)
static_assert(NPART * TEAM_MAX * 8 <= DS_MAX_CHUNKS * 4, "the gathered partials live in Shared::chunk_pref");
constexpr int TQ_LANES = 4;     // lanes that share one source point in the list walk
constexpr int TQ_PER_WARP = 32 / TQ_LANES;
constexpr int TQ_PER_CTA = 80;  // source points per team CTA by default (10 warps; A/B at KITTI shape: 48 -3 %, 64 0, 80 +1.5 %, 96 +1.3 %)
constexpr int TQ_MAX = 120;     // upper bound of source points per team CTA (warps 0..14; the solver is thread 511)
constexpr int TRED_STRIDE = NACC + 1;  // row of the per-point reduction scratch: 16 entries + the gate flag (odd: conflict-free)
static_assert(TQ_MAX * TRED_STRIDE * 8 <= DS_MAX_CHUNKS * 4, "the reduction scratch lives in Shared::chunk_pref");

// Output of the fill pass for one source point (global memory): the list holds POINT INDICES (slot * cap + k) in the
// reference's visiting order (voxel_shifts order, then insertion order), so the first strict minimum over the
// list is the reference's answer, ties included.
struct QList {
    int count;      // >= 0: idx[0..count) valid; -1: not cacheable (too many candidates)
    int full;       // points of the whole 27-voxel neighbourhood (bookkeeping of algorithmic bytes)
    int vx, vy, vz; // voxel at fill time
    int pad[3];
    double pf[3];   // position at fill time (= initial_guess * source point)
    int idx[QC_MAX];
    int tail[2];    // 320 bytes
};
static_assert(sizeof(QList) % 16 == 0 && sizeof(QList) == sizeof(QListRaw), "QList records are 16-byte aligned; Shared::rlist holds one per warp");

// A source point inside its team CTA (shared memory): state + where its candidate COORDINATES are. A warp owns 8
// points, FOUR lanes per point: lane (q8, j) walks candidates k = j, j + 4, ... The coordinates of a warp's points
// are interleaved — candidate k, component c of point q8 sits in row k / 4, column (4 q8 + k) & 31 of a
// [rows][3][32] block — so that (i) the walk (32 lanes = 8 points x 4 consecutive k of the same row) and (ii) the
// warp that stages one point's list (32 lanes = 32 consecutive k of one point) both hit 32 different banks.
// (Reading the coordinates through L1 instead was measured: every lane's load is its own L1 wavefront and the walk
// alone took 8000 cycles per iteration; one thread per point with this layout: 4500 cycles, a chain of ~30
// candidates per thread.)
struct TQHead {
    int count;      // >= 0: candidates staged; -1: not cacheable (searched again every iteration)
    int full, vx, vy, vz;
    int pad[3];
    double pf[3];   // position when the list was made
    double p[3];    // current position (TransformPoints is applied in place, Registration.cpp:55-58,160)
    double nn[4];   // nearest neighbour and distance found by a re-search inside the iteration
    double pad2;    // 120 bytes
};
static_assert(sizeof(TQHead) == 120, "TQHead layout");

struct TeamSmem {
    TQHead *heads;   // [qmax]
    double *coords;  // [warps][K / 4][3][32]
    int K;           // candidate slots per source point (multiple of 4)
};
// carve the dynamic shared memory of a team CTA for qmax source points
__device__ __forceinline__ TeamSmem team_smem(unsigned char *dyn, int dyn_bytes, int qmax) {
    TeamSmem t;
    const int head_bytes = (qmax * static_cast<int>(sizeof(TQHead)) + 15) & ~15;
    const int warps = (qmax + TQ_PER_WARP - 1) / TQ_PER_WARP;
    t.heads = reinterpret_cast<TQHead *>(dyn);
    t.coords = reinterpret_cast<double *>(dyn + head_bytes);
    t.K = (warps > 0 && dyn_bytes > head_bytes) ? 4 * min(QC_MAX / 4, (dyn_bytes - head_bytes) / (warps * 768)) : 0;
    return t;
}
// (explicit shared-space loads: through the generic pointer the compiler emits LD.E with a branch per candidate)
__device__ __forceinline__ double lds_f64(unsigned addr) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ unsigned tq_coord_addr(unsigned coords_base, int K, int li, int k) {
    return coords_base + (static_cast<unsigned>((li / TQ_PER_WARP) * (K >> 2) + (k >> 2)) * 96u +
                          static_cast<unsigned>((4 * (li & (TQ_PER_WARP - 1)) + k) & 31)) * 8u;
}
// candidate k of source point li: component c at [c * 32]
__device__ __forceinline__ double *tq_coord(const TeamSmem &ts, int li, int k) {
    return ts.coords + (static_cast<size_t>(li / TQ_PER_WARP) * (ts.K >> 2) + (k >> 2)) * 96 + ((4 * (li & (TQ_PER_WARP - 1)) + k) & 31);
}

struct TeamScratch {
    uint4 *ll;        // [2][TEAM_MAX readers][TEAM_MAX members][NPART] epoch-tagged partial systems, ping-pong by iteration parity
    double *out;      // [16] result record: pose(7) iters cand_total query_total cache_stats(3)
    QList *qrec;      // [n] per source point, written by the fill pass
    int smem_bytes;   // dynamic shared memory of the launch
    double radius_frac;  // R / voxel_size: a list stays exact while its point has moved by <= R (shorter lists for smaller R)
};

// team size for n source points at q_per_cta points per CTA; 0 when the lists would not fit in shared memory
__device__ __forceinline__ int icp_team_size(int n, int q_per_cta, int grid, int smem_bytes) {
    q_per_cta = max(1, min(q_per_cta, TQ_MAX));
    const int tmax = min(grid, TEAM_MAX);
    if ((n + q_per_cta - 1) / q_per_cta > tmax) q_per_cta = (n + tmax - 1) / tmax;  // small grid (several pipelines per GPU) / big cloud: fuller CTAs
    if (q_per_cta > TQ_MAX) return 0;
    int T = (n + q_per_cta - 1) / q_per_cta;
    T = max(T, 1);
    const int qmax = (n + T - 1) / T;
    const int head_bytes = (qmax * static_cast<int>(sizeof(TQHead)) + 15) & ~15;
    const int warps = (qmax + TQ_PER_WARP - 1) / TQ_PER_WARP;
    if (warps > 0 && 4 * ((smem_bytes - head_bytes) / (warps * 768)) < 24) return 0;
    return T;
}

// GetClosestNeighbor (core/VoxelHashMap.cpp:46-70) for one point by one warp + the list of candidates that can
// still become its nearest neighbour while it moves by <= R (QCache's exactness argument, device_ops.cuh) into *out
// (generic pointer: global memory in the fill pass, shared memory inside an iteration).
// ONE pass over the neighbourhood: every lane keeps the squared distances and point indices of its <= 8 candidates
// in registers (all loads of the neighbourhood are in flight together: one L2 round trip), the warp takes the
// minimum, and the list is filtered from the registers. Neighbourhoods with more than 256 points take two passes.
// Only for maps with max_points_per_voxel <= NN_FLAT_CAP: the team does not run on others.
constexpr int NNL_R = 8;
__device__ __noinline__ NNResult nn_search_list(const MapView &m, const V3 &q, int lane, WarpNN &w, QList *out,
                                                double cache_radius) {
    const int3 v = point_to_voxel(q.x, q.y, q.z, m.vdiv);
    const NNVoxel nv = nn_probe27(m, v, lane);
    const int cap = m.cap;
    // candidate j (reference order) -> lane j % 32, register j / 32
    const int total = nn_flatten(w, lane, nv.cnt, nv.slot);
    NNResult r;
    int count = 0;  // (an empty neighbourhood stays empty while the point stays in its voxel)
    if (total <= 32 * NNL_R) {
        double d2[NNL_R];
        int gi[NNL_R];
#pragma unroll
        for (int h = 0; h < NNL_R; h += 4) {  // (the loads of both halves are independent: one round trip)
            V3 c[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int j = (h + u) * 32 + lane;
                gi[h + u] = -1;
                if (j < total) {
                    const int vi = w.owner[j];
                    gi[h + u] = w.slot[vi] * cap + (j - w.start[vi]);
                    c[u] = ld_point24(m.points + static_cast<size_t>(gi[h + u]) * 3);
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) d2[h + u] = (gi[h + u] >= 0) ? sqnorm(c[u] - q) : DBL_MAX;
        }
        NNMin a;  // (no points: the winner's is re-read below, it is L1-hot)
#pragma unroll
        for (int u = 0; u < NNL_R; ++u) a.add(d2[u], u * 32 + lane, V3{0, 0, 0});
        if (!nn_reduce_near(a)) {
            V3 bp{0, 0, 0};
            if (total > 0) {
                const int vi = w.owner[a.bseq];
                bp = ld_point24(m.points + static_cast<size_t>(w.slot[vi] * cap + (a.bseq - w.start[vi])) * 3);
            }
            r = NNResult{total > 0 ? sqrt(a.b2) : DBL_MAX, bp, total};
        } else {  // near tie of squared distances: compare rounded roots in reference order, like the reference
            double best = DBL_MAX, best_d2 = DBL_MAX;
            int bseq = INT_MAX;
            V3 bp{0, 0, 0};
#pragma unroll
            for (int u = 0; u < NNL_R; ++u)
                if (gi[u] >= 0) {
                    const double *pp = m.points + static_cast<size_t>(gi[u]) * 3;
                    nn_consider(V3{pp[0], pp[1], pp[2]}, q, u * 32 + lane, best, best_d2, bseq, bp);
                }
            nn_reduce(best, bseq, bp);
            r = NNResult{best, bp, total};
        }
        // the candidates within d* + 2R of the point, in reference order
        if (r.d < DBL_MAX) {
            const double thr2 = nn_keep_thr2(r.d, cache_radius);
#pragma unroll
            for (int u = 0; u < NNL_R; ++u) {
                if (u * 32 < total) {  // warp-uniform
                    const bool keep = d2[u] <= thr2;  // (DBL_MAX where there is no candidate)
                    const int pos = warp_compact(keep, lane, count);
                    if (keep && pos < QC_MAX) out->idx[pos] = gi[u];
                }
            }
        }
    } else {
        r = nn_flat_search_staged(m, q, lane, w, total);
        if (r.d < DBL_MAX) {  // second pass (L1-hot)
            const double thr2 = nn_keep_thr2(r.d, cache_radius);
            constexpr int U2 = 4;
            for (int base = 0; base < total; base += 32 * U2) {
#pragma unroll
                for (int u = 0; u < U2; ++u) {
                    const int j = base + u * 32 + lane;
                    bool keep = false;
                    int g = 0;
                    if (j < total) {
                        const int vi = w.owner[j];
                        g = w.slot[vi] * cap + (j - w.start[vi]);
                        keep = sqnorm(ld_point24(m.points + static_cast<size_t>(g) * 3) - q) <= thr2;
                    }
                    const int pos = warp_compact(keep, lane, count);
                    if (keep && pos < QC_MAX) out->idx[pos] = g;
                }
            }
        }
    }
    if (count > QC_MAX) count = -1;
    if (lane == 0) {
        out->count = count;
        out->full = r.candidates;
        out->vx = v.x;
        out->vy = v.y;
        out->vz = v.z;
        out->pf[0] = q.x;
        out->pf[1] = q.y;
        out->pf[2] = q.z;
    }
    __syncwarp();
    return r;
}

// every CTA of `g`, one warp per source point: source = initial_guess * source (Registration.cpp:146-147),
// 27-voxel search, candidate list -> qrec[point]
// Scheduling: every warp takes point (its index) first; the points beyond one per warp are handed out through a ticket
// counter, so that the ~14 % of warps that would have had a second point by static assignment do not set the length of
// the pass (a point costs ~6 us) — whoever is done first takes the next one. `ticket` is zero at kernel start
// (Grid::finish re-arms it).
__device__ __noinline__ void icp_fill_pass(const Grid &g, Shared &sh, const MapView &m, const double *src, int n,
                                           const SE3 &guess, QList *qrec, double radius_frac, unsigned *ticket) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const double radius = radius_frac * m.voxel_size;
    const int nwarps = g.size * NWARPS;
    int qi = g.rank + g.size * warp;
    while (qi < n) {
        const V3 p = se3_act(guess, V3{src[3 * qi], src[3 * qi + 1], src[3 * qi + 2]});
        nn_search_list(m, p, lane, sh.wnn[warp], &qrec[qi], radius);
        unsigned t = 0;
        if (lane == 0) t = atomicAdd(ticket, 1u);
        qi = nwarps + static_cast<int>(__shfl_sync(FULL, t, 0));
    }
}

// the 16 distinct entries of one correspondence's J^T w J / J^T w r, each formed exactly as Eigen forms
// (J^T * w) * J entry by entry (icp_term's formulas, device_ops.cuh); lane j of the point's four lanes adds
// entries 4 j .. 4 j + 3 to acc
__device__ __forceinline__ void icp_term4(int j, const V3 &s, const V3 &t, double kscale, double acc[4]) {
    const V3 r = s - t;
    const double r2 = sqnorm(r);
    const double w = (kscale * kscale) * fast_rcp((kscale + r2) * (kscale + r2));  // ~1 ulp from the reference's division
    const double xw = s.x * w, yw = s.y * w, zw = s.z * w;
    double a0, a1, a2, a3;
    if (j == 0) {
        a0 = w;
        a1 = xw;
        a2 = yw;
        a3 = zw;
    } else if (j == 1) {
        a0 = zw * s.z + yw * s.y;  // (3,3)
        a1 = -(xw * s.y);          // (4,3)
        a2 = zw * s.z + xw * s.x;  // (4,4)
        a3 = -(xw * s.z);          // (5,3)
    } else if (j == 2) {
        a0 = -(yw * s.z);          // (5,4)
        a1 = yw * s.y + xw * s.x;  // (5,5)
        a2 = w * r.x;
        a3 = w * r.y;
    } else {
        a0 = w * r.z;
        a1 = -(zw * r.y) + yw * r.z;
        a2 = zw * r.x - xw * r.z;
        a3 = -(yw * r.x) + xw * r.y;
    }
    acc[0] += a0;
    acc[1] += a1;
    acc[2] += a2;
    acc[3] += a3;
}

// stage one source point's candidate list (indices -> coordinates) into the interleaved block of its owner warp;
// called by a whole warp. Lists longer than the K staged slots are not cacheable.
__device__ __forceinline__ void team_stage(const TeamSmem &sm, const MapView &m, int li, const QList *src, int lane) {
    int cnt = src->count;
    if (cnt > sm.K) cnt = -1;
    for (int k = lane; k < cnt; k += 32) {
        const V3 c = ld_point24(m.points + static_cast<size_t>(src->idx[k]) * 3);
        double *dst = tq_coord(sm, li, k);
        dst[0] = c.x;
        dst[32] = c.y;
        dst[64] = c.z;
    }
    if (lane == 0) {
        TQHead &h = sm.heads[li];
        h.count = cnt;
        h.full = src->full;
        h.vx = src->vx;
        h.vy = src->vy;
        h.vz = src->vz;
        h.pf[0] = src->pf[0];
        h.pf[1] = src->pf[1];
        h.pf[2] = src->pf[2];
    }
}

// T_icp = estimation * T_icp (Registration.cpp:161) + work counters of the iteration that was just solved. Run by the
// solver thread (BLOCK - 1, its warp owns no source point) while the other warps walk their lists for the NEXT iteration.
__device__ __noinline__ void team_accumulate(Shared &sh) {
    sh.t_icp = se3_mul_fast(sh.pending, sh.t_icp);
    sh.cand_total += sh.red[NACC + 1];
    for (int i = 0; i < 3; ++i) sh.cache_stats[i] += sh.red[NACC + 2 + i];
}

// COLD paths of the iteration live in their own functions: the loop is a latency chain executed by a handful of
// warps, and every instruction-cache line it has to skip over or fetch is paid in full (the iteration's code was
// spread over ~80 KB before this split and ran at ~15 cycles per instruction in its straight-line parts).

// two squared distances within a few ulps could round to the same root: compare rounded roots in reference order like
// GetClosestNeighbor does (whole warp calls; lanes with `near` redo their point's list)
__device__ __noinline__ void tq_exact_nn(const TeamSmem sm, int li, int l4, int cnt, bool near, double px, double py, double pz) {
    const V3 p{px, py, pz};
    double best = DBL_MAX;
    int ek = INT_MAX;
    if (near)
        for (int k = l4; k < cnt; k += TQ_LANES) {
            const double *src = tq_coord(sm, li, k);
            const double dd = norm(V3{src[0], src[32], src[64]} - p);
            if (dd < best) {
                best = dd;
                ek = k;
            }
        }
#pragma unroll
    for (int o = 1; o < TQ_LANES; o <<= 1) {
        const double ob = __shfl_xor_sync(FULL, best, o);
        const int ok2 = __shfl_xor_sync(FULL, ek, o);
        if ((ob < best) || (ob == best && ok2 < ek)) {
            best = ob;
            ek = ok2;
        }
    }
    if (near && l4 == 0) {  // the answer goes through the point's header (out-pointers would put the caller's d / np in local memory)
        const double *src = tq_coord(sm, li, ek);
        TQHead &h = sm.heads[li];
        h.nn[0] = src[0];
        h.nn[1] = src[32];
        h.nn[2] = src[64];
        h.nn[3] = best;
    }
    __syncwarp();
}

// the stale points of this iteration (queue sh.refill_q) are searched again by all warps of the CTA and their lists
// staged again; the threads that own such a point get its answer
__device__ __noinline__ void team_refill(Shared &sh, const MapView &m, const TeamSmem sm, int nref, int par, double radius) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int r = warp; r < nref; r += NWARPS) {
        const int rl = sh.refill_q[r];
        TQHead &h = sm.heads[rl];
        const V3 pq{h.p[0], h.p[1], h.p[2]};
        QList *scratch = reinterpret_cast<QList *>(&sh.rlist[warp]);
        const NNResult res = nn_search_list(m, pq, lane, sh.wnn[warp], scratch, radius);
        team_stage(sm, m, rl, scratch, lane);
        if (lane == 0) {
            h.nn[0] = res.p.x;
            h.nn[1] = res.p.y;
            h.nn[2] = res.p.z;
            h.nn[3] = res.d;
            if ((scratch->count < 0 || scratch->count > sm.K) && res.d < DBL_MAX) atomicAdd(&sh.refill_over[par], 1);
        }
        __syncwarp();
    }
    __syncthreads();
}

// (Tried: keeping the four warps of the solver's scheduler free of source points so that the solver finds its code in that
// scheduler's instruction cache - no effect, 4683 vs 4705 scans/s.)
// (Tried: running the solver's code once early per iteration on an idle thread of the same scheduler, outputs discarded, to
// warm the instruction cache for the real run - slower, 4402 vs 4510 scans/s: the solve is not fetch-bound.)
// cycle stamps inside the iteration: only in a profiling build (-DKB_PROFILE_TEAM). The iteration's code must stay small:
// it is executed once per iteration by warps that are at different places, i.e. the instruction cache sees a cyclic
// sweep over the whole loop body, and a body larger than the cache misses on every line (measured: 36 KB of loop body
// ran at 7-15 cycles per instruction whatever the data was).
#ifdef KB_PROFILE_TEAM
#define KB_WCYC(i) \
    if (dbg != nullptr && threadIdx.x == 0) dbg[24 + (i)] = static_cast<unsigned long long>(clock64())
#define KB_TCYC(i) \
    if (dbg != nullptr && threadIdx.x == 0) dbg[16 + (i)] = static_cast<unsigned long long>(clock64())
#else
#define KB_WCYC(i)
#define KB_TCYC(i)
#endif

// DataAssociation + BuildLinearSystem (Registration.cpp:60-121) for this CTA's source points, iteration j. The loop is a
// dependent chain, so what counts is the length of the per-point instruction chain: four lanes share a point (8
// points per warp), each walks a quarter of the candidate list from conflict-free shared memory, two shuffle levels
// merge them, and the 16 accumulators are split over the four lanes (one 3-level shuffle sum per warp).
//
// When is the staged list still exact? Let p_f be where it was made (d* the nearest distance then, the list = all
// points of the 27 voxels around p_f within d* + 2R of p_f), p the current position with |p - p_f| <= R, and d_S the
// smallest distance from p to the list. A point x of the CURRENT 27-voxel neighbourhood that is not in the list is
// either in the old neighbourhood, then |x - p_f| > d* + 2R and |x - p| > d* + R >= d_S; or outside it, then
// |x - p_f| >= voxel_size and |x - p| >= voxel_size - R. So the list answers exactly when the voxel is unchanged, or
// when d_S < voxel_size - R (its minimiser is then within one voxel of p, i.e. inside the current neighbourhood).
// Otherwise (moved > R, or a far match that changed voxel) the point is queued and searched again by a whole warp —
// ALL warps of the CTA serve that queue.
__device__ __forceinline__ void team_queries(uint4 *ll, Shared &sh, const MapView &m, const TeamSmem sm, const VoxelDiv vdiv, double radius_frac, int nq, int j,
                                          double max_dist, double kscale, int member, int T, unsigned tag,
                                          unsigned long long *dbg) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int l4 = lane & (TQ_LANES - 1), li = tid / TQ_LANES;
    const double voxel_size = vdiv.v;
    const double radius = radius_frac * voxel_size, r2max = radius * radius;
    const bool have = li < nq;
    const int par = j & 1;
    double *red = reinterpret_cast<double *>(sh.chunk_pref);  // [TQ_MAX][TRED_STRIDE], free during the ICP
    if (tid == BLOCK - 1 && j > 0) team_accumulate(sh);  // for iteration j - 1 (sh.red is rewritten behind two barriers)
    TQHead &t = sm.heads[have ? li : 0];
    V3 p{0.0, 0.0, 0.0};
    double d = DBL_MAX;
    V3 np{0.0, 0.0, 0.0};
    bool ok = false;
    const int nwarps_q = (nq + TQ_PER_WARP - 1) / TQ_PER_WARP;  // warps that own source points
    if (warp < nwarps_q) {
        int cnt = 0;
        bool same_voxel = false;
        if (have) {
            p = V3{t.p[0], t.p[1], t.p[2]};
            if (j > 0) p = se3_act(sh.pending, p);  // TransformPoints(estimation, source)  Registration.cpp:160
            const V3 moved = p - V3{t.pf[0], t.pf[1], t.pf[2]};
            const int3 v = point_to_voxel(p.x, p.y, p.z, vdiv);
            same_voxel = t.vx == v.x && t.vy == v.y && t.vz == v.z;
            ok = t.count >= 0 && sqnorm(moved) <= r2max;
            cnt = ok ? t.count : 0;
        }
        KB_WCYC(0);
        __syncwarp();  // all four lanes have read t.p
        if (have && l4 == 0 && j > 0) {
            t.p[0] = p.x;
            t.p[1] = p.y;
            t.p[2] = p.z;
        }
        // first strict minimum of the squared distance over the list (= reference order); s2 = second smallest
        // (equal squares count: an exact tie takes the slow exact path below). Lane l4 takes candidates l4, l4 + 4, ...:
        // row i of the warp's block, column (4 q8 + l4 + 4 i) & 31.
        double b2 = DBL_MAX, s2 = DBL_MAX;
        int bk = INT_MAX;
        const unsigned cbase = static_cast<unsigned>(__cvta_generic_to_shared(sm.coords));
        const unsigned wbase = cbase + static_cast<unsigned>((li / TQ_PER_WARP) * (sm.K >> 2)) * 768u;
        const int c0 = 4 * (li & (TQ_PER_WARP - 1)) + l4;
        constexpr int U = 4;  // (kept small: code size of the loop body matters more than trips)
        for (int i0 = 0; 4 * i0 + l4 < cnt; i0 += U) {
            double d2[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {  // independent loads and distances in flight, no branches
                const int i = i0 + u;
                const bool in = 4 * i + l4 < cnt;
                const int ii = in ? i : 0;
                const unsigned a = wbase + static_cast<unsigned>(ii) * 768u + (static_cast<unsigned>((c0 + 4 * ii) & 31) << 3);
                const V3 c{lds_f64(a), lds_f64(a + 256u), lds_f64(a + 512u)};
                const double dd = sqnorm(c - p);
                d2[u] = in ? dd : DBL_MAX;
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {  // (no NaNs here: plain compare + select instead of fmin / fmax)
                const bool lt = d2[u] < b2;
                const double hi = lt ? b2 : d2[u];
                b2 = lt ? d2[u] : b2;
                bk = lt ? 4 * (i0 + u) + l4 : bk;
                s2 = hi < s2 ? hi : s2;
            }
        }
        KB_WCYC(1);
#pragma unroll
        for (int o = 1; o < TQ_LANES; o <<= 1) {
            const double ob2 = __shfl_xor_sync(FULL, b2, o), os2 = __shfl_xor_sync(FULL, s2, o);
            const int ok2 = __shfl_xor_sync(FULL, bk, o);
            const bool take = (ob2 < b2) || (ob2 == b2 && ok2 < bk);
            const double hi = (ob2 < b2) ? b2 : ob2;  // max(b2, ob2)
            double ns2 = os2 < s2 ? os2 : s2;
            ns2 = hi < ns2 ? hi : ns2;
            bk = take ? ok2 : bk;
            b2 = (ob2 < b2) ? ob2 : b2;
            s2 = ns2;
        }
        if (cnt > 0) {
            const unsigned a = tq_coord_addr(cbase, sm.K, li, bk);
            np = V3{lds_f64(a), lds_f64(a + 256u), lds_f64(a + 512u)};
            d = sqrt(b2);
        }
        KB_WCYC(2);
        // two squares within a few ulps could round to the same root: then compare rounded roots in reference
        // order like GetClosestNeighbor does (in practice never)
        const bool near = cnt > 0 && s2 <= b2 * (1.0 + NN_TIE_REL);
        if (__any_sync(FULL, near)) {
            tq_exact_nn(sm, li, l4, cnt, near, p.x, p.y, p.z);
            if (near) {
                d = t.nn[3];
                np = V3{t.nn[0], t.nn[1], t.nn[2]};
            }
        }
        KB_WCYC(3);
        ok = ok && (same_voxel || d < (voxel_size - radius) * (1.0 - 1e-12));
        if (have && !ok && l4 == 0) sh.refill_q[atomicAdd(&sh.refill_n[par], 1)] = li;
        // this point's 16 entries of J^T w J / J^T w r (lane l4: entries 4 l4 ..) + the gate flag -> row li of the
        // reduction scratch; a stale point writes zeros now and its row again after the re-search
        if (have) {
            double acc[4] = {0.0, 0.0, 0.0, 0.0};
            const bool gate = ok && d < max_dist;  // DataAssociation's gate, Registration.cpp:72
            if (gate) icp_term4(l4, p, np, kscale, acc);
            double *row = red + li * TRED_STRIDE;
#pragma unroll
            for (int i = 0; i < 4; ++i) row[4 * l4 + i] = acc[i];
            if (l4 == 0) row[NACC] = gate ? 1.0 : 0.0;
        }
        KB_WCYC(4);
    }
    __syncthreads();
    KB_TCYC(1);
    const int nref = sh.refill_n[par];
    if (nref > 0) {  // uniform; rare
        team_refill(sh, m, sm, nref, par, radius);
        if (have && !ok) {  // answered by the re-search
            const double rd = t.nn[3];
            const V3 rp{t.nn[0], t.nn[1], t.nn[2]};
            double acc[4] = {0.0, 0.0, 0.0, 0.0};
            const bool gate = rd < max_dist;
            if (gate) icp_term4(l4, p, rp, kscale, acc);
            double *row = red + li * TRED_STRIDE;
#pragma unroll
            for (int i = 0; i < 4; ++i) row[4 * l4 + i] = acc[i];
            if (l4 == 0) row[NACC] = gate ? 1.0 : 0.0;
        }
        __syncthreads();
    }
    KB_TCYC(2);
    if (tid == 0) {  // the other parity's counters are idle now: re-arm them for the next iteration
        sh.refill_n[par ^ 1] = 0;
        sh.refill_over[par ^ 1] = 0;
    }
    // column sums without shuffles (their throughput is per SM: 8 warps x 33 shuffles cost 800 cycles): 16 parts x
    // 17 columns (16 entries + the gate flag), part g adds rows g, g + 16, ... in order; column 17 = candidate counts
    if (tid < 16 * (NACC + 1)) {
        const int part = tid / (NACC + 1), col = tid - part * (NACC + 1);
        double v = 0.0, c = 0.0;
        for (int r = part; r < nq; r += 16) {
            v += red[r * TRED_STRIDE + col];
            if (col == NACC) c += static_cast<double>(sm.heads[r].full);
        }
        sh.warp_d[part][col] = v;
        if (col == NACC) sh.warp_d[part][NACC + 1] = c;
    }
    __syncthreads();
    KB_TCYC(3);
    if (tid < NPART) {
        double v = 0.0;
        if (tid < NACC + 2) {
            double v2 = 0.0;
#pragma unroll
            for (int g = 0; g < 16; g += 2) {
                v += sh.warp_d[g][tid];
                v2 += sh.warp_d[g + 1][tid];
            }
            v += v2;
        } else if (tid == NACC + 2) {
            v = static_cast<double>(nq - nref);  // lists that were still valid
        } else if (tid == NACC + 3) {
            v = static_cast<double>(nref);  // re-searched
        } else {
            v = static_cast<double>(sh.refill_over[par]);  // re-searched and not cacheable
        }
        sh.red[tid] = v;  // (the solver's copy of the previous iteration is consumed: it was read before the last barrier)
    }
    __syncthreads();
    // one copy per reader, all threads storing (21 lanes doing the T rows one after the other took 2400 cycles):
    // element e = reader * 21 + value -> row [reader][member], 21 consecutive 16-byte chunks
    {
        uint4 *dst = ll + (static_cast<size_t>(tag & 1u) * TEAM_MAX * TEAM_MAX + member) * NPART;
        // thread -> (value = tid % 32 if < 21, readers tid / 32, tid / 32 + 16, ...): a warp stores one reader's row at a time
        const int val = lane;
        if (val < NPART) {
            const double v = sh.red[val];
            for (int reader = warp; reader < T; reader += NWARPS)
                ll_store(dst + static_cast<size_t>(reader) * TEAM_MAX * NPART + val, v, tag);
        }
    }
    KB_TCYC(4);
}

// all-gather of the T tagged partial systems. Every member WRITES its partial once per reader (ll[parity][reader][member]
// [value]: 21 x T stores of 16 bytes, coalesced 336-byte rows) so that every reader polls lines nobody else reads:
// with one shared copy the 42 x 352 polling lanes of all CTAs (64 points per CTA then) hammered the same few L2 lines and the hop took 5 us
// (measured; the members themselves arrived within 0.5 us of each other).
// Reader: thread t polls chunks t, t + 512, ... of its T x 21 (a two-line loop: the iteration's code has to stay small)
// and drops the values into shared memory; after one barrier 21 lanes of warp 15 add the members in order (the same
// bits in every team CTA) and its last lane solves.
__device__ __forceinline__ void team_gather(const uint4 *ll, Shared &sh, int T, unsigned tag) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double *g = reinterpret_cast<double *>(sh.chunk_pref);  // [T][NPART] (the reduction scratch is done with)
    const uint4 *base = ll + (static_cast<size_t>(tag & 1u) * TEAM_MAX + blockIdx.x) * TEAM_MAX * NPART;  // my private copy
    const int total = T * NPART;
    unsigned spins = 0;
#pragma unroll 1
    for (int e = threadIdx.x; e < total; e += BLOCK) {
        double v;
        while (!ll_load(&base[e], tag, &v)) {
            if (kb_spin_check(spins, WD_TEAM_GATHER, tag, static_cast<unsigned>(e))) break;
        }
        g[e] = v;
    }
    __syncthreads();
    if (warp == NWARPS - 1) {
        if (lane < NPART) {
            double s0 = 0.0, s1 = 0.0;
            int mbr = 0;
#pragma unroll 1
            for (; mbr + 1 < T; mbr += 2) {
                s0 += g[mbr * NPART + lane];
                s1 += g[(mbr + 1) * NPART + lane];
            }
            if (mbr < T) s0 += g[mbr * NPART + lane];
            sh.red[lane] = s0 + s1;
        }
        __syncwarp();
    }
}

// degenerate normal equations (no correspondences, rank-deficient geometry): the pivoted LDL^T with Eigen's zero-pivot
// rule, like the reference's JTJ.ldlt().solve(-JTr)
__device__ __noinline__ void team_solve_ldlt(const double sys[NACC], double dx[6]) {
    double JTJ[36], JTr[6], rhs[6];
    icp_expand(sys, JTJ, JTr);
#pragma unroll
    for (int i = 0; i < 6; ++i) rhs[i] = -JTr[i];
    ldlt6_solve_fast(JTJ, rhs, dx);
}
__device__ __noinline__ SE3 team_exp_large(const double dx[6]) { return se3_exp_fast(dx); }
__device__ __noinline__ bool team_norm_below(double n2, double conv) { return sqrt(n2) < conv; }

// one thread: dx = JTJ.ldlt().solve(-JTr), estimation = SE3::exp(dx), convergence test (Registration.cpp:156-157,163)
__device__ __forceinline__ void team_solve(Shared &sh, double conv, bool last_allowed) {
    double sys[NACC];
#pragma unroll
    for (int i = 0; i < NACC; ++i) sys[i] = sh.red[i];
    double dx[6];
    if (!icp_solve_schur(sys, dx)) team_solve_ldlt(sys, dx);  // structured 3x3 Schur solve; cold: pivoted LDL^T
    const double theta_sq = (dx[3] * dx[3] + dx[4] * dx[4]) + dx[5] * dx[5];
    SE3 est;
    if (theta_sq >= kEps * kEps && theta_sq < 0.01) {
        est = se3_exp_small(dx, theta_sq);
    } else {
        est = team_exp_large(dx);  // cold
    }
    double n2 = 0.0;
#pragma unroll
    for (int i = 0; i < 6; ++i) n2 += dx[i] * dx[i];
    sh.pending = est;
    // dx.norm() < convergence_criterion (:163): decided on the square unless it is within rounding of the boundary
    const double c2 = conv * conv;
    bool conv_reached = n2 < c2 * (1.0 - 1e-14);
    if (!conv_reached && n2 <= c2 * (1.0 + 1e-14)) conv_reached = team_norm_below(n2, conv);  // cold
    sh.flag = (conv_reached || last_allowed) ? 1 : 0;
}

// the iterations, on CTAs [0, T) of the launch. Precondition: icp_fill_pass + a grid barrier, map not empty,
// max_iter > 0, T = icp_team_size(...) > 0. Output in sh.result / sh.iters / sh.cand_total / ... of every team CTA.
__device__ __noinline__ void op_icp_team(const TeamScratch &ts, const Scratch &sc, Shared &sh, const MapView &m, int n,
                                         const SE3 &guess, double max_dist, double kscale, int max_iter, double conv,
                                         unsigned char *dyn_smem, int T, unsigned tag_base) {
    const int member = static_cast<int>(blockIdx.x);
    const int nq = member < n ? (n - member + T - 1) / T : 0;
    const TeamSmem sm = team_smem(dyn_smem, ts.smem_bytes, (n + T - 1) / T);
    const VoxelDiv vdiv = m.vdiv;  // (by value into the iteration: `m` itself sits in the kernel's local copy of its parameters)
    uint4 *const ll = ts.ll;
    {
        // stage this CTA's source points (member, member + T, ...): one warp per point, all warps
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        for (int li = warp; li < nq; li += NWARPS) {
            const QList *rec = &ts.qrec[member + T * li];
            team_stage(sm, m, li, rec, lane);
            if (lane == 0) {
                TQHead &h = sm.heads[li];
                h.p[0] = rec->pf[0];
                h.p[1] = rec->pf[1];
                h.p[2] = rec->pf[2];
            }
        }
    }
    if (threadIdx.x == 0) {
        sh.t_icp = se3_identity();
        sh.cand_total = 0.0;
        sh.cache_stats[0] = sh.cache_stats[1] = sh.cache_stats[2] = 0.0;
        sh.refill_n[0] = sh.refill_n[1] = 0;
        sh.refill_over[0] = sh.refill_over[1] = 0;
    }
    __syncthreads();
    if (sc.profile && member == 0 && threadIdx.x == 0) sc.dbg[33] = globaltimer_ns();
    int j = 0;
    for (;; ++j) {
        if (sc.profile == 1 && member == 0 && threadIdx.x == 0 && j < 20) sc.dbg[41 + j] = globaltimer_ns();
        const unsigned tag = tag_base + static_cast<unsigned>(j) + 1u;
        kb_mark(0x410u + (static_cast<unsigned>(j) << 12));
#ifdef KB_PROFILE_TEAM
        unsigned long long *dbg = (sc.profile == 1 && member == 0 && j == 4) ? sc.dbg : nullptr;
#else
        unsigned long long *dbg = nullptr;
#endif
#ifdef KB_PROFILE_TEAM
        const bool stamp = sc.profile == 1 && j == 4 && threadIdx.x == 0;
        if (stamp) sc.dbg[64 + 4 * member] = globaltimer_ns();
#endif
        KB_TCYC(0);
        team_queries(ll, sh, m, sm, vdiv, ts.radius_frac, nq, j, max_dist, kscale, member, T, tag, dbg);
#ifdef KB_PROFILE_TEAM
        if (stamp) sc.dbg[64 + 4 * member + 1] = globaltimer_ns();
#endif
        team_gather(ll, sh, T, tag);  // (warp 15 holds the sums: no barrier between them and its solver lane)
#ifdef KB_PROFILE_TEAM
        if (stamp) sc.dbg[64 + 4 * member + 2] = globaltimer_ns();
#endif
        KB_TCYC(6);
        if (threadIdx.x == BLOCK - 1) team_solve(sh, conv, j + 1 >= max_iter);  // warp 15 owns no source point (TQ_MAX = 120)
        __syncthreads();
        KB_TCYC(7);
        if (sh.flag) break;  // (T_icp = estimation * T_icp of this iteration: team_accumulate, off the critical path)
    }
    if (sc.profile && member == 0 && threadIdx.x == 0) sc.dbg[34] = globaltimer_ns();
    if (threadIdx.x == BLOCK - 1) {
        team_accumulate(sh);
        sh.result = se3_mul(sh.t_icp, guess);  // :166
        sh.iters = j + 1;
        sh.query_total = static_cast<double>(n) * (j + 1);
    }
    __syncthreads();
}

// result record <-> shared memory (member 0 publishes before a grid barrier, everybody reads after it)
__device__ __forceinline__ void team_publish(const TeamScratch &ts, const Shared &sh) {
    double *o = ts.out;
    o[0] = sh.result.q.x;
    o[1] = sh.result.q.y;
    o[2] = sh.result.q.z;
    o[3] = sh.result.q.w;
    o[4] = sh.result.t.x;
    o[5] = sh.result.t.y;
    o[6] = sh.result.t.z;
    o[7] = static_cast<double>(sh.iters);
    o[8] = sh.cand_total;
    o[9] = sh.query_total;
    o[10] = sh.cache_stats[0];
    o[11] = sh.cache_stats[1];
    o[12] = sh.cache_stats[2];
}
__device__ __forceinline__ void team_collect(const TeamScratch &ts, Shared &sh) {
    const double *o = ts.out;
    sh.result = SE3{{__ldcg(o + 0), __ldcg(o + 1), __ldcg(o + 2), __ldcg(o + 3)}, {__ldcg(o + 4), __ldcg(o + 5), __ldcg(o + 6)}};
    sh.iters = static_cast<int>(__ldcg(o + 7));
    sh.cand_total = __ldcg(o + 8);
    sh.query_total = __ldcg(o + 9);
    sh.cache_stats[0] = __ldcg(o + 10);
    sh.cache_stats[1] = __ldcg(o + 11);
    sh.cache_stats[2] = __ldcg(o + 12);
}

}  // namespace kb
