#!/usr/bin/env python
"""bench.py — scans/s of KissICP::RegisterFrame on synthetic LiDAR streams (BASELINE.json configs[1], [2], [3]).

Contract (driver):  python bench.py --gpus N --steps K --warmup W [--impl reference]
  * a "step" = one scan registered by one pipeline, i.e. one pass of the hot path (pipeline/KissICP.cpp:35-68).
    Default workload = BASELINE.json configs[1] ("KITTI-00-shape synthetic stream on 1xB200", 64 x 1024 rays);
    --workload ouster128 = configs[2] (128 x 1024 rays, 0.3 m voxels, per-column stamps, deskew). At N GPUs every rank
    runs its own sequence (seed = rank) — weak scaling, no collective on the data path, poses gathered at the end.
  * before the W warm-up steps each pipeline is PRIMED with --prime scans (setup, untimed) so the timed region
    sees a steady-state local map instead of an almost empty one.
  * every timed leg times exactly K consecutive scans of the stream, split into --repeats R consecutive WINDOWS (default
    one per 20 scans), each bracketed by barrier + synchronize and timed with CUDA events on the launching stream;
    every number in the line comes from the MEDIAN window time per scan (per rank), then the max over ranks; min/max and
    the per-rank medians are in `windows`. (One 20-scan window is ~3 ms: a single host hiccup used to move the result by 2x.)
  * --dump-outputs DIR: after the timed scans, rank 0 writes what the last timed scan returned to its caller as float64
    .npy files (pose.npy, preprocessed.npy, source.npy); the inputs depend only on the arguments, so two builds can be
    compared output for output.
  * value  = scans/s with the scans already resident in HBM, frames queued (kb_pipeline_register_frames, device layout)
  * e2e    = scans/s through the host-facing C-ABI call with pinned HOST buffers: H2D of every scan and D2H of every
             result inside the timed region (kb_pipeline_register_frames, host layout); `blocking_calls` is the same
             with one blocking kb_pipeline_register_frame call per scan (the reference's call shape).
  * --impl reference times the reference's CPU algorithm (the oracle port, OpenMP over the host cores; the real
    TBB/Eigen build is impossible offline — see DESIGN.md) on the same stream, same windows.
One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "kitti": {"name": "KITTI-00-shape synthetic stream (64x1024 rays, ~65k pts/scan, voxel 1.0 m, no stamps), 1 sequence per GPU",
              "metric": "scans/sec (65k-pt KITTI-shape clouds)"},
    "ouster128": {"name": "Ouster-128-shape synthetic stream (128x1024 rays, ~131k pts/scan, voxel 0.3 m, per-column stamps, deskew), 1 sequence per GPU",
                  "metric": "scans/sec (131k-pt Ouster-128-shape clouds, 0.3 m voxels)"},
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed scans of every timed leg")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--repeats", type=int, default=None,
                    help="timing windows the --steps scans are split into (default: one per 20 scans); medians are reported")
    ap.add_argument("--prime", type=int, default=100, help="scans registered before warm-up (steady-state map)")
    ap.add_argument("--workload", default="kitti", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-sample", type=int, default=60, help="scans timed by the cpu_baseline leg")
    ap.add_argument("--streams", type=int, default=4, help="multi_stream leg: S independent sequences per GPU (0 = skip)")
    ap.add_argument("--no-nn", action="store_true", help="skip the NN-kernel roofline leg")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extra", action="store_true", help="skip the f32 / profile / trajectory side legs")
    ap.add_argument("--no-clocks", action="store_true", help="diagnostic: do not sample clocks (an invalid run by the bench contract)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed scans, write what the last one returned (pose, preprocessed frame, source points) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or (args.repeats is not None and args.repeats < 1):
        ap.error("--steps and --repeats must be at least 1")
    return args


def window_sizes(args):
    """the --steps timed scans split into consecutive windows whose sizes differ by at most one"""
    R = min(args.steps, args.repeats or max(1, args.steps // 20))
    return [args.steps // R + (r < args.steps % R) for r in range(R)]


def make_lidar(workload, seed, device):
    from kiss_icp_b200 import synthetic
    return synthetic.ouster128_shape(seed=seed, device=device) if workload == "ouster128" else synthetic.kitti_shape(seed=seed, device=device)


def pipeline_config(workload):
    """KISSConfig of the workload: the reference's defaults; Ouster-128: 0.3 m voxels (SURVEY.md 8d config 3)"""
    import kiss_icp_b200 as K
    return K.load_config(voxel_size=0.3) if workload == "ouster128" else K.load_config()


def oracle_kwargs(workload):
    return {"voxel_size": 0.3} if workload == "ouster128" else {}


def common_config(args, world):
    """identical in both arms (the driver compares the two dicts)"""
    return {"workload": WORKLOADS[args.workload]["name"], "prime_scans": args.prime, "sequences": world,
            "timed_steps": args.steps, "windows": len(window_sizes(args)),
            "statistic": "median over the windows of the per-window time per scan (the --steps timed scans split into consecutive windows); max over ranks of the per-rank median time",
            "l2": "every step consumes a new scan (1.5 MB KITTI / 3 MB Ouster); the local map (the state of the stream) is legitimately L2-resident across steps"}


# ----------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed regions. In-process NVML (the counters behind
    `nvidia-smi --query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.*`): a looping nvidia-smi process needs
    ~0.4 s per sample on an 8-GPU box and was seen stalling 40 ms timed regions; the NVML calls take < 1 ms.
    Falls back to the nvidia-smi loop of B200_PROFILING.md if NVML cannot be used from Python."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
    BITS = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, index, uuid=None, period=0.01):
        self.index, self.uuid, self.period = index, uuid, period
        self.rows, self.proc, self.nvml, self.first = [], None, None, 0
        self.max_mhz, self.stop_flag, self.source, self.query_ms = None, False, None, []

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            if self.uuid:
                try:
                    h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(self.uuid)).encode())
                except Exception:
                    h = None
            if h is None:
                vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
                ids = [v for v in vis.split(",") if v.strip()]
                phys = int(ids[self.index]) if ids and all(v.strip().isdigit() for v in ids) else self.index
                h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            reasons_fn = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
            self.nvml = (pynvml, h, reasons_fn)
            self.source = "NVML in-process, %d ms period" % int(self.period * 1e3)
            threading.Thread(target=self._poll, daemon=True).start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.source = "nvidia-smi -lms 100"
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _poll(self):
        pynvml, h, reasons_fn = self.nvml
        while not self.stop_flag:
            try:
                t0 = time.perf_counter()
                sm = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                bits = int(reasons_fn(h))
                self.rows.append((sm, bits))
                self.query_ms.append((time.perf_counter() - t0) * 1e3)
            except Exception:
                pass
            time.sleep(self.period)

    def _read(self):
        for line in self.proc.stdout:
            r = [c.strip() for c in line.split(",")]
            if len(r) > 8 and r[1].replace(".", "").isdigit():
                bits = 0
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[5:9]):
                    if v.lower().startswith("active"):
                        bits |= self.BITS[name]
                if r[2].replace(".", "").isdigit():
                    self.max_mhz = max(self.max_mhz or 0.0, float(r[2]))
                self.rows.append((float(r[1]), bits))

    def wait_ready(self, timeout=20.0):
        """NVML / nvidia-smi start-up stalls the GPU for hundreds of ms: never let it land in a timed region"""
        t0 = time.perf_counter()
        while (self.proc or self.nvml) and not self.rows and time.perf_counter() - t0 < timeout:
            time.sleep(0.05)

    def mark(self):
        self.first = len(self.rows)

    def stop(self):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
        rows = self.rows[self.first:]
        sm = [r[0] for r in rows]
        reasons = sorted(name for name, bit in self.BITS.items() if any(r[1] & bit for r in rows))
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": reasons, "samples": len(sm), "source": self.source,
                "query_ms_max": float(max(self.query_ms)) if self.query_ms else None}


# ----------------------------------------------------------------------------- reference arm
def best_thread_count(O, scans, candidates, **kw):
    """the oracle's OpenMP regions are tiny (1-2k points per ICP iteration): pick the thread count
    that makes the REFERENCE fastest on this box, so the baseline is not handicapped"""
    best, best_t = None, None
    for nt in candidates:
        icp = O.KissICP(max_num_threads=nt, **kw)
        for p, t in scans[:4]:
            icp.register_frame(p, t, want_clouds=False)
        t0 = time.perf_counter()
        for p, t in scans[4:12]:
            icp.register_frame(p, t, want_clouds=False)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = nt, dt
    return best


def thread_candidates():
    n = os.cpu_count() or 1
    return sorted({min(n, x) for x in (4, 8, 16, 32, 64, n)})


def run_reference(args, rank, world):
    """the reference's CPU implementation of the path on the host cores (oracle port). At --gpus N the job is
    N independent sequences (one per GPU in our arm): here they run concurrently on the host, each with its
    share of the cores. Same windows as our arm: K scans in R windows, value = N / median window time per scan."""
    if rank != 0:
        return
    from concurrent.futures import ThreadPoolExecutor
    from oracle import oracle as O
    import torch
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    nseq = max(1, args.gpus)
    sizes = window_sizes(args)
    starts = np.cumsum([0] + sizes)
    R = len(sizes)
    head = args.prime + args.warmup
    n_total = head + args.steps
    kw = oracle_kwargs(args.workload)
    streams = []
    for sid in range(nseq):
        lidar = make_lidar(args.workload, sid, dev)
        streams.append([lidar.scan(k) for k in range(n_total)])
    ncpu = os.cpu_count() or 1
    best = best_thread_count(O, streams[0], thread_candidates(), **kw)
    nt = max(1, min(best, ncpu // nseq))
    icps = [O.KissICP(max_num_threads=nt, **kw) for _ in range(nseq)]

    def run(sid, lo, hi):
        for p, t in streams[sid][lo:hi]:
            icps[sid].register_frame(p, t, want_clouds=False)  # ctypes releases the GIL during the call

    win = []
    with ThreadPoolExecutor(nseq) as ex:
        list(ex.map(lambda sid: run(sid, 0, head), range(nseq)))
        for r in range(R):
            t0 = time.perf_counter()
            list(ex.map(lambda sid: run(sid, head + starts[r], head + starts[r + 1]), range(nseq)))
            win.append(time.perf_counter() - t0)
    dt = float(np.median(np.array(win) / sizes))  # seconds per scan
    val = nseq / dt
    cfg = common_config(args, nseq)
    line = {"impl": "reference", "metric": WORKLOADS[args.workload]["metric"], "value": val, "unit": "scans/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": cfg,
            "windows": {"ms": [w * 1e3 for w in win], "scans": sizes},
            "note": "reference CPU path = dependency-free restatement of cpp/kiss_icp (oracle port, OpenMP for TBB); the real "
                    "TBB/Eigen build needs network-fetched deps. N sequences run concurrently on the host cores.",
            "cpu_baseline": {"value": val, "unit": "scans/s", "cores": nt * nseq, "kind": "port",
                             "sample": f"{nseq} x {args.steps} scans in {R} windows after {head} untimed; {nt} OpenMP "
                                       f"threads per sequence (fastest single-sequence count of {thread_candidates()} "
                                       f"capped at cpus/sequences) on {ncpu} cpus"},
            "e2e": {"value": val, "unit": "scans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- our arm
def main():
    args = parse()
    rank, world, local = (int(os.environ.get(k, d)) for k, d in (("RANK", "0"), ("WORLD_SIZE", "1"), ("LOCAL_RANK", "0")))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import kiss_icp_b200 as K
    from kiss_icp_b200 import _native as N, sharding

    if not torch.cuda.is_available() or N.lib().kb_device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: kiss_icp_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    N.check(N.lib().kb_set_device(local))
    # torch's default stream has a NULL handle; use an explicit stream so that the library's launches and
    # the torch.cuda.Event timing share ONE stream
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    N.check(N.lib().kb_set_stream(C.c_void_p(stream.cuda_stream)))

    sampler = ClockSampler(local, getattr(torch.cuda.get_device_properties(dev), "uuid", None))
    if rank == 0 and not args.no_clocks:
        sampler.start()  # started long before the timed regions; samples before mark() are dropped

    seq = sharding.sequences_of_rank(rank, world, world)[0]
    lidar = make_lidar(args.workload, seq, dev)
    Kw, sizes = args.steps, window_sizes(args)
    starts, R = np.cumsum([0] + sizes), len(sizes)
    head = args.prime + args.warmup
    n_total = head + Kw
    scans_dev = []
    for k in range(n_total):
        p, t = lidar.scan_torch(k)
        scans_dev.append((p.contiguous(), t.contiguous()))
    L = N.lib()
    cfg = pipeline_config(args.workload)

    def make_pipeline():
        return K.KissICP(cfg)

    def tsp(t):
        return C.c_void_p(t.data_ptr()) if t.numel() else None

    def reg_dev(icp, s):
        N.check(L.kb_pipeline_register_frame_dev(icp._h, C.c_void_p(s[0].data_ptr()), s[0].shape[0], tsp(s[1]), s[1].numel()))

    def reg_host(icp, s):
        N.check(L.kb_pipeline_register_frame(icp._h, C.c_void_p(s[0].data_ptr()), s[0].shape[0], tsp(s[1]), s[1].numel()))

    def launches(icp):
        c = C.c_ulonglong(0)
        N.check(L.kb_pipeline_launch_count(icp._h, C.byref(c)))
        return c.value

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def primed(n_blocking):
        icp = make_pipeline()
        for s in scans_dev[:n_blocking]:
            reg_dev(icp, s)
        return icp

    def queued(icp, scans, layout):
        """KissICP.register_frames on raw addresses: the whole list is queued on the device, copy of frame k+1
        overlaps the registration of frame k, every frame's result (pose + counters) is read back behind the queue"""
        return icp._register_frames_raw([s[0].data_ptr() for s in scans], [s[0].shape[0] for s in scans],
                                        [s[1].data_ptr() if s[1].numel() else None for s in scans], [s[1].numel() for s in scans], layout)

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def window(fn):
        barrier()
        e0.record(stream)
        fn()
        e1.record(stream)
        barrier()
        return e0.elapsed_time(e1)

    def timed_windows(fn_of_window):
        """K scans in R windows -> (this rank's window times [ms], K x the median window time per scan, maxed over ranks)"""
        ms = [window(lambda r=r: fn_of_window(r)) for r in range(R)]
        return ms, sharding.max_over_ranks(float(np.median(np.array(ms) / sizes)) * Kw, dev)

    def win_scans(pool, r):
        off = head if len(pool) == n_total else 0  # pools hold either the whole stream or only the timed part
        return pool[off + starts[r]: off + starts[r + 1]]

    warm = scans_dev[args.prime:head]
    legs = {}

    # ---------------- value: inputs resident in HBM, frames queued (kb_pipeline_register_frames, device layout)
    icp = primed(args.prime)
    if rank == 0:
        sampler.wait_ready()  # NVML start-up perturbs the GPU for tens of ms: let it land in the warm-up
    queued(icp, warm, 2)
    if rank == 0:
        sampler.mark()
    l0 = launches(icp)
    value_poses = []
    legs["value"] = timed_windows(lambda r: value_poses.append(queued(icp, win_scans(scans_dev, r), 2)))
    gpu_launches = launches(icp) - l0
    ms_value = legs["value"][1]
    value = world * Kw / (ms_value * 1e-3)
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, L, icp, value_poses[-1][-1])

    # ---------------- the same with one blocking RegisterFrame call per scan (the reference's call shape)
    icp_b = primed(head)
    wall_dev = []

    def blocking_dev(r):
        for s in win_scans(scans_dev, r):
            t0 = time.perf_counter()
            reg_dev(icp_b, s)
            wall_dev.append(time.perf_counter() - t0)
    legs["blocking_resident"] = timed_windows(blocking_dev)

    # ---------------- e2e: host-facing call, pinned host buffers, H2D + D2H of every step inside the timed region
    def to_pinned(s):
        return (s[0].cpu().pin_memory(), s[1].cpu().pin_memory() if s[1].numel() else s[1].cpu())
    pinned_warm = [to_pinned(s) for s in warm]
    pinned = [to_pinned(s) for s in scans_dev[head:]]
    h2d = float(np.mean([p.numel() * 8 + t.numel() * 8 for p, t in pinned]))
    icp2 = primed(args.prime)
    queued(icp2, pinned_warm, 0)
    e2e_last = []
    legs["e2e"] = timed_windows(lambda r: e2e_last.append(queued(icp2, win_scans(pinned, r), 0)[-1]))
    ms_e2e = legs["e2e"][1]
    e2e_value = world * Kw / (ms_e2e * 1e-3)
    # blocking form: kb_pipeline_register_frame per scan
    icp2b = primed(head)
    wall_e2e = []

    def blocking_e2e(r):
        for s in win_scans(pinned, r):
            t0 = time.perf_counter()
            reg_host(icp2b, s)
            wall_e2e.append(time.perf_counter() - t0)
    legs["blocking_e2e"] = timed_windows(blocking_e2e)
    clocks = sampler.stop() if rank == 0 else None

    # the four pipelines saw identical inputs -> identical trajectories (determinism check)
    same = bool(np.array_equal(icp.last_pose, icp2.last_pose) and np.array_equal(icp_b.last_pose, icp2b.last_pose)
                and np.array_equal(icp.last_pose, icp_b.last_pose) and np.array_equal(e2e_last[-1], icp2.last_pose))

    # ---------------- profiling pass (untimed): the timed scans once more with the in-kernel phase timestamps ON
    # (they cost ~1 us each on the kernel's critical path, so the timed passes above run without them)
    prof_n = Kw
    prof = np.zeros((prof_n, 6))
    iters = np.zeros(prof_n)
    work = np.zeros((prof_n, 2))
    npts = np.zeros(prof_n)
    poses_local = []
    icp4 = primed(head)
    icp4.set_profiling(True)
    icp4.start_history(prof_n)
    for s in scans_dev[head:head + prof_n]:
        reg_dev(icp4, s)
    for i, st in enumerate(icp4.history()):
        prof[i] = list(st.phase_us)
        iters[i] = st.iterations
        work[i] = (st.icp_queries, st.icp_candidates)
        npts[i] = st.n_points_in
        poses_local.append(np.array(st.pose).reshape(4, 4))
    # ---------------- e2e, float32 ingestion (KITTI .bin / PointCloud2 are float32; the scans are fp32-representable)
    f32 = None
    if not args.no_extra:
        icp3 = primed(args.prime)
        queued(icp3, [(p.to(torch.float32).pin_memory(), t) for p, t in pinned_warm], 1)
        pinned32 = [(p.to(torch.float32).pin_memory(), t) for p, t in pinned]
        legs["e2e_f32"] = timed_windows(lambda r: queued(icp3, win_scans(pinned32, r), 1))
        f32 = {"value": world * Kw / (legs["e2e_f32"][1] * 1e-3), "unit": "scans/s", "h2d_bytes_per_step": h2d - 12.0 * float(np.mean([p.shape[0] for p, _ in pinned])),
               "d2h_bytes_per_step": 512.0, "same_trajectory_as_f64": bool(np.array_equal(icp3.last_pose, icp2.last_pose)),
               "note": "register_frames, float32 host frames (native KITTI/ROS payload), widened on the device"}
    # ---------------- the reference's Python call structure (python/kiss_icp/kiss_icp.py:43-75): six module calls per scan,
    # each copying its clouds in and out (KissICP(fused=False) = preprocess, voxelize x2, threshold, align, update on the
    # per-module C-ABI); host wall clock on rank 0, the K timed scans in one go
    modular = None
    if rank == 0 and world == 1 and not args.no_extra:
        try:
            icp_m = K.KissICP(cfg, fused=False)
            host_scans = [(s[0].cpu().numpy(), s[1].cpu().numpy()) for s in scans_dev[:head + Kw]]
            for pts_m, ts_m in host_scans[:head]:
                icp_m.register_frame(pts_m, ts_m)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for pts_m, ts_m in host_scans[head:]:
                icp_m.register_frame(pts_m, ts_m)
            dt_m = time.perf_counter() - t0
            modular = {"value": Kw / dt_m, "unit": "scans/s", "scans": Kw,
                       "note": "module-by-module RegisterFrame (the call structure of the reference's Python layer and of "
                               "bindings/kiss_icp_pybind.cpp): every module call copies its clouds host->device->host; one sequence, host wall clock"}
        except Exception as e:  # never lose the bench line over a side leg
            print("modular pass failed:", e, file=sys.stderr)
    # ---------------- untimed: the whole trajectory from scan 0 (for the drift metrics below)
    traj = None
    if rank == 0 and not args.no_extra:
        try:
            traj = queued(make_pipeline(), scans_dev, 2)
        except Exception as e:  # never lose the bench line over a side leg
            traj = None
            print("trajectory pass failed:", e, file=sys.stderr)
    d2h = 512.0  # sizeof(FrameResult): pose, delta, sigma, counters, stamps

    all_poses = sharding.gather_poses(np.array(poses_local), dev)  # NCCL all_gather of the trajectories
    per_rank = {name: sharding.gather_poses(np.array(ms).reshape(1, -1, 1, 1), dev).reshape(world, -1) for name, (ms, _) in legs.items()}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    def win_summary(name):
        a = per_rank[name] / sizes  # ms per scan of every window
        med = np.median(a, axis=1)
        return {"scans": sizes, "median_ms_per_scan_per_rank": [float(x) for x in med], "min_ms_per_scan": float(a.min()),
                "max_ms_per_scan": float(a.max()), "slowest_rank": int(np.argmax(med)), "scans_per_s": world / (float(med.max()) * 1e-3)}

    # ---------------- roofline of the dominant kernel (k_register_frame, one launch per scan)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    else:
        peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
    # algorithmic bytes per launch (DESIGN.md "algorithmic bytes"): ICP GetClosestNeighbor traffic
    # (24 + 27*16 + 32 per query + 24 per candidate) + one-off streams (raw scan in, result out)
    bytes_per_launch = work[:, 0] * (24 + 27 * 16 + 32) + 24.0 * work[:, 1] + 24.0 * npts + d2h
    kern_us = ms_value * 1e3 / Kw  # CUDA-event time of the median window / launches in it (queued back to back)
    achieved = float(bytes_per_launch.mean() / (kern_us * 1e-6) / 1e9)
    traffic, traffic_src = profiled_traffic("r2_register_frame")
    roofline = {"kernel": "k_register_frame (persistent cooperative, 1 launch/scan)", "bound": "hbm",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "algorithmic_bytes_per_launch": float(bytes_per_launch.mean()), "kernel_us": float(kern_us),
                "traffic": traffic, "traffic_source": traffic_src, "traffic_measured_in_this_run": False,
                "peak_source": peak_src,
                "note": "latency-bound: ~%.0f ICP iterations x %.0f queries per launch, working set L2-resident; algorithmic bytes "
                        "count the full 27-voxel neighbourhood of every query and iteration (most are served from the "
                        "candidate lists); kernel time = CUDA-event time of the median window / launches; see nn_kernel "
                        "for the bandwidth-bound NN query" % (iters.mean(), work[:, 0].mean() / max(iters.mean(), 1))}

    # side legs on rank 0 at N = 1 only (a multi-GPU run measures scaling; the CPU legs would also compete for the host cores)
    solo = world == 1
    ms_leg = multi_stream_leg(args, K, N, L, torch, dev, args.streams, cfg) if (solo and args.streams > 1 and not args.no_extra) else None
    nn = nn_leg(K, N, L, torch, dev, peak) if (solo and not args.no_nn) else None
    cpu = cpu_leg(args, lidar) if (solo and not args.no_cpu) else None
    quality = trajectory_quality(lidar, traj, cpu.pop("poses", None) if cpu else None)
    wall_dev_a, wall_e2e_a = np.array(wall_dev), np.array(wall_e2e)

    line = {"metric": WORKLOADS[args.workload]["metric"], "value": value, "unit": "scans/s", "n_gpus": world, "steps": Kw,
            "warmup": args.warmup, "ms_per_step": ms_value / Kw, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": common_config(args, world),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "scans/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / Kw,
                    "api": "KissICP.register_frames / kb_pipeline_register_frames: pinned host float64 frames in, poses out; "
                           "frames queued (H2D of scans k+1, k+2 overlaps the registration of scan k, whose launch also runs "
                           "the front end of scan k+1 on the SMs its ICP team leaves idle)"},
            "blocking_calls": {"note": "one kb_pipeline_register_frame[_dev] call per scan, host waits for every result (the reference's call shape)",
                               "value_resident": world * Kw / (legs["blocking_resident"][1] * 1e-3),
                               "e2e": world * Kw / (legs["blocking_e2e"][1] * 1e-3), "unit": "scans/s", "modular": modular},
            "e2e_f32": f32,
            "gpu_launches": int(gpu_launches),
            "windows": {name: win_summary(name) for name in legs},
            "details": {"points_per_scan": float(npts.mean()), "icp_iterations_per_scan": float(iters.mean()),
                        "icp_source_points": float((work[:, 0] / np.maximum(iters, 1)).mean()),
                        "icp_candidates_per_query": float(work[:, 1].sum() / max(work[:, 0].sum(), 1.0)),
                        "gpu_us_per_scan": {"queued_resident": ms_value * 1e3 / Kw, "queued_e2e": ms_e2e * 1e3 / Kw,
                                            "blocking_resident": legs["blocking_resident"][1] * 1e3 / Kw, "blocking_e2e": legs["blocking_e2e"][1] * 1e3 / Kw},
                        "phase_us_note": "from a separate untimed pass of blocking calls with in-kernel %globaltimer stamps ON (they add ~1 us per phase/iteration); "
                                         "icp = candidate-list pass over the map + iterations on the ICP team",
                        "phase_us": dict(zip(["preprocess", "downsample_0.5v", "downsample_1.5v", "icp", "map_update", "epilogue"],
                                             [float(x) for x in prof.mean(0)])),
                        "call_latency_ms": {"resident": {"p50": float(np.percentile(wall_dev_a, 50) * 1e3), "p99": float(np.percentile(wall_dev_a, 99) * 1e3), "max": float(wall_dev_a.max() * 1e3)},
                                            "e2e": {"p50": float(np.percentile(wall_e2e_a, 50) * 1e3), "p99": float(np.percentile(wall_e2e_a, 99) * 1e3), "max": float(wall_e2e_a.max() * 1e3)}},
                        "deterministic_replay": same, "gathered_trajectories": list(all_poses.shape),
                        "trajectory_quality": quality},
            "roofline": roofline, "nn_kernel": nn, "multi_stream": ms_leg, "cpu_baseline": cpu}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def multi_stream_leg(args, K, N, L, torch, dev, S, cfg):
    """S independent sequences on ONE GPU: S pipelines, S host threads, S CUDA streams, each persistent grid
    sized to 1/S of the SMs (SURVEY.md 8f rank 1). Reported beside the single-stream headline, never instead."""
    import threading
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    steps = args.steps
    n_total = min(args.prime, 40) + steps
    data = []
    for sid in range(S):
        lidar = make_lidar(args.workload, 100 + sid, dev)
        data.append([tuple(x.contiguous() for x in lidar.scan_torch(k)) for k in range(n_total)])
    torch.cuda.synchronize()
    pipes = [None] * S
    barrier = threading.Barrier(S + 1)
    walls = [0.0] * S
    errs = []

    def worker(sid):
        try:
            N.check(L.kb_set_device(dev.index or 0))
            N.check(L.kb_set_stream(None))                 # own non-blocking stream per pipeline
            N.check(L.kb_set_grid_blocks(max(1, sms // S)))
            icp = K.KissICP(cfg)
            pipes[sid] = icp
            seqs = data[sid]
            icp._register_frames_raw([s[0].data_ptr() for s in seqs[: n_total - steps]], [s[0].shape[0] for s in seqs[: n_total - steps]],
                                     [s[1].data_ptr() if s[1].numel() else None for s in seqs[: n_total - steps]], [s[1].numel() for s in seqs[: n_total - steps]], 2)
        except Exception as e:
            errs.append(repr(e))
        barrier.wait()
        t0 = time.perf_counter()
        try:
            tail = data[sid][n_total - steps:]
            pipes[sid]._register_frames_raw([s[0].data_ptr() for s in tail], [s[0].shape[0] for s in tail],
                                            [s[1].data_ptr() if s[1].numel() else None for s in tail], [s[1].numel() for s in tail], 2)
        except Exception as e:
            errs.append(repr(e))
        walls[sid] = time.perf_counter() - t0
        barrier.wait()

    threads = [threading.Thread(target=worker, args=(i,)) for i in range(S)]
    for t in threads:
        t.start()
    barrier.wait()
    t0 = time.perf_counter()
    barrier.wait()
    dt = time.perf_counter() - t0
    for t in threads:
        t.join()
    N.check(L.kb_set_grid_blocks(0))
    if errs:
        return {"streams": S, "error": errs[0]}
    return {"streams": S, "grid_blocks_per_stream": max(1, sms // S), "scans_per_s": S * steps / dt,
            "ms_per_scan_per_stream": float(np.mean(walls)) / steps * 1e3,
            "note": "aggregate over S concurrent sequences on one GPU (S pipelines on S streams, each launch on 1/S of the SMs), "
                    "inputs resident in HBM, frames queued, host wall clock"}


def dump_outputs(out_dir, L, icp, pose):
    """what the last timed scan returned to its caller: its pose (from kb_pipeline_register_frames) and the two clouds
    RegisterFrame returns with it (preprocessed frame, source points), all float64, ~1.6 MB per KITTI-shape scan"""
    from kiss_icp_b200 import _native as N
    n_pre, n_src = N.sz(0), N.sz(0)
    N.check(L.kb_pipeline_last_cloud_sizes(icp._h, C.byref(n_pre), C.byref(n_src)))
    pre, src = np.empty((n_pre.value, 3)), np.empty((n_src.value, 3))
    N.check(L.kb_pipeline_last_clouds(icp._h, N.ptr(pre), n_pre.value, N.ptr(src), n_src.value))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("pose", np.asarray(pose, dtype=np.float64)), ("preprocessed", pre), ("source", src)):
        np.save(os.path.join(out_dir, name + ".npy"), a)


def profiled_traffic(tag):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full summary
    (profiles/<tag>_ncu_raw_selected.csv, produced by tools/summarize_profiles.py) -> (bytes or None, source)."""
    import csv
    for t in (tag, tag.replace("r2_", "r1_")):
        path = os.path.join(ROOT, "profiles", f"{t}_ncu_raw_selected.csv")
        if not os.path.exists(path):
            continue
        scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        per_launch = {}
        for r in csv.DictReader(open(path)):
            if r["metric"] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                per_launch[r["launch"]] = per_launch.get(r["launch"], 0.0) + float(r["value"]) * scale.get(r["unit"], 1.0)
        if per_launch:
            return float(np.mean(list(per_launch.values()))), f"static: profiles/{t}_ncu_raw_selected.csv (a separate ncu --set full capture, bytes per launch)"
    return None, None


def nn_leg(K, N, L, torch, dev, peak):
    """BASELINE config 5: batched GetClosestNeighbor on a large map — the bandwidth-bound kernel."""
    from kiss_icp_b200 import synthetic
    g = torch.Generator(device="cpu")
    g.manual_seed(5)
    n_raw, n_q = 4_000_000, 1 << 20
    m = K.VoxelHashMap(1.0, 1e9, 20)
    m.add_points(synthetic.surface_cloud(n_raw, seed=5))  # dense surfaces: ~8 points per 1 m voxel like a real map
    stored = torch.from_numpy(m.point_cloud())
    sel = stored[torch.randint(0, stored.shape[0], (n_q,), generator=g)]
    q = (sel + torch.randn(n_q, 3, generator=g, dtype=torch.float64) * 0.3).to(dev).contiguous()
    outp = torch.empty_like(q)
    outd = torch.empty(n_q, dtype=torch.float64, device=dev)
    b = C.c_double(0)
    N.check(L.kb_map_query_bytes_dev(m._h, C.c_void_p(q.data_ptr()), n_q, C.byref(b)))
    stream = torch.cuda.current_stream()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > L2 (126 MB)
    def timed(variant):
        """mean ms of 10 launches (after 3 untimed), L2 flushed before each; the library reads KB_NN_KERNEL per call"""
        old = os.environ.get("KB_NN_KERNEL")
        os.environ["KB_NN_KERNEL"] = variant
        times = []
        try:
            for it in range(13):
                flush.fill_(it & 0xff)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                N.check(L.kb_map_closest_neighbors_dev(m._h, C.c_void_p(q.data_ptr()), n_q, C.c_void_p(outp.data_ptr()),
                                                       C.c_void_p(outd.data_ptr())))
                e1.record(stream)
                torch.cuda.synchronize()
                if it >= 3:
                    times.append(e0.elapsed_time(e1))
        finally:
            if old is None:
                os.environ.pop("KB_NN_KERNEL", None)
            else:
                os.environ["KB_NN_KERNEL"] = old
        return float(np.mean(times)), len(times)

    variant = "bulk" if os.environ.get("KB_NN_KERNEL") == "bulk" else "regs"
    ms, reps = timed(variant)
    other = "regs" if variant == "bulk" else "bulk"
    ms_other, _ = timed(other)
    ach = b.value / (ms * 1e-3) / 1e9
    names = {"regs": "k_nn_query (one warp per query, candidates staged in registers, next query's probes in flight)",
             "bulk": "k_nn_query_bulk (candidate blocks staged in shared memory by cp.async.bulk + mbarrier)"}
    # the ncu --set full captures: round 1 = k_nn_query, round 2 = k_nn_query_bulk
    traffic, traffic_src = profiled_traffic("r1_nn_query" if variant == "regs" else "r2_nn_query")
    return {"kernel": names[variant], "map_points": int(stored.shape[0]), "map_voxels": m.num_voxels(), "queries": n_q, "points_per_voxel": float(stored.shape[0]) / max(m.num_voxels(), 1),
            "algorithmic_bytes": b.value, "bytes_per_query": b.value / n_q, "ms": ms, "achieved": ach, "peak": peak,
            "unit": "GB/s", "frac": ach / peak, "traffic": traffic, "traffic_source": traffic_src,
            "l2": "flushed (256 MiB write) before every timed launch", "reps": reps,
            "other_variant": {"kernel": names[other], "ms": ms_other, "frac": b.value / (ms_other * 1e-3) / 1e9 / peak}}


def trajectory_quality(lidar, traj, cpu_poses):
    """KITTI-style drift of the registered trajectory against the synthetic ground truth (kiss-icp_b200/metrics.py =
    Metrics.cpp restated), for the GPU path and - over the scans the cpu_baseline leg registered - for the CPU port,
    plus the largest pose difference between the two (SURVEY.md 8f rank 4: parity drift is immaterial)."""
    if traj is None:
        return None
    try:
        from kiss_icp_b200 import metrics as M
        n = len(traj)
        gt = np.array([lidar.pose(k) for k in range(n)])
        gt = np.array([np.linalg.inv(gt[0]) @ g for g in gt])  # KISS-ICP poses are relative to the first scan
        dist = float(np.linalg.norm(np.diff(gt[:, :3, 3], axis=0), axis=1).sum())
        out = {"scans": n, "path_m": dist,
               "gpu": dict(zip(["seq_trans_pct", "seq_rot_deg_per_m", "ate_rot_rad", "ate_trans_m"],
                               list(M.sequence_error(gt, traj)) + list(M.absolute_trajectory_error(gt, traj))))}
        if cpu_poses is not None and len(cpu_poses) <= n:
            m = len(cpu_poses)
            out["cpu_port"] = dict(zip(["scans", "seq_trans_pct", "seq_rot_deg_per_m", "ate_rot_rad", "ate_trans_m"],
                                       [m] + list(M.sequence_error(gt[:m], cpu_poses)) + list(M.absolute_trajectory_error(gt[:m], cpu_poses))))
            out["gpu_same_scans"] = dict(zip(["seq_trans_pct", "seq_rot_deg_per_m", "ate_rot_rad", "ate_trans_m"],
                                             list(M.sequence_error(gt[:m], traj[:m])) + list(M.absolute_trajectory_error(gt[:m], traj[:m]))))
            out["max_abs_pose_diff_gpu_vs_cpu_port"] = float(np.abs(traj[:m] - cpu_poses).max())
        return out
    except Exception as e:
        return {"error": repr(e)}


def cpu_leg(args, lidar):
    """oracle (port of the reference CPU path) on the host cores, bounded sample of the same stream; best OpenMP
    thread count and the 1-thread figure (SURVEY.md 8d)."""
    from oracle import oracle as O
    kw = oracle_kwargs(args.workload)
    n = min(args.cpu_sample, args.steps)
    scans = [lidar.scan(k) for k in range(args.prime + n)]
    nt = best_thread_count(O, scans, thread_candidates(), **kw)
    icp = O.KissICP(max_num_threads=nt, **kw)
    poses = []
    for p, t in scans[:args.prime]:
        icp.register_frame(p, t, want_clouds=False)
        poses.append(np.array(icp.pose))
    t0 = time.perf_counter()
    for p, t in scans[args.prime:]:
        icp.register_frame(p, t, want_clouds=False)
        poses.append(np.array(icp.pose))
    dt = time.perf_counter() - t0
    # 1 thread: a short sample on a map primed with 30 scans (bounded: ~1-2 s)
    n1 = min(12, n)
    one = O.KissICP(max_num_threads=1, **kw)
    for p, t in scans[:30]:
        one.register_frame(p, t, want_clouds=False)
    t1 = time.perf_counter()
    for p, t in scans[30:30 + n1]:
        one.register_frame(p, t, want_clouds=False)
    dt1 = time.perf_counter() - t1
    return {"poses": np.array(poses), "value": n / dt, "unit": "scans/s", "cores": nt, "kind": "port", "ms_per_scan": dt / n * 1e3,
            "one_thread": {"value": n1 / dt1, "ms_per_scan": dt1 / n1 * 1e3, "sample": f"{n1} scans after 30 priming scans, 1 OpenMP thread"},
            "sample": f"{n} scans after {args.prime} untimed priming scans of the same stream (seed 0); OpenMP threads "
                      f"picked as fastest of {thread_candidates()} on {os.cpu_count()} cpus"}


if __name__ == "__main__":
    main()
