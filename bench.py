#!/usr/bin/env python
"""Benchmark of the sonar front end (BASELINE.json metric: sonar frames/sec, CFAR + ICP).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--frames F] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE config 4, the configuration the metric is quoted on): a synthetic bag replay --
F = 4096 polar sonar frames (512 beams x 512 range bins, uint8) per step and per GPU, rendered from a
moving vehicle with odometry; every frame goes through CFAR (SOCA 40/10, Pfa 0.1) + amplitude gate ->
polar->Cartesian cloud -> voxel-medoid down-sample -> radius outlier removal -> scan match (ICP, 20
iterations, window of 3 previous frames).  One step = one batch through sfe_frontend_*.

  value   frames/s with the frames already resident in HBM (sfe_frontend_run_dev), CUDA-event timed
  e2e     the same batch through the host-buffer C-ABI call (sfe_frontend_run_host): pinned host frames
          are copied in inside the timed region, results are copied back
  roofline  the CFAR kernel of the step (HBM bound): algorithmic bytes / its CUDA-event time
  cpu_baseline  the CPU oracle (oracle/: reference cfar.cpp compiled unmodified + restated cloud/ICP
          code) on a bounded sample of the same frames, one thread
  --impl reference   the reference arm: that CPU path on all host cores (rank 0 only under torchrun)

  config3_icp   BASELINE config 3 (2 000 x 20 000-point scan matches, 20 iterations and the shipped checkers) on
          rank 0: pairs/s over 8 waves of 148 problems, ms per wave
  config5   BASELINE config 5: a FIXED backlog of 80 000 such pairs held by rank 0, sharded over the N ranks
          (strong scaling): pair batches leave rank 0 by grouped NCCL send/recv (sonar_slam_b200/dist.py), are
          solved while the next batch arrives, and the 48-byte results come back by NCCL gather; pairs/s with and
          without the scatter in the timed region

Multi-GPU: one process per GPU (torchrun).  The headline `value` shards frames by rank (weak scaling: F frames
per GPU per step) with no collective on the data path; config5 is the path with a real exchange (scatter of pair
batches from rank 0, gather of SE(2) results).  NCCL's own log is not suppressed or redirected by environment;
what it prints on stdout while communicators come up or go down is diverted to stderr (file descriptor level) so
that stdout stays the one JSON line.
"""
import argparse
import atexit
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

TAU_SOCA = 2.749063720096473   # CFAR(40, 10, 0.1, 10).threshold_factor_SOCA (tests/golden/cfar_tau.json)
R = B = 512
METRIC = "sonar frames/sec (CFAR+ICP)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--frames", type=int, default=4096, help="frames per step and per GPU")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--chunk", type=int, default=256, help="frames per host->device copy chunk (e2e)")
    ap.add_argument("--cpu-sample", type=int, default=1024, help="frames of the bounded CPU-baseline sample")
    ap.add_argument("--minimizer", default="point", choices=["point", "plane"],
                    help="ICP error minimiser: point = the shipped PointToPointErrorMinimizer (icp.yaml:20); plane = the "
                         "PointToPlaneErrorMinimizer icp.yaml:18-19 keeps commented out (normals: knn 5), both arms")
    ap.add_argument("--pairs", type=int, default=80000, help="config 5: size of the scan-match backlog (0: skip)")
    ap.add_argument("--pair-steps", type=int, default=2, help="config 5: timed steps (after one warm-up step)")
    ap.add_argument("--pair-chunks", type=int, default=8, help="config 5: pieces per shard in the pipelined scatter")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (rank 0) as DIR/<name>.npy, to compare two builds")
    return ap.parse_args()


NCU_SUMMARY = os.path.join("profiles", "r02_ncu_full_summaries.json")
NCU_KEY = "prof_cfar_u8gate4"


def ncu_traffic_per_frame():
    """(dram read+write bytes per frame, source) of the pipeline's CFAR kernel.  ncu cannot run inside a timed
    bench (it replays kernels), so this is STATIC: read from this round's committed `ncu --set full` capture of the
    same kernel on a 4096-frame launch (tools/prof_cfar.py 4096 u8 bits); (None, reason) if that file is absent."""
    try:
        with open(os.path.join(REPO, NCU_SUMMARY)) as f:
            d = json.load(f)[NCU_KEY]

        def gb(v):
            x, unit = v.split()
            return float(x) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}[unit]
        return (gb(d["dram__bytes_read.sum"]) + gb(d["dram__bytes_write.sum"])) / 4096.0, \
            f"static: {NCU_SUMMARY}[{NCU_KEY}] (ncu --set full of the same kernel, 4096-frame launch)"
    except Exception as e:  # noqa: BLE001
        return None, f"no committed ncu capture ({type(e).__name__})"


def measured_peak():
    try:
        with open(os.path.join(REPO, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:  # noqa: BLE001
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.proc, self.lines, self.first = gpu_index, None, [], 0

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True).start()
            atexit.register(self._kill)   # an exception on the way must not leave the poller behind
        except Exception:  # noqa: BLE001
            self.proc = None

    def _kill(self):
        if self.proc is not None and self.proc.poll() is None:
            self.proc.terminate()

    def mark(self):
        """The timed region starts here: lines that arrived earlier (start-up, rendering, warm-up) are not counted.
        nvidia-smi needs a few hundred ms before its first line (longer with eight of them starting at once), so it is
        started well before the timed region and only what it prints from here on is reported."""
        self.first = len(self.lines)

    def keep_load_until(self, n, load, timeout=6.0):
        """The timed region of a short run can still be over before `n` lines have arrived since mark(): keep the
        same load running, untimed, until they are in -- they are still clocks under this workload.  Returns the
        number of extra load calls."""
        extra, t_end = 0, time.perf_counter() + timeout
        while (self.proc is not None and self.proc.poll() is None and len(self.lines) - self.first < n
               and time.perf_counter() < t_end):
            load()
            extra += 1
        return extra

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for l in self.lines[self.first:]:
            p = [x.strip() for x in l.split(",")]
            if len(p) < 8:
                continue
            try:
                sm.append(float(p[1]))
                smax.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm), "lines_before_timed_region_not_counted": self.first}


def parse_cpulist(text):
    """'0-3,8,10-11' -> [0, 1, 2, 3, 8, 10, 11] (the sysfs cpulist format)."""
    cpus = []
    for part in text.strip().split(","):
        if not part:
            continue
        a, _, b = part.partition("-")
        cpus += list(range(int(a), int(b or a) + 1))
    return cpus


def bind_near_gpu(pci_domain, pci_bus, pci_device, sysfs="/sys/bus/pci/devices"):
    """Multi-rank runs: restrict this rank's threads to the CPUs next to its GPU (sysfs local_cpulist of the PCI
    device) BEFORE it allocates pinned host memory, so the pinned frames are first-touched on the GPU's own NUMA
    node.  Eight ranks pulling 53 GB/s each through whichever socket the scheduler happened to start them on is what
    made the N = 8 `e2e` swing between 1.31 and 1.59 M frames/s.  Returns a description for the bench line; never
    raises (a box without the sysfs entry keeps the scheduler's placement)."""
    try:
        path = os.path.join(sysfs, f"{pci_domain:04x}:{pci_bus:02x}:{pci_device:02x}.0", "local_cpulist")
        with open(path) as f:
            near = set(parse_cpulist(f.read()))
        allowed = os.sched_getaffinity(0)
        pick = sorted(near & allowed)
        if not pick or len(pick) == len(allowed):
            return {"bound": False, "why": "no narrower local cpulist", "usable_cpus": len(allowed)}
        os.sched_setaffinity(0, pick)
        return {"bound": True, "cpus": len(pick), "of_usable": len(allowed), "source": path}
    except Exception as e:  # noqa: BLE001
        return {"bound": False, "why": f"{type(e).__name__}: {e}"}


# ------------------------------------------------------------------------------------ CPU side
def _cpu_geometry(bearings):
    from oracle import featx_ref
    return featx_ref.Geometry(30.0 / R, R, bearings)


_W = {}


def _cpu_init(bearings):
    from oracle import oracle as orc
    try:  # one thread per worker process: the pool is the parallelism
        import cv2
        cv2.setNumThreads(1)
    except Exception:  # noqa: BLE001
        pass
    _W["geo"] = _cpu_geometry(bearings)
    _W["prm"] = orc.IcpParams(smooth_length=0, max_iterations=20, minimizer=_W.get("minimizer", 0))


def _cpu_cloud(img):
    from oracle import pipeline_ref
    return pipeline_ref.slam_cloud(pipeline_ref.frame_cloud(img, _W["geo"], tau=TAU_SOCA, use_reference=True))


def _cpu_match(job):
    from oracle import oracle as orc, pipeline_ref
    src, parts, guess = job
    tgt = np.concatenate(parts) if parts else np.zeros((0, 2), np.float32)
    if len(tgt):
        tgt, _ = orc.downsample(tgt, 0.5)
    if len(src) < 50 or len(tgt) < 50:
        return 7
    return orc.icp(src, tgt, guess, _W["prm"])["status"]


def cpu_pipeline(frames, poses, bearings, pool=None):
    """The reference's CPU path on `frames` (oracle chain); returns seconds taken."""
    from oracle import pipeline_ref
    t0 = time.perf_counter()
    mapper = pool.map if pool else lambda f, xs: [f(x) for x in xs]
    clouds = mapper(_cpu_cloud, list(frames))
    jobs = []
    for i in range(len(frames)):
        guess = pipeline_ref.between(poses[i - 1], poses[i]) if i > 0 else np.eye(3, dtype=np.float32)
        parts = [pipeline_ref.transform_points(clouds[k], pipeline_ref.between(poses[i - 1], poses[k]))
                 for k in range(max(0, i - 3), i)]
        jobs.append((clouds[i], parts, guess))
    mapper(_cpu_match, jobs)
    return time.perf_counter() - t0


def host_cores():
    """(cores this process may run on, cores the machine reports).  A `fork` pool sized by os.cpu_count() ignores
    cgroup / affinity limits and oversubscribes a restricted box (the round-1 reference arm swung 3.6x between two
    runs for that reason); the affinity mask is what the scheduler will actually give us."""
    try:
        usable = len(os.sched_getaffinity(0))
    except AttributeError:
        usable = os.cpu_count() or 1
    return usable, os.cpu_count() or usable


def run_reference(args):
    """--impl reference: the CPU path on all usable host cores, bounded sample per step, median of the steps."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    import torch  # noqa: F401  (frame renderer)
    from sonar_slam_b200 import synth
    cores, reported = host_cores()
    _W["minimizer"] = 1 if args.minimizer == "plane" else 0   # (inherited by the forked workers)
    n = max(16, min(8 * cores, 1024))
    d = synth.make_trajectory_frames(n, seed=0)
    frames, poses = d["frames"].numpy(), d["poses_odom"]
    ctx = mp.get_context("fork")
    with ctx.Pool(cores, initializer=_cpu_init, initargs=(d["bearings"],)) as pool:
        for _ in range(max(1, args.warmup)):   # warm-up on the FULL sample: page-in, pool start-up, CPU clocks
            cpu_pipeline(frames, poses, d["bearings"], pool)
        secs = [cpu_pipeline(frames, poses, d["bearings"], pool) for _ in range(args.steps)]
    t = float(np.median(secs))
    from oracle import oracle as orc
    val = n / t
    line = {"metric": METRIC, "value": val, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": "config4-pipeline: bounded sample of the bag replay per step",
                       "frames_per_step": n, "image": [R, B], "icp_iterations": 20, "window": 3,
                       "icp_minimizer": args.minimizer,
                       "timing": "median of the timed steps; every step is the full sample",
                       "step_seconds": [round(x, 4) for x in secs]},
            "cpu_baseline": {"value": val, "unit": "frames/s", "cores": cores, "cores_reported_by_os": reported,
                             "kind": "reference+port" if orc.have_reference() else "port",
                             "sample": f"{n} frames/step, frame-parallel over {cores} processes (= len(os.sched_"
                                       f"getaffinity(0)); os.cpu_count() = {reported}): CFAR = reference cfar.cpp "
                                       "compiled unmodified (oracle/_ref) when present, cv2.remap, restated "
                                       "libpointmatcher/PCL filters + ICP (oracle/), keyframe clouds as SLAM reads "
                                       "them (lateral sign flip, slam_ros.py:169-170)"},
            "e2e": {"value": val, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------ GPU side
DUMP_FRAMES = 4096   # --dump-outputs: per-frame results of at most this many frames (a seeded sample of larger steps)
DUMP_CLOUDS = 256    # and the filtered clouds of at most this many of them (<= 256 x cap_points x 8 B = 16 MiB)


def last_step_outputs(ctx, fe, F):
    """What the last sfe_frontend_run_dev call left on the device, read as its caller reads it
    (sfe_frontend_results_dev): for a fixed seeded sample of the F frames (all of them up to DUMP_FRAMES) the scan-match
    result T, iterations, inliers, status and the size of the filtered cloud, and the clouds themselves (x, y rows,
    concatenated in frame order) of a seeded sub-sample.  Integer outputs are stored as float64 (exact)."""
    r = fe.results_dev()
    rng = np.random.default_rng(0)
    frames = np.sort(rng.choice(F, min(F, DUMP_FRAMES), replace=False))
    cloud_frames = np.sort(rng.choice(frames, min(len(frames), DUMP_CLOUDS), replace=False))
    out = {"frame_index": frames.astype(np.float64), "T": ctx.to_host(r["T"], (F, 3, 3), np.float32)[frames]}
    for k in ("iterations", "inliers", "status", "cloud_count"):
        out[k] = ctx.to_host(r[k], (F,), np.int32)[frames].astype(np.float64)
    stride, count = r["cloud_stride"], ctx.to_host(r["cloud_count"], (F,), np.int32)
    clouds = [ctx.to_host(r["cloud_xy"] + int(f) * stride * 8, (min(int(count[f]), stride), 2), np.float32)
              for f in cloud_frames]
    out["cloud_frame_index"] = cloud_frames.astype(np.float64)
    out["cloud_xy"] = np.concatenate(clouds) if clouds else np.zeros((0, 2), np.float32)
    return out


def dump_outputs(directory, arrays):
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def make_pair_backlog(P, device, n_scenes=32, ns=2000, nt=20000):
    """Config 3 / 5 input on `device`: P (source, target, guess) records tiled from `n_scenes` seeded scenes of
    synth.make_icp_pair (SURVEY 8(d) config 3: 2 000-point scan vs 20 000-point submap, identity guess).  The solver
    keeps no state between problems, so repeating scenes does not help it; the bytes moved are those of P distinct
    pairs.  Scenes whose thinned target falls short of `nt` points are skipped (records have a fixed size)."""
    import torch
    from sonar_slam_b200 import synth
    src, tgt, seed = [], [], 0
    while len(src) < n_scenes:
        a, b, _ = synth.make_icp_pair(seed, n_source=ns, n_target=nt)
        seed += 1
        if len(a) == ns and len(b) == nt:
            src.append(a), tgt.append(b)
    src_s = torch.from_numpy(np.stack(src)).to(device)
    tgt_s = torch.from_numpy(np.stack(tgt)).to(device)
    idx = torch.arange(P, device=device) % n_scenes
    return src_s[idx].contiguous(), tgt_s[idx].contiguous(), torch.eye(3, device=device).repeat(P, 1, 1).contiguous()


def run_ours(args):
    import torch
    import torch.distributed as dist
    from sonar_slam_b200 import _lib, ops, pipeline, synth
    from sonar_slam_b200 import dist as sdist
    from sonar_slam_b200.bruce_slam.feature_extraction import FeatureExtraction

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- this benchmark has no CPU fallback for the product path")
    torch.cuda.set_device(local)
    clocks = ClockSampler(local)   # started now, counted from clocks.mark() at the start of the timed region
    clocks.start()
    if world > 1:
        # NCCL's log is left alone (NCCL_DEBUG / NCCL_DEBUG_FILE are whatever the caller set; the driver counts ranks
        # in it).  stdout carries the one JSON line, so what NCCL prints there while the communicators come up (its
        # version line, NCCL_DEBUG=INFO output) is sent to stderr by pointing file descriptor 1 at stderr until the
        # first collective and the first send/recv have completed -- and again after the JSON line is out.
        opts = None
        try:  # high-priority communication stream: send/recv kernels are scheduled as soon as an SM frees up
            opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
        except Exception:  # noqa: BLE001
            opts = None
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local), pg_options=opts)
            warm = torch.zeros(1, device="cuda")
            dist.all_reduce(warm)
            if rank == 0:  # both directions of every (0, r) pair: the scatter's sends and the gather's
                for q in dist.batch_isend_irecv([dist.P2POp(dist.isend, warm, r) for r in range(1, world)]):
                    q.wait()
            else:
                for q in dist.batch_isend_irecv([dist.P2POp(dist.irecv, warm, 0)]):
                    q.wait()
            dist.gather(warm, [torch.zeros(1, device="cuda") for _ in range(world)] if rank == 0 else None, dst=0)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    F, K, W = args.frames, args.steps, args.warmup
    numa = {"bound": False, "why": "single rank"}
    if world > 1:
        prop = torch.cuda.get_device_properties(local)
        numa = bind_near_gpu(getattr(prop, "pci_domain_id", 0), prop.pci_bus_id, prop.pci_device_id)

    # ---- synthetic bag replay for this rank (frames stay resident in HBM; > L2 by far: F*256 KiB).  Every rank replays
    #      the SAME seeded bag: the stages' cost follows the scene (detections, cloud sizes), and with one scene per
    #      rank the max over ranks measured the unluckiest scene (+7 % at N = 8), not the parallel overhead
    d = synth.make_trajectory_frames(F, seed=0, device=f"cuda:{local}")
    frames_dev, poses = d["frames"], d["poses_odom"]
    fx = FeatureExtraction()
    fx.generate_map_xy(synth.Ping(0, None, 30.0 / R, R, d["bearings"]))
    ctx = ops.context(local)
    maps = _lib.Maps(ctx, fx.map_x, fx.map_y, R, B, fx.width, fx.height)
    mini = _W["minimizer"] = 1 if args.minimizer == "plane" else 0
    fe = pipeline.FrontEnd(ctx, maps, max_frames=F, tau=TAU_SOCA,
                           icp=_lib.IcpParams(smooth_length=0, max_iterations=20, minimizer=mini))
    host_frames_t = torch.empty((F, R, B), dtype=torch.uint8, pin_memory=True)
    host_frames_t.copy_(frames_dev)
    host_frames = host_frames_t.numpy()
    out = fe.alloc_results(F)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident leg (no stage events inside the timed loop)
    for _ in range(W):
        fe.run_dev(frames_dev.data_ptr(), poses, F)
    barrier()
    clocks.mark()
    l0 = ctx.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        fe.run_dev(frames_dev.data_ptr(), poses, F)
    e1.record()
    barrier()
    dev_ms = max_over_ranks(e0.elapsed_time(e1))
    launches = ctx.launches - l0
    # read now: the legs below run on the same handle and overwrite the results
    outputs = last_step_outputs(ctx, fe, F) if args.dump_outputs and rank == 0 else None

    # ---- end-to-end leg: host buffers in, results out, through one C-ABI call per step
    for _ in range(W):
        fe.run_host(host_frames, poses, chunk_frames=args.chunk, out=out)
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        fe.run_host(host_frames, poses, chunk_frames=args.chunk, out=out)
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)

    # ---- separate pass with per-stage CUDA events on the launch stream (the roofline's kernel time, stage shares)
    fe.set_timing(True)
    for _ in range(K):
        fe.run_dev(frames_dev.data_ptr(), poses, F)
    stage = fe.get_timing()
    fe.set_timing(False)

    def _load():
        fe.run_dev(frames_dev.data_ptr(), poses, F)
        torch.cuda.synchronize()
    extra_load = clocks.keep_load_until(3, _load)
    clk = clocks.stop()
    clk["untimed_load_steps_while_sampling"] = extra_load
    barrier()

    matched = int((out["status"] == 0).sum())
    stats = torch.tensor([float(matched), float(out["npoints"].mean())], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)

    # ---- config 3 (rank 0) and config 5 (all ranks): 2 000 x 20 000-point scan matches
    cfg3, cfg5 = None, None
    prm20 = _lib.IcpParams(smooth_length=0, max_iterations=20, minimizer=mini)
    try:
        if rank == 0:
            P3 = 8 * torch.cuda.get_device_properties(local).multi_processor_count
            s3, t3, g3 = make_pair_backlog(P3, f"cuda:{local}", n_scenes=16)
            cfg3 = {"pairs": P3, "source_points": 2000, "target_points": 20000, "waves": 8}
            for name, prm in (("fixed20", prm20), ("checkers", _lib.IcpParams(minimizer=mini))):
                for _ in range(2):
                    r3 = sdist.unpack_results(sdist._default_icp(s3, t3, g3, prm))
                ts = []
                for _ in range(3):
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    r3 = sdist.unpack_results(sdist._default_icp(s3, t3, g3, prm))
                    b.record()
                    torch.cuda.synchronize()
                    ts.append(a.elapsed_time(b))
                ms = float(np.median(ts))
                cfg3[name] = {"pairs_per_s": P3 / (ms * 1e-3), "ms_per_wave_of_148": ms / 8, "ms": ms,
                              "mean_iterations": float(r3["iterations"].float().mean().item()),
                              "converged": int((r3["status"] == 0).sum().item())}
            del s3, t3, g3
        if args.pairs > 0:
            P5 = args.pairs
            sa, ta, ga = make_pair_backlog(P5, f"cuda:{local}") if rank == 0 else (None, None, None)
            barrier()

            def timed(fn, reps):
                """max over ranks of the device time of `fn` (CUDA events on this rank's stream), per repetition"""
                barrier()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(reps):
                    res = fn()
                b.record()
                barrier()
                return max_over_ranks(a.elapsed_time(b)) / reps, res

            # (a) the whole step: pipelined scatter -> solve -> gather (the product path, sonar_slam_b200/dist.py)
            step = lambda: sdist.run_pair_backlog(P5, 2000, 20000, prm20, sa, ta, ga, chunks=args.pair_chunks)
            timed(step, 1)
            ms_step, packed = timed(step, args.pair_steps)
            # (b) its parts, each alone: one-shot scatter; solve + gather on the resident shard
            ms_scatter, shard = timed(lambda: sdist.scatter_pairs(P5, 2000, 20000, sa, ta, ga), 1)
            solve = lambda: sdist.gather_pair_results(sdist._default_icp(*shard, prm20), P5)
            timed(solve, 1)
            ms_solve, packed2 = timed(solve, args.pair_steps)
            if rank == 0:
                r5 = sdist.unpack_results(packed)
                same = bool(torch.equal(packed, packed2))
                per_pair = (2000 + 20000) * 8 + 36
                cfg5 = {"pairs_total": P5, "scaling": "strong (fixed backlog)", "n_gpus": world,
                        "pairs_per_s_incl_scatter_gather": P5 / (ms_step * 1e-3),
                        "pairs_per_s_without_scatter": P5 / (ms_solve * 1e-3),
                        "ms_step_pipelined": ms_step, "ms_solve_and_gather_resident": ms_solve,
                        "ms_scatter_alone": ms_scatter,
                        "scatter_GBps_from_rank0": (P5 - P5 // world) * per_pair / (ms_scatter * 1e-3) / 1e9 if world > 1 else None,
                        "scatter_bytes": (P5 - P5 // world) * per_pair if world > 1 else 0,
                        "gather_bytes": P5 * 4 * sdist.RESULT_WORDS if world > 1 else 0,
                        "chunks_per_shard": args.pair_chunks, "timed_steps": args.pair_steps,
                        "converged": int((r5["status"] == 0).sum().item()),
                        "pipelined_equals_resident_results": same,
                        "transport": "grouped NCCL send/recv (dist.batch_isend_irecv) + NCCL gather" if world > 1 else "none (one rank)"}
            del sa, ta, ga, shard
    except Exception as e:  # noqa: BLE001
        cfg5 = {"error": f"{type(e).__name__}: {e}"}
        if world > 1:
            raise

    if rank == 0:
        peak, peak_src = measured_peak()
        total_ms = sum(v[0] for v in stage.values())
        cfar_ms, cfar_calls = stage["cfar"]
        cfar_bytes = F * R * B * (1 + 1 / 8)            # uint8 image in, bit plane out, per launch
        achieved = cfar_bytes / (cfar_ms / max(1, cfar_calls) * 1e-3) / 1e9
        traffic_pf, traffic_src = ncu_traffic_per_frame()
        line = {
            "metric": METRIC, "value": world * F * K / (dev_ms * 1e-3), "unit": "frames/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "config4-pipeline: synthetic bag replay, CFAR(SOCA 40/10, Pfa 0.1, gate 65) -> "
                                   "cloud -> voxel 0.5 m -> outlier(1.0 m, 5) -> keyframe cloud (x, -z) -> ICP 20 "
                                   "iterations vs 3-frame submap",
                       "frames_per_step_per_gpu": F, "image": [R, B], "image_dtype": "u8", "icp_iterations": 20,
                       "icp_minimizer": args.minimizer,
                       "window": 3, "sharding": "frames by rank (every rank replays the same seeded bag), no data-path collective",
                       "l2": f"inputs larger than L2 ({F * R * B / 2**20:.0f} MiB of frames per step)",
                       "host_numa_binding_rank0": numa,
                       "frames_matched_last_step": int(stats[0].item()),
                       "mean_cloud_points": float(stats[1].item() / world)},
            "clocks": clk,
            "e2e": {"value": world * F * K / e2e_s, "unit": "frames/s",
                    "h2d_bytes_per_step": F * R * B + F * 4 * 9 * 4, "d2h_bytes_per_step": F * (36 + 16)},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "cfar_u8_gate4_kernel<SOCA, bits>", "achieved": achieved,
                         "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": (traffic_pf * F) if traffic_pf else None, "traffic_source": traffic_src,
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": cfar_bytes,
                         "kernel_ms_per_launch": cfar_ms / max(1, cfar_calls),
                         "timing": "CUDA events on the launch stream around the kernel, separate pass after the "
                                   "timed steps (the timed `value` loop carries no stage events)"},
            "stage_share": {k: (v[0] / total_ms if total_ms else None) for k, v in stage.items()},
            "stage_ms_per_step": {k: v[0] / K for k, v in stage.items()},
            "config3_icp": cfg3, "config5": cfg5,
        }
        # config 2 (SURVEY 8(d) primary definition: float32 frames in, uint8 mask out), same run
        try:
            x = frames_dev.float()
            for _ in range(3):
                ops.cfar(x, "SOCA", 20, 5, TAU_SOCA, gate=65)
            ts = []
            for _ in range(10):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                ops.cfar(x, "SOCA", 20, 5, TAU_SOCA, gate=65)
                b.record()
                torch.cuda.synchronize()
                ts.append(a.elapsed_time(b))
            by = F * R * B * 5
            ach = by / (float(np.median(ts)) * 1e-3) / 1e9
            line["roofline_config2_cfar_f32"] = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s",
                                                 "frac": ach / peak, "frac_of_8TBps_nominal": ach / 8000.0,
                                                 "ms_median_of_10": float(np.median(ts)), "frames": F,
                                                 "algorithmic_bytes_per_launch": by,
                                                 "note": "outside the timed pipeline steps; includes the flag memset and "
                                                         "the exact-path sweep launch"}
            del x
        except Exception as e:  # noqa: BLE001
            line["roofline_config2_cfar_f32"] = {"error": str(e)}
        # CPU baseline on a bounded sample (N = 1 only)
        if world == 1:
            try:
                from oracle import oracle as orc
                n = min(args.cpu_sample, F)
                _cpu_init(d["bearings"])
                sample = frames_dev[:n].cpu().numpy()
                secs = cpu_pipeline(sample, poses[:n], d["bearings"])
                usable, reported = host_cores()
                line["cpu_baseline"] = {"value": n / secs, "unit": "frames/s", "cores": 1,
                                        "kind": "reference+port" if orc.have_reference() else "port",
                                        "sample": f"first {n} frames of the step ({secs:.1f} s), one thread ({usable} "
                                                  f"usable host cores, os.cpu_count() = {reported}): reference cfar.cpp "
                                                  "(unmodified, oracle/_ref) + cv2.remap + restated libpointmatcher/PCL "
                                                  "filters and ICP (oracle/)"}
            except Exception as e:  # noqa: BLE001
                line["cpu_baseline"] = {"error": str(e)}
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    if world > 1:
        sys.stdout.flush()
        os.dup2(2, 1)  # communicator tear-down messages (NCCL_DEBUG=INFO) must not follow the JSON line on stdout
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
