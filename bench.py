#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric (GICP scans/sec) on BASELINE.json's configs.

    python bench.py [--config c2|c3|c4|c5] [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

--config c2 (default, BASELINE configs[1], the configuration the metric is quoted on): scan-to-scan odometry.
    A synthetic 64-beam stream of 100 scans, 131072 rays each (tools/gen_lidar.py); per scan
        VoxelGrid (130k -> ~30k)  ->  setInputSource(new) + setInputTarget(previous filtered) + align()
    with the odometry settings of SURVEY.md 8d/C2 (50 outer / 20 inner BFGS iterations, corr 1.0 m, tf_eps 1e-3,
    k-NN(20) covariances).  Source AND target index + covariances are rebuilt for every scan, exactly like the
    reference's callers (PointCloudOdometry.cc:265-267).
      value          scans/s of ONE scan stream through lb_odometry_* (the library's pipelined form of that chain:
                     scan k+1 is filtered and indexed while scan k is in its align kernel, `depth` aligns in flight;
                     results identical to the per-scan calls, checked here), inputs resident in HBM, CUDA events.
                     A step = one batch of --scans-per-step (16) consecutive scans.
      e2e            the same pipeline with HOST (pinned) buffers: H2D of every raw scan, D2H of its filtered cloud and
                     of the pose inside the timed region.
      sequential     THE DROP-IN SEAM: the blocking per-scan C-ABI calls the reference's callers make (lb_voxel_filter,
                     lb_gicp_set_source / set_target, lb_gicp_align), one scan at a time, device-resident inputs, L2
                     flushed between scans.  sequential_e2e: the same calls with HOST buffers (copies inside the
                     timed region).  These are what `icp_->align()` inside LOCUS's queue-depth-1 lidar callback sees.
--config c3 (BASELINE configs[2], the shape north_star's ">= 100x" is stated on): scan-to-submap localization.
    ~30k-point filtered scan vs the 500000-point rolling submap built from 40 posed scans of the same scene
    (SURVEY 8d), localization settings (corr 0.2 m, tf_eps 1e-5, 50 inner), prior = true pose off by a few cm.
    Blocking per-scan calls (the seam).  A step = one scan.
      value / e2e    the submap stays resident between scans (set_target once; SURVEY 8d: "submap index built once,
                     reused"); device-resident / host buffers.
      variants.submap_rebuilt_every_scan   set_target(submap) before every align: index + k-NN(20) covariances of
                     the 500k points rebuilt per scan, which is what LOCUS's callers do today.
--config c4 (BASELINE configs[3]): c3 with one independent stream per GPU (seeds 10..17), torchrun, no collective.
--config c5 (BASELINE configs[4], dense stress): 1M-ray scan -> VoxelGrid ~200k vs a resident 10M-point map; the
    roofline object is the NN-search kernel (the HBM-bound kernel of this path) on the scan's 200k queries.
--impl reference: the CPU arm = oracle/ (C port of the reference; the reference itself needs PCL/ROS and cannot be
    built here), all host threads, the same config, each step a bounded sample of the b200 arm's step (one scan).
--dump-outputs DIR: after the timed steps, what the headline arm returned in its LAST timed step, as DIR/<name>.npy
    (float32 / float64; rank 0's stream).  c2: per scan of the step, the pipeline's pose and align result
    (final_transformation, converged, iterations, n_correspondences, delta, n_filtered); c3-c5: the same for the step's
    one scan plus its filtered cloud (filtered_cloud, x y z intensity).  The inputs are generated from fixed seeds and
    the step's scans depend only on the arguments, so two builds run with the same arguments can be compared output
    for output.

N>1 (torchrun): one independent scan stream per GPU (weak scaling, no data-path collective); barrier + device sync
on both sides of the timed region, max over ranks.
"""
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

from tools import gen_lidar as G  # noqa: E402

POINT_STEP = 32
N_STREAM = 100          # distinct scans of the c2 stream (SURVEY 8d: "stream of 100 scans")
CONFIGS = {
    "c2": dict(name="C2 scan-to-scan odometry", beams=64, az=2048, voxels=30000, n_stream=N_STREAM,
               gicp=dict(max_iterations=50, max_inner=20, corr_dist=1.0, tf_eps=1e-3, k=20)),
    "c3": dict(name="C3 scan-to-submap localization", beams=64, az=2048, voxels=30000, n_stream=24, map_scans=40,
               submap=500_000, gicp=dict(max_iterations=50, max_inner=50, corr_dist=0.2, tf_eps=1e-5, k=20)),
    "c4": dict(name="C4 batched scan-to-submap localization (one stream per GPU)", beams=64, az=2048, voxels=30000,
               n_stream=24, map_scans=40, submap=500_000,
               gicp=dict(max_iterations=50, max_inner=50, corr_dist=0.2, tf_eps=1e-5, k=20)),
    "c5": dict(name="C5 dense stress", beams=128, az=8192, voxels=200_000, n_stream=6, map_scans=24, submap=10_000_000, merge="subsample",
               gicp=dict(max_iterations=50, max_inner=50, corr_dist=0.2, tf_eps=1e-5, k=20)),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default=os.environ.get("LB_CONFIG", "c2"), choices=sorted(CONFIGS))
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--scans-per-step", type=int, default=int(os.environ.get("LB_BATCH", "16")),
                    help="c2: one step = one batch of this many consecutive scans of the stream (b200 arm)")
    ap.add_argument("--depth", type=int, default=int(os.environ.get("LB_DEPTH", "8")),
                    help="c2: registration workers of the odometry pipeline (aligns in flight)")
    ap.add_argument("--pipeline-ppc", type=int, default=int(os.environ.get("LB_PIPE_PPC", "1024")),
                    help="c2: align_points_per_cta of the pipeline's registration workers (sequential arm: library default 512)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-baseline-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--leaf", type=float, default=0.0, help="fixed VoxelGrid leaf (skips the bisection; profiling aid)")
    ap.add_argument("--stream-scans", type=int, default=0, help="distinct scans of the stream (0 = the config's; profiling aid)")
    ap.add_argument("--profile", action="store_true",
                    help="profiling aid for ncu: the blocking per-scan calls only (no pipeline, no e2e arm, no CPU baseline)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the timed path returned in its last step as DIR/<name>.npy "
                         "(c2: the pipeline's results for the step's scans; c3-c5: the align result and the filtered scan)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.profile):
        ap.error("--dump-outputs writes the outputs of the b200 arm's timed path (not with --impl reference or --profile)")
    return args


# ------------------------------------------------------------------------------------------ helpers
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region.  NVML in a thread (a few microseconds per
    query) when nvidia_ml_py is importable; otherwise an `nvidia-smi -lms` subprocess.  (Eight nvidia-smi pollers on
    an 8-GPU box visibly slowed the arm they ran next to, so the in-process NVML path is preferred.)"""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index, period_s=0.1):     # an NVML query every 10 ms was measured to stall the blocking calls it sampled
        self.index = index
        self.period = period_s
        self.rows = []
        self.proc = None
        self.nvml = None
        self.stop_flag = False
        self.sm, self.mx, self.reasons = [], None, set()

    def _visible_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[self.index])
            except (ValueError, IndexError):
                return None          # UUID list: let the nvidia-smi path deal with it
        return self.index

    def start(self):
        if os.environ.get("LB_NO_SAMPLER"):      # diagnostic: is the sampling itself perturbing the arm it watches?
            return
        try:
            import pynvml
            pynvml.nvmlInit()
            idx = self._visible_index()
            if idx is None:
                raise RuntimeError("no integer device index")
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll_nvml(self):
        N = self.nvml
        names = [("hw_slowdown", "nvmlClocksEventReasonHwSlowdown"), ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown"),
                 ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown"), ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap")]
        masks = [(n, getattr(N, a, 0)) for n, a in names]
        while not self.stop_flag:
            try:
                self.sm.append(float(N.nvmlDeviceGetClockInfo(self.h, N.NVML_CLOCK_SM)))
                r = int(N.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                for n, m in masks:
                    if m and (r & m):
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(self.period)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if os.environ.get("LB_NO_SAMPLER"):
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": "disabled (LB_NO_SAMPLER)"}
        if self.nvml is not None:
            self.stop_flag = True
            self.thread.join(timeout=2)
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.mx,
                    "reasons": sorted(self.reasons), "samples": len(self.sm), "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for nme, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvidia-smi"}


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def seq(i, n=None):
    """position in the stream of the i-th scan handed to a pipelined arm: forward through the stream, then back
    (ping-pong), so that consecutive scans are always neighbouring poses however many scans a run needs"""
    n = N_STREAM if n is None else n
    p = 2 * (n - 1)
    r = i % p
    return r if r < n else p - r


def stream_seed(rank, config="c2"):
    """scan stream s -> GPU s: independent streams, one per rank (SURVEY 8e); rank 0 is the N=1 workload.
    c4: seeds 10..17 (SURVEY 8d)"""
    return (10 + rank) if config == "c4" else (2 + 8 * rank)


def make_stream(rank, n_scans=N_STREAM, beams=64, az=2048, config="c2"):
    scene, poses, blobs = G.stream(stream_seed(rank, config), n_scans, beams, az)
    return poses, blobs


def aggregate(dist, device, times_ms, steps, world):
    """max over ranks of the per-rank device times; whole-job throughput = all ranks' scans / that time.
    steps: scans per rank behind each time (one number, or one per entry of times_ms)"""
    import torch
    t = torch.tensor(list(times_ms), dtype=torch.float64, device=device)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    tmax = [float(x) for x in t]
    counts = list(steps) if isinstance(steps, (list, tuple)) else [steps] * len(tmax)
    return tmax, [c * world / (x / 1e3) if x > 0 else 0.0 for c, x in zip(counts, tmax)]


def bisect_leaf(count_fn, target, lo=0.02, hi=2.0, rounds=18):
    """VoxelGrid leaf such that the filter output is ~target points (SURVEY 8d: "leaf chosen once by bisection")"""
    for _ in range(rounds):
        mid = 0.5 * (lo + hi)
        if count_fn(mid) > target:
            lo = mid
        else:
            hi = mid
    return float(np.float32(0.5 * (lo + hi)))


def oracle_voxel_fn(O, limits=False):
    def fn(blob, leaf):
        if limits:
            return O.voxel_filter(blob, POINT_STEP, leaf, float_fields=G.FLOAT_FIELDS, filter_field_offset=G.Z_OFF,
                                  limit_min=-100.0, limit_max=100.0)["out"]
        return O.voxel_filter(blob, POINT_STEP, leaf, float_fields=G.FLOAT_FIELDS)["out"]
    return fn


def describe(args, world, cfg):
    """config object of the JSON line: a pure function of the command line, identical in both --impl arms"""
    g = cfg["gicp"]
    gi = "GICP (<=%d outer, %d inner BFGS, corr %.1f m, tf_eps %g, kNN(%d) covariances)" % (
        g["max_iterations"], g["max_inner"], g["corr_dist"], g["tf_eps"], g["k"])
    rays = cfg["beams"] * cfg["az"]
    w = {"name": args.config, "raw_points_per_scan": rays, "streams": world, "parallelism": "stream-per-gpu x%d" % world,
         "optimizer": "bfgs (reference-exact)", "distinct_scans_per_stream": cfg["n_stream"]}
    if args.config == "c2":
        w["workload"] = ("C2 scan-to-scan odometry: %d-ray synthetic 64-beam scan -> VoxelGrid ~%dk -> %s against the "
                         "previous filtered scan" % (rays, cfg["voxels"] // 1000, gi))
        w["index"] = ("blocking-call arms: the caller hands over source AND target for every scan, like the reference's callers; "
                      "the library recognises a target that equals the previous source bit for bit and adopts its index + "
                      "covariances (the CPU arm rebuilds both, as the reference does); pipeline arms: each filtered scan's index + "
                      "covariances computed once and adopted as the next registration's target (bit-identical poses; "
                      "variants.pipeline_rebuild_both_clouds rebuilds them)")
        w["l2"] = ("inputs larger than L2: %d distinct raw scans of %.1f MB cycled; blocking-call arms: L2 flushed "
                   "between scans by a 256 MiB write" % (cfg["n_stream"], rays * POINT_STEP / 1e6))
        w["pipeline"] = "lb_odometry: 1 VoxelGrid stage + %d registration workers, %d source points per align CTA, one scan stream" % (
            args.depth, args.pipeline_ppc)
        w["scans_per_step"] = args.scans_per_step
        w["step"] = ("one batch of %d consecutive scans of the stream submitted to the pipeline (the reference arm's "
                     "step is a bounded sample of that batch: one scan)" % args.scans_per_step)
    else:
        w["workload"] = ("%s: %d-ray synthetic %d-beam scan -> VoxelGrid ~%dk -> %s against the %d-point submap "
                         "(%s union of %d posed scans of the same scene), prior = true pose off by <= 5 cm / 0.4 deg"
                         % (cfg["name"], rays, cfg["beams"], cfg["voxels"] // 1000, gi, cfg["submap"],
                            "randomly subsampled" if cfg.get("merge") == "subsample" else "voxel-merged", cfg["map_scans"]))
        w["index"] = ("submap index + covariances built once and kept while the submap is unchanged (value, e2e); "
                      "rebuilt before every align in variants.submap_rebuilt_every_scan (what LOCUS's callers do)")
        w["l2"] = "L2 flushed between scans by a 256 MiB write"
        w["pipeline"] = "blocking per-scan calls (the drop-in seam): lb_voxel_filter, lb_gicp_set_source, lb_gicp_align(prior)"
        w["scans_per_step"] = 1
        w["step"] = "one scan"
    return w


# ------------------------------------------------------------------------------------------ workload data
def build_data(args, cfg, rank, voxel_fn, voxel_limits_fn):
    """synthetic inputs of this rank's stream: raw scans, poses, VoxelGrid leaf, and for c3-c5 the submap + priors.
    voxel_fn(blob, leaf) -> filtered blob without limits (submap merge); voxel_limits_fn: with z limits (scan leaf)."""
    seed = stream_seed(rank, args.config)
    t0 = time.time()
    if args.config == "c2":
        scene, poses, blobs = G.stream(seed, cfg["n_stream"], cfg["beams"], cfg["az"])
        d = {"poses": poses, "blobs": blobs}
    else:
        w = G.c3_workload(seed, cfg["n_stream"], voxel_fn, n_map_scans=cfg["map_scans"], n_submap=cfg["submap"],
                          beams=cfg["beams"], az=cfg["az"], merge=cfg.get("merge", "voxel"))
        d = {"poses": w["poses"], "blobs": w["blobs"], "submap": w["submap"], "submap_leaf": w["submap_leaf"],
             "guesses": w["guesses"], "union_points": w["union_points"]}
    leaf = args.leaf if args.leaf > 0 else bisect_leaf(lambda l: voxel_limits_fn(d["blobs"][0], l).shape[0], cfg["voxels"])
    d["leaf"] = float(np.float32(leaf))
    d["gen_s"] = time.time() - t0
    return d


# ------------------------------------------------------------------------------------------ CPU arm
def oracle_params(O, g, threads):
    return O.default_params(transformation_epsilon=g["tf_eps"], corr_dist_threshold=g["corr_dist"],
                            max_iterations=g["max_iterations"], max_inner_iterations=g["max_inner"],
                            k_correspondences=g["k"], num_threads=threads)


def cpu_filter(O, blob, leaf):
    r = O.voxel_filter(blob, POINT_STEP, leaf, float_fields=G.FLOAT_FIELDS, filter_field_offset=G.Z_OFF,
                       limit_min=-100.0, limit_max=100.0)
    return np.ascontiguousarray(r["out"]).view(np.float32).reshape(-1, 8)


_CPU_THREADS = {}


def pick_cpu_threads(O, probe):
    """The reference parallelises covariances + NN look-ups with OpenMP (objective serial); on a many-core host more
    threads is not always faster, so give the CPU arm its best thread count (untimed probe of one scan)."""
    if "n" in _CPU_THREADS:
        return _CPU_THREADS["n"]
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (4, 8, 16, 32, 64, ncpu) if c <= ncpu})
    best, best_t = cands[0], None
    for c in cands:
        t0 = time.perf_counter()
        probe(c)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = c, dt
    _CPU_THREADS["n"] = best
    return best


PROBE_PAIRS = 30        # scans per config on which the reference's own sensitivity to summation order is measured
PROBE_CHUNKS = (64, 256, 1024, 4096, 16384)


def run_cpu_arm(args, cfg, data, budget_s=None, max_steps=None, rebuild_target=False, probe=None):
    """Times the oracle (C port of the reference, OpenMP like the reference: covariances + NN look-ups parallel,
    objective serial) on the same stream, one scan per step.  returns (scans_per_s, n_scans, {key: pose}, cores).
    c2: key = (previous position, position); c3-c5: key = position."""
    from oracle import oracle as O
    O.build()
    g, leaf, blobs = cfg["gicp"], data["leaf"], data["blobs"]
    poses = {}
    if args.config == "c2":
        f0 = cpu_filter(O, blobs[0], leaf)
        f1 = cpu_filter(O, blobs[1], leaf)
        cores = pick_cpu_threads(O, lambda c: O.gicp_align(f1, f0, oracle_params(O, g, c)))
        prm = oracle_params(O, g, cores)
        prev, n, t_total, i = f0, 0, 0.0, 1
        while True:
            t0 = time.perf_counter()
            cur = cpu_filter(O, blobs[seq(i, len(blobs))], leaf)
            res = O.gicp_align(cur, prev, prm)
            t_total += time.perf_counter() - t0
            key = (seq(i - 1, len(blobs)), seq(i, len(blobs)))
            poses[key] = res["T"]
            if probe is not None and len(probe) < PROBE_PAIRS:
                probe[key] = (lambda a=cur, b=prev: O.gicp_align(a, b, prm))
            prev = cur
            n += 1; i += 1
            if max_steps is not None and n >= max_steps:
                break
            if budget_s is not None and (t_total >= budget_s or n >= len(blobs) - 1):
                break
        return n / t_total, n, poses, cores
    sub = np.ascontiguousarray(data["submap"], dtype=np.float32)
    f0 = cpu_filter(O, blobs[0], leaf)
    tgt, t_prep = None, 0.0
    if rebuild_target:
        cores = min(os.cpu_count() or 1, 64)
    else:
        t_prep0 = time.perf_counter()
        tgt = O.PreparedTarget(sub, oracle_params(O, g, min(os.cpu_count() or 1, 64)))     # covariances do not depend on the thread count
        t_prep = time.perf_counter() - t_prep0
        cores = pick_cpu_threads(O, lambda c: tgt.align(f0, oracle_params(O, g, c), guess=data["guesses"][0]))
    prm = oracle_params(O, g, cores)
    n, t_total = 0, 0.0
    while True:
        j = n % len(blobs)
        t0 = time.perf_counter()
        cur = cpu_filter(O, blobs[j], leaf)
        res = O.gicp_align(cur, sub, prm, guess=data["guesses"][j]) if rebuild_target else tgt.align(cur, prm, guess=data["guesses"][j])
        t_total += time.perf_counter() - t0
        poses[j] = res["T"]
        if probe is not None and tgt is not None and len(probe) < PROBE_PAIRS:
            probe[j] = (lambda a=cur, jj=j: tgt.align(a, prm, guess=data["guesses"][jj]))
        n += 1
        if max_steps is not None and n >= max_steps:
            break
        if budget_s is not None and (t_total >= budget_s or n >= len(blobs)):
            break
    data["cpu_submap_prepare_s"] = t_prep
    if probe is not None:
        data["_cpu_target"] = tgt            # kept alive for the (untimed) re-association probes; closed by the caller
    elif tgt is not None:
        tgt.close()
    return n / t_total, n, poses, cores


def reassociation_probe(cpu_poses, probe):
    """How far does the REFERENCE's own pose move when only the association of its double sums changes (partial sums
    over blocks of 512 / 4096 correspondences; oracle.set_sum_chunk)?  Untimed.  returns {key: max (dt, dr) over the
    probes}.  Pairs that do not move are 'decisive': there, and only there, a parallel implementation can be held to
    the 1e-4 bar (tests/test_oracle.py::test_reference_pose_depends_on_summation_order, DESIGN.md "Numerics")."""
    from oracle import oracle as O
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import fixtures as F
    out = {}
    for key, rerun in probe.items():
        worst = (0.0, 0.0)
        for c in PROBE_CHUNKS:
            O.set_sum_chunk(c)
            try:
                d = F.pose_delta(cpu_poses[key], rerun()["T"])
            finally:
                O.set_sum_chunk(0)
            worst = (max(worst[0], d[0]), max(worst[1], d[1]))
        out[key] = worst
    return out


def reference_arm(args, cfg, workload):
    """--impl reference: rank 0 only; the same config, one scan per step"""
    from oracle import oracle as O
    O.build()
    G.WORKERS = max(1, min(16, (os.cpu_count() or 1)))
    data = build_data(args, cfg, 0, oracle_voxel_fn(O), oracle_voxel_fn(O, limits=True))
    workload["leaf_m"] = data["leaf"]
    if "submap_leaf" in data:
        workload["submap_leaf_m"] = data["submap_leaf"]
    run_cpu_arm(args, cfg, data, max_steps=max(1, min(args.warmup, 2)))            # warm-up
    sps, n, _, cores = run_cpu_arm(args, cfg, data, max_steps=max(1, args.steps))
    what = "scans of the same stream" if args.config == "c2" else "scans against the kept submap (kd-tree + covariances prepared once, %.1f s, untimed)" % data.get("cpu_submap_prepare_s", 0.0)
    line = {"impl": "reference", "metric": "gicp_scans_per_sec", "value": sps, "unit": "scans/s", "n_gpus": args.gpus,
            "steps": n, "warmup": args.warmup, "ms_per_step": 1000.0 / sps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32 points / f64 accumulation", "data": "synthetic",
            "config": workload,
            "cpu_baseline": {"value": sps, "unit": "scans/s", "cores": cores, "kind": "port",
                             "sample": "%d %s (oracle/: C port of multithreaded_gicp + PCL VoxelGrid; the reference "
                                       "itself needs PCL/ROS, unbuildable here)" % (n, what)},
            "e2e": {"value": sps, "unit": "scans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ main
def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cfg = dict(CONFIGS[args.config])
    if args.stream_scans > 0:
        cfg["n_stream"] = max(3, args.stream_scans)
    workload = describe(args, world, cfg)

    if args.impl == "reference":
        if rank == 0:
            reference_arm(args, cfg, workload)
        return

    # ray-cast this rank's scans before CUDA is touched (the worker pool forks)
    G.WORKERS = max(1, min(16, (os.cpu_count() or 1) // max(1, world)))
    seed = stream_seed(rank, args.config)
    t_gen0 = time.time()
    if args.config == "c2":
        scene, poses_, blobs_ = G.stream(seed, cfg["n_stream"], cfg["beams"], cfg["az"])
        pre = {"poses": poses_, "blobs": blobs_}
    else:
        scene, poses_, blobs_ = G.stream(seed, cfg["n_stream"], cfg["beams"], cfg["az"])
        pre = {"poses": poses_, "blobs": blobs_, "world": G.submap_cloud(scene, seed, cfg["map_scans"], cfg["beams"], cfg["az"])}
    G.WORKERS = 1

    import torch
    import locus_b200
    from locus_b200 import api

    if locus_b200.device_count() <= 0:
        raise SystemExit("bench.py: no CUDA device; locus_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        os.environ.setdefault("NCCL_DEBUG", "WARN")      # keep NCCL's version banner off stdout: one JSON line only
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    ctx = BenchCtx(args, cfg, workload, rank, world, local_rank, dist, torch, locus_b200, api)
    ctx.prepare(pre, time.time() - t_gen0)
    if args.config == "c2":
        line = run_c2(ctx)
    else:
        line = run_submap(ctx)
    if rank == 0 and line is not None:
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


class BenchCtx:
    """everything the b200 arms share: handles, buffers, timers"""

    def __init__(self, args, cfg, workload, rank, world, local_rank, dist, torch, locus_b200, api):
        self.args, self.cfg, self.workload = args, cfg, workload
        self.rank, self.world, self.local_rank, self.dist = rank, world, local_rank, dist
        self.torch, self.lb, self.api = torch, locus_b200, api
        self.L = locus_b200.lib()
        self.stream = torch.cuda.Stream(device=local_rank)
        self.fields = locus_b200.xyzi_fields()
        self.fa = api.VoxelGridB200._fields(self.fields)
        self.vg = locus_b200.VoxelGridB200(local_rank, stream=self.stream.cuda_stream)
        self.gicp = locus_b200.GicpB200(local_rank, stream=self.stream.cuda_stream)
        g, gc = self.gicp, cfg["gicp"]
        g.setMaximumIterations(gc["max_iterations"]); g.setMaximumOptimizerIterations(gc["max_inner"])
        g.setMaxCorrespondenceDistance(gc["corr_dist"]); g.setTransformationEpsilon(gc["tf_eps"])
        g.setCorrespondenceRandomness(gc["k"]); g.setRANSACIterations(0)
        g.setOptimizer(locus_b200.LB_OPT_BFGS); g.setExecution(locus_b200.LB_EXEC_STREAM_ORDERED)
        self.implementation = {"execution": "stream-ordered (search grids with TMA-staged candidates + cooperative solve grid per outer iteration), "
                                            "exact (per-point) objective evaluation",
                               "optimizer": "bfgs (reference-exact)"}
        if os.environ.get("LB_CELL"):            # tuning aid: fixed voxel-hash cell size instead of the automatic one
            g.setIndexCellSize(float(os.environ["LB_CELL"]))
            workload["index_cell_size"] = float(os.environ["LB_CELL"])
        if os.environ.get("LB_OPT"):             # tuning aid: 1 = Gauss-Newton inner solve (north_star's 6x6 solve; not reference-exact)
            g.setOptimizer(int(os.environ["LB_OPT"]))
            workload["optimizer"] = "gauss-newton" if int(os.environ["LB_OPT"]) else workload["optimizer"]
        if os.environ.get("LB_EXEC"):
            g.setExecution(int(os.environ["LB_EXEC"]))
            self.implementation["execution"] = "lb_execution %d (LB_EXEC)" % int(os.environ["LB_EXEC"])
        self.n_out = C.c_size_t(0)
        self.res = api.GicpResult()

    def check(self, s):
        if s != 0:
            raise RuntimeError("locus_b200 status %d: %s" % (s, self.L.lb_last_error_string().decode()))

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def gpu_voxel_fn(self, limits):
        vg = self.lb.VoxelGridB200(self.local_rank)
        if limits:
            vg.setFilterFieldName("z"); vg.setFilterLimits(-100.0, 100.0)

        def fn(blob, leaf):
            vg.setLeafSize(leaf)
            return vg.filter(blob, POINT_STEP, self.fields)
        return fn

    def prepare(self, pre, gen_s):
        torch, cfg, args = self.torch, self.cfg, self.args
        self.blobs, self.poses = pre["blobs"], pre["poses"]
        t0 = time.time()
        if "world" in pre:
            if cfg.get("merge", "voxel") == "subsample":
                sub, sleaf = G.subsample_to(pre["world"], cfg["submap"]), 0.0
            else:
                sub, sleaf = G.voxel_merge_to(pre["world"], cfg["submap"], self.gpu_voxel_fn(False))
            self.submap, self.workload["submap_leaf_m"] = sub, sleaf
            self.guesses = [G.perturbed_prior(self.poses[i], 100 + i) for i in range(len(self.blobs))]
            self.union_points = int(len(pre["world"]))
        fl = self.gpu_voxel_fn(True)
        self.leaf = float(np.float32(args.leaf)) if args.leaf > 0 else bisect_leaf(lambda l: fl(self.blobs[0], l).shape[0], cfg["voxels"])
        self.workload["leaf_m"] = self.leaf
        self.setup_s = {"ray_casting": gen_s, "leaf_and_submap": time.time() - t0}
        self.vg.setFilterFieldName("z"); self.vg.setFilterLimits(-100.0, 100.0); self.vg.setLeafSize(self.leaf)
        self.nraw = self.blobs[0].size // POINT_STEP
        with torch.cuda.stream(self.stream):
            self.d_scans = [torch.from_numpy(b).cuda(non_blocking=False) for b in self.blobs]
            self.d_filt = [torch.empty(self.nraw * POINT_STEP, dtype=torch.uint8, device="cuda") for _ in range(2)]
            self.flush = torch.empty(64 * 1024 * 1024, dtype=torch.int32, device="cuda")
        self.h_scans = [torch.from_numpy(b).pin_memory() for b in self.blobs]
        self.h_filt = [torch.empty(self.nraw * POINT_STEP, dtype=torch.uint8).pin_memory() for _ in range(2)]
        torch.cuda.synchronize()

    def timed_calls(self, step_fn, positions, warm_positions):
        """blocking per-scan calls: CUDA events around every scan (L2 flushed before each, outside the events).
        returns (device ms summed over the timed scans, wall s, launches)"""
        torch = self.torch
        for p in warm_positions:
            step_fn(p, False)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in positions]
        self.barrier()
        l0 = self.gicp.launchCount() + self.vg.launchCount()
        t0 = time.perf_counter()
        for k, p in enumerate(positions):
            with torch.cuda.stream(self.stream):
                self.flush.fill_(k)                       # L2 flush: 256 MiB write, outside the event pair
                ev[k][0].record(self.stream)
            step_fn(p, True)
            ev[k][1].record(self.stream)
        self.barrier()
        wall = time.perf_counter() - t0
        return sum(a.elapsed_time(b) for a, b in ev), wall, self.gicp.launchCount() + self.vg.launchCount() - l0


def kernel_shares(gicp, vg_ms, names=("align_persistent", "knn_cov", "index_build")):
    out = {}
    for n in names:
        ms, cnt = gicp.kernelTime(n)
        out[n] = {"ms_avg": ms, "launches": int(cnt)}
    out["voxel_grid"] = {"ms_avg": vg_ms}
    return out


def pose_deltas(cpu_poses, gpu_poses, spread=None):
    """GPU pose vs the CPU arm's on the same inputs; with `spread` (reassociation_probe) also split by whether the
    reference itself reproduces its pose to the bar under a re-association of its sums"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import fixtures as F
    seen, d = set(), {}
    for k, T in gpu_poses:
        if k in cpu_poses and k not in seen:
            seen.add(k)
            d[k] = F.pose_delta(cpu_poses[k], T)
    if not d:
        return None
    dt = np.array([v[0] for v in d.values()]); dr = np.array([v[1] for v in d.values()])
    ok = (dt <= 1e-4) & (dr <= 1e-4)
    out = {"max_dt_m": float(dt.max()), "max_dr_rad": float(dr.max()), "median_dt_m": float(np.median(dt)),
           "median_dr_rad": float(np.median(dr)), "pairs": len(d), "pairs_within_bar": int(ok.sum()),
           "bar": "1e-4 m / 1e-4 rad (north_star)"}
    if spread:
        keys = [k for k in d if k in spread]
        if keys:
            dec = [k for k in keys if spread[k][0] <= 1e-4 and spread[k][1] <= 1e-4]
            sens = [k for k in keys if k not in dec]
            out["reference_reassociated"] = {
                "what": "the CPU arm against ITSELF with the double sums of its objective re-associated (partial sums over "
                        "blocks of %s correspondences; same terms, same arithmetic)" % "/".join(str(c) for c in PROBE_CHUNKS),
                "pairs_probed": len(keys), "pairs_where_the_reference_reproduces_itself_to_the_bar": len(dec),
                "max_dt_m": float(max(spread[k][0] for k in keys)), "max_dr_rad": float(max(spread[k][1] for k in keys)),
                "gpu_max_dt_m_on_those_decisive_pairs": float(max([d[k][0] for k in dec], default=0.0)),
                "gpu_max_dr_rad_on_those_decisive_pairs": float(max([d[k][1] for k in dec], default=0.0)),
                "gpu_max_dt_m_on_the_other_pairs": float(max([d[k][0] for k in sens], default=0.0)),
                "note": "where the reference's BFGS line search stalls on the float32 noise floor of its objective, the last "
                        "bits of f pick the branch: its pose then moves by up to millimetres under ANY re-association of the "
                        "sums, which a parallel reduction cannot avoid; the 1e-4 bar is attainable on the decisive pairs only"}
    return out


def gicp_outputs(results, n_filtered):
    """what lb_gicp_align returns to its caller for each scan of a step (timings left out: they are not results)"""
    return {"final_transformation": np.array([list(r.final_transformation) for r in results], dtype=np.float32).reshape(-1, 4, 4),
            "converged": np.array([r.converged for r in results], dtype=np.float64),
            "iterations": np.array([r.iterations for r in results], dtype=np.float64),
            "n_correspondences": np.array([r.n_correspondences for r in results], dtype=np.float64),
            "delta": np.array([r.delta for r in results], dtype=np.float64),
            "n_filtered": np.array(n_filtered, dtype=np.float64)}


def dump_outputs(path, arrays):
    """--dump-outputs: one float32 / float64 array per file, DIR/<name>.npy.  The largest is one filtered scan
    (c5: ~200k points x 4 floats), far below 64 MB in all."""
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(path, name + ".npy"), a)


# ------------------------------------------------------------------------------------------ c2
def run_c2(ctx):
    args, cfg, workload, torch, L, lb, api = ctx.args, ctx.cfg, ctx.workload, ctx.torch, ctx.L, ctx.lb, ctx.api
    gicp, vg, fa, fields, nraw, res, n_out = ctx.gicp, ctx.vg, ctx.fa, ctx.fields, ctx.nraw, ctx.res, ctx.n_out
    n_str = len(ctx.blobs)
    state = {"n_prev": 0, "prev_pos": None, "poses": [], "iters": [], "evals": [], "ncorr": [], "nsrc": []}

    def step(pos, record, host):
        """one scan through the blocking C-ABI calls (the seam); host: pinned host buffers in and out"""
        i = state.setdefault("flip", 0)
        state["flip"] = i ^ 1
        if host:
            cur, prv, src = ctx.h_filt[i], ctx.h_filt[i ^ 1], ctx.h_scans[pos]
        else:
            cur, prv, src = ctx.d_filt[i], ctx.d_filt[i ^ 1], ctx.d_scans[pos]
        m = 0 if host else 1
        ctx.check(L.lb_voxel_filter(vg._h, C.c_void_p(src.data_ptr()), nraw, POINT_STEP, fa, len(fields), None, 0,
                                    C.c_void_p(cur.data_ptr()), nraw, C.byref(n_out), None, m, m))
        n_cur = n_out.value
        if state["n_prev"]:
            ctx.check(L.lb_gicp_set_source(gicp._h, C.c_void_p(cur.data_ptr()), n_cur, POINT_STEP, 0, -1, m))
            ctx.check(L.lb_gicp_set_target(gicp._h, C.c_void_p(prv.data_ptr()), state["n_prev"], POINT_STEP, 0, -1, m, None))
            ctx.check(L.lb_gicp_align(gicp._h, None, C.byref(res)))
            if host:
                state["h2d"] = nraw * POINT_STEP + (n_cur + state["n_prev"]) * POINT_STEP
                state["d2h"] = n_cur * POINT_STEP + C.sizeof(api.GicpResult)
            if record:
                state["poses"].append(((state["prev_pos"], pos), np.array(res.final_transformation, dtype=np.float32).reshape(4, 4)))
                state["iters"].append(res.iterations); state["evals"].append(res.n_objective_evals)
                state["ncorr"].append(res.n_correspondences); state["nsrc"].append(n_cur)
        state["n_prev"], state["prev_pos"] = n_cur, pos

    def blocking_arm(host, n_timed):
        for k in ("poses", "iters", "evals", "ncorr", "nsrc"):
            state[k] = []
        state["n_prev"], state["prev_pos"] = 0, None
        n_timed = min(n_timed, n_str - 1)
        warm = list(range(min(4, n_str - 1), -1, -1))         # ... 2, 1, 0: ends on scan 0, the timed scans are 1, 2, ...
        return ctx.timed_calls(lambda p, rec: step(p, rec, host), list(range(1, n_timed + 1)), warm) + (n_timed,)

    # ---- the seam, device-resident inputs: per-kernel timers, launch counting, the poses of the parity check
    sampler = ClockSampler(ctx.local_rank)
    gicp.resetKernelTimes(True)
    vg.avgCallMs()
    sampler.start()
    n_scans = args.steps * args.scans_per_step            # scans in the timed region of the pipelined arms
    n_warm = max(args.warmup, 3) * args.scans_per_step
    # first pass with the per-kernel CUDA-event timers on (kernel shares, cycle counters); they cost ~100 event records per
    # scan, so the reported number comes from a second pass without them
    seq_ms, seq_wall, seq_launches, n_seq = blocking_arm(False, n_str - 1)
    clocks_seq = sampler.stop()        # clocks under this arm's load; the timed pass below runs without the sampling thread
    shares = kernel_shares(gicp, vg.avgCallMs())
    k_seq_ms = shares["align_persistent"]["ms_avg"]
    probe_rounds = gicp.kernelTime("probe_rounds")[0]
    dbg = [gicp.kernelTime("debug%d" % i)[0] for i in range(4)]
    dbg6, dbg7, dbg8 = (gicp.kernelTime("debug%d" % i)[0] for i in (6, 7, 8))
    if os.environ.get("LB_SNAP"):     # debugging aid: per-CTA publish / completion times of one collective
        snapP = [gicp.kernelTime("snapP%d" % i)[0] for i in range(64)]
        snapC = [gicp.kernelTime("snapC%d" % i)[0] for i in range(64)]
        sys.stderr.write("SNAP publish ns: %s\nSNAP complete ns: %s\n" % (snapP, snapC))
    gicp.resetKernelTimes(False)
    seq_allocs = 0
    if not args.profile:
        a0 = gicp.kernelTime("dbuf_allocs")[0]
        if os.environ.get("LB_ALLOC_TRACE"): sys.stderr.write("[bench] seam, timed pass begins\n"); sys.stderr.flush()
        seq_ms, seq_wall, seq_launches, n_seq = blocking_arm(False, n_str - 1)
        if os.environ.get("LB_ALLOC_TRACE"): sys.stderr.write("[bench] seam, timed pass ends\n"); sys.stderr.flush()
        seq_allocs = int(gicp.kernelTime("dbuf_allocs")[0] - a0)
    gpu_poses = list(state["poses"])
    iters = np.array(state["iters"], dtype=np.float64); evals = np.array(state["evals"], dtype=np.float64)
    ncorr = np.array(state["ncorr"], dtype=np.float64); nsrc = np.array(state["nsrc"], dtype=np.float64)
    if args.profile:
        if ctx.rank == 0:
            print(json.dumps({"profile_run": True, "metric": "gicp_scans_per_sec", "value": n_seq / (seq_ms * 1e-3),
                              "unit": "scans/s (blocking per-scan calls; NOT a bench value when run under a profiler)",
                              "steps": args.steps, "warmup": args.warmup, "config": workload, "gpu_launches": int(seq_launches),
                              "kernels": shares}))
        return None
    # ---- the seam with HOST buffers (copies inside the timed region)
    seqh_ms, seqh_wall, _, n_seqh = blocking_arm(True, min(n_seq, 50))
    seq_h2d, seq_d2h = state.get("h2d", 0), state.get("d2h", 0)

    # ---- the odometry pipeline (lb_odometry_*): value (device-resident inputs) and e2e (host buffers)
    props = torch.cuda.get_device_properties(ctx.local_rank)
    l2_bytes = int(getattr(props, "L2_cache_size", 126 * 1024 * 1024))
    scan_bytes = nraw * POINT_STEP
    odo = lb.OdometryB200(ctx.local_rank, depth=args.depth, max_points=nraw, max_point_step=POINT_STEP)
    odo.voxel.setFilterFieldName("z"); odo.voxel.setFilterLimits(-100.0, 100.0); odo.voxel.setLeafSize(ctx.leaf)
    odo.setGicpParams(**dict({k: getattr(gicp._p, k) for k, _ in api.GicpParams._fields_},
                             align_points_per_cta=args.pipeline_ppc))
    h_fout = [torch.empty(nraw * POINT_STEP, dtype=torch.uint8).pin_memory() for _ in range(2 * args.depth + 4)]
    torch.cuda.synchronize()
    tick2i = {}

    def submit_device(i):
        return odo.submit(ctx.d_scans[seq(i, n_str)].data_ptr(), nraw, POINT_STEP, fa, mem=lb.LB_MEM_DEVICE)

    def submit_host(i):
        return odo.submit(ctx.h_scans[seq(i, n_str)].data_ptr(), nraw, POINT_STEP, fa, mem=lb.LB_MEM_HOST,
                          filtered_out=h_fout[i % len(h_fout)].data_ptr(), mem_filtered=lb.LB_MEM_HOST)

    def pipelined_run(odo, submit_fn, steps, warmup):
        """K scans of one stream through the pipeline; returns (device ms, results of the timed scans, launches)"""
        warmup = max(warmup, 3 * args.depth)     # every registration worker sizes its buffers before the timed region
        for i in range(1 + warmup):
            submit_fn(i)
        while odo.pending():
            r = odo.next()
            if r.status != 0:
                raise RuntimeError("lb_odometry: status %d: %s" % (r.status, r.error.decode(errors="replace")))
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ctx.barrier()
        st0 = odo.stageTimes()
        l0 = odo.launchCount()
        a0 = gicp.kernelTime("dbuf_allocs")[0]           # device allocations of the process so far
        ev0.record(ctx.stream)
        out = []
        for k in range(steps):
            tick2i[submit_fn(1 + warmup + k)] = 1 + warmup + k
            r = odo.next(block=False)
            while r is not None:
                out.append(r)
                r = odo.next(block=False) if odo.pending() else None
        while odo.pending():
            out.append(odo.next())
        ctx.barrier()
        ev1.record(ctx.stream)
        torch.cuda.synchronize()
        state["allocs_timed_region"] = gicp.kernelTime("dbuf_allocs")[0] - a0
        for r in out:
            if r.status != 0 or not r.has_pose:
                raise RuntimeError("lb_odometry: ticket %d status %d: %s" % (r.ticket, r.status, r.error.decode(errors="replace")))
        st1 = odo.stageTimes()
        nf = max(1, st1["filtered"] - st0["filtered"]); nr = max(1, st1["registered"] - st0["registered"])
        state["stages"] = {"voxel_stage_busy_ms_per_scan": 1e3 * (st1["voxel_busy_s"] - st0["voxel_busy_s"]) / nf,
                           "voxel_stage_wait_ms_per_scan": 1e3 * (st1["voxel_wait_s"] - st0["voxel_wait_s"]) / nf,
                           "worker_busy_ms_per_scan": 1e3 * (st1["workers_busy_s"] - st0["workers_busy_s"]) / nr,
                           "worker_wait_ms_per_scan": 1e3 * (st1["workers_wait_s"] - st0["workers_wait_s"]) / nr}
        return ev0.elapsed_time(ev1), out, odo.launchCount() - l0

    def equals_sequential(results):
        seq_T = {key: T for key, T in gpu_poses}
        same, compared = True, 0
        for r in results:
            i = tick2i[int(r.ticket)]
            key = (seq(i - 1, n_str), seq(i, n_str))
            T = np.array(r.gicp.final_transformation, dtype=np.float32).reshape(4, 4)
            if key in seq_T:
                compared += 1
                same = same and np.array_equal(T, seq_T[key])
        return bool(same), compared

    sampler = ClockSampler(ctx.local_rank)
    sampler.start()
    for g in (odo.gicp(i) for i in range(args.depth)):
        g.resetKernelTimes(2)          # only the event pair around the align kernel (the roofline's live duration)
    dev_ms, p_out, launches_timed = pipelined_run(odo, submit_device, n_scans, n_warm)
    allocs_timed = state["allocs_timed_region"]       # device allocations inside the timed region (steady state: 0)
    clocks = sampler.stop()
    stages_device = dict(state["stages"])
    kt = [odo.gicp(i).kernelTime("align_persistent") for i in range(args.depth)]
    for g in (odo.gicp(i) for i in range(args.depth)):
        g.resetKernelTimes(False)
    k_n = sum(n for _, n in kt)
    k_ms = sum(ms * n for ms, n in kt) / k_n if k_n else 0.0
    pipe_same, pipe_compared = equals_sequential(p_out)      # same scans, same kernels: bit-identical poses expected
    if args.dump_outputs and ctx.rank == 0:                   # p_out is in submission order: the last step's scans are last
        last = p_out[-args.scans_per_step:]
        dump_outputs(args.dump_outputs, gicp_outputs([r.gicp for r in last], [r.n_filtered for r in last]))
    e2e_ms, e_out, _ = pipelined_run(odo, submit_host, n_scans, n_warm)
    e2e_h2d = args.scans_per_step * nraw * POINT_STEP
    e2e_d2h = args.scans_per_step * (int(np.mean([r.n_filtered for r in e_out])) * POINT_STEP + C.sizeof(api.OdometryResult))

    variants = {}
    # ---- variant (information only, N = 1): the pipeline WITHOUT cloud sharing -- both clouds' index + covariances rebuilt
    # for every registration, which is what the reference's callers make the reference do
    if ctx.world == 1 and os.environ.get("LB_SHARE_VARIANT", "1") != "0":
        try:
            odo2 = lb.OdometryB200(ctx.local_rank, depth=args.depth, max_points=nraw, max_point_step=POINT_STEP)
            odo2.setCloudSharing(False)
            odo2.voxel.setFilterFieldName("z"); odo2.voxel.setFilterLimits(-100.0, 100.0); odo2.voxel.setLeafSize(ctx.leaf)
            odo2.setGicpParams(**dict({k: getattr(gicp._p, k) for k, _ in api.GicpParams._fields_},
                                      align_points_per_cta=args.pipeline_ppc))
            sub2 = lambda i: odo2.submit(ctx.d_scans[seq(i, n_str)].data_ptr(), nraw, POINT_STEP, fa, mem=lb.LB_MEM_DEVICE)  # noqa: E731
            sh_ms, sh_out, _ = pipelined_run(odo2, sub2, n_scans, n_warm)
            same, compared = equals_sequential(sh_out)
            variants["pipeline_rebuild_both_clouds"] = {
                "value": n_scans / (sh_ms * 1e-3), "unit": "scans/s", "equals_sequential": same, "scans_timed": n_scans,
                "stages": dict(state["stages"]),
                "note": "lb_odometry_set_cloud_sharing(0): source AND target index + covariances rebuilt for every registration, "
                        "like the reference's callers do; same poses as the default (sharing on), bit for bit"}
            odo2.close()
        except Exception as ex:          # the variant must never take the bench line down
            variants["pipeline_rebuild_both_clouds"] = {"error": str(ex)[:200]}
    # ---- variant (information only, N = 1): north_star's Gauss-Newton inner solve instead of the reference's BFGS
    if ctx.world == 1 and not os.environ.get("LB_OPT"):
        keep = list(gpu_poses)
        gicp.setOptimizer(lb.LB_OPT_GAUSS_NEWTON)
        gn_ms, _, _, n_gn = blocking_arm(False, min(n_seq, 30))
        gicp.setOptimizer(lb.LB_OPT_BFGS)
        variants["gauss_newton"] = {"value": n_gn / (gn_ms * 1e-3), "unit": "scans/s", "mode": "blocking per-scan calls",
                                    "poses": list(state["poses"]),
                                    "note": "6x6 Gauss-Newton inner solve (BASELINE north_star wording); NOT the headline: "
                                            "its pose differs from the reference's BFGS result by more than the 1e-4 bar"}
        gpu_poses = keep

    # max over ranks (device time), whole-job aggregate
    tmax, vals = aggregate(ctx.dist, "cuda", [dev_ms, e2e_ms, seq_ms, seqh_ms], [n_scans, n_scans, n_seq, n_seqh], ctx.world)
    dev_ms_max, e2e_ms_max, seq_ms_max, seqh_ms_max = tmax
    value, e2e_value, seq_value, seqh_value = vals
    odo.close()
    if ctx.rank != 0:
        return None

    # roofline of the dominant kernel (persistent align: K4 correspondences + K5 objective resident on device).
    # algorithmic bytes per launch (SURVEY 8d): It * (88*Ns + E * 80*m), It = outer iterations, E = evals per outer.
    peak, peak_src = measured_peak_hbm()
    bytes_per_launch = float(np.mean(iters * 88.0 * nsrc + evals * 80.0 * ncorr)) if len(iters) else 0.0
    achieved = (bytes_per_launch / (k_ms * 1e-3)) / 1e9 if k_ms > 0 else 0.0
    roofline = {"bound": "hbm", "kernel": ALIGN_KERNELS,
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None,
                "traffic": align_traffic(float(iters.mean()) if len(iters) else 0.0), "peak_source": peak_src,
                "algorithmic_bytes_per_launch": bytes_per_launch,
                "avg_launch_ms": k_ms, "launches_timed": int(k_n), "avg_launch_ms_sequential": k_seq_ms,
                "kernel_share_of_sequential_step": (k_seq_ms / (seq_ms_max / n_seq)) if seq_ms_max else None,
                "aligns_in_flight_mean": (k_ms / (dev_ms_max / n_scans)) if dev_ms_max else None,
                "objective_evaluations_per_align": float(evals.mean()) if len(evals) else None,
                "note": "working set (<= 5 MB) is L2/register-resident: this kernel is bound by the latency of its chain of "
                        "dependent grid-wide reductions (one per objective evaluation of the reference's BFGS line search), "
                        "not by HBM (SURVEY H3); fraction reported for information.  avg_launch_ms is measured inside the "
                        "pipelined timed region, avg_launch_ms_sequential with the kernel alone on the GPU"}

    line = {"metric": "gicp_scans_per_sec", "value": value, "unit": "scans/s", "n_gpus": ctx.world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 points / f64 accumulation", "data": "synthetic", "config": workload,
            "clocks": clocks, "gpu_launches": int(launches_timed), "implementation": ctx.implementation,
            "e2e": {"value": e2e_value, "unit": "scans/s", "h2d_bytes_per_step": int(e2e_h2d),
                    "d2h_bytes_per_step": int(e2e_d2h), "ms_per_step": e2e_ms_max / args.steps,
                    "ms_per_scan": e2e_ms_max / n_scans},
            "roofline": roofline,
            "ms_per_scan": dev_ms_max / n_scans,
            "sequential": {"value": seq_value, "unit": "scans/s", "ms_per_scan": seq_ms_max / n_seq, "scans_timed": n_seq,
                           "gpu_launches": int(seq_launches), "clocks": clocks_seq, "device_allocations": seq_allocs,
                           "note": "THE DROP-IN SEAM: blocking per-scan C-ABI calls (what icp_->align() inside LOCUS's "
                                   "queue-depth-1 lidar callback sees), device-resident inputs, L2 flushed between scans"},
            "sequential_e2e": {"value": seqh_value, "unit": "scans/s", "ms_per_scan": seqh_ms_max / n_seqh, "scans_timed": n_seqh,
                               "h2d_bytes_per_scan": int(seq_h2d), "d2h_bytes_per_scan": int(seq_d2h),
                               "note": "the same blocking calls with HOST (pinned) buffers: raw scan H2D, filtered cloud D2H, "
                                       "source and target clouds H2D, pose D2H, all inside the timed region"},
            "pipeline_equals_sequential": pipe_same, "pipeline_scans_compared": pipe_compared,
            "pipeline_device_allocations": int(allocs_timed),
            "pipeline_stages": dict(stages_device, note="host wall clock per scan inside the timed region (value arm): the "
                                    "VoxelGrid stage is serial, the registration workers run %d-wide" % args.depth),
            "input_pool": {"distinct_scans": n_str, "bytes": n_str * scan_bytes, "l2_bytes": l2_bytes},
            "setup_s": ctx.setup_s,
            "per_scan": {"outer_iterations_mean": float(iters.mean()) if len(iters) else None,
                         "objective_evals_mean": float(evals.mean()) if len(evals) else None,
                         "correspondences_mean": float(ncorr.mean()) if len(ncorr) else None,
                         "source_points_mean": float(nsrc.mean()) if len(nsrc) else None,
                         "kernels_sequential": shares, "cell_probe_rounds_total": probe_rounds,
                         "align_last_launch_cycles": {"total": dbg[0], "block_reduce_publish": dbg[1],
                                                      "slot_wait_sum": dbg[2], "collectives": dbg[3], "leader_scalar_before_fdf": dbg6, "poll_rounds_thread0": dbg7,
                                                      "poll_publish_to_done_thread0": dbg8},
                         "wall_s_timed_region": seq_wall}}

    if ctx.world == 1 and not args.no_cpu_baseline:
        # CPU baseline on a bounded sample of the same stream, and pose delta GPU vs CPU on those scans
        data = {"leaf": ctx.leaf, "blobs": ctx.blobs}
        probe = {}
        sps, n, cpu_poses, cores = run_cpu_arm(args, cfg, data, budget_s=args.cpu_baseline_seconds, probe=probe)
        spread = reassociation_probe(cpu_poses, probe)
        line["cpu_baseline"] = {"value": sps, "unit": "scans/s", "cores": cores, "kind": "port",
                                "sample": "%d consecutive scans of the same stream, same leaf (oracle/: C port of "
                                          "multithreaded_gicp + PCL VoxelGrid); threads = fastest of {4..%d}" % (n, os.cpu_count() or 1)}
        line["speedup_vs_cpu"] = {"pipelined_e2e": e2e_value / sps, "pipelined_device": value / sps,
                                  "seam_sequential_e2e": seqh_value / sps, "seam_sequential_device": seq_value / sps}
        pd = pose_deltas(cpu_poses, gpu_poses, spread)
        if pd:
            line["pose_delta_vs_cpu"] = pd
        for v in variants.values():
            pd = pose_deltas(cpu_poses, v.get("poses", []))
            if pd:
                v["pose_delta_vs_cpu"] = pd
    for v in variants.values():
        v.pop("poses", None)
    if variants:
        line["variants"] = variants
    return line


# ------------------------------------------------------------------------------------------ c3 / c4 / c5
def run_submap(ctx):
    args, cfg, workload, torch, L, lb, api = ctx.args, ctx.cfg, ctx.workload, ctx.torch, ctx.L, ctx.lb, ctx.api
    gicp, vg, fa, fields, nraw, res, n_out = ctx.gicp, ctx.vg, ctx.fa, ctx.fields, ctx.nraw, ctx.res, ctx.n_out
    n_str = len(ctx.blobs)
    n_map = int(ctx.submap.shape[0])
    sub_blob = np.ascontiguousarray(ctx.submap, dtype=np.float32)          # (n, 3) float32, stride 12
    with torch.cuda.stream(ctx.stream):
        d_map = torch.from_numpy(sub_blob.reshape(-1)).cuda()
    h_map = torch.from_numpy(sub_blob.reshape(-1)).pin_memory()
    torch.cuda.synchronize()
    state = {"poses": [], "iters": [], "evals": [], "ncorr": [], "nsrc": []}
    guesses = [np.ascontiguousarray(g, dtype=np.float32).reshape(16) for g in ctx.guesses]

    def set_target(host):
        p = h_map if host else d_map
        ctx.check(L.lb_gicp_set_target(gicp._h, C.c_void_p(p.data_ptr()), n_map, 12, 0, -1, 0 if host else 1, None))

    def step(pos, record, host, rebuild):
        m = 0 if host else 1
        cur = ctx.h_filt[0] if host else ctx.d_filt[0]
        src = ctx.h_scans[pos] if host else ctx.d_scans[pos]
        ctx.check(L.lb_voxel_filter(vg._h, C.c_void_p(src.data_ptr()), nraw, POINT_STEP, fa, len(fields), None, 0,
                                    C.c_void_p(cur.data_ptr()), nraw, C.byref(n_out), None, m, m))
        n_cur = n_out.value
        ctx.check(L.lb_gicp_set_source(gicp._h, C.c_void_p(cur.data_ptr()), n_cur, POINT_STEP, 0, -1, m))
        if rebuild:
            set_target(host)
        ctx.check(L.lb_gicp_align(gicp._h, guesses[pos].ctypes.data_as(C.c_void_p), C.byref(res)))
        if host:
            state["h2d"] = nraw * POINT_STEP + n_cur * POINT_STEP + (n_map * 12 if rebuild else 0)
            state["d2h"] = n_cur * POINT_STEP + C.sizeof(api.GicpResult)
        if record:
            state["poses"].append((pos, np.array(res.final_transformation, dtype=np.float32).reshape(4, 4)))
            state["iters"].append(res.iterations); state["evals"].append(res.n_objective_evals)
            state["ncorr"].append(res.n_correspondences); state["nsrc"].append(n_cur)

    def arm(host, rebuild, n_timed, warm, timers=False):
        for k in ("poses", "iters", "evals", "ncorr", "nsrc"):
            state[k] = []
        t0 = time.perf_counter()
        set_target(host)                                 # the resident submap: built once (first align), then kept
        step(0, False, host, False)
        state["submap_first_build_s"] = time.perf_counter() - t0
        if timers:                                       # per-kernel averages without the one-off build of the submap
            gicp.resetKernelTimes(True)
            vg.avgCallMs()
        pos = [(1 + k) % n_str for k in range(n_timed)]
        return ctx.timed_calls(lambda p, rec: step(p, rec, host, rebuild), pos, [(n_str - 1 - k) % n_str for k in range(warm)]) + (n_timed,)

    n_timed = max(1, args.steps)
    warm = max(args.warmup, 3)
    sampler = ClockSampler(ctx.local_rank)
    gicp.resetKernelTimes(True)
    vg.avgCallMs()
    sampler.start()
    # first pass with the per-kernel CUDA-event timers on (kernel shares); the reported number comes from a second pass
    # without them (~100 event records per scan)
    dev_ms, wall, launches, _ = arm(False, False, n_timed, warm, timers=True)
    shares = kernel_shares(gicp, vg.avgCallMs())
    first_build_s = state["submap_first_build_s"]
    gicp.resetKernelTimes(False)
    dev_ms, wall, launches, _ = arm(False, False, n_timed, warm)
    clocks = sampler.stop()
    if args.dump_outputs and ctx.rank == 0:      # res, n_out and d_filt[0] still hold the last timed scan's results
        n = n_out.value
        cloud = ctx.d_filt[0][:n * POINT_STEP].cpu().numpy().view(np.float32).reshape(n, POINT_STEP // 4)
        dump_outputs(args.dump_outputs, dict(gicp_outputs([res], [n]),
                                             filtered_cloud=np.ascontiguousarray(cloud[:, [0, 1, 2, 4]])))   # x y z intensity
    gpu_poses = list(state["poses"])
    iters = np.array(state["iters"], dtype=np.float64); evals = np.array(state["evals"], dtype=np.float64)
    ncorr = np.array(state["ncorr"], dtype=np.float64); nsrc = np.array(state["nsrc"], dtype=np.float64)
    e2e_ms, _, _, _ = arm(True, False, n_timed, warm)
    e2e_h2d, e2e_d2h = state.get("h2d", 0), state.get("d2h", 0)
    gicp.resetKernelTimes(True)
    vg.avgCallMs()
    n_reb = max(1, min(n_timed, 10))
    reb_ms, _, reb_launches, _ = arm(False, True, n_reb, 2)
    reb_shares = kernel_shares(gicp, vg.avgCallMs())
    gicp.resetKernelTimes(False)
    reb_poses = list(state["poses"])
    rebh_ms, _, _, _ = arm(True, True, n_reb, 2)

    nn = None
    if args.config == "c5":
        nn = nn_search_roofline(ctx, d_map, n_map)
    rolling = None
    if args.config != "c5":
        try:
            rolling = rolling_submap_arm(ctx, d_map, n_map, guesses, n_timed, warm)
        except Exception as ex:          # the variant must never take the bench line down
            rolling = {"error": str(ex)[:300]}

    tmax, vals = aggregate(ctx.dist, "cuda", [dev_ms, e2e_ms, reb_ms, rebh_ms], [n_timed, n_timed, n_reb, n_reb], ctx.world)
    if ctx.rank != 0:
        return None
    value, e2e_value, reb_value, rebh_value = vals
    peak, peak_src = measured_peak_hbm()
    k_ms = shares["align_persistent"]["ms_avg"]
    bytes_per_launch = float(np.mean(iters * 88.0 * nsrc + evals * 80.0 * ncorr)) if len(iters) else 0.0
    achieved = (bytes_per_launch / (k_ms * 1e-3)) / 1e9 if k_ms > 0 else 0.0
    if nn is not None:
        roofline = nn
    else:
        roofline = {"bound": "hbm", "kernel": ALIGN_KERNELS + " -- target = the 500k submap",
                    "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None, "traffic": None,
                    "peak_source": peak_src, "algorithmic_bytes_per_launch": bytes_per_launch, "avg_launch_ms": k_ms,
                    "launches_timed": shares["align_persistent"]["launches"],
                    "kernel_share_of_step": (k_ms / (tmax[0] / n_timed)) if tmax[0] else None,
                    "note": "latency-bound chain of dependent grid-wide reductions (one per objective evaluation), working set "
                            "L2-resident: fraction for information (SURVEY H3)"}
    line = {"metric": "gicp_scans_per_sec", "value": value, "unit": "scans/s", "n_gpus": ctx.world, "steps": n_timed,
            "warmup": warm, "ms_per_step": tmax[0] / n_timed, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 points / f64 accumulation", "data": "synthetic", "config": workload,
            "clocks": clocks, "gpu_launches": int(launches), "implementation": ctx.implementation,
            "e2e": {"value": e2e_value, "unit": "scans/s", "h2d_bytes_per_step": int(e2e_h2d), "d2h_bytes_per_step": int(e2e_d2h),
                    "ms_per_step": tmax[1] / n_timed},
            "roofline": roofline,
            "submap": {"points": n_map, "union_points": ctx.union_points, "first_build_s_incl_upload_and_first_scan": first_build_s},
            "setup_s": ctx.setup_s,
            "per_scan": {"outer_iterations_mean": float(iters.mean()), "objective_evals_mean": float(evals.mean()),
                         "correspondences_mean": float(ncorr.mean()), "source_points_mean": float(nsrc.mean()),
                         "kernels": shares, "wall_s_timed_region": wall},
            "variants": {"submap_rebuilt_every_scan": {
                "value": reb_value, "unit": "scans/s", "ms_per_scan": tmax[2] / n_reb, "scans_timed": n_reb,
                "e2e": {"value": rebh_value, "unit": "scans/s", "ms_per_scan": tmax[3] / n_reb},
                "gpu_launches": int(reb_launches), "kernels": reb_shares,
                "equals_resident_submap": bool(all(np.array_equal(T, dict(gpu_poses).get(p)) for p, T in reb_poses if p in dict(gpu_poses))),
                "note": "lb_gicp_set_target(submap) before every align: the 500k-point index and k-NN(20) covariances rebuilt "
                        "per scan, what LOCUS's callers do today (setInputTarget clears them, gicp.h:196-200)"}}}
    if rolling is not None:
        line["variants"]["rolling_submap"] = rolling
    if ctx.world == 1 and not args.no_cpu_baseline:
        data = {"leaf": ctx.leaf, "blobs": ctx.blobs, "submap": ctx.submap, "guesses": ctx.guesses}
        probe = {}
        sps, n, cpu_poses, cores = run_cpu_arm(args, cfg, data, budget_s=args.cpu_baseline_seconds, probe=probe)
        spread = reassociation_probe(cpu_poses, probe) if args.config != "c5" else None
        if data.get("_cpu_target") is not None:
            data.pop("_cpu_target").close()
        line["cpu_baseline"] = {"value": sps, "unit": "scans/s", "cores": cores, "kind": "port",
                                "sample": "%d scans of the same stream against the kept submap (kd-tree + covariances prepared "
                                          "once, %.1f s, untimed); oracle/: C port of multithreaded_gicp + PCL VoxelGrid" % (n, data.get("cpu_submap_prepare_s", 0.0))}
        pd = pose_deltas(cpu_poses, gpu_poses, spread)
        if pd:
            line["pose_delta_vs_cpu"] = pd
        line["speedup_vs_cpu"] = {"seam_e2e": e2e_value / sps, "seam_device": value / sps}
        if args.config != "c5":
            sps_r, n_r, _, cores_r = run_cpu_arm(args, cfg, data, max_steps=2, rebuild_target=True)
            line["variants"]["submap_rebuilt_every_scan"]["cpu_baseline"] = {
                "value": sps_r, "unit": "scans/s", "cores": cores_r, "kind": "port", "sample": "%d scans, submap kd-tree + covariances rebuilt per align" % n_r}
            line["variants"]["submap_rebuilt_every_scan"]["speedup_vs_cpu"] = {"seam_e2e": rebh_value / sps_r, "seam_device": reb_value / sps_r}
    return line


def rolling_submap_arm(ctx, d_map, n_map, guesses, n_timed, warm, keyframe_every=5, window=20.0):
    """SURVEY 8f row f3: the map lives in an lb_submap object and CHANGES while the stream is registered against it, the way
    LOCUS's lidar callback drives its mapper (Locus.cc:522-543): every `keyframe_every`-th scan is a keyframe -- its
    aligned points are inserted (InsertPoints), the window is cropped (Refresh, box_filter_size 20 m) and the target is
    refreshed: index rebuilt, covariances computed for the NEW points only.  All on the device; blocking calls."""
    torch, L, lb, gicp, vg = ctx.torch, ctx.L, ctx.lb, ctx.gicp, ctx.vg
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import fixtures as F
    m = lb.SubmapB200(ctx.local_rank, resolution=0.5 * float(ctx.workload.get("submap_leaf_m", 0.06)))
    n0 = m.insert_device(d_map.data_ptr(), n_map, 12, 0)
    aligned = torch.empty(ctx.nraw * 16, dtype=torch.uint8, device="cuda")
    res, n_out = ctx.res, ctx.n_out
    n_str = len(ctx.blobs)
    stats = {"keyframes": 0, "inserted": 0, "removed": 0, "err": []}

    def step(pos, timed):
        cur, src = ctx.d_filt[0], ctx.d_scans[pos]
        ctx.check(L.lb_voxel_filter(vg._h, C.c_void_p(src.data_ptr()), ctx.nraw, POINT_STEP, ctx.fa, len(ctx.fields), None, 0,
                                    C.c_void_p(cur.data_ptr()), ctx.nraw, C.byref(n_out), None, 1, 1))
        n_cur = n_out.value
        ctx.check(L.lb_gicp_set_source(gicp._h, C.c_void_p(cur.data_ptr()), n_cur, POINT_STEP, 0, -1, 1))
        ctx.check(L.lb_gicp_set_target_submap(gicp._h, m._h))
        ctx.check(L.lb_gicp_align(gicp._h, guesses[pos].ctypes.data_as(C.c_void_p), C.byref(res)))
        T = np.array(res.final_transformation, dtype=np.float32).reshape(4, 4)
        if timed:
            stats["err"].append(F.pose_delta(ctx.poses[pos], T))
            stats["k"] = stats.get("k", 0) + 1
            if stats["k"] % keyframe_every == 0:         # keyframe: the aligned scan enters the map, the window moves
                ctx.check(L.lb_gicp_transform_source(gicp._h, None, C.c_void_p(aligned.data_ptr()), 16, 0, -1, 1))
                stats["inserted"] += m.insert_device(aligned.data_ptr(), n_cur, 16, 0)
                stats["removed"] += m.Refresh(T[:3, 3], window)
                stats["keyframes"] += 1

    pos = [(1 + k) % n_str for k in range(n_timed)]
    dev_ms, wall, launches = ctx.timed_calls(lambda p, rec: step(p, rec), pos, [(n_str - 1 - k) % n_str for k in range(warm)])
    tmax, vals = aggregate(ctx.dist, "cuda", [dev_ms], [n_timed], ctx.world)
    out = {"value": vals[0], "unit": "scans/s", "ms_per_scan": tmax[0] / n_timed, "scans_timed": n_timed,
           "keyframes": stats["keyframes"], "keyframe_every": keyframe_every, "window_half_size_m": window,
           "map_points_start": int(n0), "map_points_end": int(m.size()), "points_inserted": int(stats["inserted"]),
           "points_cropped": int(stats["removed"]),
           "pose_error_vs_truth": {"max_dt_m": float(max(e[0] for e in stats["err"])), "max_dr_rad": float(max(e[1] for e in stats["err"]))},
           "note": "lb_submap_* + lb_gicp_set_target_submap: the map is resident and rolling; a keyframe costs one index rebuild "
                   "of the map plus k-NN covariances of the inserted points only (cached per point afterwards)"}
    m.close()
    return out


def nn_search_roofline(ctx, d_map, n_map):
    """c5: the NN-search kernel (the HBM-bound kernel of the path) on the filtered scan's queries against the resident
    10M-point map, at the library's automatic voxel-hash cell.  Algorithmic bytes = SURVEY 8d's candidate-scan figure
    B_nn = Nq (16 + 16 c + 8), c = target points a query visits (counted on the device)."""
    gicp, torch, L = ctx.gicp, ctx.torch, ctx.L
    q = ctx.d_filt[0]
    ctx.check(L.lb_voxel_filter(ctx.vg._h, C.c_void_p(ctx.d_scans[0].data_ptr()), ctx.nraw, POINT_STEP, ctx.fa, len(ctx.fields),
                                None, 0, C.c_void_p(q.data_ptr()), ctx.nraw, C.byref(ctx.n_out), None, 1, 1))
    nq = int(ctx.n_out.value)
    idx = torch.empty(nq, dtype=torch.int32, device="cuda"); d2 = torch.empty(nq, dtype=torch.float32, device="cuda")
    call = lambda: ctx.check(L.lb_gicp_nn_target(gicp._h, C.c_void_p(q.data_ptr()), nq, POINT_STEP, C.c_void_p(idx.data_ptr()),  # noqa: E731
                                                 C.c_void_p(d2.data_ptr()), 1))
    call()
    gicp.resetKernelTimes(True)
    for k in range(5):
        ctx.flush.fill_(k)
        call()
    ms, n = gicp.kernelTime("nn_query")
    c = gicp.kernelTime("debug4")[0] / float(nq)
    cell = gicp.kernelTime("cell_tgt")[0]
    dense = gicp.kernelTime("dense_tgt")[0]
    first_ms, far_ms, n_second = gicp.kernelTime("nn_query_first")[0], gicp.kernelTime("nn_query_far")[0], gicp.kernelTime("debug6")[0]
    gicp.resetKernelTimes(False)
    peak, peak_src = measured_peak_hbm()
    b = nq * (16.0 + 16.0 * c + 8.0)
    ach = b / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
    staged = first_ms > 0
    return {"bound": "hbm", "kernel": ("nn_query_staged_kernel<TMA> + nn_query_far_kernel (exact 1-NN of the scan's points in the 10M-point map; 32 queries "
                                       "per warp, candidates staged through shared memory with cp.async.bulk)") if staged else
                                      "nn_query_warp_kernel (exact 1-NN of the scan's points in the 10M-point map; one query per warp)",
            "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak if peak else None,
            "traffic": ncu_traffic("nn_query_staged_kernel" if staged else "nn_query_warp_kernel"), "peak_source": peak_src, "algorithmic_bytes_per_launch": b,
            "avg_launch_ms": ms, "launches_timed": int(n), "queries": nq, "map_points": n_map, "candidates_per_query": c,
            "cell_m": cell, "cell": "automatic", "queries_per_s": nq / (ms * 1e-3) if ms else 0.0,
            "map_points_in_cells_with_more_than_32_points": dense,
            "kernel_choice": "points in dense cells > 10 % of the map -> nn_query_warp_kernel (32 lanes share one query's candidates), else the "
                             "staged kernels (first_look / second kernel times below are 0 when the warp kernel ran)",
            "first_look_kernel_ms": first_ms, "second_kernel_ms": far_ms, "queries_left_to_second_kernel": n_second,
            "bytes_model": "B_nn = Nq (16 + 16 c + 8) (SURVEY 8d), c = target points THIS kernel fetches per query (its first look is a "
                           "ball of half a cell, not the 3x3x3 block the round-1 kernel scanned: the same answers from ~5x fewer "
                           "bytes, so queries_per_s, not the fraction, is the figure to compare across rounds)"}


ALIGN_KERNELS = ("the kernels of one align() -- per outer iteration loop_nn_kernel + loop_far_kernel (K4: exact 1-NN correspondences, "
                 "Mahalanobis) and loop_solve_kernel (K5 objective + BFGS, cooperative grid); 'launch' below = one align()")


def align_traffic(iterations_per_align):
    """DRAM bytes of one align() from the committed ncu capture: per-launch bytes of its three kernels x outer iterations."""
    parts = [ncu_traffic(k) for k in ("loop_nn_kernel", "loop_far_kernel", "loop_solve_kernel")]
    if any(p is None for p in parts) or iterations_per_align <= 0:
        return None
    return float(sum(parts) * iterations_per_align)


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed ncu --set full capture
    (profiles/traffic.json, written by tools/summarize_ncu.py traffic); None when no capture is committed."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
        return float(t[kernel]["dram_bytes_per_launch"])
    except (OSError, KeyError, ValueError):
        return None


if __name__ == "__main__":
    main()
