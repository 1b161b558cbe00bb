#!/usr/bin/env python
"""bench.py -- headline benchmark: BASELINE.json's metric, "vSLAM frames/s (AKAZE+match+RANSAC, 1080p ~5k kp)".

One frame PAIR of the workload is the sequence cv-sfm runs for a two-view initialisation (cv-sfm/src/lib.rs:2200-2204, 1375-1412):
  AKAZE extract of both 1920x1080 f32 frames (~5k keypoints each, one batched pass)
  -> symmetric brute-force Hamming 2-NN match (rule d0 + 24 <= d1, cross-check)
  -> calibrated bearings of the matched keypoints (f = 1000 px, c = (960, 540))
  -> Arrsac(1e-7, Xoshiro256++).initialization_hypotheses(8192).max_candidate_hypotheses(1024) + EightPoint
     (the two-view consensus of vslam-sandbox/src/main.rs:112-117), every stage on the GPU, nothing returns to the host in between.
A "step" is one batch of PAIRS_PER_STEP such pairs (declared in config); metric = frames/s = 2 * pairs / time.
N>1: every rank processes its own frame pairs (independent -> weak scaling, no data-path collective).

  value : device-resident frames, results stay in HBM; CUDA events, max over ranks
  e2e   : the host entry point cvb_two_view_frames: pinned HOST frames in, keypoints / descriptors / matches / pose / inliers back
          on the host, copies inside the timed region
  roofline : dominant HBM-modelled kernel: algorithmic bytes / CUDA-event duration (instrumented pass) + the RANSAC kernels' figures
  cpu_baseline : the CPU oracle (restated reference, -O3) on this box's host cores, bounded sample, all-core and 1-thread

`--impl reference` times the reference's CPU implementation (the oracle port; the Rust original cannot be built: no cargo/rustc
in the image) on the same workload and prints the same JSON line.
"""
import argparse
import ctypes as C
import json
import os

# many contexts (streams) are pipelined: give every stream its own hardware queue (default 8 would alias unrelated contexts
# onto one queue and serialise them); must be set before the CUDA context exists
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "vSLAM frames/s (AKAZE+match+RANSAC, 1080p ~5k kp) at 1/2/4/8 B200"     # BASELINE.json, verbatim
W, H = 1920, 1080
MAXF = 5000            # maximum_features -> exactly "~5k keypoints" per frame
BETTER_BY = 24         # cv-sfm/src/settings.rs:397-399
POOL_PAIRS = 8         # 16 distinct frames = 133 MB > 126 MB L2: step inputs are never L2-resident
PAIRS_PER_STEP = 16    # one step = one batch of 16 frame pairs (32 frames)
FOCAL, CX, CY = 1000.0, 960.0, 540.0
ARRSAC = dict(threshold=1e-7, initialization_hypotheses=8192, max_candidate_hypotheses=1024)      # vslam-sandbox/src/main.rs:112-117
ALG_BYTES_PER_FRAME = 4 * (13 * 11016000 + 3 * 40759200 + 4 * 2073600)   # SURVEY.md 8(d): 1.095 GB
WORKLOAD = ("configs[1]+[2]: AKAZE extract x2 + symmetric Hamming 2-NN + ARRSAC(1e-7, init 8192, max_cand 1024)/eight-point, "
            "2 frames 1920x1080 f32, ~5k kp/frame")


def make_pool(npairs, seed0=0):
    from tests.synth import synth_frame, warp_frame
    frames = []
    for i in range(npairs):
        a = synth_frame(seed0 + i)
        frames.append(np.stack([a, warp_frame(a, 1000 + seed0 + i)]))
    return frames


class ClockSampler(threading.Thread):
    """NVML clocks / throttle reasons sampled during the timed regions."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index, pci=None):
        super().__init__(daemon=True)
        self.index, self.pci, self.samples, self.stop_flag = index, pci, [], False

    def run(self):
        # NVML in-process (the library nvidia-smi itself reads): spawning nvidia-smi ten times a second inside the timed
        # region takes driver locks for tens of ms and throttles the launching threads
        try:
            import pynvml as N
            N.nvmlInit()
            h = N.nvmlDeviceGetHandleByPciBusId(self.pci.encode()) if self.pci else N.nvmlDeviceGetHandleByIndex(self.index)
            reasons_fn = getattr(N, "nvmlDeviceGetCurrentClocksEventReasons", None) or N.nvmlDeviceGetCurrentClocksThrottleReasons
            bits = [(0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap")]
            mx = N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM)
            while not self.stop_flag:
                r = reasons_fn(h)
                self.samples.append([str(N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)), str(mx)] +
                                    ["Active" if r & b else "Not Active" for b, _ in bits])
                time.sleep(0.02)
            return
        except Exception:
            pass
        while not self.stop_flag:          # fallback: the nvidia-smi query line of the profiling recipe
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.25)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples if len(s) > 2 + i)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(self.samples[0][1]) if self.samples[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------ CPU reference arm
def cpu_reference_pair(pair, threads):
    """The reference's CPU path (oracle port) on one frame pair: extract both frames, symmetric 2-NN match, calibrate, ARRSAC +
    eight-point.  Returns (seconds, matches, inliers or None, bearings)."""
    from oracle import pyoracle as O
    O.set_num_threads(threads)      # torchrun exports OMP_NUM_THREADS=1; the CPU arm may use every host thread
    t0 = time.perf_counter()
    ks, ds = [], []
    for f in pair:
        k, d = O.Akaze(maximum_features=MAXF).extract(f)
        ks.append(k); ds.append(d)
    fi, fd = O.hamming_knn(ds[0], ds[1], 2)
    ri, rd = O.hamming_knn(ds[1], ds[0], 2)
    fwd = np.where(fd[:, 0] + BETTER_BY <= fd[:, 1], fi[:, 0].astype(np.int64), -1)
    rev = np.where(rd[:, 0] + BETTER_BY <= rd[:, 1], ri[:, 0].astype(np.int64), -1)
    pairs = np.array([(i, j) for i, j in enumerate(fwd) if j >= 0 and rev[j] == i], np.int64).reshape(-1, 2)
    ba, bb = calibrate_np(ks[0][pairs[:, 0]]), calibrate_np(ks[1][pairs[:, 1]])
    cfg = O.arrsac_cfg(ARRSAC["threshold"], initialization_hypotheses=ARRSAC["initialization_hypotheses"],
                       max_candidate_hypotheses=ARRSAC["max_candidate_hypotheses"])
    r = O.arrsac(cfg, 0, ba, bb, O.rng_xoshiro(0)) if len(pairs) else None
    return time.perf_counter() - t0, len(pairs), (None if r is None else r[2]), (ba, bb)


def calibrate_np(kps):
    """cv-pinhole CameraIntrinsics::calibrate, identical to cv_b200/pinhole.py (no import of the product in the CPU arm)."""
    y = (kps["y"].astype(np.float64) - CY) / FOCAL
    x = (kps["x"].astype(np.float64) - CX - 0.0 * y) / FOCAL
    n = np.sqrt(x * x + y * y + 1.0)
    return np.stack([x / n, y / n, 1.0 / n], 1)


def run_reference(args, rank, world):
    if rank != 0:
        return
    frames = make_pool(2)
    cores = os.cpu_count()
    for i in range(min(args.warmup, 1)):
        cpu_reference_pair(frames[i % 2], cores)
    steps = args.steps                       # one frame pair (~5 s of CPU work) per step
    t = [cpu_reference_pair(frames[i % 2], cores) for i in range(steps)]
    sec = sum(x[0] for x in t) / steps
    fps = 2.0 / sec
    sec1 = cpu_reference_pair(frames[0], 1)[0]      # the reference's default build is unthreaded (akaze/README.md:22)
    line = {"metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": min(args.warmup, 1), "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": WORKLOAD, "maximum_features": MAXF, "detector_threshold": 0.001, "better_by": BETTER_BY, "arrsac": ARRSAC,
                       "pairs_per_step": 1, "note": "one frame pair per step (the GPU arm's step is a batch of "
                                                    f"{PAIRS_PER_STEP} pairs); frames/s is step-size independent"},
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
                             "single_thread_value": 2.0 / sec1,
                             "sample": f"{steps} frame pair(s), matches {t[0][1]}, inliers {0 if t[0][2] is None else len(t[0][2])}; C restatement of "
                                       "rust-cv akaze/space/arrsac/eight-point (oracle/, -O3 -march=x86-64-v3 -ffp-contract=off), OpenMP at the reference's "
                                       "rayon sites and over independent hypotheses; single_thread_value = the same pair on 1 thread"},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def allpairs64(rank, world, local_rank, dev, cap):
    """BASELINE configs[3]: 64 synthetic 1080p frames sharded round-robin, extract all, ONE packed all-gather of descriptors, all
    2 016 frame pairs matched symmetrically (pairs partitioned over the ranks).  CUDA-event times, max over ranks."""
    import torch
    import torch.distributed as dist
    from cv_b200 import AkazeConfig, dist as D, multi
    from tests.synth import synth_frame, warp_frame
    F = 64
    mine = D.shard_frames(F, rank, world)
    bases = {}
    frames = []
    for g in mine:        # 4 base textures, every frame a distinct warp (smooth camera path); content only has to yield ~5k keypoints
        b = g % 4
        if b not in bases:
            bases[b] = synth_frame(500 + b)
        frames.append(bases[b] if g < 4 else warp_frame(bases[b], 2000 + g, shift=(0.9 * (g // 4), -0.6 * (g // 4))))
    imgs = torch.from_numpy(np.stack(frames)).to(dev)
    ctx = multi.make_context(local_rank)
    cfg = AkazeConfig(maximum_features=cap)
    tm = {}
    multi.extract_and_match_all_pairs(ctx, cfg, imgs, F, cap=cap, better_by=BETTER_BY, timing=tm)        # warm-up: workspaces, graphs
    if world > 1:
        dist.barrier()
    tm = {}
    counts, res = multi.extract_and_match_all_pairs(ctx, cfg, imgs, F, cap=cap, better_by=BETTER_BY, timing=tm)
    t = torch.tensor([tm["extract_ms"], tm["match_ms"], tm["gather_ms"], tm["total_ms"]], dtype=torch.float64, device=dev)
    c = torch.tensor([tm["comparisons"], float(sum(len(v) for v in res.values()))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
    t, c = t.cpu().numpy(), c.cpu().numpy()
    ctx.close()
    return {"frames": F, "frame_pairs": F * (F - 1) // 2, "keypoints_per_frame_mean": float(np.mean(list(counts.values()))),
            "extract_frames_per_s": F / (t[0] * 1e-3), "match_Gcmp_per_s": c[0] / (t[1] * 1e-3) / 1e9, "comparisons": c[0], "matches_total": int(c[1]),
            "extract_ms": t[0], "match_ms": t[1], "total_ms": t[3], "collective": "one all_gather_into_tensor of the packed descriptors (NCCL over NVLink)",
            "collective_us": t[2] * 1e3, "collective_bytes": tm["gather_bytes"], "pairs_this_rank": tm["pairs"], "pairs_matched_during_gather": tm["local_pairs"],
            "timing": "CUDA events on the rank's stream, max over ranks; the match time includes waiting for the all-gather"}


def track256(rank, world, ctxs):
    """BASELINE configs[4]: the cv-sfm registration loop over a 256-frame synthetic track -- per frame
    Arrsac(1e-5, init 16384, max_cand 1024, est/block 256) + LambdaTwist on ~2 000 FeatureWorldMatches (20 % outliers), then
    LinearEigenTriangulator on every landmark with >= 3 inlier observations.  Every rank runs its own track (replicas, weak scaling);
    the frames of a track are independent registrations, handed to the contexts' host threads.  Host API (host pointers in, results
    on the host), wall clock."""
    import cv_b200
    from tests.geom_util import world_homog
    from tests.synth import helix_track, landmark_observations
    F = int(os.environ.get("CVB_BENCH_TRACK_FRAMES", "256"))
    cloud, frames = helix_track(1 + rank, F, 20000, 2000, 0.2)
    worlds = [world_homog(cloud[fr["ids"]]) for fr in frames]
    regs = [None] * F
    nthreads = len(ctxs)

    def register(k, c):
        ars = (cv_b200.Arrsac(1e-5, cv_b200.Xoshiro256PlusPlus(100 + k), ctx=ctxs[c]).initialization_hypotheses(16384)
               .max_candidate_hypotheses(1024).estimations_per_block(256))
        regs[k] = ars.model_inliers(cv_b200.LambdaTwist(), frames[k]["bearing"], worlds[k])

    def sweep(first, count):
        lock, nxt = threading.Lock(), [first]

        def worker(c):
            while True:
                with lock:
                    k = nxt[0]
                    if k >= first + count:
                        return
                    nxt[0] = k + 1
                register(k, c)
        th = [threading.Thread(target=worker, args=(c,)) for c in range(nthreads)]
        for t in th:
            t.start()
        for t in th:
            t.join()
    sweep(0, min(F, 2 * nthreads))                 # warm-up: workspaces of every context
    t0 = time.perf_counter()
    sweep(0, F)
    t_reg = time.perf_counter() - t0
    # feature tracks of bounded length (the first 8 inlier observations of a landmark): the reference's cheirality rule
    # (cv-geom/src/triangulation.rs:120-127) rejects a landmark as soon as ONE of its views sees it from the far side of the world
    # origin, which over four full turns of the orbit would be nearly every landmark
    ids, poses, bearings, offsets = landmark_observations(frames, regs, max_obs=8)
    from cv_b200.geom import POSE_DTYPE
    parr = np.zeros(len(poses), POSE_DTYPE)
    parr["r"] = np.array([p[0] for p in poses]).reshape(-1, 9); parr["t"] = np.array([p[1] for p in poses]).reshape(-1, 3)
    tri = cv_b200.LinearEigenTriangulator()
    tri.triangulate_batch(parr, bearings, offsets)
    t0 = time.perf_counter()
    pts, ok = tri.triangulate_batch(parr, bearings, offsets)
    t_tri = time.perf_counter() - t0
    inl = [0 if r is None else len(r[2]) for r in regs]
    good = [float(fr["good"][r[2]].mean()) for fr, r in zip(frames, regs) if r is not None and len(r[2])]
    xyz = pts[ok, :3] / pts[ok, 3:4]
    err = np.linalg.norm(xyz - cloud[np.array(ids)[ok]], axis=1) if ok.any() else np.array([np.nan])
    return {"frames": F, "matches_per_frame": 2000, "outlier_fraction": 0.2, "registered": int(sum(r is not None for r in regs)),
            "inliers_per_frame_mean": float(np.mean(inl)), "inlier_purity_mean": float(np.mean(good)) if good else None,
            "registration_ms_total": t_reg * 1e3, "registrations_per_s": F / t_reg, "host_threads": nthreads,
            "landmarks": len(ids), "observations": len(poses), "max_observations_per_landmark": 8, "triangulated_ok": int(ok.sum()), "triangulation_ms": t_tri * 1e3,
            "landmarks_per_s": len(ids) / t_tri if t_tri > 0 else None, "median_landmark_error": float(np.median(err)),
            "arrsac": {"threshold": 1e-5, "initialization_hypotheses": 16384, "max_candidate_hypotheses": 1024, "estimations_per_block": 256},
            "timing": "host API (host pointers in, results on the host), wall clock, this rank's replica"}


def dump_outputs(out_dir, pairs, pair_dev, slot, cap):
    """--dump-outputs: what the device-resident path hands its caller for each frame pair of the last timed step, as .npy files
    (float32 holds every index and keypoint field exactly; at most ~47 MB for 16 pairs of 5 000 keypoints per frame).  The pairs
    run again, one at a time on context 0, after the timed region: a pair's result depends only on its frames and its generator
    seed (the pair index), so it is the result the timed step computed.
      keypoints   [N, 7]  x, y, response, size, angle, octave, class_id; frame a then frame b of each pair, in pair order
      descriptors [N, 64] descriptor bytes, rows as in keypoints
      matches     [M, 2]  keypoint index in frame a, keypoint index in frame b; in pair order
      inliers     [I]     consensus inliers as indices into the pair's matches; in pair order
      poses       [P, 12] consensus model (rotation row-major, translation); zero where none was found
      counts      [P, 6]  pair index, keypoints in a, keypoints in b, matches, inliers, model found"""
    from cv_b200._lib import KP_DTYPE
    kps, descs, matches, inliers, poses, counts = [], [], [], [], [], []
    for i in pairs:
        pair_dev(i, 0)                  # returns with the context's stream drained
        na, nb = slot.n.cpu().numpy().tolist()
        npairs, ninl, found = slot.cnt.cpu().numpy()[:3].tolist()
        kp = np.frombuffer(slot.kp.cpu().numpy().tobytes(), KP_DTYPE)
        desc = slot.desc.cpu().numpy().reshape(2 * cap, 64)
        for lo, n in ((0, na), (cap, nb)):
            kps.append(np.stack([kp[f][lo:lo + n].astype(np.float32) for f in KP_DTYPE.names], 1))
            descs.append(desc[lo:lo + n].astype(np.float32))
        matches.append(slot.pairs.cpu().numpy()[:2 * npairs].reshape(-1, 2).astype(np.float32))
        inliers.append(slot.inl.cpu().numpy()[:ninl].astype(np.float32))
        poses.append(slot.model.cpu().numpy() if found else np.zeros(12))
        counts.append([i, na, nb, npairs, ninl, found])
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("keypoints", np.concatenate(kps)), ("descriptors", np.concatenate(descs)), ("matches", np.concatenate(matches)),
                    ("inliers", np.concatenate(inliers)), ("poses", np.stack(poses)), ("counts", np.array(counts, np.float64))):
        np.save(os.path.join(out_dir, name + ".npy"), a)


def bind_to_gpu_numa_node(props):
    """Run this process (and the pinned buffers it first-touches) on the CPUs local to the GPU's PCIe root, like a deployed
    service would; silently skipped when sysfs does not expose the topology."""
    try:
        bus = f"{props.pci_domain_id:04x}:{props.pci_bus_id:02x}:{props.pci_device_id:02x}.0"
        cpus = set()
        for part in open(f"/sys/bus/pci/devices/{bus}/local_cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
    except Exception:
        pass


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cvb200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step's frame pairs to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path only")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    import torch
    import torch.distributed as dist
    import cv_b200
    from cv_b200._lib import KP_DTYPE
    from cv_b200.geom import ArrsacCfg, Pose, Rng, _lib as geom_lib
    from cv_b200.pair import Intrinsics, bind as pair_bind
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if os.environ.get("CVB_BENCH_NUMA_BIND", "1") == "1":
        bind_to_gpu_numa_node(torch.cuda.get_device_properties(local_rank))
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    K, Wm = args.steps, max(args.warmup, 3)          # timing rule: at least 3 warm-up steps
    NCTX = int(os.environ.get("CVB_BENCH_CONTEXTS", "16"))   # 16 contexts x (main + auxiliary stream) = the 32 hardware queues: more contexts alias queues   # contexts (stream + workspace + host thread each) pipelined on the GPU

    frames = make_pool(POOL_PAIRS, seed0=100 * rank)
    ctxs = [cv_b200.Context(local_rank) for _ in range(NCTX)]
    ctx = ctxs[0]
    lib = ctx.lib
    geom_lib(ctx)
    pair_bind(lib)
    akaze_cfg = cv_b200.AkazeConfig(maximum_features=MAXF).to_c()
    intr = Intrinsics(FOCAL, FOCAL, CX, CY, 0.0)
    acfg = ArrsacCfg()
    lib.cvb_arrsac_default_cfg(C.byref(acfg), ARRSAC["threshold"])
    acfg.initialization_hypotheses = ARRSAC["initialization_hypotheses"]
    acfg.max_candidate_hypotheses = ARRSAC["max_candidate_hypotheses"]
    cap = MAXF
    d_pool = [torch.from_numpy(p).to(dev) for p in frames]
    h_pool = [torch.from_numpy(p).pin_memory() for p in frames]

    class Slot:
        """Everything one context owns: device result buffers, pinned host result buffers, its consensus generator (pair_dev
        seeds it per pair; pair_host carries it across frame pairs, like the two_view_consensus object of a VSlam instance)."""
        def __init__(self):
            self.kp = torch.empty(2 * cap * KP_DTYPE.itemsize, dtype=torch.uint8, device=dev)
            self.desc = torch.zeros(2 * cap * 64, dtype=torch.uint8, device=dev)
            self.n = torch.zeros(2, dtype=torch.int32, device=dev)
            self.pairs = torch.zeros(cap * 2, dtype=torch.int32, device=dev)
            self.inl = torch.zeros(cap, dtype=torch.int32, device=dev)
            self.cnt = torch.zeros(4, dtype=torch.int32, device=dev)      # n_pairs, n_inliers, found
            self.model = torch.zeros(12, dtype=torch.float64, device=dev)
            self.h_kp = torch.empty(2 * cap * KP_DTYPE.itemsize, dtype=torch.uint8).pin_memory()
            self.h_desc = torch.empty(2 * cap * 64, dtype=torch.uint8).pin_memory()
            self.h_pairs = torch.empty(cap * 2, dtype=torch.int32).pin_memory()
            self.h_inl = torch.empty(cap, dtype=torch.int32).pin_memory()
            self.h_n = (C.c_uint32 * 2)()
            self.h_np, self.h_ni, self.h_found = C.c_uint32(), C.c_uint32(), C.c_int32()
            self.h_model = Pose()
            self.rng = Rng()
            lib.cvb_rng_seed_xoshiro256pp(C.byref(self.rng), 0)
            self.stats = (C.c_uint32 * 16)()
            self.pairs_done = 0
            self.t_busy = 0.0
    slots = [Slot() for _ in range(NCTX)]

    def pair_dev(i, c):
        """device-resident: frames already in HBM, results stay in HBM; one synchronisation (the generator commit).  The
        consensus generator is seeded with the pair index, so pair i's result does not depend on which context ran it."""
        cx, s = ctxs[c], slots[c]
        img = d_pool[i % POOL_PAIRS]
        lib.cvb_rng_seed_xoshiro256pp(C.byref(s.rng), i)
        cx.check(lib.cvb_akaze_extract_batch_dev(cx.handle, C.byref(akaze_cfg), img.data_ptr(), 2, W, H, s.kp.data_ptr(), s.desc.data_ptr(), cap,
                                                 s.n.data_ptr()))
        cx.check(lib.cvb_two_view_pair_dev(cx.handle, s.kp.data_ptr(), s.desc.data_ptr(), s.n.data_ptr(),
                                           s.kp.data_ptr() + cap * KP_DTYPE.itemsize, s.desc.data_ptr() + cap * 64, s.n.data_ptr() + 4, cap,
                                           BETTER_BY, C.byref(intr), C.addressof(acfg), C.addressof(s.rng), s.pairs.data_ptr(), cap,
                                           s.cnt.data_ptr(), s.model.data_ptr(), s.inl.data_ptr(), s.cnt.data_ptr() + 4, s.cnt.data_ptr() + 8))
        cx.check(lib.cvb_arrsac_commit_rng(cx.handle, C.addressof(s.rng), s.stats))

    def pair_host(i, c):
        """end to end: pinned host frames in, every result back on the host"""
        cx, s = ctxs[c], slots[c]
        img = h_pool[i % POOL_PAIRS]
        cx.check(lib.cvb_two_view_frames(cx.handle, C.addressof(akaze_cfg), img.data_ptr(), W, H, BETTER_BY, C.byref(intr), C.addressof(acfg),
                                         C.addressof(s.rng), s.h_kp.data_ptr(), s.h_desc.data_ptr(), cap, s.h_n, s.h_pairs.data_ptr(),
                                         C.byref(s.h_np), C.byref(s.h_model), s.h_inl.data_ptr(), C.byref(s.h_ni), C.byref(s.h_found)))

    def run_pairs(fn, first, count, nthreads=NCTX):
        """`count` pairs handed out dynamically to one host thread per context (the blocking C calls release the GIL)"""
        lock, nxt = threading.Lock(), [first]

        def worker(c):
            while True:
                with lock:
                    i = nxt[0]
                    if i >= first + count:
                        return
                    nxt[0] = i + 1
                t0 = time.perf_counter()
                fn(i, c)
                slots[c].t_busy += time.perf_counter() - t0
                slots[c].pairs_done += 1
        th = [threading.Thread(target=worker, args=(c,)) for c in range(nthreads)]
        for t in th:
            t.start()
        for t in th:
            t.join()

    def barrier():
        for cx in ctxs:
            cx.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def reset_rngs():
        for s in slots:
            lib.cvb_rng_seed_xoshiro256pp(C.byref(s.rng), 0)
            s.pairs_done = 0; s.t_busy = 0.0

    # ---- setup (not a warm-up step): every (context, input buffer) pair captures its extraction graph; workspaces are allocated
    for c in range(NCTX):
        for i in range(POOL_PAIRS):
            pair_dev(i, c)
    barrier()
    try:
        pr = torch.cuda.get_device_properties(local_rank)
        pci = f"{pr.pci_domain_id:08x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
    except Exception:
        pci = None
    sampler = ClockSampler(local_rank, pci)
    sampler.start()

    # ---- value: device-resident, W warm-up steps then exactly K timed steps of PAIRS_PER_STEP pairs
    reset_rngs()
    run_pairs(pair_dev, 0, Wm * PAIRS_PER_STEP)
    barrier()
    l0 = sum(cx.launch_count() for cx in ctxs)
    for s in slots:
        s.pairs_done = 0; s.t_busy = 0.0
    t0 = time.perf_counter()
    ctx.timer_begin()                      # CUDA events on context 0's stream, which is idle here and again at timer_end
    run_pairs(pair_dev, Wm * PAIRS_PER_STEP, K * PAIRS_PER_STEP)     # every worker returns with its stream drained (generator commit)
    ms = ctx.timer_end()
    wall_ms = (time.perf_counter() - t0) * 1e3
    barrier()
    assert ms > 0.5 * wall_ms or wall_ms < 1.0, f"device timer {ms} ms disagrees with wall clock {wall_ms} ms"
    launches = sum(cx.launch_count() for cx in ctxs) - l0
    from cv_b200 import dist as D
    value, ms_max = D.aggregate_throughput(2.0 * K * PAIRS_PER_STEP, ms, dev)      # frames of all ranks / max-over-ranks device time
    dev_busy = [round(s.t_busy / max(s.pairs_done, 1) * 1e3, 3) for s in slots]
    stats0 = [int(x) for x in slots[0].stats]
    n_kp = slots[0].n.cpu().numpy().tolist()
    cnt0 = slots[0].cnt.cpu().numpy().tolist()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, range((Wm + K - 1) * PAIRS_PER_STEP, (Wm + K) * PAIRS_PER_STEP), pair_dev, slots[0], cap)

    # ---- e2e: host entry point, pinned host buffers, copies inside the timed region
    reset_rngs()
    run_pairs(pair_host, 0, Wm * PAIRS_PER_STEP)
    barrier()
    for s in slots:
        s.pairs_done = 0; s.t_busy = 0.0
    t0 = time.perf_counter()
    cpu0 = time.process_time()
    run_pairs(pair_host, Wm * PAIRS_PER_STEP, K * PAIRS_PER_STEP)
    ms_e2e = (time.perf_counter() - t0) * 1e3     # blocking host API: wall clock over the K steps (all results on the host)
    host_cpu_ms_per_pair = (time.process_time() - cpu0) * 1e3 / (K * PAIRS_PER_STEP)
    barrier()
    s0 = slots[0]
    nb_max = (cap + 63) // 64 + 1
    nraw = 8192 * 8 + 8192 * 8 // 4 + 64 + nb_max * (64 * 8 + 64 * 8 // 4 + 64)     # geom.cu: arrsac_run_dev
    h2d_step = PAIRS_PER_STEP * (2 * W * H * 4 + 4 * nraw + 160)                  # frames + the consensus generator's draw stream + control block
    d2h_step = PAIRS_PER_STEP * (2 * cap * (KP_DTYPE.itemsize + 64) + cap * 8 + cap * 4 + 16 + 96 + 8 + 160)
    e2e_value, _ = D.aggregate_throughput(2.0 * K * PAIRS_PER_STEP, ms_e2e, dev)
    per_rank = torch.tensor([2.0 * K * PAIRS_PER_STEP / (ms_e2e * 1e-3), h2d_step * K / (ms_e2e * 1e-3) / 1e9, host_cpu_ms_per_pair],
                            dtype=torch.float64, device=dev)
    per_rank_all = [torch.zeros_like(per_rank) for _ in range(world)]
    if world > 1:
        dist.all_gather(per_rank_all, per_rank)
    else:
        per_rank_all = [per_rank]
    per_rank_all = [[round(float(v), 3) for v in t.cpu().tolist()] for t in per_rank_all]
    e2e_busy = [round(s.t_busy / max(s.pairs_done, 1) * 1e3, 3) for s in slots]
    e2e_pairs = [s.pairs_done for s in slots]
    sampler.stop_flag = True
    sampler.join(timeout=2)

    # ---- parity of the benchmarked result: pair 0 through the host entry point vs the CPU oracle on the same bearings
    inliers_equal_oracle = None
    ransac = None
    if rank == 0:
        try:
            lib.cvb_rng_seed_xoshiro256pp(C.byref(s0.rng), 0)
            pair_host(0, 0)
            npairs, ninl = int(s0.h_np.value), int(s0.h_ni.value)
            kp = np.frombuffer(s0.h_kp.numpy().tobytes(), dtype=KP_DTYPE)
            pr_ = s0.h_pairs.numpy()[:2 * npairs].reshape(-1, 2).astype(np.int64)
            ba, bb = calibrate_np(kp[:cap][pr_[:, 0]]), calibrate_np(kp[cap:2 * cap][pr_[:, 1]])
            gpu_inl = s0.h_inl.numpy()[:ninl].astype(np.int64)
            from oracle import pyoracle as O      # checker only
            O.set_num_threads(os.cpu_count())
            want = O.arrsac(O.arrsac_cfg(ARRSAC["threshold"], initialization_hypotheses=ARRSAC["initialization_hypotheses"],
                                         max_candidate_hypotheses=ARRSAC["max_candidate_hypotheses"]), 0, ba, bb, O.rng_xoshiro(0))
            inliers_equal_oracle = bool(want is not None and int(s0.h_found.value) == 1 and np.array_equal(want[2].astype(np.int64), gpu_inl))
            # single-call latencies of the consensus stage alone (host API, data upload included)
            ars = cv_b200.Arrsac(ARRSAC["threshold"], cv_b200.Xoshiro256PlusPlus(0), ctx=ctx).initialization_hypotheses(
                ARRSAC["initialization_hypotheses"]).max_candidate_hypotheses(ARRSAC["max_candidate_hypotheses"])
            for _ in range(3):       # the second call with the same buffers captures the run's graph; time replays only
                ars.model_inliers(cv_b200.EightPoint(), ba, bb)
            lat = []
            for _ in range(7):
                t0 = time.perf_counter()
                ars.model_inliers(cv_b200.EightPoint(), ba, bb)
                lat.append((time.perf_counter() - t0) * 1e3)
            lat.sort()
            ransac = {"config": "Arrsac(1e-7, Xoshiro256++).initialization_hypotheses(8192).max_candidate_hypotheses(1024) + EightPoint",
                      "matches": npairs, "inliers": ninl, "single_call_latency_ms": lat[len(lat) // 2], "single_call_latency_ms_max": lat[-1],
                      "note": "median (and maximum) of 7 isolated calls through the host API (upload, every kernel, download); inside the pipelined step its kernels overlap other pairs"}
        except Exception as ex:   # never fail the headline line on the cross-check
            ransac = {"error": repr(ex)}

    # ---- BASELINE configs[3] (multi-frame all-pairs workload; the one place the path has a collective)
    ap64 = None
    if os.environ.get("CVB_BENCH_ALLPAIRS", "1") == "1":
        try:
            ap64 = allpairs64(rank, world, local_rank, dev, cap)
        except Exception as ex:      # secondary block: never fail the headline line
            ap64 = {"error": repr(ex)}

    # ---- BASELINE configs[4] (P3P registration + triangulation over a 256-frame track; one replica per rank)
    tr256 = None
    if os.environ.get("CVB_BENCH_TRACK", "1") == "1":
        try:
            tr256 = track256(rank, world, ctxs)
        except Exception as ex:
            tr256 = {"error": repr(ex)}
        if world > 1:          # every rank takes part in the reduction, whatever happened to its replica
            v = torch.tensor([tr256.get("registration_ms_total", 0.0), tr256.get("triangulation_ms", 0.0)], dtype=torch.float64, device=dev)
            dist.all_reduce(v, op=dist.ReduceOp.MAX)
            v = v.cpu().tolist()
            if "error" not in tr256:
                tr256["replicas"] = world
                tr256["registrations_per_s_all_ranks"] = world * tr256["frames"] / (v[0] * 1e-3)
                tr256["landmarks_per_s_all_ranks"] = world * tr256["landmarks"] / (v[1] * 1e-3) if v[1] > 0 else None

    # ---- roofline: instrumented pass (per-kernel CUDA events on the launching stream, one context, no overlap)
    ctx.profile(True)
    PK = 6
    for i in range(PK):
        pair_dev(i, 0)
    rep = ctx.profile_report()
    ctx.profile(False)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"
    tot_ms = sum(v["ms"] for v in rep.values())
    top = max(rep.items(), key=lambda kv: kv[1]["ms"]) if rep else (None, None)
    kernels = {k: {"launches_per_pair": v["launches"] / PK, "ms_per_pair": v["ms"] / PK, "share": v["ms"] / tot_ms if tot_ms else 0,
                   "alg_GBps": (v["bytes"] / (v["ms"] * 1e-3) / 1e9) if v["ms"] > 0 and v["bytes"] > 0 else None} for k, v in rep.items()}
    hb = {k: v for k, v in rep.items() if v["bytes"] > 0 and k != "k_hamming_knn"}      # the matcher's 64 B/cmp is a streaming model, not traffic
    dom = max(hb.items(), key=lambda kv: kv[1]["ms"])
    achieved = dom[1]["bytes"] / (dom[1]["ms"] * 1e-3) / 1e9
    traffic, traffic_src = None, None
    try:      # DRAM bytes per launch of the dominant kernel from the committed ncu capture (profiles/), not measured live
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(dom[0])
        if tj:
            traffic, traffic_src = tj["dram_bytes_per_launch"], tj["source"]
    except Exception:
        pass
    fps_rank = value / world
    roofline = {"bound": "hbm", "kernel": dom[0], "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "launch_ms": dom[1]["ms"] / dom[1]["launches"], "bytes_per_launch": dom[1]["bytes"] / dom[1]["launches"],
                "timing": "per-kernel CUDA events on the launching stream, separate instrumented pass of the same pairs (one context, no overlap)",
                "pipeline_alg_GBps": fps_rank * ALG_BYTES_PER_FRAME / 1e9, "pipeline_frac": fps_rank * ALG_BYTES_PER_FRAME / 1e9 / hbm_peak,
                "top_kernel_by_time": top[0], "kernels": kernels}
    knn = rep.get("k_hamming_knn")
    gcmp = (knn["bytes"] / 64.0) / (knn["ms"] * 1e-3) / 1e9 if knn and knn["ms"] > 0 else None
    # RANSAC scoring figure (SURVEY.md 8d): (hypothesis, datum) predicates per second of the scoring kernels
    sc = [rep.get("k_ars_score_init"), rep.get("k_ars_score_block")]
    ransac_scoring = None
    if sc[0] and stats0[1]:
        init_pairs = 32 * (stats0[8] + stats0[9])          # predicates the two scoring stages actually evaluated
        ransac_scoring = {"init_models": stats0[1], "init_predicates": init_pairs, "score_init_ms": sc[0]["ms"] / PK,
                          "predicates_per_s": init_pairs / (sc[0]["ms"] / PK * 1e-3) if sc[0]["ms"] > 0 else None,
                          "sprt_pass": stats0[2], "sprt_commit_rounds": stats0[3], "block_iterations": stats0[4], "draws": stats0[5],
                          "exact_fallbacks": stats0[10], "sprt_lazy_words": stats0[11], "sprt_repairs": stats0[12], "sprt_walk_steps": stats0[13]}

    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        sec, nm_cpu, inl_cpu, _ = cpu_reference_pair(frames[0], os.cpu_count())      # ~5 s of CPU work
        sec1 = cpu_reference_pair(frames[0], 1)[0]                                  # ~20 s: the reference's default build is unthreaded
        cpu = {"value": 2.0 / sec, "unit": "frames/s", "cores": os.cpu_count(), "kind": "port", "single_thread_value": 2.0 / sec1,
               "sample": f"1 frame pair of the same workload (2 extracts, symmetric match, ARRSAC: {nm_cpu} matches, "
                         f"{0 if inl_cpu is None else len(inl_cpu)} inliers) on all host threads, and the same pair on 1 thread; C restatement of the "
                         "reference (oracle/, -O3), OpenMP at the reference's rayon sites and over independent hypotheses"}
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": Wm,
                "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32+f64", "data": "synthetic",
                "config": {"workload": WORKLOAD, "pairs_per_step": PAIRS_PER_STEP, "frames_per_step_per_gpu": 2 * PAIRS_PER_STEP,
                           "keypoints_per_frame": n_kp, "matches": cnt0[0], "inliers": cnt0[1], "maximum_features": MAXF,
                           "detector_threshold": 0.001, "better_by": BETTER_BY, "arrsac": ARRSAC, "intrinsics": [FOCAL, FOCAL, CX, CY],
                           "pipelining": f"{NCTX} contexts (CUDA stream + workspace + host thread + consensus generator each) take pairs from a "
                                         "shared queue; extraction is one CUDA graph per context",
                           "l2": f"inputs rotate over a pool of {2 * POOL_PAIRS} distinct frames ({2 * POOL_PAIRS * W * H * 4 / 1e6:.0f} MB > 126 MB L2)",
                           "setup": "graph capture / allocation pass over every (context, input) pair before the warm-up steps"},
                "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": h2d_step, "d2h_bytes_per_step": d2h_step,
                        "host_threads": NCTX, "timed_region_ms": ms_e2e, "mean_call_ms": sum(e2e_busy) / len(e2e_busy),
                        "pairs_per_thread": e2e_pairs,
                        "per_rank": {"columns": ["frames_per_s", "h2d_GBps", "host_cpu_ms_per_pair"], "rows": per_rank_all}},
                "timed_region_ms": ms_max, "mean_pair_latency_ms": sum(dev_busy) / len(dev_busy),
                "gpu_launches": int(launches), "roofline": roofline, "hamming_Gcmp_per_s": gcmp, "ransac_two_view": ransac,
                "ransac_scoring": ransac_scoring, "allpairs64": ap64, "track256": tr256, "inliers_equal_oracle": inliers_equal_oracle, "cpu_baseline": cpu,
                "clocks": sampler.summary()}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
