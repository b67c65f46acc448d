#!/usr/bin/env python
"""bench.py -- mocap frame-sets/s of the B200 marker-tracking core (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One "step" = one pass of the hot path (S1 blob detection -> S2 epipolar matching -> S3 DLT
triangulation + reprojection error, one launch group per batch) over one batch of synthetic
frame-sets.  Workload at N = 1: BASELINE config 2 -- 4 cameras, 4 markers, 10 000 frame-sets of
640x480 uint8 per step, resident in HBM (12.3 GB >> L2, so every step reads HBM; the batch cycles
through 4096 distinct frame-sets rendered on the device).  N > 1: one process per GPU (torchrun),
every rank owns its own 10 000-frame-set shard of the stream (round-robin ownership, weak scaling)
and the ranks exchange ONE NCCL all-gather of 3D track records per batch.
--workload c8m16: 8 cameras, 16 markers, 4000 distinct frame-sets per GPU per step -- at N = 1
BASELINE config 3 (S1-S3 plus one bundle adjustment S4 per 1000 frame-sets, all on the device), at
N > 1 config 4 (S1-S3 + the all-gather).  Every rank asserts that the timed batch carries no
overflow flag, checks its first frame-sets against the oracle and (config 3) that S4 converged to
the true rig; a failed check fails the run.

Printed JSON line (rank 0): value = whole-job frame-sets/s with inputs resident in HBM;
e2e = the same through the host-buffer C-ABI call (pinned host frames, H2D + D2H inside the
timed region); roofline = the dominant kernel (k_pipeline_fused, or the stream kernel of the
three-kernel pipeline on heavy frame-sets) against the measured HBM peak, traffic from the
committed ncu capture while the kernels are the ones that were profiled; cpu_baseline = the oracle port (the reference's own cv2/numpy/scipy call sequence) on
this box's host cores on a bounded sample.

--impl reference times the reference's CPU implementation (oracle port: the reference is
Python and /root/reference does not exist on the GPU box) on all host cores, same workload
shape, bounded sample per step.
"""
import os

# one worker PROCESS per host core is how the CPU arm fans out; BLAS / OpenMP / cv2 pools inside every worker
# would oversubscribe the box 128-fold, so they are pinned to one thread before numpy / scipy / cv2 are imported
for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS", "NUMEXPR_NUM_THREADS", "VECLIB_MAXIMUM_THREADS"):
    os.environ[_v] = "1"

import argparse
import importlib
import json
import math
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_CAM, N_MARKERS, BATCH = 4, 4, 10000
POOL = 4096                      # distinct rendered frame-sets per GPU (SURVEY 8(d): >= 4096); the batch cycles through them
CPU_POOL = 250                   # host-rendered frame-sets of the same generator for the CPU arm
WITH_BA = False                  # config 3: one bundle adjustment per BA_BATCH frame-sets
BA_BATCH = 1000
BA_MAX_ERR = 2.0                 # tracks whose reprojection error exceeds this (px^2) are not handed to S4
WIDTH, HEIGHT = 640, 480
MAX_ROOTS = 16
MAX_GROUPS = 4096
HBM_FALLBACK_GBS = 6650.0        # /opt/skills/guides/B200_PROFILING.md fallback


# ------------------------------------------------------------------------------------------------
def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 6 and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def make_pool():
    synth = importlib.import_module("low-cost-mocap_b200.synth")
    return synth.make_frame_pool(N_CAM, N_MARKERS, min(CPU_POOL, 250 if N_CAM <= 4 else 100), seed=0)


# ------------------------------------------------------------------------------------------------
# CPU side: the oracle port, one worker process per core (the reference itself is single-threaded
# Python; frame-sets are independent, so fanning out over processes is the most it can use)
_W = {}


def _cpu_init(K, poses):
    import cv2
    cv2.setNumThreads(1)
    from oracle.ref_port import RefPort
    _W["port"] = RefPort([K] * len(poses))
    _W["poses"] = poses


def _cpu_range(rng):
    """One task = one contiguous range of frame-sets (a handful of tasks per worker, so the dispatcher thread is
    idle).  Frames are inherited through fork as H x W x 3 arrays -- the layout the reference's _find_dot receives
    (helpers.py:143) -- so tasks carry two integers and no image bytes travel through pipes."""
    port, poses, frames3 = _W["port"], _W["poses"], _W["frames3"]
    lo, hi = rng
    got = 0
    for index in range(lo, hi):
        frame_set = frames3[index % len(frames3)]
        pts = [port.find_dot(img) for img in frame_set]
        e, o, _ = port.match_and_triangulate(pts, poses)
        got += len(e)
    return got


def cpu_pass(pool_obj, n_sets, n_workers):
    n_tasks = min(n_sets, 4 * n_workers)
    edges = [round(i * n_sets / n_tasks) for i in range(n_tasks + 1)]
    tasks = [(edges[i], edges[i + 1]) for i in range(n_tasks) if edges[i + 1] > edges[i]]
    t0 = time.perf_counter()
    got = pool_obj.map(_cpu_range, tasks, chunksize=1)
    return time.perf_counter() - t0, sum(got)


def host_cores():
    """CPUs this process may actually use: the affinity mask, capped by the container's cgroup CPU quota (a GPU box
    shows all 128 hardware threads in the mask but grants a fraction of them)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:                       # cgroup v2: "<quota> <period>" or "max <period>"
            q, p = f.read().split()[:2]
            if q != "max":
                quota = float(q) / float(p)
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f, open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as g:
                q, p = float(f.read()), float(g.read())
                if q > 0:
                    quota = q / p
        except Exception:
            pass
    if quota is not None:
        n = max(1, min(n, int(math.ceil(quota))))
    return n


class CpuArm:
    """The reference's CPU path (oracle port: the reference's own cv2 / numpy / scipy call sequence, pinned
    bit-exact to it) fanned out over the host cores.  The SAME object times the GPU arm's cpu_baseline leg and
    the --impl reference arm, so the two agree."""

    def __init__(self, frames, K, poses):
        import multiprocessing as mp
        self.cores = host_cores()
        self.K, self.poses = K, poses
        # 3-channel frames as the reference's capture loop hands them to _find_dot; built once, outside every timed region
        n3 = min(len(frames), 256 if frames.shape[1] <= 4 else 96)
        _W["frames3"] = np.ascontiguousarray(np.repeat(frames[:n3, :, :, :, None], 3, axis=4))
        _cpu_init(K, poses)
        _cpu_range((0, 1))                             # untimed: first-call imports and page-ins (seconds on a fresh box)
        t0 = time.perf_counter()                       # single core first (the reference is single-threaded Python)
        n = 0
        while time.perf_counter() - t0 < 3.0:
            _cpu_range((n, n + 1))
            n += 1
        self.single_core = n / (time.perf_counter() - t0)
        self.pool = mp.get_context("fork").Pool(self.cores, initializer=_cpu_init, initargs=(K, poses))
        cpu_pass(self.pool, 2 * self.cores, self.cores)        # spin the workers up (imports, page tables)
        t, _ = cpu_pass(self.pool, 4 * self.cores, self.cores)
        self.rate_probe = 4 * self.cores / t

    def sample_for(self, seconds, batch):
        """frame-sets per pass: at least 64 per worker so that start-up and the tail are amortised"""
        return int(min(max(batch, 64 * self.cores), max(64 * self.cores, seconds * self.rate_probe)))

    def run(self, n_sets):
        t, _ = cpu_pass(self.pool, n_sets, self.cores)
        return t

    def report(self, value, sample_text):
        eff = value / (self.cores * self.single_core)
        if eff < 0.5:
            print(f"bench.py: WARNING: CPU arm parallel efficiency {eff:.2f} < 0.5 ({value:.0f} frame-sets/s on {self.cores} "
                  f"cores vs {self.single_core:.0f} on one): the CPU figure understates the box", file=sys.stderr, flush=True)
        aff = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        return {"value": value, "unit": "frame-sets/s", "cores": self.cores, "kind": "port", "sample": sample_text,
                "single_core_value": self.single_core, "parallel_efficiency": eff,
                "cpus_in_affinity_mask": aff, "cores_note": "cores = min(affinity mask, cgroup CPU quota)"}

    def close(self):
        self.pool.close()
        self.pool.join()


def compare_with_oracle(ref, out):
    """3D-point distance between the GPU results of a timed step and the cpu_baseline leg's oracle output."""
    n = out["n"][:len(ref)].cpu().numpy()
    obj = out["obj"][:len(ref)].cpu().numpy()
    worst, same_count, points = 0.0, True, 0
    for b, o in enumerate(ref):
        same_count = same_count and (len(o) == int(n[b]))
        if len(o) and len(o) == int(n[b]):
            worst = max(worst, float(np.abs(obj[b, :len(o)] - o).max()))
            points += len(o)
    return {"frame_sets": len(ref), "points": points, "point_counts_equal": bool(same_count),
            "max_abs_3d_difference": worst, "tolerance": 1e-7}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    frames, truth, poses, K = make_pool()
    arm = CpuArm(frames, K, poses)
    cores = arm.cores
    # size one step so that the whole run (K timed steps + W quarter-size warm-up steps) takes about two and a
    # half minutes on this box; never fewer than 64 frame-sets per worker (start-up and tail amortised)
    step_s = max(0.25, 150.0 / (args.steps + 0.25 * args.warmup))
    sample = arm.sample_for(step_s, BATCH)
    for _ in range(args.warmup):
        arm.run(max(16 * cores, sample // 4))
    t = 0.0
    for _ in range(args.steps):
        t += arm.run(sample)
    arm.close()
    value = sample * args.steps / t
    line = {
        "impl": "reference", "metric": f"mocap frame-sets/s ({N_CAM}-cam 640x480 synthetic, blob+epipolar+DLT)",
        "value": value, "unit": "frame-sets/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8 pixels -> int64 moments -> f64 geometry", "data": "synthetic",
        "config": {"workload": f"BASELINE config {'2' if N_CAM == 4 else '3/4 shape'}: {N_CAM} cameras, {N_MARKERS} markers, 640x480 uint8 frame-sets; "
                               f"bounded sample of {sample} frame-sets per step of the {BATCH}-frame-set batch",
                   "cameras": N_CAM, "markers": N_MARKERS, "frame_sets_per_step": sample},
        "cpu_baseline": arm.report(value, f"{sample} frame-sets per step x {args.steps} steps, one worker process per core"),
        "e2e": {"value": value, "unit": "frame-sets/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def render_pool_on_device(torch, dev, n_sets, seed, chunk=256):
    """[n_sets, C, H, W] uint8 on the device: the synthetic stream of low-cost-mocap_b200/synth.py (same rig, same
    marker random walk and separation rule -- those run on the host, they are cheap), rendered with torch: uniform
    noise <= 40 under the threshold, every marker a Gaussian spot of peak 255.  Excluded from every timed region.
    Also returns the true 3D points [n_sets, M, 3]."""
    synth = importlib.import_module("low-cost-mocap_b200.synth")
    st = synth.MarkerStream(N_CAM, N_MARKERS, seed=seed)
    uv = np.empty((n_sets, N_CAM, N_MARKERS, 2))
    truth = np.empty((n_sets, N_MARKERS, 3))
    for b in range(n_sets):
        pts, uvs, _ = st.next_frame_set(render=False)
        uv[b], truth[b] = uvs, pts
    g = torch.Generator(device=dev)
    g.manual_seed(1234 + seed)
    frames = torch.empty((n_sets, N_CAM, HEIGHT, WIDTH), dtype=torch.uint8, device=dev)
    sig = torch.from_numpy(st.sigmas).to(dev)                                     # [C, M]
    r = 9
    off = torch.arange(2 * r + 2, device=dev)
    for b0 in range(0, n_sets, chunk):
        b1 = min(n_sets, b0 + chunk)
        fr = torch.randint(0, 41, (b1 - b0, N_CAM, HEIGHT, WIDTH), dtype=torch.uint8, device=dev, generator=g)
        u = torch.from_numpy(uv[b0:b1, :, :, 0]).to(dev)                          # [b, C, M]
        v = torch.from_numpy(uv[b0:b1, :, :, 1]).to(dev)
        xs = (torch.floor(u).long() - r)[..., None, None] + off[None, None, None, None, :]     # [b, C, M, 1, P]
        ys = (torch.floor(v).long() - r)[..., None, None] + off[None, None, None, :, None]     # [b, C, M, P, 1]
        d2 = (xs.double() - u[..., None, None]) ** 2 + (ys.double() - v[..., None, None]) ** 2
        val = torch.floor(255.0 * torch.exp(-d2 / (2.0 * sig[None, :, :, None, None] ** 2))).to(torch.uint8)
        ok = (xs >= 0) & (xs < WIDTH) & (ys >= 0) & (ys < HEIGHT)
        img = (torch.arange(b1 - b0, device=dev)[:, None] * N_CAM + torch.arange(N_CAM, device=dev)[None, :])[:, :, None, None, None]
        idx = (img * HEIGHT + ys.clamp(0, HEIGHT - 1)) * WIDTH + xs.clamp(0, WIDTH - 1)
        val = torch.where(ok, val, torch.zeros((), dtype=torch.uint8, device=dev))
        fr.view(-1).scatter_reduce_(0, idx.reshape(-1), val.reshape(-1), "amax")
        frames[b0:b1] = fr
    return frames, truth, st.poses, st.K


# the sources the S1-S3 kernels (the ones a roofline.traffic figure belongs to) are built from
STREAM_KERNEL_SOURCES = ("common.cuh", "geom.cuh", "blob_device.cuh", "blob_holes.cuh", "match_device.cuh", "fused_common.cuh", "fused_device.cuh",
                         "fused_kernel.cu", "blob_kernels.cu", "match_kernels.cu")


def csrc_hash():
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "low-cost-mocap_b200", "csrc")
    for f in STREAM_KERNEL_SOURCES:
        with open(os.path.join(d, f), "rb") as fh:
            h.update(f.encode()); h.update(fh.read())
    return h.hexdigest()[:16]


def committed_traffic(workload, kernel_prefix):
    """DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture of this workload
    (profiles/traffic_<workload>.json, written by tools/ncu_traffic.py from the raw ncu CSV next to it); null when no
    capture exists for the configuration or when the kernels have changed since it was taken."""
    path = os.path.join(ROOT, "profiles", f"traffic_{workload}.json")
    try:
        with open(path) as f:
            t = json.load(f)
    except Exception:
        return None, None
    if not t.get("kernel", "").startswith(kernel_prefix):
        return None, f"profiles/traffic_{workload}.json is for {t.get('kernel')}"
    if t.get("csrc_sha") != csrc_hash():
        return None, f"profiles/traffic_{workload}.json predates the current kernels (csrc {t.get('csrc_sha')} != {csrc_hash()})"
    return int(t["dram_bytes_read"]) + int(t["dram_bytes_write"]), f"profiles/traffic_{workload}.json <- {t.get('source')}"


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, out, ba_R=None, ba_t=None):
    """What the caller of the timed path receives for the last timed step, one <name>.npy per array: the track
    buffers of mocap_pipeline_dev (obj, err, n, flags, and track_xy when S4 runs) and the refined poses of that
    step's bundle adjustments.  Slots at and past n[b] hold no result and are written as zero, so that two builds
    can be compared array for array."""
    n = out["n"].cpu().numpy()
    unused = np.arange(out["obj"].shape[1])[None, :] >= n[:, None]                 # [B, R]
    arrays = {"obj": out["obj"].cpu().numpy().astype(np.float64), "err": out["err"].cpu().numpy().astype(np.float64),
              "n": n.astype(np.float32), "flags": out["flags"].cpu().numpy().astype(np.float32)}
    arrays["obj"][unused] = 0
    arrays["err"][unused] = 0
    if "track_xy" in out:
        arrays["track_xy"] = out["track_xy"].cpu().numpy().astype(np.float32)
        arrays["track_xy"][unused] = 0
    if ba_R is not None:
        arrays["ba_R"] = np.stack([r.cpu().numpy() for r in ba_R]).astype(np.float64)
        arrays["ba_t"] = np.stack([t.cpu().numpy() for t in ba_t]).astype(np.float64)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes (limit {DUMP_LIMIT_BYTES})")
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def run_gpu_arm(args):
    import torch
    import torch.distributed as dist
    pkg = importlib.import_module("low-cost-mocap_b200")
    sharding = importlib.import_module("low-cost-mocap_b200.sharding")
    synth = pkg.synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch N > 1 with: python -m torch.distributed.run --nproc-per-node N bench.py --gpus N ...")
    with_ba = WITH_BA and world == 1 and not args.no_ba            # BASELINE config 3 (N = 1); config 4 (N > 1) has no S4
    cpu_res = None
    if rank == 0 and not args.profile:
        # CPU baseline FIRST, before this process owns a CUDA context (forking worker processes out of such a
        # process is slow and unsafe): the oracle port on this box's host cores, bounded sample of the same workload
        # (frames from the same generator, rendered on the host)
        frames, truth, poses, K = make_pool()
        arm = CpuArm(frames, K, poses)
        sample = arm.sample_for(12.0, BATCH)
        t_cpu = arm.run(sample)
        arm.close()
        s4_cpu = None
        if with_ba:                                                 # one residual-vector evaluation of the reference's S4, bounded sample
            obs, ps, Kt, _ = synth.make_tracks(N_CAM, 256, seed=3, missing_frac=0.1)
            t0 = time.perf_counter()
            _W["port"].ba_residuals(_W["port"].poses_to_params(ps), obs)
            s4_cpu = (time.perf_counter() - t0) / 256
        cpu_res = (arm, sample, t_cpu, s4_cpu)
        del frames

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    # max_groups is a bound on the matcher's enumeration per root, not a buffer: 16 markers in 8 views reach tens of
    # thousands of candidate groups for some layouts (the reference enumerates them all, helpers.py:222-238)
    ctx = pkg.MocapContext(N_CAM, WIDTH, HEIGHT, device=local, max_roots=MAX_ROOTS, max_groups=MAX_GROUPS)

    # every rank owns BATCH frame-sets of the global stream of world*BATCH (round-robin ownership); each rank renders
    # its own pool of POOL distinct frame-sets (seed = rank), the batch cycles through it
    pool_dev, truth, poses, K = render_pool_on_device(torch, dev, POOL, seed=rank)
    ctx.set_cameras([K] * N_CAM, poses)
    if POOL == BATCH:
        batch = pool_dev
    else:
        batch = pool_dev[torch.arange(BATCH, device=dev) % POOL].contiguous()      # [BATCH, C, H, W] uint8
    first_sets = batch[:8].cpu().numpy()
    del pool_dev
    torch.cuda.empty_cache()
    # the matcher writes straight into the all-gather send buffer (one flat allocation); two buffers in turn,
    # so that on the multi-GPU path batch k's tracks travel while batch k+1 is being processed
    n_bufs = 2 if (world > 1 or with_ba) else 1
    track_bufs = [sharding.TrackBuffer(BATCH, MAX_ROOTS, dev) for _ in range(n_bufs)]
    outs = [tb.views for tb in track_bufs]
    pending = [None] * n_bufs
    bytes_per_step = batch.numel()
    step_no = [0]

    # S4 per BA_BATCH frame-sets (config 3): observations and poses live on the device; the solve starts from the
    # perturbed rig every time (SURVEY 8(d): rotvec sigma 0.03, t sigma 0.05) and runs on a side stream, so that it
    # overlaps the next step's pass over HBM
    if with_ba:
        n_sub = BATCH // BA_BATCH
        for o in outs:
            o["track_xy"] = torch.empty((BATCH, MAX_ROOTS, N_CAM, 2), dtype=torch.int32, device=dev)
        cap = BA_BATCH * MAX_ROOTS
        ba_obs = [{"obs": torch.empty((cap, N_CAM, 2), dtype=torch.float64, device=dev),
                   "mask": torch.empty((cap, N_CAM), dtype=torch.uint8, device=dev),
                   "n": torch.zeros((1,), dtype=torch.int32, device=dev)} for _ in range(n_bufs * n_sub)]
        start = synth.perturb_poses(poses, seed=10)
        R0 = torch.from_numpy(np.stack([np.asarray(p["R"]) for p in start])).to(dev).contiguous()
        t0_ = torch.from_numpy(np.stack([np.asarray(p["t"]).reshape(3) for p in start])).to(dev).contiguous()
        ba_R = [R0.clone() for _ in range(n_bufs * n_sub)]
        ba_t = [t0_.clone() for _ in range(n_bufs * n_sub)]
        ba_rep = [None] * (n_bufs * n_sub)
        # the n_sub solves of a step are independent.  k_ba_solve is one cooperative grid whose serial sections (dense
        # solves, tridiagonalisation) leave most of it waiting at barriers: several solves side by side, each on a share of
        # the SMs (own context = own workspace, own stream), overlap one solve's serial sections with another's tiles
        # (tools/ba_grid_probe.py: 4 solves of 18 800 points take 5.24 ms one after the other on 148 CTAs, 3.87 ms as
        # 2 x 74 CTAs, 5.18 ms for SIX as 3 x 49)
        ba_k = max(1, min(int(args.ba_streams), n_sub))
        if ba_k > 1:
            sms = torch.cuda.get_device_properties(dev).multi_processor_count
            ba_ctx = [pkg.MocapContext(N_CAM, WIDTH, HEIGHT, device=local, max_roots=MAX_ROOTS) for _ in range(ba_k)]
            for c_ in ba_ctx:
                c_.set_cameras([K] * N_CAM, poses)
                c_.set_ba_grid(max(1, sms // ba_k))
        else:
            ba_ctx = [ctx]
        sides = [torch.cuda.Stream(device=dev) for _ in range(ba_k)]
        tracks_ready = [torch.cuda.Event() for _ in range(n_bufs)]
        ba_done = [None] * n_bufs
        ba_ms_events = []

    def run_s4(k, timed):
        """tracks of buffer k -> n_sub bundle adjustments, enqueued on the side stream"""
        main = torch.cuda.current_stream(dev)
        tracks_ready[k].record(main)
        done = []
        for q, side in enumerate(sides):
            with torch.cuda.stream(side):
                side.wait_event(tracks_ready[k])
                for j in range(q, n_sub, len(sides)):
                    i = k * n_sub + j
                    sl = slice(j * BA_BATCH, (j + 1) * BA_BATCH)
                    tr = {key: outs[k][key][sl] for key in ("track_xy", "n", "err")}
                    ba_ctx[q].tracks_to_observations_dev(tr, max_err=BA_MAX_ERR, capacity=cap, out=ba_obs[i])
                    ba_R[i].copy_(R0); ba_t[i].copy_(t0_)
                    if timed:
                        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        ea.record(side)
                    ba_rep[i] = ba_ctx[q].bundle_adjust_dev(ba_obs[i]["obs"], ba_obs[i]["mask"], ba_R[i], ba_t[i], n_points=ba_obs[i]["n"], report=ba_rep[i])
                    if timed:
                        eb.record(side)
                        ba_ms_events.append((ea, eb))
                ev = torch.cuda.Event()
                ev.record(side)
                done.append(ev)
        ba_done[k] = done

    def step(timed=False):
        k = step_no[0] % n_bufs
        step_no[0] += 1
        if pending[k] is not None:
            pending[k].wait()                # this buffer's previous all-gather has read it
            pending[k] = None
        if with_ba and ba_done[k] is not None:
            for ev in ba_done[k]:
                torch.cuda.current_stream(dev).wait_event(ev)        # the S4 that read this buffer has finished
        ctx.pipeline(batch, out=outs[k])
        if with_ba:
            run_s4(k, timed)
        if world > 1:
            # ONE NCCL all-gather per batch, enqueued behind the pipeline kernel; consumers read views
            _, pending[k] = track_bufs[k].all_gather(async_op=True)

    def drain():
        for k, w in enumerate(pending):
            if w is not None:
                w.wait()
                pending[k] = None
        if with_ba:
            for evs in ba_done:
                for ev in evs or []:
                    torch.cuda.current_stream(dev).wait_event(ev)

    def sync_all():
        drain()
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    # clocks / throttle reasons are sampled from the warm-up through the end of the timed region
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(3, args.warmup)):
        step()
    sync_all()

    # ---- timed region: resident inputs -----------------------------------------------------
    ctx.enable_kernel_timing(True)
    ctx.detect_kernel_ms(reset=True)
    def all_launches():
        return ctx.launch_count() + (sum(c_.launch_count() for c_ in ba_ctx if c_ is not ctx) if with_ba else 0)
    launches0 = all_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    e0.record()
    for _ in range(args.steps):
        step(timed=True)
    drain()                                  # the stream now waits for the last all-gathers / bundle adjustments: inside the timed region
    e1.record()
    sync_all()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    launches = all_launches() - launches0
    if world > 1:
        launches += args.steps              # the NCCL all-gather kernel
    kern_ms, kern_n = ctx.detect_kernel_ms(reset=True)
    ctx.enable_kernel_timing(False)
    clocks = sampler.stop() if rank == 0 else None
    value = BATCH * world * args.steps / (ms_total * 1e-3)

    # ---- checks on every rank: no capacity overflow anywhere in the timed batch; the first frame-sets against the oracle
    out = outs[(step_no[0] - 1) % n_bufs]
    if args.dump_outputs and rank == 0:                  # before the e2e leg, which reuses the S4 buffers
        last = ((step_no[0] - 1) % n_bufs) * n_sub if with_ba else 0
        dump_outputs(args.dump_outputs, out, *((ba_R[last:last + n_sub], ba_t[last:last + n_sub]) if with_ba else ()))
    flags_set = int((out["flags"] != 0).sum().item())
    problems = []
    if flags_set:
        bits = 0
        for v in torch.unique(out["flags"]).tolist():
            bits |= int(v)
        problems.append(f"rank {rank}: {flags_set} frame-sets of the timed batch carry MOCAP_F_* overflow flags (bits {bits:#x})")
    _cpu_init(K, poses)
    port = _W["port"]
    ref = []
    for fs in first_sets:
        pts = [port.find_dot(np.repeat(img[:, :, None], 3, axis=2)) for img in fs]
        e, o, _ = port.match_and_triangulate(pts, poses)
        ref.append(np.asarray(o, dtype=np.float64).reshape(-1, 3))
    parity = compare_with_oracle(ref, out)
    if not parity["point_counts_equal"] or parity["max_abs_3d_difference"] > 1e-7:
        problems.append(f"rank {rank}: parity against the oracle failed: {parity}")
    s4 = None
    if with_ba:
        reps = [ctx.decode_ba_report(r) for r in ba_rep]
        Rn, tn = ba_R[-1].cpu().numpy(), ba_t[-1].cpu().numpy()
        sc = np.linalg.norm(np.stack([np.asarray(p["t"]).reshape(3) for p in poses])) / np.linalg.norm(tn)
        rot_err = max(float(np.abs(Rn[c] - np.asarray(poses[c]["R"])).max()) for c in range(N_CAM))
        t_err = max(float(np.abs(tn[c] * sc - np.asarray(poses[c]["t"]).reshape(3)).max()) for c in range(N_CAM))
        ba_ms = [a.elapsed_time(b) for a, b in ba_ms_events]
        s4 = {"solves_per_step": n_sub, "frame_sets_per_solve": BA_BATCH, "points_per_solve": int(np.mean([r["n_residuals"] for r in reps])),
              "max_err_px2": BA_MAX_ERR, "ms_per_solve": float(np.median(ba_ms)), "ms_per_solve_max": float(np.max(ba_ms)),
              "launches_per_solve": 3, "status": sorted(set(r["status"] for r in reps)),
              "cost_initial": float(np.mean([r["cost_initial"] for r in reps])), "cost_final": float(np.mean([r["cost_final"] for r in reps])),
              "optimality": float(np.max([r["optimality"] for r in reps])),
              "prefit_iterations": float(np.mean([r["prefit_iterations"] for r in reps])), "n_fev": float(np.mean([r["n_fev"] for r in reps])),
              "phase_ms": [float(v) for v in np.mean([r["phase_ms"] for r in reps], axis=0)],
              "pose_error_vs_true_rig": {"rotation_max_abs": rot_err, "translation_max_abs_after_scale": t_err},
              "overlap": "side stream; the solves of step k run while step k+1 streams",
              "side_streams": ba_k, "ctas_per_solve": torch.cuda.get_device_properties(dev).multi_processor_count // ba_k}
        if any(r["status"] not in (1, 2, 3, 4) for r in reps) or rot_err > 2e-2 or t_err > 5e-2:
            problems.append(f"rank {rank}: S4 did not converge to the true rig: {s4}")
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, problems)
        problems = [p for lst in gathered for p in lst]
    if problems:
        if rank == 0:
            print("bench.py: RESULT CHECK FAILED\n  " + "\n  ".join(problems), file=sys.stderr, flush=True)
        raise SystemExit(3)

    if args.profile:
        if rank == 0:
            print(json.dumps({"profile_only": True, "ms_per_step": ms_total / args.steps, "kernel_ms": kern_ms, "s4": s4}), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- e2e: host buffers ------------------------------------------------------------------------
    host_frames = torch.empty(batch.shape, dtype=torch.uint8).pin_memory()
    host_frames.copy_(batch)
    host_out = {"obj": torch.empty((BATCH, MAX_ROOTS, 3), dtype=torch.float64).pin_memory(),
                "err": torch.empty((BATCH, MAX_ROOTS), dtype=torch.float64).pin_memory(),
                "n": torch.empty((BATCH,), dtype=torch.int32).pin_memory(),
                "flags": torch.empty((BATCH,), dtype=torch.int32).pin_memory()}
    d2h = sum(v.numel() * v.element_size() for v in host_out.values())
    e2e_steps = max(1, min(args.steps, 3))
    if not with_ba:
        def e2e_step():                                              # the C-ABI host entry point: returns with results in host memory
            ctx.pipeline_host(host_frames, out=host_out)
        e2e_api = "mocap_pipeline_host (H2D in chunks overlapped with compute, D2H of the tracks)"
    else:
        # config 3 through host buffers: frames travel H2D in chunks (copy stream, two device buffers), every chunk
        # goes through mocap_pipeline_tracks_dev, every BA_BATCH frame-sets through S4, tracks and poses travel D2H
        chunk = BA_BATCH
        stage = [torch.empty((chunk,) + tuple(batch.shape[1:]), dtype=torch.uint8, device=dev) for _ in range(2)]
        copy_s = torch.cuda.Stream(device=dev)
        host_R = torch.empty((BATCH // chunk, N_CAM, 3, 3), dtype=torch.float64).pin_memory()
        host_t = torch.empty((BATCH // chunk, N_CAM, 3), dtype=torch.float64).pin_memory()
        d2h += host_R.numel() * 8 + host_t.numel() * 8
        dev_out = ctx.alloc_tracks(BATCH, dev)
        dev_out["track_xy"] = outs[0]["track_xy"]

        def e2e_step():
            main = torch.cuda.current_stream(dev)
            copied = [None, None]
            used = [None, None]
            for ci in range(BATCH // chunk):
                bi = ci % 2
                with torch.cuda.stream(copy_s):
                    if used[bi] is not None:
                        copy_s.wait_event(used[bi])
                    stage[bi].copy_(host_frames[ci * chunk:(ci + 1) * chunk], non_blocking=True)
                    ev = torch.cuda.Event(); ev.record(copy_s); copied[bi] = ev
                main.wait_event(copied[bi])
                sl = slice(ci * chunk, (ci + 1) * chunk)
                tr = {key: dev_out[key][sl] for key in ("obj", "err", "n", "flags", "track_xy")}
                ctx.pipeline(stage[bi], out=tr)
                ev = torch.cuda.Event(); ev.record(main); used[bi] = ev
                ctx.tracks_to_observations_dev(tr, max_err=BA_MAX_ERR, capacity=cap, out=ba_obs[0])
                ba_R[0].copy_(R0); ba_t[0].copy_(t0_)
                ctx.bundle_adjust_dev(ba_obs[0]["obs"], ba_obs[0]["mask"], ba_R[0], ba_t[0], n_points=ba_obs[0]["n"], report=ba_rep[0])
                host_R[ci].copy_(ba_R[0], non_blocking=True); host_t[ci].copy_(ba_t[0], non_blocking=True)
            for key in ("obj", "err", "n", "flags"):
                host_out[key].copy_(dev_out[key], non_blocking=True)
            torch.cuda.synchronize(dev)
        e2e_api = ("MocapContext.pipeline(want_tracks) + tracks_to_observations_dev + bundle_adjust_dev per 1000 frame-sets, frames H2D in "
                   "chunks from pinned memory on a copy stream, tracks and refined poses D2H")
    e2e_step()                                                      # warm-up (allocates staging)
    sync_all()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize(dev)
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    e2e_value = BATCH * world * e2e_steps / float(dt.item())
    same = bool((host_out["n"].to(dev) == out["n"]).all().item())

    split = os.environ.get("MOCAP_PIPELINE") == "split" or (os.environ.get("MOCAP_PIPELINE") is None and N_CAM * N_MARKERS > 48)
    kernel_name = ("k_threshold_segments_c1 (stream kernel of the three-kernel pipeline)" if split
                   else "k_pipeline_fused (threshold + blob reduce + match/DLT in one pass)")
    traffic, traffic_src = committed_traffic(args.workload, "k_threshold_segments" if split else "k_pipeline_fused")
    if rank == 0:
        peak, peak_src = measured_peak()
        # algorithmic bytes: C*W*H bytes per frame-set, read exactly once; per launch of the timed kernel:
        # step bytes * steps / launches
        alg_bytes = bytes_per_step * args.steps / kern_n if kern_n else None
        achieved = alg_bytes / (kern_ms * 1e-3) / 1e9 if kern_ms > 0 else None
        arm, sample, t_cpu, s4_cpu = cpu_res
        stages = "S1 blob + S2 epipolar + S3 DLT" + (f" + S4 bundle adjustment per {BA_BATCH} frame-sets" if with_ba else "")
        config_no = "2" if N_CAM == 4 else ("3" if with_ba else ("4" if world > 1 else "3 without S4"))
        cpu_rep = arm.report(sample / t_cpu, f"{sample} frame-sets of the same workload (S1-S3), one worker process per core")
        if with_ba:
            n_par = 1 + 7 * (N_CAM - 1)
            cpu_rep["s4_note"] = ("S1-S3 only: the reference's S4 on one 1000-frame batch cannot be timed in a bounded sample -- one residual-vector "
                                  f"evaluation costs {s4_cpu * 1e3:.2f} ms per point on one core (measured on 256 points), i.e. "
                                  f"{s4_cpu * s4['points_per_solve']:.1f} s per evaluation and {s4_cpu * s4['points_per_solve'] * (n_par + 1):.0f} s per "
                                  f"finite-difference Jacobian ({n_par + 1} evaluations) of such a batch")
        line = {
            "metric": f"mocap frame-sets/s ({N_CAM}-cam 640x480 synthetic, {'blob+epipolar+DLT' + ('+bundle adjustment' if with_ba else '')})",
            "value": value, "unit": "frame-sets/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8 pixels -> int64 moments -> f64 geometry", "data": "synthetic",
            "config": {"workload": (f"BASELINE config {config_no}: {N_CAM} cameras, {N_MARKERS} markers, {BATCH} frame-sets "
                                    f"of 640x480 uint8 per GPU per step, {stages}"),
                       "cameras": N_CAM, "markers": N_MARKERS, "frame_sets_per_step_per_gpu": BATCH,
                       "distinct_frame_sets": POOL, "limits": {"max_roots": MAX_ROOTS, "max_groups": MAX_GROUPS}, "l2": f"inputs ({BATCH * N_CAM * 307200 / 1e9:.1f} GB per step) larger than L2, no flush needed",
                       "parallelism": f"frame-set round-robin over {world} GPU(s), one NCCL all-gather of tracks per batch" if world > 1 else "single GPU"},
            "e2e": {"value": e2e_value, "unit": "frame-sets/s", "h2d_bytes_per_step": int(bytes_per_step),
                    "d2h_bytes_per_step": int(d2h), "steps": e2e_steps, "matches_resident_path": same, "api": e2e_api,
                    "bound": "PCIe: the frames cross the link once (55 GB/s measured); only more GPUs (one link each) move this figure"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": kernel_name, "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": (achieved / peak) if achieved else None, "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": int(alg_bytes) if alg_bytes else None,
                         "avg_launch_ms": kern_ms, "launches_timed": kern_n,
                         "whole_step_frac": (bytes_per_step * args.steps / (ms_total * 1e-3) / 1e9) / peak},
            "cpu_baseline": cpu_rep,
            "parity_vs_oracle": parity, "overflow_flags_in_timed_batch": flags_set,
            "clocks": clocks,
        }
        if s4:
            line["s4"] = s4
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c4m4", choices=["c4m4", "c8m16"],
                    help="c4m4 (default): BASELINE config 2, the configuration the metric is quoted on; c8m16: 8 cameras, 16 markers, 4000 "
                         "frame-sets per GPU per step -- at N = 1 BASELINE config 3 (S1-S3 plus one S4 per 1000 frame-sets), at N > 1 "
                         "config 4 (S1-S3, round-robin shards, one NCCL all-gather of tracks per batch)")
    ap.add_argument("--ba-streams", type=int, default=4,
                    help="c8m16 with S4: the solves of a step side by side on this many contexts / streams, each on a share of the SMs")
    ap.add_argument("--no-ba", action="store_true", help="c8m16 at N = 1 without S4 (the S1-S3 figure of the config-3 shape)")
    ap.add_argument("--profile", action="store_true",
                    help="resident steps only (no e2e, no CPU baseline): for runs under ncu; prints no bench line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0) as DIR/<name>.npy, float32 / float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the b200 implementation")
    if args.workload == "c8m16":
        global N_CAM, N_MARKERS, BATCH, POOL, MAX_ROOTS, MAX_GROUPS, WITH_BA
        N_CAM, N_MARKERS, BATCH, POOL, MAX_ROOTS, MAX_GROUPS, WITH_BA = 8, 16, 4000, 4000, 64, 1 << 16, True
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
