#!/usr/bin/env python
"""bench.py — stereo-pairs/sec of the B200-native stereo point+line front-end (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run, one rank per GPU)
  python bench.py --impl reference ...                     (the CPU path timed on the host cores; rank 0 only)
  python bench.py ... --dump-outputs DIR                   (also write what the last timed step returned, DIR/<name>.npy)

One "step" = one pass of the hot path (ORB + LSD/LBD extraction of both images, L/R stereo association,
frame-to-frame tracking, robust Gauss-Newton pose) over one batch of B consecutive synthetic stereo pairs of a
KITTI-00-shape stream (BASELINE.json configs[1]).  `value` = pairs/s with the batch already resident in HBM
(device time, CUDA events on the library's stream, max over ranks); `e2e` = the same metric through the
reference-facing C-ABI call plf_process_batch with pinned HOST buffers (H2D of the images and D2H of the per-frame
results inside the timed region).  Rank 0 prints ONE JSON line.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "pl-slam_b200"))

METRIC = "stereo_pairs_per_sec"
UNIT = "pairs/s"
KITTI = dict(width=1242, height=375, fx=718.856, fy=718.856, cx=607.1928, cy=185.2157, b=0.537165719)  # kitti00-02.yaml:2-10
EUROC = dict(width=752, height=480, fx=458.654, fy=457.296, cx=367.215, cy=248.375, b=0.110077842)     # euroc_params.yaml:2,8

# BASELINE.json configs: [1] = kitti (the headline: what `metric` is quoted on and what the driver runs), [2] = euroc,
# [4] = lowtex.  `n_kp / m_lines / lbar` only feed the SURVEY 8(d) byte formula when the measured counts are unknown.
CONFIGS = {
    "kitti": dict(cam=KITTI, prm=dict(orb_nfeatures=1500, lsd_nfeatures=200),
                  workload="kitti00_shape_synthetic_stream_1242x375_orb1500_lsd200_tracking", batch=1536, lbar=90,
                  world=lambda seed: dict(seed=7), stream=lambda seed: dict(seed=42 + seed)),
    "euroc": dict(cam=EUROC, prm=dict(orb_nfeatures=1200, lsd_nfeatures=300, max_iters=5, max_iters_ref=10),
                  workload="euroc_mh_shape_synthetic_stream_752x480_orb1200_lsd300_full_frontend_pose_refine", batch=1536, lbar=80,
                  world=lambda seed: dict(seed=8, length=40.0, n_quads=220, n_segs=120, half_width=5.0, half_height=3.0),
                  stream=lambda seed: dict(seed=43 + seed, step=0.08, yaw_deg=0.8)),
    "lowtex": dict(cam=KITTI, prm=dict(orb_nfeatures=150, lsd_nfeatures=0),
                   workload="low_texture_lines_dominant_synthetic_stream_1242x375_orb150_lsd_all", batch=1536, lbar=120,
                   world=None, stream=lambda seed: dict(seed=17 + seed, noise=2)),
}
# Sequences of different ranks (BASELINE config 4: one independent sequence per GPU) are independent TRAJECTORIES (stream seed +
# rank: own motion, own image noise) through the SAME synthetic world.  Weak scaling wants equal work per GPU: with one world
# per rank (the first round-2 measurement, profiles/r02_scale_n8_heterogeneous.json) the scene content made the summed kernel
# time of a step range from 124 to 158 ms across the 8 ranks (region growing 45 .. 69 ms), and because the ranks meet at the
# per-step pose all-gather the whole job ran at the pace of the heaviest sequence - 0.78 "efficiency" that measured the
# scenes, not the system.
CFG = CONFIGS["kitti"]
CAM, PRM, WORKLOAD = CFG["cam"], CFG["prm"], CFG["workload"]


def select_config(name):
    global CFG, CAM, PRM, WORKLOAD
    CFG = CONFIGS[name]
    CAM, PRM, WORKLOAD = CFG["cam"], CFG["prm"], CFG["workload"]


def algorithmic_bytes_per_pair(w, h, s=1.2, n_kp=1500, m_lines=200, lbar=90):
    """SURVEY.md §8(d): BYTES_PER_PAIR = 2*(ORB + LSD + LBD) + MATCH."""
    A0 = w * h
    A = [round(w / 1.2 ** k) * round(h / 1.2 ** k) for k in range(4)]
    S = sum(A)
    Ns = round(w * s) * round(h * s)
    orb = A0 + 2 * sum(A[1:]) + 2 * S + 56 * n_kp
    lsd = A0 + 2 * Ns + 8 * Ns + 8 * Ns + 6 * Ns + 16 * m_lines
    lbd = A0 + 4 * A0 + min(4 * A0, 63 * lbar * 4 * m_lines) + 32 * m_lines
    match = 2 * 32 * n_kp + 4 * n_kp + 2 * 32 * m_lines + 4 * m_lines
    return dict(orb=orb, lsd=lsd, lbd=lbd, match=match, pair=2 * (orb + lsd + lbd) + match, Ns=Ns, A0=A0, S=S, A=A,
                chunks=(round(h * s) + 14) // 16, lbar=lbar)


# Bytes per IMAGE of each kernel, two ways:
#   survey = the term of SURVEY.md 8(d)'s per-image formula this kernel implements (what `frac_hbm` is judged on);
#   design = what this implementation's data layout moves by construction (extra maps / records it reads or writes).
# The measured DRAM bytes (ncu --set full, profiles/ncu_traffic_per_image.json) are reported next to both.
def kernel_bytes(name, ab, n_kp, m_lines):
    A0, Ns, A, S = ab["A0"], ab["Ns"], ab["A"], ab["S"]
    ch = 4 * 1024 * ab["chunks"]
    t = {                        # (survey, design)
        "orb.k_resize_exact": (sum(A[:3]) + sum(A[1:]),) * 2,        # read level k-1, write level k
        "orb.k_fast_nms": (S, S + 8 * n_kp),                          # read the pyramid once (+ candidates out)
        "orb.k_select_sort": (24 * n_kp, 8 * n_kp + 28 * n_kp),
        "orb.k_ic_angle": (961 * n_kp,) * 2,
        "orb.k_orb_blur7": (2 * S,) * 2,                              # read + write every level
        "orb.k_rbrief": (32 * n_kp, 512 * n_kp + 32 * n_kp),         # survey: descriptors out; design: + the 37x37 patches read
        "lsd.k_blur_q8": (2 * A0,) * 2,
        "lsd.k_resize_exact": (A0 + Ns,) * 2,
        # d = defined pixels (gradient above the threshold), ~ Ns / 8 on the KITTI-shape stream
        "lsd.k_lsd_grad": (Ns + 8 * Ns, Ns + (16 + 8) * (Ns // 8)),   # survey: read u8, write f32 mag + angle; design: 16 B record + (index, |g|^2) list entry, defined pixels only
        "lsd.k_lsd_rowhist": (4 * Ns, 6 * (Ns // 8) + ch),            # survey: half of the 8 Ns "write + read bin-sort index"; design: read |g|^2, write the u16 bin, chunk counters
        "lsd.k_lsd_binscan": (2 * ch,) * 2,
        "lsd.k_lsd_scatter": (4 * Ns, 6 * (Ns // 8) + ch + 4 * (Ns // 8)),   # design: read (index, bin) + bases, write the order
        "lsd.k_lsd_grow": (6 * Ns, 6 * Ns),                           # SURVEY 8(d): read angle + r/w used mask
        "lsd.k_lsd_rects": (3 * 8 * Ns // 4, 2 * (4 + 4) * (Ns // 8) + 4 * (Ns // 8)),   # design: 2 passes of (point, record li) + 1 of the point list
        "lsd.k_keylines": (16 * m_lines, 16 * 1200 + 68 * 1200),
        "lbd.k_blur5_sobel": (A0 + 4 * A0,) * 2,
        "lbd.k_lbd": (63 * ab["lbar"] * 4 * m_lines + 32 * m_lines,) * 2,
    }
    return t.get(name, (None, None))


def render_pool(cam, n, seed):
    from plslam_b200 import synth      # input generator (not the oracle)
    world = synth.corridor_world() if CFG["world"] is None else synth.World(**CFG["world"](seed))
    return [(L, R) for (L, R, _) in synth.stream(cam, n, world=world, **CFG["stream"](seed))]


def fill_batch(pool, B, dstL, dstR):
    """Ping-pong over the rendered frames so that consecutive pairs are always neighbours on the trajectory."""
    n = len(pool)
    period = list(range(n)) + list(range(n - 2, 0, -1)) if n > 2 else list(range(n))
    for k in range(B):
        L, R = pool[period[k % len(period)]]
        dstL[k] = L
        dstR[k] = R


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except ValueError:
                continue
            for nm, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


DUMP_FRAMES = 16            # frames of the last batch whose features --dump-outputs writes (fixed, seeded sample)
DUMP_MAX_BYTES = 64 << 20


def collect_outputs(fe, results, poses, B, all_poses=None):
    """What this rank's caller of the timed path receives for its last step, as float32 / float64 arrays: every field
    of the per-frame results (plf_batch_download), the device-resident poses (plf_batch_device_poses; with more than
    one rank also the all-gathered poses of every rank, rank-major, as device_poses_all_ranks) and the stereo features
    (plf_get_frame) of DUMP_FRAMES frames drawn with a fixed seed, concatenated in frame order with their counts.
    Call before anything else runs a batch: plf_get_frame reads the last one."""
    out = {f"result_{f}": results[f].astype(np.float64) for f in results.dtype.names}
    out["device_poses"] = poses.cpu().numpy().astype(np.float64)
    if all_poses is not None:
        out["device_poses_all_ranks"] = all_poses.cpu().numpy().astype(np.float64)
    frames = np.sort(np.random.default_rng(0).choice(B, size=min(DUMP_FRAMES, B), replace=False))
    feats = [fe.get_frame(int(k)) for k in frames]
    out["features_frame"] = frames.astype(np.float64)
    out["features_n_pt"] = np.array([len(f["pt_pl"]) for f in feats], np.float64)
    out["features_n_ls"] = np.array([len(f["ls_spl"]) for f in feats], np.float64)
    for name in feats[0]:
        a = np.concatenate([f[name] for f in feats])
        out[f"features_{name}"] = a.astype(np.float32 if a.dtype in (np.uint8, np.float32) else np.float64)
    return out


def write_outputs(d, arrays):
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {total / 2**20:.1f} MB (limit {DUMP_MAX_BYTES >> 20} MB)")
    d = Path(d)
    d.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(d / f"{name}.npy", a)
    print(f"bench.py: wrote {len(arrays)} arrays ({total / 2**20:.1f} MB) to {d}", file=sys.stderr)


def cpu_baseline_run(n_frames, threads=None):
    """(pairs/s, worker processes, seconds) of the CPU path on n_frames rendered pairs; the worker pool is started
    before the clock and one untimed pass warms it up."""
    from oracle import baseline
    pool = render_pool(CAM, n_frames, seed=0)
    with baseline.Workers(CAM, pool, PRM, threads=threads) as w:
        w.run(min(len(pool), w.threads))
        t0 = time.perf_counter()
        w.run()
        dt = time.perf_counter() - t0
        return len(pool) / dt, w.threads, dt


def run_reference(args, rank):
    """--impl reference: the CPU path (cv2 ORB / LSD / BFMatcher + C restatements of LBD / GN) on the host cores."""
    if rank != 0:
        return
    from oracle import baseline
    cores = baseline.effective_cores()     # affinity mask capped by the cgroup CPU quota, if any
    n = max(8, min(4 * cores, 512))        # bounded sample per step: a few waves over all cores
    pool = render_pool(CAM, min(n, 24), seed=0)
    pairs = [pool[i % len(pool)] for i in range(n)]
    with baseline.Workers(CAM, pairs, PRM) as w:     # worker processes started once, outside the timed region
        for _ in range(max(args.warmup, 1)):
            w.run(max(cores, 8))
        t0 = time.perf_counter()
        for _ in range(args.steps):
            w.run()
        dt = time.perf_counter() - t0
        print("bench.py reference arm: last step %.2f s extraction on %d processes + %.2f s sequential tracking/pose"
              % (w.last_split[0], w.threads, w.last_split[1]), file=sys.stderr)
    v = n * args.steps / dt
    line = dict(metric=METRIC, value=v, unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=1e3 * dt / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="u8/f32/f64",
                data="synthetic", impl="reference",
                config=dict(workload=WORKLOAD, bench_config=args.config, pairs_per_step=n, **PRM),
                cpu_baseline=dict(value=v, unit=UNIT, cores=w.threads, kind="port", host_cpus=os.cpu_count(),
                                  sample=f"{n} pairs/step x {args.steps} steps: cv2 4.13 ORB+LSD+BFMatcher + C LBD/GN, {w.threads} worker processes"
                                         f" ({os.cpu_count()} CPUs visible); last step {w.last_split[0]:.2f} s extraction + {w.last_split[1]:.2f} s sequential tracking/pose"),
                e2e=dict(value=v, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    emit(line)


_REAL_STDOUT = None


def emit(line: dict):
    """The one JSON line goes to the process's original stdout; everything else (NCCL banners, library chatter) was
    redirected to stderr at start-up."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, data)
    else:
        sys.stdout.write(data.decode()); sys.stdout.flush()


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)           # stdout of this process (and of any library writing to fd 1) -> stderr
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=os.environ.get("PLF_BENCH_CONFIG", "kitti"), choices=sorted(CONFIGS),
                    help="BASELINE.json workload: kitti = configs[1] (the headline, default), euroc = configs[2], lowtex = configs[4]")
    ap.add_argument("--batch", type=int, default=int(os.environ.get("PLF_BENCH_BATCH", "0")),
                    help="stereo pairs per step per GPU (default: the config's; reduced automatically if it would not fit)")
    ap.add_argument("--pool", type=int, default=24, help="distinct rendered frames (ping-ponged to fill a batch)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--overlap-profile", action="store_true", help="also report per-kernel times measured with two batches in flight (overlapped)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (per-frame results, device poses, the features "
                         "of a fixed sample of frames) as DIR/<name>.npy; the inputs depend only on the arguments")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    select_config(args.config)
    rank = int(os.environ.get("RANK", "0")); local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if args.warmup < 3:
        args.warmup = 3

    import torch
    import plslam_b200 as plf
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    w, h = CAM["width"], CAM["height"]
    B = args.batch or CFG["batch"]
    per_pair = 0.062e9 * (w * h) / (1242 * 375)       # HBM per pair (LSD maps once, extraction outputs for 2 batch parities)
    free_b, _tot = torch.cuda.mem_get_info()
    fit = int((free_b * 0.85 - 4e9) / per_pair)
    if B > fit:
        print(f"bench.py: batch {B} -> {max(fit, 8)} (free HBM {free_b / 1e9:.0f} GB)", file=sys.stderr)
        B = max(fit, 8)
    lim = plf.default_limits()
    lim.max_batch = B; lim.max_keypoints = 4096; lim.max_segments = 8192; lim.max_lines = 1024
    fe = plf.Frontend(camera=CAM, limits=lim, device=local_rank, **PRM)
    pool = render_pool(CAM, args.pool, seed=rank)            # rank r tracks its own sequence (BASELINE config 4)
    hostL = torch.empty((B, h, w), dtype=torch.uint8, pin_memory=True)
    hostR = torch.empty((B, h, w), dtype=torch.uint8, pin_memory=True)
    fill_batch(pool, B, hostL.numpy(), hostR.numpy())
    ext = torch.cuda.ExternalStream(fe.stream, device=torch.device("cuda", local_rank))
    side = torch.cuda.Stream()                                # the pose exchange runs here, beside the library's streams
    pose_buf = torch.zeros((B, 16), dtype=torch.float64, device="cuda")
    gather_buf = torch.zeros((world * B, 16), dtype=torch.float64, device="cuda") if world > 1 else None

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def gather_poses():
        """The path's only exchange (SURVEY 8e): the B poses of the oldest batch in flight go device-to-device into
        pose_buf behind that batch's match phase (plf_batch_device_poses) and, with more than one rank, through ONE
        NCCL all-gather - no host round trip.  Call before the batch is downloaded."""
        with torch.cuda.stream(side):
            fe.batch_device_poses(B, pose_buf.data_ptr(), side.cuda_stream)
            if dist is not None:
                dist.all_gather_into_tensor(gather_buf, pose_buf)

    # ---- warm-up through the public call (also builds every lazily allocated buffer)
    last = None
    for _ in range(args.warmup):
        fe.batch_upload_raw(B, hostL.data_ptr(), hostR.data_ptr())
        fe.batch_run(B)
        gather_poses()
        last = fe.batch_download(B)
    barrier()
    free_after, _tot = torch.cuda.mem_get_info(local_rank)
    print(f"bench.py: HBM in use after warm-up {(_tot - free_after) / 1e9:.1f} GB ({(_tot - free_after) / 1e6 / B:.1f} MB per pair)", file=sys.stderr)
    stats = {k: float(np.mean([r[k] for r in last[1:]])) for k in ("n_kp_l", "n_lines_l", "n_stereo_pt", "n_stereo_ls", "n_matched_pt", "n_matched_ls", "n_inliers_pt", "n_inliers_ls")}
    tracked = float(np.mean([r["status"] == 0 for r in last[1:]]))
    # the gathered poses are the ones the host sees (checked once, outside the timed regions)
    side.synchronize()
    dt_host = np.stack([r["DT"].reshape(16) for r in last])
    pose_ok = bool(np.array_equal(pose_buf.cpu().numpy(), dt_host))
    if dist is not None:
        pose_ok = pose_ok and bool(np.array_equal(gather_buf[rank * B:(rank + 1) * B].cpu().numpy(), dt_host))
    if not pose_ok:
        raise SystemExit("bench.py: device-resident pose gather does not match the downloaded results")

    # ---- `value`: batch resident in HBM, K x (plf_batch_run + device-resident pose exchange), device time
    fe.batch_upload_raw(B, hostL.data_ptr(), hostR.data_ptr())
    fe.sync()
    sampler = None
    if rank == 0:                               # one nvidia-smi sampler per job, not per rank (they cost host CPU)
        sampler = ClockSampler(local_rank); sampler.start()
    l0 = fe.launches
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_host0 = time.perf_counter()
    with torch.cuda.stream(ext):
        e0.record(ext)
        depth = min(3, args.steps)             # up to three batches in flight: extraction of batch i+2 / i+1 overlaps the
        for _ in range(depth):                 # latency-bound LSD region growing and the match phase of batch i
            fe.batch_run(B)
        for _ in range(args.steps - depth):
            gather_poses()
            fe.batch_download_array(B)
            fe.batch_run(B)
        for _ in range(depth):
            gather_poses()
            last_res = fe.batch_download_array(B)
        ext.wait_stream(side)                   # the last pose exchange is inside the timed region
        e1.record(ext)
    barrier()
    host_ms = (time.perf_counter() - t_host0) * 1e3
    dev_ms = e0.elapsed_time(e1)
    launches = fe.launches - l0
    clocks = sampler.stop() if sampler else None
    try:   # device-clock timeline of the last two (overlapping) batches: [batch][E,G,M][start,end] in ms
        timeline = [[[round(float(x), 2) for x in ph] for ph in b] for b in fe.debug_timeline()]
    except Exception:
        timeline = None

    dumped = collect_outputs(fe, last_res, pose_buf, B, gather_buf) if args.dump_outputs and rank == 0 else None

    # ---- `e2e`: pinned host buffers -> plf_batch_upload + run + pose exchange + download, K steps
    # (software-pipelined like a streaming caller: the H2D of batch i+1 is issued while batch i runs; every step still
    #  uploads its own 2*B images and downloads its own B results inside the timed region; up to 3 batches in flight)
    barrier()
    t0 = time.perf_counter()
    issued = done = 0
    while done < args.steps:
        while issued < args.steps and issued - done < 3:
            fe.batch_upload_raw(B, hostL.data_ptr(), hostR.data_ptr())
            fe.batch_run(B)
            issued += 1
        gather_poses()
        res = fe.batch_download_array(B)
        done += 1
    barrier()
    e2e_s = time.perf_counter() - t0

    # ---- per-kernel device times (one extra profiled pass, outside both timed regions)
    fe.sync()
    fe.profile_enable(True)
    fe.batch_run(B)
    stages = [(n, ms) for n, ms in fe.profile_read() if n != "start"]
    fe.batch_download_array(B)
    fe.profile_enable(False)

    overlapped = None
    if args.overlap_profile:   # same marks with the E/G/M pipeline left on: two batches in flight, second batch reported
        fe.profile_enable(2)
        fe.batch_run(B); fe.batch_run(B)
        marks = fe.profile_read()
        fe.batch_download_array(B); fe.batch_download_array(B)
        fe.profile_enable(False)
        overlapped = [(n, round(ms, 3)) for n, ms in marks]

    mine = dict(rank=rank, dev_ms_per_step=round(dev_ms / args.steps, 3), host_ms_per_step=round(host_ms / args.steps, 3),
                e2e_ms_per_step=round(e2e_s * 1e3 / args.steps, 3), timeline=timeline,
                serial_kernel_ms=round(sum(ms for _, ms in stages), 3),
                grow_ms=next((round(ms, 3) for n, ms in stages if "grow" in n), None))
    per_rank = [mine]
    t = torch.tensor([dev_ms, e2e_s * 1e3], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        per_rank = [None] * world
        dist.all_gather_object(per_rank, mine)
    dev_ms, e2e_ms = float(t[0]), float(t[1])
    if rank == 0:
        total_pairs = world * B * args.steps
        value = total_pairs / (dev_ms * 1e-3)
        e2e_v = total_pairs / (e2e_ms * 1e-3)
        peak, peak_src = measured_peaks()
        ab = algorithmic_bytes_per_pair(w, h, 1.2, int(round(stats["n_kp_l"])), int(round(stats["n_lines_l"])), CFG["lbar"])
        step_ms = sum(ms for _, ms in stages)
        tp = ROOT / "profiles" / "ncu_traffic_per_image.json"      # dram bytes per image from the committed ncu --set full capture
        ncu_bytes = {}
        if tp.exists() and args.config == "kitti":
            try:
                ncu_bytes = json.loads(tp.read_text())
            except Exception:
                ncu_bytes = {}
        ktab = []
        for name, ms in stages:
            sb, db = kernel_bytes(name, ab, stats["n_kp_l"], stats["n_lines_l"])
            gbs = (sb * 2 * B / (ms * 1e-3) / 1e9) if (sb and ms > 0) else None
            dram = ncu_bytes.get(name)
            ktab.append(dict(kernel=name, ms=round(ms, 4), share=round(ms / step_ms, 4) if step_ms else None,
                             survey_bytes_per_image=int(sb) if sb else None, algo_gbs=round(gbs, 1) if gbs else None,
                             frac_hbm=round(gbs / peak, 4) if gbs else None,
                             design_bytes_per_image=int(db) if db else None,
                             dram_bytes_per_image=int(dram) if dram else None,
                             dram_gbs=round(dram * 2 * B / (ms * 1e-3) / 1e9, 1) if (dram and ms > 0) else None))
        dom = max(ktab, key=lambda r: r["ms"]) if ktab else None
        roof = None
        if dom and dom["algo_gbs"]:
            traffic = dom["dram_bytes_per_image"] * 2 * B if dom["dram_bytes_per_image"] else None
            roof = dict(kernel=dom["kernel"], bound="hbm", achieved=dom["algo_gbs"], peak=peak, unit="GB/s",
                        frac=round(dom["algo_gbs"] / peak, 5), traffic=traffic, peak_source=peak_src,
                        bytes="SURVEY 8(d) term of this kernel x 2B images per launch / its launch time (CUDA events, serialised pass)",
                        traffic_source=(ncu_bytes.get("_source") if traffic else None),
                        note=("share of step %.0f%%; region growing is a sequential greedy partition per image: latency-bound, "
                              "reported against HBM for completeness" % (100 * dom["share"])) if "grow" in dom["kernel"] else None)
        # PER-GPU figures: `value` is the whole-job aggregate over `world` ranks, the peak is one GPU's
        whole = dict(algorithmic_bytes_per_pair=ab["pair"], per="gpu", achieved_gbs=round(ab["pair"] * value / world / 1e9, 1),
                     frac_hbm=round(ab["pair"] * value / world / 1e9 / peak, 4))
        line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=dev_ms / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
                    dtype="u8/f32/f64", data="synthetic",
                    config=dict(workload=WORKLOAD, bench_config=args.config, pairs_per_step_per_gpu=B, image=[w, h], **PRM,
                                rendered_frames=args.pool,
                                l2="per-step working set %.0f MB (images + pyramids + LSD maps) >> 126 MB L2" % (B * 36.0 * w * h / 465750),
                                features_per_frame=stats, tracked_fraction=tracked,
                                exchange="device-resident pose copy (+ one NCCL all-gather when n_gpus > 1) per step, inside both timed regions",
                                sequences="one independent trajectory per rank (stream seed + rank) through the same synthetic world: equal work per GPU",
                                rank_serial_kernel_ms=[round(min(r["serial_kernel_ms"] for r in per_rank), 1),
                                                       round(max(r["serial_kernel_ms"] for r in per_rank), 1)]),
                    e2e=dict(value=e2e_v, unit=UNIT, h2d_bytes_per_step=2 * B * w * h,
                             d2h_bytes_per_step=B * ctypes.sizeof(plf.plf_frame_result), ms_per_step=e2e_ms / args.steps),
                    gpu_launches=int(launches), clocks=clocks, roofline=roof, pipeline_vs_hbm=whole,
                    pipeline_timeline_ms=dict(phases=["E", "G", "M"], last_two_batches=timeline), per_rank=per_rank,
                    kernels=ktab)
        if overlapped:
            line["kernels_overlapped"] = overlapped
        if dumped is not None:
            write_outputs(args.dump_outputs, dumped)
        if world == 1 and not args.no_cpu_baseline:
            n_cpu = 48                         # ~12 s of single-core CPU work (0.25 s per pair)
            v, c, dt = cpu_baseline_run(n_cpu, None)
            line["cpu_baseline"] = dict(value=v, unit=UNIT, cores=c, kind="port", host_cpus=os.cpu_count(),
                                        sample="%d rendered pairs of the same stream, one pass (%.1f s): cv2 4.13 ORB+LSD+BFMatcher + C LBD/GN, "
                                               "%d worker processes (%d CPUs visible)" % (n_cpu, dt, c, os.cpu_count()))
        emit(line)
    fe.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
