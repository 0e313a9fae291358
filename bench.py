#!/usr/bin/env python
"""Benchmark of the batched VIO hot path (BASELINE.json metric: batched VIO image frames/s).

  python bench.py --gpus 1 --steps 40 --warmup 6            # this repo's CUDA path
  python bench.py --impl reference --steps 40 --warmup 6     # the CPU path (oracle port) on all host cores
  torchrun --nproc-per-node N bench.py --gpus N ...          # one rank per GPU, sequences sharded (weak scaling)

A "step" = one 752x480 image per sequence through processImage (+ processFeatures on published frames)
for all S sequences of the rank (app/larvioMain.cpp:107-114).  Workload = BASELINE.json configs[2]:
64 batched synthetic sequences per GPU, 200 tracks, 30-pose window, MSCKF-only.
Prints ONE JSON line on rank 0 (contract in the task statement).
"""
import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from larvio_b200.config import Config          # noqa: E402
from larvio_b200 import synth                  # noqa: E402

W_IMG, H_IMG = 752, 480
B0 = W_IMG * H_IMG
# FP64 peak is not in MEASURED_PEAKS.json (bf16 + HBM only): nominal B200 FP64 vector rate, stated as such.
FP64_PEAK_TF = 37.0        # nominal B200 FP64 (vector = tensor); replaced by the DGEMM probe below when it runs


def probe_fp64_peak(device, n=8192, reps=3):
    """FP64 denominator measured like MEASURED_PEAKS.json measures bf16 (SURVEY 8d asks for it): best of `reps` cuBLAS
    DGEMMs n^3, CUDA-event timed, after one warm-up.  A library call used ONLY as the yardstick, never on the path."""
    import torch
    a = torch.randn(n, n, dtype=torch.float64, device=device); b = torch.randn(n, n, dtype=torch.float64, device=device)
    torch.matmul(a, b)
    best = None
    for _ in range(reps):
        if device.type == "cuda":
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(); e0.record(); torch.matmul(a, b); e1.record(); torch.cuda.synchronize()
            dt = e0.elapsed_time(e1) * 1e-3
        else:
            t0 = time.perf_counter(); torch.matmul(a, b); dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return 2.0 * n ** 3 / best / 1e12
def load_ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch and per sequence from the newest committed `ncu --set full`
    summary (profiles/*_ncu_traffic.json, written by scripts/ncu_summary.py on the GPU box)."""
    import glob
    out = {}; newest = None
    for f in sorted(glob.glob(os.path.join(ROOT, "profiles", "*_ncu_traffic.json"))):      # later tags override earlier captures
        try:
            d = json.load(open(f))
            for k, v in d["kernels"].items():
                name = k.replace("void ", "").split("<")[0].strip()
                out[name] = v["dram_bytes_per_launch"] / max(v.get("sequences_per_launch", 64), 1)
            newest = f
        except Exception:
            continue
    return out, (os.path.relpath(newest, ROOT) if newest else None)


def effective_cores():
    """Host cores this process may actually use: the scheduler affinity mask capped by the cgroup CPU quota (a container
    can see 64 CPUs in os.cpu_count() and be allowed 16)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    if quota:
        n = max(1, min(n, int(quota + 0.5)))
    return n


def load_cfg(args):
    if getattr(args, "workload", "C") == "E":
        # BASELINE configs[4] per GPU: 400 tracks, 50-pose window, 4x5 grid of 1-D inverse-depth SLAM features (20 in the state)
        return Config.load(os.path.join(ROOT, "configs", "euroc_mono.yaml"), max_features_in_one_grid=1, feature_idp_dim=1,
                           aug_grid_rows=4, aug_grid_cols=5, min_distance=14, sw_size=args.window, max_features_num=args.tracks)
    if getattr(args, "workload", "C") == "D":
        # BASELINE configs[3] per GPU: 1-D inverse-depth hybrid (5x6 grid, one SLAM feature per cell), online extrinsic / td /
        # IMU-intrinsic calibration.  Not the headline workload; selectable for measurements of the hybrid path.
        return Config.load(os.path.join(ROOT, "configs", "euroc_mono.yaml"), max_features_in_one_grid=1, feature_idp_dim=1,
                           calib_imu_instrinsic=1, estimate_extrin=1, estimate_td=1, sw_size=args.window, max_features_num=args.tracks)
    return Config.load(os.path.join(ROOT, "configs", "euroc_mono.yaml"), max_features_in_one_grid=0,
                       sw_size=args.window, max_features_num=args.tracks)


# ----------------------------------------------------------------------------- data generation (fork pool)
_GEN_CFG = None


def _gen_one(a):
    seq_index, n_frames = a
    import cv2
    cv2.setNumThreads(1)
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(1)          # one BLAS thread per generator process (one process per core)
    except Exception:
        pass
    return synth.make_sequence(_GEN_CFG, seq_index, n_frames)


def generate(cfg_raw, seq_ids, n_frames, procs):
    """Render the seeded sequences on the host cores.  The result is cached on local disk (LVB_BENCH_CACHE, default
    /tmp/lvb_bench_cache; "off" disables) keyed by config + ids + length, so the arms the driver runs back to back on one
    box (reference first, then this repo's) replay byte-identical inputs without rendering them twice."""
    global _GEN_CFG
    import hashlib
    import pickle
    cache = os.environ.get("LVB_BENCH_CACHE", "/tmp/lvb_bench_cache")
    path = None
    if cache != "off" and seq_ids:
        key = hashlib.sha1(json.dumps([cfg_raw, list(seq_ids), n_frames], sort_keys=True, default=str).encode()).hexdigest()[:20]
        path = os.path.join(cache, "seqs_%s.pkl" % key)
        try:
            with open(path, "rb") as f:
                return pickle.load(f)
        except Exception:
            pass
    _GEN_CFG = cfg_raw
    with mp.get_context("fork").Pool(min(procs, len(seq_ids))) as pool:
        out = pool.map(_gen_one, [(s, n_frames) for s in seq_ids], chunksize=1)
    if path:
        try:
            os.makedirs(cache, exist_ok=True)
            tmp = path + ".%d.tmp" % os.getpid()
            with open(tmp, "wb") as f:
                pickle.dump(out, f, protocol=4)
            os.replace(tmp, path)
        except Exception:
            pass
    return out


# ----------------------------------------------------------------------------- CPU arm: oracle port, one worker per core
def _cpu_worker(conn, cfg_raw, seqs):
    import cv2
    cv2.setNumThreads(1)
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(1)          # one BLAS thread per worker: one sequence per core
    except Exception:
        pass
    from oracle.frontend import ImageProcessorOracle
    from oracle.backend import LarVioOracle
    from oracle import backend_c, orb
    orb.use_compiled(True)                # compiled ORB (oracle/orb_c.cpp), bit-identical to the numpy one
    BE = backend_c.LarVioOracleC if backend_c.supported(cfg_raw) else LarVioOracle      # compiled filter where it covers the config
    st = []
    for sq in seqs:
        st.append(dict(fe=ImageProcessorOracle(cfg_raw), be=BE(cfg_raw), imu=[], k=0, seq=sq, t_fe=0.0, t_be=0.0, n_be=0))
        st[-1]["be"].set_initial_state(sq.img_t[0], sq.gt_q[0], sq.gt_p[0], sq.gt_v[0], np.zeros(3), np.zeros(3))
    conn.send("ready")
    while True:
        cmd = conn.recv()
        if cmd[0] == "quit":
            break
        a, b = cmd[1], cmd[2]
        cpu0 = time.process_time(); w0 = time.perf_counter()
        for j in range(a, b):
            for s in st:
                sq = s["seq"]
                k2 = synth.imu_window(sq, s["k"], sq.img_t[j])
                s["imu"].extend(sq.imu[s["k"]:k2].tolist()); s["k"] = k2
                t0 = time.perf_counter()
                msg = s["fe"].process_image(sq.images[j], sq.img_t[j], np.array(s["imu"]).reshape(-1, 7))
                t1 = time.perf_counter()
                s["t_fe"] += t1 - t0
                if msg is not None:
                    try:
                        s["be"].process_features(msg, s["imu"])
                    except NotImplementedError:
                        pass
                    s["t_be"] += time.perf_counter() - t1; s["n_be"] += 1
        util = (time.process_time() - cpu0) / max(time.perf_counter() - w0, 1e-9)
        conn.send(("done", sum(s["t_fe"] for s in st), sum(s["t_be"] for s in st), sum(s["n_be"] for s in st), util))
        for s in st:
            s["t_fe"] = s["t_be"] = 0.0; s["n_be"] = 0


def cpu_arm_description(cfg_raw):
    """What the CPU arm runs (cpu_baseline.sample): the oracle with its compiled pieces switched on."""
    from oracle import backend_c
    if backend_c.supported(cfg_raw):
        return "cv2 4.13 C++ for the OpenCV calls + compiled ORB (oracle/orb_c.cpp) + compiled filter (oracle/backend_c.cpp, g++ -O3, pinned to golden vectors of the reference's own larvio.cpp and to the numpy oracle to 1e-9), Python glue"
    return "cv2 4.13 C++ for the OpenCV calls + compiled ORB (oracle/orb_c.cpp) + numpy f64 filter (oracle/backend.py: the compiled filter covers pure MSCKF only), Python glue"


class CpuArm:
    def __init__(self, cfg_raw, seqs, cores):
        from oracle import backend_c, orb
        backend_c.load(); orb.use_compiled(True); orb.use_compiled(False)      # build the compiled oracle pieces once, before forking
        ctx = mp.get_context("fork")
        self.cores = min(cores, len(seqs))
        self.conns = []; self.procs = []
        for w in range(self.cores):
            pa, ch = ctx.Pipe()
            p = ctx.Process(target=_cpu_worker, args=(ch, cfg_raw, seqs[w::self.cores]), daemon=True)
            p.start()
            self.conns.append(pa); self.procs.append(p)
        for c in self.conns:
            c.recv()

    def run(self, a, b):
        t0 = time.perf_counter()
        for c in self.conns:
            c.send(("run", a, b))
        res = [c.recv() for c in self.conns]
        dt = time.perf_counter() - t0
        self.last_util = float(np.mean([r[4] for r in res]))      # mean per-worker CPU utilisation (1.0 = a core to itself)
        return dt, sum(r[1] for r in res), sum(r[2] for r in res), sum(r[3] for r in res)

    def close(self):
        for c in self.conns:
            c.send(("quit",))
        for p in self.procs:
            p.join(timeout=5)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock / throttle-reason samples DURING the timed region: an NVML polling thread (5 ms period; the timed
    region of a default run is a few hundred ms, too short for an `nvidia-smi -lms` child to even start)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index, period=0.005):
        self.sm = []; self.bits = 0; self.mx = None; self.ok = False; self.stop_flag = False; self.period = period
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            return
        self.th = threading.Thread(target=self._loop, daemon=True)
        self.th.start()

    def _loop(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.bits |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
            except Exception:
                pass
            time.sleep(self.period)

    def reset(self):
        self.sm = []; self.bits = 0

    def stop(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[])
        if not self.ok:
            return out
        self.stop_flag = True
        self.th.join(timeout=2)
        if self.sm:
            out = dict(sm_mhz=float(np.median(self.sm)), sm_min_mhz=float(min(self.sm)), sm_max_mhz=self.mx,
                       reasons=sorted(v for k, v in self.REASONS.items() if self.bits & k), samples=len(self.sm))
        return out


# ----------------------------------------------------------------------------- roofline models
def kernel_models(S_sub, stats, n_frames, n_sub):
    """ALGORITHMIC bytes (HBM-bound kernels) or FP64 flops per LAUNCH-SET (all launches of that kernel in one frame of one
    sub-batch), DESIGN.md 4 / SURVEY.md 8(d): per-unit figure x the units processed.  `stats` are the device-side work counters of
    the profiled frames summed over sub-batches (lvb_get_stats), so point/row counts are measured, not assumed.  The caller
    divides by the measured number of launches per launch-set."""
    lk_pts, orb_desc, det_runs, msgs, upd, sum_r, sum_rdd, sum_rows, qr_runs, sum_rcc = [float(x) for x in stats[:10]]
    sum_rncd = float(stats[15])
    nl = max(n_frames * n_sub, 1)          # launch-sets
    m = {}
    m["clahe_lut_kernel"] = ("hbm", B0 * S_sub, "read 752x480 u8 per sequence")
    m["clahe_apply_kernel"] = ("hbm", 2 * B0 * S_sub, "read + write 752x480 u8 per sequence")
    m["pyrdown_kernel"] = ("hbm", (B0 + B0 // 4 + B0 // 4 + B0 // 16) * S_sub, "SURVEY F3: both levels")
    m["blur7_kernel"] = ("hbm", 2 * B0 * S_sub, "SURVEY F4")
    m["corner_kernel"] = ("hbm", B0 * det_runs / nl, "SURVEY F5: one pass over 752x480 u8 of the sequences that detect")
    m["lk_kernel"] = ("hbm", 6060.0 * lk_pts / nl, "6060 B per point-track (SURVEY F6)")
    m["orb_gate_kernel"] = ("hbm", 2986.0 * orb_desc / nl, "2986 B per descriptor (SURVEY F7)")
    m["be_gemm_kernel"] = ("fp64", ((2.0 * sum_rncd + 2.0 * sum_rdd) / nl) if upd else None, "T = H P over the nonzero columns (2 r nc d) + P -= Y^T Y (2 r d^2); S = T H^T not counted")
    m["be_qr_kernel"] = ("fp64", (2.0 * sum_rcc / nl) if qr_runs else None, "2 R nc^2 per compression")
    return m


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=120)
    ap.add_argument("--warmup", type=int, default=6)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--seqs", type=int, default=None, help="sequences per GPU (BASELINE configs[2] and [3]: 64; configs[4]: 128)")
    ap.add_argument("--tracks", type=int, default=None)
    ap.add_argument("--window", type=int, default=None)
    ap.add_argument("--preroll", type=int, default=None,
                    help="untimed frames every arm runs before --warmup so that the sliding window is full (30 poses at 10 Hz publishing = 60 frames)")
    ap.add_argument("--cpu-frames", type=int, default=12, help="timed frames per sequence of the bounded cpu_baseline sample (after the pre-roll)")
    ap.add_argument("--profile-steps", type=int, default=8)
    ap.add_argument("--workload", choices=["C", "D", "E"], default="C",
                    help="C = BASELINE configs[2] (MSCKF-only, the headline); D = configs[3] per GPU (1-D IDP hybrid + online calibration); "
                         "E = configs[4] per GPU (128 sequences, 400 tracks, 50-pose window, 20 SLAM features)")
    ap.add_argument("--streams", type=int, default=4,
                    help="sub-batches per GPU, each an independent handle/stream driven by its own host thread")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the run, write what the last timed step of each timed pass returned (publish flags, filter states of "
                         "every sequence) as DIR/<name>.npy in float64, so that two builds can be compared on identical inputs")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.warmup < 3:
        args.warmup = 3
    # per-workload defaults; the pre-roll fills the sliding window (2 frames per pose at 10 Hz publishing) and, in the hybrid
    # workloads, passes the 5 s after which SLAM features are promoted (larvio.cpp:1974)
    wd = {"C": dict(seqs=64, tracks=200, window=30, preroll=70), "D": dict(seqs=64, tracks=200, window=30, preroll=120),
          "E": dict(seqs=128, tracks=400, window=50, preroll=130)}[args.workload]
    for key, val in wd.items():
        if getattr(args, key) is None:
            setattr(args, key, val)
    S, K, Wm = args.seqs, args.steps, args.warmup
    PR = max(args.preroll, 0)
    cfg = load_cfg(args)
    workload = {"C": "configs[2]: %d batched synthetic 752x480@20Hz+200Hz-IMU sequences per GPU, %d tracks, %d-pose window, MSCKF-only",
                "D": "configs[3] per GPU: %d batched synthetic sequences, %d tracks, %d-pose window, 1-D IDP hybrid (5x6 grid) + online extrinsic/td/IMU-intrinsic calibration",
                "E": "configs[4] per GPU: %d batched synthetic sequences, %d tracks, %d-pose window, 1-D IDP hybrid with a 4x5 grid (20 SLAM features in the state)"}[args.workload] % (S, args.tracks, args.window)
    config = dict(workload=workload, preroll_frames=PR, sequences_per_gpu=S, sub_batches_per_gpu=args.streams, tracks=args.tracks, window=args.window, image="752x480 u8",
                  l2_policy="each step reads a fresh %.1f MB image batch and touches >250 MB of per-sequence state (> 126 MB L2)" % (S * B0 / 1e6),
                  inputs=("one pool of %d seeded sequences (seed 1234+i)" % S) + ("" if world == 1 else
                          ", rendered cooperatively by the %d ranks, exchanged over NCCL, replayed on every GPU rotated by rank*%d/%d" % (world, S, world)))
    if os.environ.get("LVB_NO_GRAPH"):
        config["no_graph"] = True                                    # debugging switch: stream launches instead of one graph per step
    ncores = effective_cores()

    # ------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        if rank != 0:
            return 0
        n_frames = PR + Wm + K + args.profile_steps          # same length as the GPU arm renders (shared input cache)
        seqs = generate(cfg.raw, list(range(S)), n_frames, ncores)
        arm = CpuArm(cfg.raw, seqs, ncores)
        arm.run(0, PR + Wm)                      # untimed: fill the sliding window, then the warm-up steps
        dt, tfe, tbe, nbe = arm.run(PR + Wm, PR + Wm + K)
        util = arm.last_util
        arm.close()
        val = S * K / dt
        line = dict(metric="batched VIO frames/sec", value=val, unit="frames/s", n_gpus=args.gpus, steps=K, warmup=Wm,
                    ms_per_step=1e3 * dt / K, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="u8+f32 front end, f64 filter",
                    data="synthetic", config=config, impl="reference",
                    cpu_baseline=dict(value=val, unit="frames/s", cores=arm.cores, kind="port", os_cpu_count=os.cpu_count(), worker_cpu_utilisation=util,
                                      sample="%d sequences x %d frames after a %d-frame pre-roll; %s; one worker process per core" % (S, K, PR + Wm, cpu_arm_description(cfg.raw)),
                                      fe_ms_per_frame=1e3 * tfe / (S * K), be_ms_per_update=1e3 * tbe / max(nbe, 1)),
                    e2e=dict(value=val, unit="frames/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ our arm
    n_frames = PR + Wm + K + args.profile_steps
    # One pool of S seeded sequences per job.  With N ranks every rank renders S/N of them on its share of the host
    # cores (before CUDA is touched: the generator forks), the pool is exchanged with one NCCL all_gather per field,
    # and rank r replays the pool rotated by r*S/N - so host-side image synthesis does not grow with the GPU count
    # while every GPU still steps S distinct sequences.
    from larvio_b200 import dist as ldist
    seq_ids = ldist.shard_sequences(S, rank, world) if world > 1 else list(range(S))
    t_gen = time.time()
    seqs = generate(cfg.raw, seq_ids, n_frames, max(1, ncores // max(world, 1))) if seq_ids else []
    t_gen = time.time() - t_gen
    cpu_baseline = None
    if rank == 0 and world == 1 and args.cpu_frames > 0:
        # bounded sample of the same workload at the same steady state: one sequence per usable core, pre-rolled like the GPU arm
        ncpu = min(S, ncores)
        nf = min(args.cpu_frames, n_frames - PR)
        arm = CpuArm(cfg.raw, seqs[:ncpu], ncores)
        arm.run(0, PR)
        dt, tfe, tbe, nbe = arm.run(PR, PR + nf)
        util = arm.last_util
        arm.close()
        cpu_baseline = dict(value=ncpu * nf / dt, unit="frames/s", cores=arm.cores, kind="port", os_cpu_count=os.cpu_count(), worker_cpu_utilisation=util,
                            sample="%d sequences (one per core) x %d frames after a %d-frame pre-roll of the same workload; %s" % (ncpu, nf, PR, cpu_arm_description(cfg.raw)),
                            fe_ms_per_frame=1e3 * tfe / (ncpu * nf), be_ms_per_update=1e3 * tbe / max(nbe, 1))

    import torch
    import torch.distributed as dist
    from larvio_b200 import api
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        pool = ldist.share_sequences(seqs, S, rank, world, device=torch.device("cuda", local_rank))
        rot = (rank * S) // world
        seqs = pool[rot:] + pool[:rot]
    NSUB = max(1, min(args.streams, S))
    bounds = [(S * i) // NSUB for i in range(NSUB + 1)]          # sub-batch i owns sequences [bounds[i], bounds[i+1])

    def make_batches():
        bs = []
        for i in range(NSUB):
            lo, hi = bounds[i], bounds[i + 1]
            bb = api.Batch(cfg, n_seq=hi - lo, device=local_rank)
            for s in range(lo, hi):
                bb.set_initial_state(s - lo, seqs[s].img_t[0], seqs[s].gt_q[0], seqs[s].gt_p[0], seqs[s].gt_v[0], np.zeros(3), np.zeros(3))
            bs.append(bb)
        return bs

    batches = make_batches()
    last_pub = [None] * NSUB              # what the newest step of sub-batch i returned to its caller
    last_states = [None] * NSUB
    frames_host = np.stack([np.stack([seqs[s].images[j] for s in range(S)]) for j in range(n_frames)])   # [F][S][H][W]
    pinned = torch.from_numpy(frames_host).pin_memory()
    t_img = np.stack([[seqs[s].img_t[j] for s in range(S)] for j in range(n_frames)])
    # per-frame IMU increments per sequence (app/larvioMain.cpp:98-102), pre-packed so that the timed loop
    # appends them to the caller-owned buffers with one vectorised assignment
    k = [0] * S
    inc = []
    for j in range(n_frames):
        rows = []
        for s in range(S):
            k2 = synth.imu_window(seqs[s], k[s], seqs[s].img_t[j]); rows.append(seqs[s].imu[k[s]:k2]); k[s] = k2
        m = np.array([len(r) for r in rows])
        mm = int(m.max()) if len(m) else 0
        arr = np.zeros((S, max(mm, 1), 7))
        for s, r in enumerate(rows):
            arr[s, :len(r)] = r
        inc.append((m, arr))
    IMU_STRIDE = 96

    def sub_pass(i, mode, lo_f, hi_f, state):
        """Driver loop of sub-batch i over frames [lo_f, hi_f) (app/larvioMain.cpp:87-117 for its sequences)."""
        bb = batches[i]
        lo, hi = bounds[i], bounds[i + 1]
        n = hi - lo
        imu, n_imu = state[i]
        ar = np.arange(n)
        for j in range(lo_f, hi_f):
            m, arr = inc[j]
            m = m[lo:hi]; arr = arr[lo:hi]
            mm = arr.shape[1]
            cols = n_imu[:, None] + np.arange(mm)[None, :]
            valid = np.arange(mm)[None, :] < m[:, None]
            rr = np.broadcast_to(ar[:, None], cols.shape)[valid]; cc = cols[valid]
            imu["t"][rr, cc] = arr[:, :, 0][valid]; imu["gyro"][rr, cc] = arr[:, :, 1:4][valid]; imu["acc"][rr, cc] = arr[:, :, 4:7][valid]
            n_imu += m.astype(np.int32)
            if mode == "dev":
                last_pub[i] = bb.step(dev_frames[j, lo:hi].data_ptr(), t_img[j, lo:hi], imu, n_imu, images_on_device=True)
            else:
                last_pub[i] = bb.step(pinned[j, lo:hi].numpy(), t_img[j, lo:hi], imu, n_imu)
                last_states[i] = bb.get_states()

    def run_pass(mode, lo_f, hi_f, state):
        if NSUB == 1:
            sub_pass(0, mode, lo_f, hi_f, state)
            return
        ths = [threading.Thread(target=sub_pass, args=(i, mode, lo_f, hi_f, state)) for i in range(NSUB)]
        for t in ths:
            t.start()
        for t in ths:
            t.join()

    def fresh_state():
        return [(np.zeros((bounds[i + 1] - bounds[i], IMU_STRIDE), api.IMU_DTYPE), np.zeros(bounds[i + 1] - bounds[i], np.int32)) for i in range(NSUB)]

    def launches_total():
        return sum(bb.launches for bb in batches)

    def all_states():
        return np.concatenate([bb.get_states() for bb in batches], 0)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reset_batch():
        nonlocal batches
        for bb in batches:
            bb.close()
        batches = make_batches()

    # ---- device-resident pass: `value`
    dev_frames = pinned.to("cuda", non_blocking=False)
    st = fresh_state()
    sampler = ClockSampler(local_rank) if rank == 0 else None      # NVML polling thread (5 ms period), started before the pre-roll so that
    run_pass("dev", 0, PR + Wm, st)          # untimed: pre-roll to a full sliding window, then the warm-up steps
    barrier()
    if sampler:
        sampler.reset()                      # ... it is already running when the timed region starts: only samples from here on count
    l0 = launches_total()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record(); t0 = time.perf_counter()
    run_pass("dev", PR + Wm, PR + Wm + K, st)
    e1.record(); torch.cuda.synchronize(); wall = time.perf_counter() - t0
    ms_dev = max(e0.elapsed_time(e1), 1e3 * wall * 0.0)     # each step ends with a stream sync, so events == wall
    barrier()
    dump = {}
    if args.dump_outputs:
        dump.update(published=np.concatenate(last_pub), states=all_states())
    clocks = sampler.stop() if sampler else None
    launches = launches_total() - l0
    # steady-state evidence: sliding-window fill and state dimension of every sequence right after the timed region
    ic = np.array([bb.debug_icore(q) for bb in batches for q in range(bb.S)])
    steady = dict(window_poses_mean=float(ic[:, 2].mean()), window_poses_min=int(ic[:, 2].min()), state_dim_mean=float(ic[:, 7].mean()),
                  window_capacity=int(args.window), slam_features_in_state_mean=float(ic[:, 22].mean()))
    # ---- per-kernel profile on the next frames (not part of the timed region)
    prof = {}
    prof_stats = []
    if args.profile_steps > 0:
        stats0 = [bb.stats() for bb in batches]
        for bb in batches:
            bb.profile(True)
        for i in range(NSUB):                      # one sub-batch at a time: per-kernel times without co-running streams
            sub_pass(i, "dev", PR + Wm + K, n_frames, st)
        for bb in batches:
            for kname, (ms, cnt) in bb.profile_get().items():
                a0, c0 = prof.get(kname, (0.0, 0))
                prof[kname] = (a0 + ms, c0 + cnt)
            bb.profile(False)
        prof_stats = [[a1 - a0 for a0, a1 in zip(s0, bb.stats())] for s0, bb in zip(stats0, batches)]
    states_dev = all_states()
    # ---- end-to-end pass: `e2e` (fresh filters, same frames, host buffers)
    reset_batch()
    st = fresh_state()
    run_pass("dev", 0, PR, st)               # untimed pre-roll (device-resident frames), then warm-up through the host-buffer path
    run_pass("e2e", PR, PR + Wm, st)
    barrier()
    e2 = torch.cuda.Event(enable_timing=True); e3 = torch.cuda.Event(enable_timing=True)
    e2.record(); t0 = time.perf_counter()
    run_pass("e2e", PR + Wm, PR + Wm + K, st)
    e3.record(); torch.cuda.synchronize(); wall_e2e = time.perf_counter() - t0
    ms_e2e = max(e2.elapsed_time(e3), 0.0)
    if args.dump_outputs:
        dump.update(e2e_published=np.concatenate(last_pub), e2e_states=np.concatenate(last_states))
    t = torch.tensor([ms_dev, ms_e2e], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        # trajectory gather (SURVEY §8e): final states of every rank to all ranks over NCCL
        mine = torch.from_numpy(all_states()).cuda()
        gathered = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(gathered, mine)
    ms_dev, ms_e2e = float(t[0]), float(t[1])
    if rank == 0:
        value = world * S * K / (ms_dev / 1e3)
        e2e_val = world * S * K / (ms_e2e / 1e3)
        # roofline of the dominant kernel
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0)); peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
        global FP64_PEAK_TF
        fp64_src = "nominal 37 TFLOP/s (not in MEASURED_PEAKS.json)"
        try:
            FP64_PEAK_TF = float(probe_fp64_peak(torch.device("cuda", local_rank)))
            fp64_src = "measured: cuBLAS DGEMM 8192^3 burst, this run"
        except Exception as ex:                                   # the probe must never take the bench down
            fp64_src += "; probe failed: %s" % type(ex).__name__
        tot = sum(v[0] for v in prof.values()) or 1.0
        top = sorted(prof.items(), key=lambda kv: -kv[1][0]) or [("none", (0.0, 0))]
        kernel_share = {kname: dict(ms_per_launch=v[0] / max(v[1], 1), launches=v[1], share=v[0] / tot) for kname, v in top}
        dom_by_time = top[0][0]
        pstats = [sum(x) for x in zip(*prof_stats)] if prof_stats else [0] * 16
        if pstats[4]:
            steady.update(mean_update_rows_r=pstats[5] / pstats[4], mean_stacked_rows=pstats[7] / pstats[4], qr_runs_per_update=pstats[8] / pstats[4])
        lk_paths = dict(point_tracks=pstats[0], iterations=pstats[10], slow_path_iterations=pstats[11], slow_path_setups=pstats[12], tile_restages=pstats[13],
                        iterations_per_point_track=(pstats[10] / pstats[0] if pstats[0] else None),
                        ransac_runs_with_8_to_13_points=pstats[14])
        models = kernel_models(S // NSUB, pstats, args.profile_steps, NSUB)
        roofs = {}
        for kname, v in top:
            mdl = models.get(kname)
            if not mdl or not mdl[1]:
                continue
            per_launch_ms = v[0] / max(v[1], 1)
            per_launch = mdl[1] * (args.profile_steps * NSUB) / max(v[1], 1)      # launch-set figure / launches per launch-set
            if mdl[0] == "hbm":
                ach = per_launch / (per_launch_ms * 1e-3) / 1e9
                roofs[kname] = dict(bound="hbm", achieved=ach, peak=hbm_peak, unit="GB/s", frac=ach / hbm_peak, algorithmic_bytes_per_launch=per_launch, basis=mdl[2])
            else:
                ach = per_launch / (per_launch_ms * 1e-3) / 1e12
                roofs[kname] = dict(bound="fp64", achieved=ach, peak=FP64_PEAK_TF, unit="TFLOP/s", frac=ach / FP64_PEAK_TF, flops_per_launch=per_launch, basis=mdl[2])
        # the roofline object describes the most expensive kernel that has a byte / flop model (per-sequence latency kernels such as
        # the RANSAC replay have no meaningful one); `dominant_by_time` names the top kernel by device time whatever it is
        dom, (dom_ms, dom_n) = next(((kname, v) for kname, v in top if kname in roofs), top[0])
        ncu_traffic, ncu_src = load_ncu_traffic()
        roof = dict(kernel=dom, dominant_by_time=dom_by_time, bound="hbm", achieved=None, peak=hbm_peak, unit="GB/s", frac=None, traffic=(ncu_traffic[dom] * (S // NSUB) if dom in ncu_traffic else None),
                    traffic_source=("%s (ncu --set full, cold cache, per launch, scaled to the sequences of one launch)" % ncu_src) if ncu_src else None, peak_source=peak_src,
                    ms_per_launch=dom_ms / max(dom_n, 1))
        if dom in roofs:
            roof.update({kk: roofs[dom][kk] for kk in ("bound", "achieved", "peak", "unit", "frac")})
            roof["basis"] = roofs[dom]["basis"]
        # SURVEY 8(d): step-level roofline = sum_k launches_k * max(bytes_k / BW_hbm, flops_k / peak_fp64) over the measured kernel time
        bound_ms = 0.0
        for kname, v in top:
            if kname in roofs:
                rk = roofs[kname]
                per = (rk["algorithmic_bytes_per_launch"] / (hbm_peak * 1e9) if rk["bound"] == "hbm" else rk["flops_per_launch"] / (FP64_PEAK_TF * 1e12)) * 1e3
                bound_ms += per * v[1]
        step_roof = dict(bound_ms=bound_ms, measured_kernel_ms=tot, frac=bound_ms / tot, fp64_peak_tflops=FP64_PEAK_TF, fp64_peak_source=fp64_src,
                         note="kernels without a byte/flop model (bookkeeping, <10% of the time) contribute 0 to bound_ms")
        # per-frame EKF-update time (BASELINE metric, second half): back-end kernels of the profiled frames per published batch frame
        be_ms = sum(v[0] for kname, v in prof.items() if kname.startswith("be_"))
        n_pub = max(pstats[3] / float(S), 1e-9)                      # published (sequence, frame) messages / sequences
        ekf_ms = dict(batch_ms_per_published_frame=be_ms / n_pub, per_sequence_ms=be_ms / n_pub / S,
                      note="sum of be_* kernel durations over the profiled frames; batch of %d sequences in %d sub-batches" % (S, NSUB))
        line = dict(metric="batched VIO frames/sec", value=value, unit="frames/s", n_gpus=world, steps=K, warmup=Wm,
                    ms_per_step=ms_dev / K, higher_is_better=True, scaling="weak", vs_baseline=None,
                    dtype="u8+f32 front end, f64 filter", data="synthetic", config=config,
                    e2e=dict(value=e2e_val, unit="frames/s", h2d_bytes_per_step=int(S * B0 + S * 10 * 56), d2h_bytes_per_step=int(S * 17 * 8 + S * 32 * 4 + S)),
                    gpu_launches=int(launches), clocks=clocks, roofline=roof, kernels=kernel_share, kernel_rooflines=roofs, work_counters=pstats,
                    steady_state=steady, lk_paths=lk_paths, ekf_update_ms=ekf_ms, step_roofline=step_roof, cpu_baseline=cpu_baseline, gen_seconds=t_gen, wall_dev_s=wall, wall_e2e_s=wall_e2e)
        print(json.dumps(line))
        if args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in dump.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), np.asarray(arr, np.float64))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
