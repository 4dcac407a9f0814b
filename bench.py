#!/usr/bin/env python3
"""bench.py -- frames/sec of the hot path (ORB extract + brute-force Hamming match [+ local BA]) at 1920x1080, ~2000 kpts.

Contract: `python bench.py --gpus N --steps K --warmup W [--impl reference]` prints ONE JSON line on rank 0.
  * a "step" = one pass of the hot path over one batch of synthetic frames per GPU (--batch frames of one stream;
    frame t is matched against frame t-1, the first frame against the last frame of the previous step);
  * `value`  = whole-job frames/s with the frames already resident in HBM (device-side timing, max over ranks);
  * `e2e`    = the same metric through the C ABI with HOST (pinned) buffers: H2D of every frame and D2H of keypoints,
               descriptors and match pairs inside the timed region;
  * `roofline` = the dominant kernel's algorithmic bytes / its CUDA-event duration against MEASURED_PEAKS.json;
  * `cpu_baseline` / `--impl reference` = the CPU oracle (a port of the reference; the reference itself needs
    OpenCV/g2o and cannot be built here) timed on this box's host cores on a bounded sample of the same workload.
  * `--dump-outputs DIR` writes what the last timed step returned (keypoints, descriptors, match pairs, its last local-BA window)
    as DIR/<name>.npy; the inputs are seeded, so two builds run with the same arguments can be compared output for output.
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
# Up to 17 streams carry work at once here (the front end + 16 local-BA windows).  The driver multiplexes streams onto
# CUDA_DEVICE_MAX_CONNECTIONS hardware queues (default 8): a window whose stream shares a queue with the front end is serialised behind
# the 2-3 steps of front-end work the device-resident arm keeps queued, which is the suspected cause of that arm's occasional
# collapse (DESIGN.md section 6).  Give every stream its own queue; must be set before the CUDA context exists.
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

W, H = 1920, 1080
TARGET_KPTS = 2000
METRIC = "frames/sec (ORB+match+local BA) @1920x1080, 2000 kpts"
LOWE, CHECK_ORI = 0.8, True  # robust matcher as constructed by frame_tracker (module/frame_tracker.cc:98)
# Local BA runs asynchronously next to the front end, like the reference's mapping thread (mapping_module.cc:63,206): the windows of
# LBA_BATCH_STEPS consecutive steps are solved by ONE b200_lba_solve_batch call (lockstep launch sequence), up to LBA_INFLIGHT such
# batches are in flight on their own streams, and every window submitted inside a timed region is joined before the closing event.
LBA_BATCH_STEPS = float(os.environ.get("B200_BENCH_LBA_BATCH_STEPS", "1"))   # may be fractional: 0.5 = two batches per step
LBA_INFLIGHT = int(os.environ.get("B200_BENCH_LBA_INFLIGHT", "4"))


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="frames per GPU per step")
    ap.add_argument("--min-area", type=int, default=0, help="Preprocessing.min_size; 0 = search for ~2000 keypoints")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-lba", action="store_true")
    ap.add_argument("--no-tracking", action="store_true", help="skip the second workload (device-resident track_local_map chain)")
    ap.add_argument("--lba-every", type=int, default=16, help="one local-BA window (50 keyframes / 10k landmarks) per this many frames")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last timed step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    return args


# ---------------------------------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md): nvidia-smi in the background during the timed region
# ---------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            p = [x.strip() for x in r.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0]))
                smax.append(float(p[1]))
                power.append(float(p[2]))
            except ValueError:
                continue
            for n, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle on the host cores (kind "port")
# ---------------------------------------------------------------------------------------------------------------------
def usable_cpus():
    """Host cores this process may actually use: affinity mask and cgroup CPU quota, not just os.cpu_count()."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period) + 0.5)))
    except (OSError, ValueError):
        pass
    return max(1, n)


def cpu_frames_per_sec(frames, min_area, budget_s, threads=None, lba_problem=None, lba_every=16):
    """The CPU oracle on `threads` host threads: extract + match (pthread pool, one frame per task) and, when
    lba_problem is given, one local-BA solve per `lba_every` frames (one window per thread).
    Returns (frames/s, n_frames, threads, mean matches, n_lba)."""
    from concurrent.futures import ThreadPoolExecutor

    from oracle import pyoracle as O
    O.lib()
    threads = max(1, min(threads or usable_cpus(), 512))
    frames = np.ascontiguousarray(np.stack(frames))
    t0 = time.perf_counter()
    O.frontend_batch(frames, 2, min_area, LOWE, CHECK_ORI, 1)     # calibration on one thread
    per_frame = (time.perf_counter() - t0) / 2.0
    n = int(max(threads, min(16 * threads, budget_s * threads / max(per_frame, 1e-3))))
    if lba_problem is not None:
        n = max(lba_every, (n // lba_every) * lba_every)
    t0 = time.perf_counter()
    counts, matches = O.frontend_batch(frames, n, min_area, LOWE, CHECK_ORI, threads)
    n_lba = 0
    if lba_problem is not None:
        n_lba = n // lba_every
        with ThreadPoolExecutor(min(threads, n_lba)) as ex:
            list(ex.map(lambda _: O.lba_solve(lba_problem)["n_outliers"], range(n_lba)))
    dt = time.perf_counter() - t0
    return n / dt, n, threads, float(matches.mean()), n_lba


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from workloads import synth
    frames = synth.make_stream(8, W, H, stream=0)
    min_area = args.min_area or 7000
    # calibrate min_area with the oracle itself (no GPU code on this arm)
    if not args.min_area:
        from oracle import pyoracle as O
        lo, hi = 800, 20000
        for _ in range(8):
            mid = (lo + hi) // 2
            n = len(O.orb_extract(frames[0], min_area=mid)["kps"])
            if abs(n - TARGET_KPTS) <= 0.03 * TARGET_KPTS:
                lo = hi = mid
                break
            if n > TARGET_KPTS:
                lo = mid
            else:
                hi = mid
        min_area = (lo + hi) // 2
    per_step = []
    total_frames = 0
    threads = usable_cpus()
    budget = max(1.0, min(args.cpu_seconds, 120.0 / max(1, args.steps + args.warmup)))
    lba_problem = None if args.no_lba else synth.make_ba_problem(50, 10, 10000, seed=0, model="stereo")
    for s in range(args.warmup + args.steps):
        fps, n, threads, _, _ = cpu_frames_per_sec(frames, min_area, budget, threads, lba_problem, args.lba_every)
        if s >= args.warmup:
            per_step.append((n, n / fps))
            total_frames += n
    t = sum(x[1] for x in per_step)
    value = total_frames / t
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t / max(1, len(per_step)), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "configs[1]: 1920x1080 synthetic stream, ~2000 kpts, ORB extract + brute-force match vs previous frame"
                               + ("" if args.no_lba else f" + one local BA (50 KF / 10k landmarks, stereo) per {args.lba_every} frames") + " (CPU oracle port)",
                   "min_area": int(min_area), "frames_per_step": int(per_step[0][0]) if per_step else 0},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": threads, "kind": "port",
                         "sample": f"{total_frames} frames of the synthetic 1080p stream, extract + match (+ local BA), {threads} threads "
                                   "(oracle/: C restatement of the reference; the reference itself needs OpenCV/g2o)"},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------------------------------
def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa_note = bind_to_gpu_numa_node(torch, local_rank) if world > 1 else None
    if numa_note and os.environ.get("B200_BENCH_VERBOSE"):
        print(f"[bench] rank {rank}: {numa_note}", file=sys.stderr, flush=True)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from stella_vslam_b200 import _lib, feature, multi_gpu
    from workloads import synth
    from stella_vslam_b200._lib import check, lib, ptr
    L = lib()
    B = args.batch

    # ---- synthetic workload: one 1080p stream per rank -------------------------------------------------------------
    frames_np = np.stack(synth.make_stream(B, W, H, stream=rank))
    calib = frames_np[0] if rank == 0 else synth.make_stream(1, W, H, stream=0)[0]
    prm = feature.orb_params()
    min_area = args.min_area
    if not min_area:  # Preprocessing.min_size searched once so that stream 0 / frame 0 yields 2000 +- 3 % keypoints (SURVEY F2)
        lo, hi = 800, 20000
        for _ in range(10):
            mid = (lo + hi) // 2
            ex = feature.orb_extractor(prm, mid, device=local_rank)
            n = len(ex.extract(calib)[0])
            ex.close()
            if abs(n - TARGET_KPTS) <= 0.03 * TARGET_KPTS:
                lo = hi = mid
                break
            if n > TARGET_KPTS:
                lo = mid
            else:
                hi = mid
        min_area = (lo + hi) // 2

    ex = feature.orb_extractor(prm, min_area, device=local_rank, max_batch=B)
    hx = ex._h
    stride = L.b200_orb_max_keypoints(hx, W, H)
    check(L.b200_orb_reserve(hx, W, H, B))
    hm = C.c_void_p()
    check(L.b200_matcher_create(local_rank, C.byref(hm)))
    stream = torch.cuda.current_stream()
    check(L.b200_orb_set_stream(hx, C.c_void_p(stream.cuda_stream), 0))
    check(L.b200_matcher_set_stream(hm, C.c_void_p(stream.cuda_stream), 0))
    # the sequential resolve pass of the matcher (64 warps on the whole chip) runs on the matcher's side stream under the NEXT step's
    # extraction; its inputs must survive until then, so torch owns TWO sets of result buffers used by alternate steps
    check(L.b200_matcher_set_async_resolve(hm, 1))

    class ResultSet:
        """slot 0 = last frame of the previous step, slots 1..B = this step's frames"""
        def __init__(self):
            self.kps = torch.zeros((B + 1, stride, 6), dtype=torch.float32, device=dev)
            self.desc = torch.zeros((B + 1, stride, 32), dtype=torch.uint8, device=dev)
            self.counts = torch.zeros(B + 1, dtype=torch.int32, device=dev)
            self.pairs = torch.zeros((B, stride, 2), dtype=torch.int32, device=dev)
            self.n_pairs = torch.zeros(B, dtype=torch.int32, device=dev)
            self.angle_ptr = self.kps.data_ptr() + 12  # &kps[0].angle

    sets = [ResultSet(), ResultSet()]
    off = (torch.arange(B + 1, dtype=torch.int32, device=dev) * stride).contiguous()
    frames_dev = torch.from_numpy(frames_np).to(dev)
    gathered = torch.zeros((world, B, 2), dtype=torch.int32, device=dev) if world > 1 else None
    stream_id = multi_gpu.assign_streams(world, world, rank)[0]   # one stream per GPU (BASELINE config 5)
    assert stream_id == rank
    step_no = [0]

    # local BA: one KITTI-sized window (BASELINE config 4) per --lba-every frames
    n_lba = 0 if args.no_lba else max(1, B // args.lba_every)
    lba_pool, lba_handles, lba_problem = None, [], None
    lba_preps = {}
    if n_lba:
        from concurrent.futures import ThreadPoolExecutor

        from stella_vslam_b200 import optimize
        lba_problem = synth.make_ba_problem(50, 10, 10000, seed=rank, model="stereo")
        lba_handles = [optimize.local_bundle_adjuster(device=local_rank) for _ in range(LBA_INFLIGHT)]
        lba_pool = ThreadPoolExecutor(LBA_INFLIGHT)
    lba_state = {"launches": 0, "windows": 0, "pending": 0, "next": 0, "ref": None, "last": None}
    lba_inflight = []   # (future, handle index)

    def lba_prep(hidx, n):
        key = (hidx, n)
        if key not in lba_preps:
            lba_preps[key] = lba_handles[hidx].prepare_batch([lba_problem] * n)
        return lba_preps[key]

    def lba_run(hidx, n):
        prep = lba_prep(hidx, n)
        launches = lba_handles[hidx].optimize_prepared_batch(prep)
        st = prep["st"][n - 1]
        return launches, n, (list(st.iterations), st.n_outliers)

    def lba_collect(fut):
        launches, n, sig = fut.result()
        lba_state["launches"] += launches
        lba_state["windows"] += n
        if lba_state["ref"] is None:
            lba_state["ref"] = sig
        assert sig == lba_state["ref"], "local-BA windows of the same problem disagree"

    def lba_dispatch(n):
        hidx = lba_state["next"]
        lba_state["next"] = (hidx + 1) % LBA_INFLIGHT
        lba_state["last"] = (hidx, n)
        for item in [it for it in lba_inflight if it[1] == hidx]:   # the handle's previous batch must be done
            lba_collect(item[0])
            lba_inflight.remove(item)
        lba_inflight.append((lba_pool.submit(lba_run, hidx, n), hidx))

    def lba_submit():
        if not n_lba:
            return
        lba_state["pending"] += n_lba
        per_batch = max(1, int(round(n_lba * LBA_BATCH_STEPS)))
        while lba_state["pending"] >= per_batch:
            lba_dispatch(per_batch)
            lba_state["pending"] -= per_batch

    def lba_join(keep=None):
        """keep=None: only make room (at most LBA_INFLIGHT batches in flight); keep=0: flush the pending windows and join everything."""
        if not n_lba:
            return
        if keep == 0:
            if lba_state["pending"]:
                lba_dispatch(lba_state["pending"])
                lba_state["pending"] = 0
            while lba_inflight:
                lba_collect(lba_inflight.pop(0)[0])
            return
        while len(lba_inflight) > LBA_INFLIGHT:
            lba_collect(lba_inflight.pop(0)[0])

    def step_device():
        lba_submit()
        step_frontend_device()
        lba_join()

    def step_frontend_device():
        cur, prv = sets[step_no[0] & 1], sets[(step_no[0] & 1) ^ 1]
        step_no[0] += 1
        # previous step's last frame becomes slot 0
        cur.kps[0].copy_(prv.kps[B])
        cur.desc[0].copy_(prv.desc[B])
        cur.counts[0:1].copy_(prv.counts[B:B + 1])
        check(L.b200_orb_bind_outputs(hx, C.c_void_p(cur.kps[1].data_ptr()), C.c_void_p(cur.desc[1].data_ptr()), C.c_void_p(cur.counts[1:].data_ptr()), stride))
        check(L.b200_orb_extract_device(hx, C.c_void_p(frames_dev.data_ptr()), W, H, W, W * H, B, None, 0))
        # (joins the previous step's resolve first, then enqueues distances + top-K on this stream and the resolve on the side stream)
        check(L.b200_match_bruteforce_device(hm, B, C.c_void_p(cur.desc.data_ptr()), C.c_void_p(cur.angle_ptr), 24, C.c_void_p(off[1:].data_ptr()),
                                             C.c_void_p(cur.counts[1:].data_ptr()), C.c_void_p(cur.desc.data_ptr()), C.c_void_p(cur.angle_ptr), 24, None,
                                             C.c_void_p(off.data_ptr()), C.c_void_p(cur.counts.data_ptr()), stride, stride, LOWE, int(CHECK_ORI),
                                             C.c_void_p(cur.pairs.data_ptr()), stride, C.c_void_p(cur.n_pairs.data_ptr())))
        if world > 1:  # gather the per-stream records (keypoint and match counts) of the step whose resolve has just been joined: NCCL over NVLink
            multi_gpu.gather_records(torch.stack([prv.counts[1:], prv.n_pairs], 1), world, gathered)

    def frontend_join():
        check(L.b200_matcher_join(hm))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: device-resident -----------------------------------------------------------------------------------------
    # The timed region is EXACTLY args.steps steps between two barriers; it is repeated REPEATS times back to back and the median
    # repeat is reported (min / p10 / max beside it) -- one region of 20 steps is ~0.1 s, too short to be stable on its own.
    REPEATS = max(1, int(os.environ.get("B200_BENCH_REPEATS", "5")))
    for _ in range(max(args.warmup, 3)):
        step_device()
    lba_join(0)
    frontend_join()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    rep_ms, lba_launches_value = [], 0
    for rep in range(REPEATS):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        lba_state["launches"] = lba_state["windows"] = 0
        e0.record()
        for _ in range(args.steps):
            step_device()
        lba_join(0)          # every window submitted inside the timed region has completed
        frontend_join()      # ... and so has the resolve pass of the last step
        e1.record()
        barrier()
        assert lba_state["windows"] == n_lba * args.steps
        lba_launches_value = lba_state["launches"]
        rep_ms.append(multi_gpu.max_over_ranks(e0.elapsed_time(e1), dev, world))
    clocks = sampler.stop() if rank == 0 else None
    ms_total = float(np.median(rep_ms))
    last = sets[(step_no[0] - 1) & 1]
    n_kp = last.counts[1:].cpu().numpy()
    n_mt = last.n_pairs.cpu().numpy()
    if args.dump_outputs and rank == 0:
        lba_last = None
        if n_lba:
            prep = lba_preps[lba_state["last"]]
            w = prep["n"] - 1
            lba_last = (prep["pose"][w], prep["pts"][w], prep["outl"][w][:prep["arr"][w].n_edges])
        dump_outputs(args.dump_outputs, last.kps[1:].cpu().numpy(), last.desc[1:].cpu().numpy(), n_kp, last.pairs.cpu().numpy(), n_mt, lba_last)
    value = multi_gpu.frames_per_second(B, args.steps, world, ms_total)
    repeat_stats = {"repeats": REPEATS, "ms_per_step": [m / args.steps for m in rep_ms], "median": ms_total / args.steps,
                    "min": min(rep_ms) / args.steps, "p10": float(np.percentile(rep_ms, 10)) / args.steps, "max": max(rep_ms) / args.steps}

    # ---- per-kernel device times from an UNCONTENDED pass (front end alone, then one local-BA batch alone, both after the timed
    #      regions): stage events taken while other streams co-run measure the co-runner too
    check(L.b200_orb_enable_timing(hx, 1))
    check(L.b200_matcher_enable_timing(hm, 1))
    stage_runs, match_runs = [], []
    for _ in range(3):
        step_frontend_device()
        frontend_join()
        torch.cuda.synchronize()
        check(L.b200_orb_sync(hx))
        stage_runs.append(ex.stage_ms())
        t_ms = [C.c_float(), C.c_float()]
        for i in range(2):
            check(L.b200_matcher_stage_ms(hm, i, C.byref(t_ms[i])))
        match_runs.append([t_ms[0].value, t_ms[1].value])
    stage_ms = [float(x) for x in np.median(np.array(stage_runs), axis=0)]
    match_ms = [float(x) for x in np.median(np.array(match_runs), axis=0)]
    check(L.b200_orb_enable_timing(hx, 0))
    check(L.b200_matcher_enable_timing(hm, 0))
    raw_counts = np.zeros(B, np.int32)
    check(L.b200_orb_raw_corner_counts(hx, ptr(raw_counts), B))
    lba_kernel_ms, lba_batch_windows = None, 0
    if n_lba:
        hd = lba_handles[0]
        Lb = hd._L
        Lb.b200_lba_enable_profile.argtypes = [C.c_void_p, C.c_int]
        Lb.b200_lba_kernel_ms.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_int)]
        lba_batch_windows = 16   # SURVEY 8d: >= 32 problems for an L2-exceeding footprint would be 0.5 GB more; 16 windows = 230 MB > L2
        prep16 = hd.prepare_batch([lba_problem] * lba_batch_windows)
        hd.optimize_prepared_batch(prep16)
        Lb.b200_lba_enable_profile(hd._h, 1)
        hd.optimize_prepared_batch(prep16)
        Lb.b200_lba_enable_profile(hd._h, 0)
        lba_kernel_ms = []
        for kk in range(8):
            v_, n_ = C.c_float(), C.c_int()
            Lb.b200_lba_kernel_ms(hd._h, kk, C.byref(v_), C.byref(n_))
            lba_kernel_ms.append((v_.value, n_.value))
        lba_iters = sum(prep16["st"][0].iterations)

    # ---- second workload ("tracking step", rank 0): the device-resident chain undistort -> can_observe -> projection match -> pose
    #      optimisation (b200_track_local_map) over the B frames the extractor has just left in HBM, one synthetic local map per frame
    tracking = None
    if not args.no_tracking and rank == 0:
        tracking = tracking_workload(ex, sets[(step_no[0] - 1) & 1], B, W, H, stride, peak_for_tracking(), args)

    # ---- e2e: host buffers through the reference-facing C ABI calls ---------------------------------------------------
    # Two host result sets used by alternate steps (like the device arm): the synchronous matcher call of step k runs on a worker
    # thread while the main thread already uploads and extracts step k + 1 -- what a streaming application does with two synchronous
    # calls.  Everything (uploads, kernels, downloads, both calls of every step) is inside the timed region and joined before it ends.
    from concurrent.futures import ThreadPoolExecutor as _TPE
    cap = stride
    h_frames = _lib.pinned_empty((B, H, W), np.uint8)
    h_frames[:] = frames_np

    class HostSet:
        def __init__(self):
            self.kps = _lib.pinned_empty((B + 1, cap), _lib.KP_DTYPE)
            self.desc = _lib.pinned_empty((B + 1, cap, 32), np.uint8)
            self.counts = _lib.pinned_empty((B + 1,), np.int32)
            self.pairs = _lib.pinned_empty((B, cap, 2), np.int32)
            self.npairs = _lib.pinned_empty((B,), np.int32)
            self.counts[:] = 0
            self.angle = self.kps.ctypes.data + 12

    hsets = [HostSet(), HostSet()]
    h_off = (np.arange(B + 1, dtype=np.int32) * cap).astype(np.int32)
    check(L.b200_orb_bind_outputs(hx, None, None, None, 0))
    check(L.b200_orb_set_stream(hx, None, 1))
    check(L.b200_matcher_set_stream(hm, None, 1))
    check(L.b200_matcher_set_async_resolve(hm, 0))
    match_pool = _TPE(1)
    e2e_no = [0]
    match_futs = [None, None]

    def match_host(hs):
        check(L.b200_match_bruteforce(hm, B, ptr(hs.desc), C.c_void_p(hs.angle), 24, C.c_void_p(h_off[1:].ctypes.data),
                                      C.c_void_p(hs.counts[1:].ctypes.data), ptr(hs.desc), C.c_void_p(hs.angle), 24, None, ptr(h_off), ptr(hs.counts),
                                      LOWE, int(CHECK_ORI), ptr(hs.pairs), cap, ptr(hs.npairs)))

    def step_e2e():
        lba_submit()
        step_frontend_e2e()
        lba_join()

    def step_frontend_e2e():
        k = e2e_no[0]
        e2e_no[0] += 1
        cur, prv = hsets[k & 1], hsets[(k & 1) ^ 1]
        if match_futs[k & 1] is not None:      # the matcher call that last read this set (step k - 2) must have returned
            match_futs[k & 1].result()
        cur.kps[0] = prv.kps[B]
        cur.desc[0] = prv.desc[B]
        cur.counts[0] = prv.counts[B]
        check(L.b200_orb_extract(hx, ptr(h_frames), W, H, W, W * H, B, None, 0, C.c_void_p(cur.kps[1:].ctypes.data), C.c_void_p(cur.desc[1:].ctypes.data),
                                 cap, C.c_void_p(cur.counts[1:].ctypes.data)))
        match_futs[k & 1] = match_pool.submit(match_host, cur)

    def e2e_join():
        for i in range(2):
            if match_futs[i] is not None:
                match_futs[i].result()
                match_futs[i] = None

    for _ in range(max(args.warmup, 3)):
        step_e2e()
    lba_join(0)
    e2e_join()
    e2e_runs = []
    for rep in range(REPEATS):
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_e2e()
        lba_join(0)
        e2e_join()
        torch.cuda.synchronize()
        e2e_runs.append(multi_gpu.max_over_ranks(time.perf_counter() - t0, dev, world))
    h_last = hsets[(e2e_no[0] - 1) & 1]
    h_counts, h_npairs = h_last.counts, h_last.npairs
    e2e_s = float(np.median(e2e_runs))
    e2e_value = world * B * args.steps / e2e_s
    assert np.array_equal(h_counts[1:], n_kp), "host path and device path disagree on keypoint counts"
    assert np.array_equal(h_npairs, n_mt), "host path and device path disagree on match counts"
    n_live = int(h_counts.sum())
    # bytes that cross PCIe per step, counted from the buffers the calls copy: frames up; keypoints / descriptors / counts down;
    # both sides of every matched pair up again (the host-buffer matcher takes host descriptors) and the pairs down; per local-BA
    # window its observations, poses and landmarks up and the optimised poses / landmarks / outlier flags down
    h2d = B * W * H + 2 * (32 + 24) * B * cap + 4 * 4 * B
    d2h = 4 * B + (24 + 32) * B * cap + 4 * B + 8 * B * cap
    if n_lba:
        pr_ = lba_problem
        E_, K_, L_ = len(pr_["e_pose"]), len(pr_["pose_cw"]), len(pr_["points"])
        h2d += n_lba * (E_ * (4 + 4 + 1 + 1 + 1 + 12 + 4 + 4) + K_ * (4 + 152) + L_ * (4 + 24))
        d2h += n_lba * (E_ + K_ * 56 + L_ * 24)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- roofline: every kernel of the step, the dominant one on top ------------------------------------------------------------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured" if "hbm_gbs" in peaks else "fallback"
    sizes = [(W, H)]
    sf = np.float32(1.0)
    for _ in range(1, 8):
        sf = np.float32(1.2) * sf
        sizes.append((int(np.floor(W / float(sf) + 0.5)), int(np.floor(H / float(sf) + 0.5))))
    P = sum(w * h for w, h in sizes)
    p0, p7 = sizes[0][0] * sizes[0][1], sizes[-1][0] * sizes[-1][1]
    N = float(n_kp.mean())
    raw_c = float(raw_counts.mean())     # counted by the FAST kernel itself (b200_orb_raw_corner_counts)
    # algorithmic bytes per unit (SURVEY.md section 8d), every stage counted once.  Front end: per frame; matcher: per (frame, previous
    # frame) pair; local BA: per window and LM iteration
    alg = {
        "pyramid": (P - p7) + (P - p0),
        "fast_nms_gridmax": P + 16 * raw_c,
        "select": 16 * raw_c + 16 * N,
        # blur fused into the descriptor: it reads the (37+6)^2 neighbourhood of every keypoint instead of the whole level twice
        "blur_orient_describe": 43 * 43 * N + 32 * N + 28 * N,
        "match_topk": (N + N) * 32 + N * 8 * 4,
        "match_resolve": N * 8 * 4 + N * 32 + 8 * N,
    }
    unit_ms = {"pyramid": stage_ms[0], "fast_nms_gridmax": stage_ms[1], "select": stage_ms[2], "blur_orient_describe": stage_ms[4],
               "match_topk": match_ms[0], "match_resolve": match_ms[1]}
    kernels = {}
    for nm, ms in unit_ms.items():
        gbs = alg[nm] * B / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
        kernels[nm] = {"ms_per_step": ms, "launches_per_step": 7 if nm == "pyramid" else 1, "alg_bytes_per_unit": float(alg[nm]), "units_per_launch": B,
                       "achieved_gbs": gbs, "frac": gbs / peak_gbs}
    if lba_kernel_ms:
        E_, K_, L_ = len(lba_problem["e_pose"]), len(lba_problem["pose_cw"]), len(lba_problem["points"])
        Kf_ = int((np.asarray(lba_problem["pose_fixed"]) == 0).sum())
        lba_alg = {   # SURVEY 8d, per window and iteration (Hpl records are 160 B here: 144 B + padding to whole sectors)
            "lba_landmark_build": E_ * (24 + 160) + L_ * (24 + 72 + 24),
            "lba_pose_rows": E_ * 24 + K_ * (56 + 288 + 48),
            "lba_schur": E_ * 160 + L_ * 72 + (6 * Kf_) ** 2 * 8,
            "lba_cholesky": (6 * Kf_) ** 2 * 8 * 2,
            # back-substitution + chi2 of the trial state + accept / reject (one kernel since round 2b)
            "lba_backsub_trial": E_ * 160 + L_ * 48 + E_ * 24 + L_ * 24 + E_ * 8,
        }
        idx = {"lba_landmark_build": 1, "lba_pose_rows": 2, "lba_schur": 3, "lba_cholesky": 4, "lba_backsub_trial": 5}
        windows_per_step = n_lba
        for nm, kk in idx.items():
            tot_ms, n_int = lba_kernel_ms[kk]
            # the profiled batch launched n_int repetitions for lba_iters useful LM iterations (the rest ran empty); time per useful launch
            per_launch = tot_ms / max(lba_iters, 1)
            gbs = lba_alg[nm] * lba_batch_windows / (per_launch * 1e-3) / 1e9 if per_launch > 0 else 0.0
            kernels[nm] = {"ms_per_step": tot_ms * windows_per_step / lba_batch_windows, "launches_per_step": n_int * windows_per_step / lba_batch_windows,
                           "alg_bytes_per_unit": float(lba_alg[nm]), "units_per_launch": lba_batch_windows, "ms_per_launch": per_launch,
                           "achieved_gbs": gbs, "frac": gbs / peak_gbs}
    dom = max(kernels, key=lambda k_: kernels[k_]["ms_per_step"])
    # DRAM traffic per launch of every kernel from the committed `ncu --set full` captures of the same kernels at the same sizes
    # (profiles/r2_ncu_full_*.csv: dram__bytes_read.sum + dram__bytes_write.sum; 64 frames / 16 windows per launch like `achieved`).
    # ncu replays kernels, so the capture cannot be re-taken inside a timed bench; the file travels with the repository.
    traffic = ncu_traffic_per_launch()
    for nm, tb in traffic.items():
        if nm in kernels:
            kernels[nm]["dram_bytes_per_launch_ncu"] = tb
    roofline = {"kernel": dom, "bound": "hbm", "achieved": kernels[dom]["achieved_gbs"], "peak": peak_gbs, "unit": "GB/s",
                "frac": kernels[dom]["frac"], "traffic": traffic.get(dom), "traffic_source": "profiles/r2_ncu_full_{frontend,lba}.csv" if dom in traffic else None,
                "peak_source": peak_src,
                "note": ("per-kernel times come from an uncontended pass after the timed regions (front end alone; one batch of "
                         f"{lba_batch_windows} local-BA windows alone, profiling mode); dominant = largest device time per step over ALL kernels. "
                         "FAST is integer-ALU-bound and the matcher POPC-bound by construction; the HBM fraction is reported as the contract asks. "
                         "traffic: bytes per launch from the committed ncu captures (profiles/), not re-measured in this run"),
                "kernels": kernels}

    cpu = cpu1 = cv2_stage = None
    if not args.no_cpu_baseline:
        fps, n, threads, mean_matches, n_cpu_lba = cpu_frames_per_sec(list(frames_np[:8]), min_area, args.cpu_seconds, None, lba_problem,
                                                                      args.lba_every)
        cpu = {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
               "sample": f"{n} frames of the same synthetic 1080p stream (extract + match vs previous frame) + {n_cpu_lba} local-BA windows "
                         f"on {threads} host threads; scalar C restatement (-O3, no SIMD): BASELINE.md's probe puts the reference's OpenCV "
                         "primitives at ~2.5x this per core, so read the ratio against this port as an upper bound"}
        # B-1 (BASELINE.md section 3): ONE thread, the reference's default build (USE_OPENMP OFF, src/stella_vslam/CMakeLists.txt:120)
        fps1, n1, _, _, n1_lba = cpu_frames_per_sec(list(frames_np[:8]), min_area, min(args.cpu_seconds, 8.0), 1, lba_problem, args.lba_every)
        cpu1 = {"value": fps1, "unit": "frames/s", "cores": 1, "kind": "port", "sample": f"{n1} frames + {n1_lba} local-BA windows on one thread"}
        # B-3: the ORB stage alone assembled from the real cv2 primitives (resize, FAST per cell, GaussianBlur), one thread -- a sanity
        # anchor for the absolute speed of "the reference's OpenCV path"; IC angle / rBRIEF / match / BA are not in it
        try:
            import cv2
            cv2.setNumThreads(1)
            t0 = time.perf_counter()
            reps_cv = 0
            det = cv2.FastFeatureDetector_create(20, True, cv2.FAST_FEATURE_DETECTOR_TYPE_9_16)
            while time.perf_counter() - t0 < 3.0:
                lev = frames_np[reps_cv % B]
                for l in range(8):
                    if l:
                        lev = cv2.resize(lev, sizes[l], interpolation=cv2.INTER_LINEAR)
                    hh, ww = lev.shape
                    for y in range(19, hh - 19 - 6, 64):
                        for x in range(19, ww - 19 - 6, 64):
                            det.detect(lev[y:min(y + 70, hh - 19), x:min(x + 70, ww - 19)])
                    cv2.GaussianBlur(lev, (7, 7), 2, sigmaY=2, borderType=cv2.BORDER_REFLECT_101)
                reps_cv += 1
            cv2_stage = {"value": reps_cv / (time.perf_counter() - t0), "unit": "frames/s", "cores": 1,
                         "what": "cv2 pyramid + per-cell FAST + GaussianBlur only (Python loop over cells included), cv2 " + cv2.__version__}
        except Exception as exc:  # cv2 missing on the box: the number is optional
            cv2_stage = {"unavailable": str(exc)[:100]}

    names = ["pyramid", "fast_nms_gridmax", "select", "blur(fused)", "blur_orient_describe"]
    line = {
        "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic",
        "config": {"workload": "configs[1]: 1920x1080 synthetic stream, ~2000 kpts, ORB extract + brute-force match vs previous frame",
                   "frames_per_gpu_per_step": B, "min_area": int(min_area), "keypoints_per_frame_mean": float(N),
                   "matches_per_frame_mean": float(n_mt.mean()), "raw_fast_corners_per_frame_mean": raw_c,
                   "l2": f"inputs larger than L2: {B} frames x {W * H / 1e6:.2f} MB + {B} pyramids",
                   "timing": f"median of {REPEATS} timed regions of {args.steps} steps each (repeat_stats)",
                   "numa_binding_rank0": numa_note,
                   "lba": (f"{n_lba} local-BA windows per step (one per {args.lba_every} frames): 50 keyframes (10 fixed), 10000 landmarks, "
                           f"{len(lba_problem['e_pose'])} stereo observations, 5+10 LM iterations, solved asynchronously next to the front end "
                           f"(b200_lba_solve_batch: {max(1, int(round(n_lba * LBA_BATCH_STEPS)))} windows per launch sequence, up to {LBA_INFLIGHT} batches in flight; "
                           f"all joined inside the timed region; inputs are host buffers in both arms -- the ABI of the mapping thread)")
                   if n_lba else "disabled"},
        "clocks": clocks,
        "repeat_stats": repeat_stats,
        "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": 1e3 * e2e_s / args.steps, "repeats_ms_per_step": [1e3 * t / args.steps for t in e2e_runs],
                "note": "synchronous host-buffer calls b200_orb_extract / b200_match_bruteforce / b200_lba_solve_batch; the matcher call of "
                        "step k runs on a worker thread while step k+1 uploads and extracts (two host result sets); all joined inside the timed region"},
        "gpu_launches": 12 * args.steps + lba_launches_value,   # per step: 7 resize + FAST + select + describe + top-K + resolve
        "roofline": roofline,
        "cpu_baseline": cpu,
        "cpu_baseline_1thread": cpu1,
        "cv2_orb_stage_1thread": cv2_stage,
        "stage_ms": {n_: stage_ms[i] for i, n_ in enumerate(names + ["extract_total"])},
        "tracking": tracking,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


DUMP_LIMIT_BYTES = 60 << 20        # the whole dump, .npy headers included, stays under 64 MB


def dump_outputs(out_dir, kps, desc, counts, pairs, n_pairs, lba):
    """Write what one step returns to its caller as DIR/<name>.npy (float32; the local-BA window in float64), so that two builds can be
    compared output for output.  Per frame: its keypoints (x, y, size, angle, response, octave), rBRIEF descriptors (one byte per
    column) and (frame, previous frame) match pairs, concatenated in frame order; `frames` lists the frames written.  If all frames
    would exceed DUMP_LIMIT_BYTES, a fixed, seeded sample of frames is written.  lba: (pose_cw, points, outlier flags) of the step's
    last local-BA window, or None."""
    counts, n_pairs = counts.astype(np.int64), n_pairs.astype(np.int64)
    lba_bytes = sum(a.size * 8 for a in lba) if lba is not None else 0
    frame_bytes = 4 * (counts * (6 + 32) + n_pairs * 2 + 3)
    frames = np.arange(len(counts))
    if frame_bytes.sum() + lba_bytes > DUMP_LIMIT_BYTES:
        order = np.random.default_rng(0).permutation(len(counts))
        frames = np.sort(order[:np.searchsorted(np.cumsum(frame_bytes[order]), DUMP_LIMIT_BYTES - lba_bytes, side="right")])
    kp = np.concatenate([kps[f, :counts[f]] for f in frames])
    kp[:, 5] = kp[:, 5].view(np.int32)          # the octave column holds int32 bits
    out = {"frames": frames, "keypoint_counts": counts[frames], "keypoints": kp,
           "descriptors": np.concatenate([desc[f, :counts[f]] for f in frames]),
           "match_counts": n_pairs[frames], "match_pairs": np.concatenate([pairs[f, :n_pairs[f]] for f in frames])}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))
    if lba is not None:
        for name, a in zip(("lba_pose_cw", "lba_points", "lba_outliers"), lba):
            np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


def bind_to_gpu_numa_node(torch, local_rank):
    """One process per GPU: run this rank (and first-touch its pinned host buffers) on the CPU socket the GPU hangs off.  With eight ranks
    on a two-socket host the end-to-end arm moves 8 x 157 MB per step over PCIe; buffers on the far socket cross the inter-socket link.
    Best effort: silently does nothing where sysfs does not expose the topology.  B200_BENCH_NUMA=0 disables it."""
    if os.environ.get("B200_BENCH_NUMA", "1") == "0":
        return "disabled"
    try:
        pr = torch.cuda.get_device_properties(local_rank)
        bdf = "%04x:%02x:%02x.0" % (getattr(pr, "pci_domain_id", 0), pr.pci_bus_id, pr.pci_device_id)
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        if node < 0:
            return f"{bdf}: no NUMA node reported"
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if not allowed:
            return f"{bdf}: node {node} has no allowed CPU"
        os.sched_setaffinity(0, allowed)
        return f"{bdf}: NUMA node {node}, {len(allowed)} CPUs"
    except Exception as exc:  # containers without sysfs topology, old torch without pci ids ...
        return f"unavailable ({type(exc).__name__})"


def ncu_traffic_per_launch():
    """kernel name of `roofline.kernels` -> DRAM bytes (read + write) per launch, from profiles/r2_ncu_full_*.csv (tools/ncu_summary.py)."""
    import csv
    names = {"resize_kernel": "pyramid", "fast_cells_kernel": "fast_nms_gridmax", "select_kernel": "select", "describe_kernel": "blur_orient_describe",
             "topk_tc_kernel": "match_topk", "resolve_kernel": "match_resolve", "landmark_kernel<0>": "lba_landmark_build", "pose_rows_kernel": "lba_pose_rows",
             "schur_mma_kernel": "lba_schur", "chol_solve_kernel": "lba_cholesky", "backsub_kernel": "lba_backsub_trial"}
    out, seen = {}, {}
    for fn in ("r2_ncu_full_frontend.csv", "r2_ncu_full_lba.csv"):
        path = os.path.join(ROOT, "profiles", fn)
        if not os.path.exists(path):
            continue
        rows = list(csv.reader(open(path)))
        hdr, units = rows[0], rows[1]
        ir, iw, ik = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum"), hdr.index("Kernel Name")
        scale = {"Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0, "Gbyte": 1e9}
        for r in rows[2:]:
            key = next((v for k, v in names.items() if k in r[ik]), None)
            if key is None:
                continue
            b = float(r[ir]) * scale.get(units[ir], 1.0) + float(r[iw]) * scale.get(units[iw], 1.0)
            if key == "pyramid":     # seven launches per step: sum the first seven
                if seen.get(key, 0) < 7:
                    out[key] = out.get(key, 0.0) + b
                    seen[key] = seen.get(key, 0) + 1
            elif key not in out:
                out[key] = b
    return out


def peak_for_tracking():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", 6650.0))
    except Exception:
        return 6650.0


def tracking_workload(ex, last, B, W, H, stride, peak_gbs, args):
    """frames/s of tracking_module::track_local_map's GPU-shaped part (search_local_landmarks + pose optimisation) for B frames whose
    keypoints never leave the GPU.  The local map of every frame is synthetic (workloads/synth.py::make_tracking_frame) and lives in host
    buffers -- the reference's map database does -- so every call uploads it and downloads the results: that IS the end-to-end call."""
    from oracle import pyoracle as O          # cpu_baseline leg only
    from stella_vslam_b200 import _lib, tracking
    from workloads import synth
    cam = dict(model="perspective", fx=1000.0, fy=1000.0, cx=W / 2.0, cy=H / 2.0, fxb=0.0, cols=float(W), rows=float(H), setup="monocular")
    counts = last.counts[1:].cpu().numpy()
    kps_all = np.ascontiguousarray(last.kps[1:].cpu().numpy()).view(_lib.KP_DTYPE).reshape(B, stride)
    desc_all = last.desc[1:].cpu().numpy()
    frames = [dict(synth.make_tracking_frame(kps_all[f, :counts[f]], desc_all[f, :counts[f]], cam, ex.orb_params_.scale_factors_, seed=900 + f,
                                             pre_matched_frac=0.0), frame=f, kp_landmark=None) for f in range(B)]
    tr = tracking.local_map_tracker(ex, cam)
    packed = tr.pack(frames, stride)
    for _ in range(3):
        tr.run_packed(packed)
    walls, stages = [], []
    for _ in range(max(5, args.steps // 2)):
        t0 = time.perf_counter()
        tr.run_packed(packed)
        walls.append(time.perf_counter() - t0)
        stages.append(tr.stage_ms())
    wall = float(np.median(walls))
    st = {k: float(np.median([s_[k] for s_ in stages])) for k in stages[0]}
    n_lm = float(np.mean([len(fr["landmarks"]["pos_w"]) for fr in frames]))
    n_kp = float(counts.mean())
    n_match = float(np.mean([T.n_matches for T in packed[0]]))
    n_valid = float(np.mean([T.n_valid for T in packed[0]]))
    h2d = int(sum(len(fr["landmarks"]["pos_w"]) * (24 + 24 + 4 + 4 + 32 + 2) for fr in frames))
    d2h = int(sum(len(fr["landmarks"]["pos_w"]) * (1 + 4) for fr in frames) + B * (stride * 5 + 16 * 8 + 24))
    # compulsory bytes per frame of every stage (inputs once + outputs once)
    alg = {"undistort_observe": n_kp * (24 + 24 + 9) + n_lm * (56 + 2 + 21), "grid": n_kp * (8 + 4) + 64 * 48 * 8,
           "candidates": n_lm * (32 + 18) + n_kp * (32 + 9) + n_match * 8, "resolve": n_lm * (8 + 4) + n_kp,
           "edges": n_lm * 4 + n_kp * (24 + 4 + 1) + (n_match) * (48 + 4 + 24), "pose_optimize": n_match * (48 + 2)}
    kern = {k: {"ms_per_step": st[k], "alg_bytes_per_unit": float(v), "units_per_launch": B,
                "achieved_gbs": v * B / (st[k] * 1e-3) / 1e9 if st[k] > 0 else 0.0} for k, v in alg.items()}
    for k in kern:
        kern[k]["frac"] = kern[k]["achieved_gbs"] / peak_gbs
    dom = max(kern, key=lambda k_: kern[k_]["ms_per_step"])
    # CPU baseline: the oracle's stage-by-stage composition on one thread, a few frames
    t0, n_cpu = time.perf_counter(), 0
    prm = ex.orb_params_
    while n_cpu < min(B, 4) or (time.perf_counter() - t0 < 3.0 and n_cpu < B):
        fr = frames[n_cpu]
        ref = O.track_local_map(cam, kps_all[n_cpu, :counts[n_cpu]], desc_all[n_cpu, :counts[n_cpu]], fr, prm.scale_factors_, prm.inv_level_sigma_sq_,
                                prm.log_scale_factor_)
        assert ref["n_matches"] == packed[0][n_cpu].n_matches and ref["n_valid"] == packed[0][n_cpu].n_valid, "tracking chain disagrees with the oracle"
        n_cpu += 1
    cpu_fps = n_cpu / (time.perf_counter() - t0)
    return {"metric": "frames/sec (track_local_map: undistort + can_observe + projection match + pose optimisation) @1920x1080, 2000 kpts",
            "value": B / (st["chain"] * 1e-3), "unit": "frames/s", "ms_per_step": st["chain"],
            "config": {"workload": f"{B} frames device-resident after extraction, one local map of ~{n_lm:.0f} landmarks per frame (host buffers)",
                       "keypoints_per_frame_mean": n_kp, "landmarks_per_frame_mean": n_lm, "matches_per_frame_mean": n_match,
                       "inliers_per_frame_mean": n_valid, "launches_per_step": 9},
            "e2e": {"value": B / wall, "unit": "frames/s", "ms_per_step": 1e3 * wall, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "stage_ms": st,
            "roofline": {"kernel": dom, "bound": "hbm", "achieved": kern[dom]["achieved_gbs"], "peak": peak_gbs, "unit": "GB/s", "frac": kern[dom]["frac"],
                         "traffic": None, "kernels": kern,
                         "note": "compulsory bytes (inputs once + outputs once); these kernels are latency-bound: one warp per frame in the sequential "
                                 "resolve, one CTA per frame in the pose optimiser"},
            "cpu_baseline_1thread": {"value": cpu_fps, "unit": "frames/s", "cores": 1, "kind": "port",
                                     "sample": f"{n_cpu} frames through oracle.pyoracle.track_local_map (results checked against the GPU chain)"}}


if __name__ == "__main__":
    sys.exit(main())
