#!/usr/bin/env python
"""Benchmark of the LINEMOD match hot path (BASELINE.json: frames/sec @640x480 vs template-bank size).

  python bench.py --gpus N --steps K --warmup W              our CUDA path
  python bench.py --impl reference --gpus N --steps K ...    the reference's CPU algorithm on the host cores

Workload (configs[1] of BASELINE.json): one object, 3115 templates (89 views x 35 variants), 150 features
per modality at level 0 / 75 at level 1, T = [4, 8], 640x480 frames, threshold 75 (the caller's value,
linemod_and_levelup_test.py:324).  No datasets exist offline: bank and frames are synthetic
(6dpose_b200/synth.py), frames are generated as quantized label images with the fixture frame's
statistics and 8 planted templates each.  A "step" = Detector::match of one frame after quantization
(the cv2 quantization front-end is upstream of the accelerated path and identical for both arms).

value  = frames/s with the frame ring resident in HBM, steps enqueued back to back on the detector's
         stream, timed with CUDA events on that stream (max over ranks).
e2e    = frames/s through the C-ABI call a binding makes (lm_match_quantized): label images in pinned host
         memory -> H2D -> stages -> D2H of the kept records -> host finisher (sort/unique), one blocking
         call per frame.
N > 1  : the template bank is sharded over the ranks (strong scaling), every rank sees every frame, the
         per-rank result blocks are all-gathered (NCCL) every step.
"""
import argparse
import ctypes
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--templates", type=int, default=3115, help="templates per object")
    ap.add_argument("--objects", type=int, default=1, help="objects (classes) in the bank: config 4 = 6 x 3115")
    ap.add_argument("--no-extras", action="store_true", help="N=1: skip the real-data arm, threshold sweep, front-end, ICP blocks")
    ap.add_argument("--features", type=int, default=150)
    ap.add_argument("--width", type=int, default=640)
    ap.add_argument("--height", type=int, default=480)
    ap.add_argument("--threshold", type=float, default=75.0)
    ap.add_argument("--ring", type=int, default=176, help="distinct frames cycled through (176 x 768 KB > 126 MB L2)")
    ap.add_argument("--cpu-frames", type=int, default=3, help="frames of the same workload timed for cpu_baseline")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--lanes", type=int, default=0,
                    help="frames in flight per GPU for `value`: one handle (stream + buffers) per lane, frames "
                         "alternate between lanes so that the small kernels of one frame fill the tail of another "
                         "(default: 3 on one GPU, 6 with the bank sharded: a shard's kernels are short chains)")
    ap.add_argument("--exchange", default="fused", choices=["fused", "nccl"],
                    help="N>1: record exchange fused into the refinement kernel (peer stores over NVLink) or one "
                         "NCCL all-gather of result blocks per frame (the baseline)")
    ap.add_argument("--shards", default="interleaved", choices=["interleaved", "contiguous"],
                    help="N>1: template shard layout (interleaved: rank r takes templates r, r+N, ...: even candidate load)")
    ap.add_argument("--no-parity", action="store_true", help="skip the in-run result check against the oracle")
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the match list of the last timed step (what lm_finish hands a caller) "
                         "as DIR/matches_<field>.npy, to compare two builds on the same inputs")
    return ap.parse_args()


T_PYR = [4, 8]


def make_workload(args, n_frames):
    synth = importlib.import_module("6dpose_b200.synth")
    cids = tuple("%02d_template" % (k + 1) for k in range(max(args.objects, 1)))
    bank = synth.synth_bank(args.templates, num_features=args.features, levels=2, seed=args.seed, variants=35, class_ids=cids)
    frames = []
    for i in range(n_frames):
        q, _ = synth.synth_frame(args.width, args.height, levels=2, seed=1000 + i, bank=bank, plant=8, T=T_PYR)
        frames.append(q)
    return bank, frames


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(smax)) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_arms(args, bank, frames, n_frames):
    """The reference's algorithm on the host cores, two ways: oracle/_ref = the reference's own
    linemodLevelup.cpp compiled unmodified (single-threaded, like the reference), and the OpenMP-over-
    templates port in oracle/lm_oracle.cpp on every core.  Returns a dict of fps per arm."""
    from oracle import oracle
    packed = bank.pack(bank.class_ids(), 4)
    threads = os.cpu_count() or 1
    arms = {"port_all_cores": (lambda q: oracle.match(q, T_PYR, packed, args.threshold, n_threads=threads), threads),
            "port_1_thread": (lambda q: oracle.match(q, T_PYR, packed, args.threshold, n_threads=1), 1)}
    try:
        from oracle import ref as oref
        if oref.available():
            arms["reference_1_thread"] = (lambda q: oref.match(q, T_PYR, packed, args.threshold), 1)
    except ImportError:
        pass
    out = {}
    for name, (fn, cores) in arms.items():
        fn(frames[0])  # warm-up (page in, thread pool)
        t0 = time.perf_counter()
        for i in range(n_frames):
            fn(frames[i % len(frames)])
        dt = time.perf_counter() - t0
        out[name] = {"fps": n_frames / dt, "cores": cores, "seconds": dt}
    return out


def best_cpu_arm(arms):
    name = max(arms, key=lambda k: arms[k]["fps"])
    kind = "reference" if name.startswith("reference") else "port"
    return name, kind


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_frames = min(max(args.steps, 1), 32)  # a bounded sample of full frames: the whole run stays within minutes
    bank, frames = make_workload(args, min(n_frames, 8))
    arms = cpu_arms(args, bank, frames, n_frames)
    name, kind = best_cpu_arm(arms)
    fps = arms[name]["fps"]
    out = {
        "impl": "reference", "metric": metric_name(args),
        "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": n_frames, "warmup": 1,
        "ms_per_step": 1e3 / fps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u8/u16", "data": "synthetic",
        "config": workload_config(args, 1),
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": arms[name]["cores"], "kind": kind,
                         "sample": "%d full frames of the same workload per arm; fastest arm reported (%s)" % (n_frames, name),
                         "arms": arms},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    try:  # poseRefine on the host: the numpy/scipy restatement (oracle/icp_oracle.py), one hypothesis
        from oracle import icp_oracle
        gold = np.load(os.path.join(ROOT, "tests", "golden", "icp_case1.npz"))
        x, y = [int(v) for v in gold["xy_shift_0"]]
        t0 = time.perf_counter()
        icp_oracle.pose_refine(gold["scene_shift_0"], gold["model"], gold["K"], gold["K"], gold["R"], gold["t"].reshape(3), x, y)
        out["icp_cpu"] = {"ms_per_hypothesis": (time.perf_counter() - t0) * 1e3, "kind": "port (numpy/scipy, 1 thread)"}
    except Exception as e:
        out["icp_cpu"] = {"error": repr(e)}
    emit(json.dumps(out))


def oracle_expected(args, packed, quantized, world):
    """The reference's result for one frame of the workload (CPU oracle, test infrastructure: the checker only)."""
    from oracle import oracle
    threads = max(1, (os.cpu_count() or 1) // max(world, 1))
    return oracle.match(quantized, T_PYR, packed, args.threshold, n_threads=min(threads, 64))


DUMP_BYTES = 60 * 10 ** 6   # rows of a dump; with the .npy headers the files stay under 64 MB


def dump_outputs(out_dir, matches):
    """One .npy per field of a match list, one row per match: similarity float32, the integer fields float64 (exact).  A
    list of more than DUMP_BYTES is cut to a fixed, seeded sample of its rows, kept in order."""
    os.makedirs(out_dir, exist_ok=True)
    dtypes = {f: np.float32 if f == "similarity" else np.float64 for f in matches.dtype.names}
    row_bytes = sum(np.dtype(t).itemsize for t in dtypes.values())
    if len(matches) * row_bytes > DUMP_BYTES:
        matches = matches[np.sort(np.random.default_rng(0).choice(len(matches), DUMP_BYTES // row_bytes, replace=False))]
    for f, t in dtypes.items():
        np.save(os.path.join(out_dir, "matches_%s.npy" % f), matches[f].astype(t))


def same_matches(got, want):
    if len(got) != len(want):
        return False
    return (all(np.array_equal(got[k], want[k]) for k in ("x", "y", "template_id", "similarity"))
            and np.array_equal(got["class_index"], want["class_idx"]))


def _device_loop_fps(torch, nat, stream, threshold, steps):
    """frames/s of `steps` enqueues of the frame currently bound to `nat`, CUDA events on its stream."""
    for _ in range(5):
        nat.enqueue(threshold)
    nat.complete()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        nat.enqueue(threshold)
    e1.record(stream)
    nat.complete()
    return steps / (e0.elapsed_time(e1) / 1e3)


def real_data_arm(lib, torch, local):
    """The reference's own fixture frame (linemodLevelup/test/case1/0000_*) against its full allScales bank (2989
    templates, Detector() = 63 features, T = {5, 8}; test.cpp:174-181), thresholds 80 (the reference's invocation) and 75
    (61 912 coarse candidates, SURVEY 6): results checked against the lists the compiled reference produced
    (tests/golden/expected_allScales_full.npz).  One frame repeated, i.e. L2-resident inputs: a candidate-load check of
    the kernels on real data, not a second headline."""
    g = os.path.join(ROOT, "tests", "golden")
    from oracle import golden
    packed, T = golden.allscales_full_bank()
    fr = np.load(os.path.join(g, "frames_case1.npz"))
    q = [[np.ascontiguousarray(fr["full_l%d_m%d" % (l, m)]) for m in range(2)] for l in range(2)]
    exp = np.load(os.path.join(g, "expected_allScales_full.npz"))
    nat = lib.NativeDetector(T, device=local)
    nat.load_bank(packed, 4)
    stream = torch.cuda.ExternalStream(nat.stream(), device=local)
    ts = [torch.from_numpy(q[l][m]).cuda() for l in range(2) for m in range(2)]
    rows, cols = [q[0][0].shape[0], q[1][0].shape[0]], [q[0][0].shape[1], q[1][0].shape[1]]
    hq = [[torch.from_numpy(q[l][m]).pin_memory().numpy() for m in range(2)] for l in range(2)]
    out = {"workload": "fixture frame 640x480 x allScales (2989 templates, 63 features/modality at L0, T=[5,8]); one frame "
                       "repeated (inputs L2-resident), 1 frame in flight", "thresholds": {}}
    for thr in (80.0, 75.0):
        got = nat.match_quantized(hq, thr)
        want = exp["full_%g" % thr]
        ok = len(got) == len(want) and all(np.array_equal(got[k], want[k]) for k in ("x", "y", "template_id", "similarity"))
        c = nat.counters()
        nat.bind_quantized_device([t.data_ptr() for t in ts], rows, cols)
        fps = _device_loop_fps(torch, nat, stream, thr, 100)
        nat.set_timing(50)
        for _ in range(50):
            nat.enqueue(thr)
        nat.complete()
        st = nat.stage_times_us()
        nat.set_timing(0)
        t0 = time.perf_counter()
        for _ in range(50):
            nat.match_quantized(hq, thr)
        e2e = 50 / (time.perf_counter() - t0)
        out["thresholds"]["%g" % thr] = {"matches": int(len(got)), "identical_to_compiled_reference": bool(ok),
                                         "coarse_candidates": c["coarse_candidates"], "frames_per_s": fps,
                                         "e2e_frames_per_s": e2e, "stage_us": st}
    nat.close()
    return out


def threshold_sweep(lib, torch, local, args, packed, ring, rows, cols):
    """Candidate-rate sweep on the synthetic workload (SURVEY 8d): thresholds 75 and 90, one frame in flight."""
    nat = lib.NativeDetector(T_PYR, device=local)
    nat.load_bank(packed, 4)
    stream = torch.cuda.ExternalStream(nat.stream(), device=local)
    out = {}
    for thr in (75.0, 90.0):
        nat.bind_quantized_device(ring[0][1], rows, cols)
        nat.enqueue(thr)
        nat.complete()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n = 64
        e0.record(stream)
        for i in range(n):
            nat.bind_quantized_device(ring[i % len(ring)][1], rows, cols)
            nat.enqueue(thr)
        e1.record(stream)
        nat.complete()
        c = nat.counters()
        out["%g" % thr] = {"frames_per_s_1_lane": n / (e0.elapsed_time(e1) / 1e3), "coarse_candidates_last_frame": c["coarse_candidates"],
                           "kept_last_frame": c["kept"]}
    nat.close()
    return out


def pose_pipeline(lib, local):
    """BASELINE.json config 3 as ONE figure: raw RGB-D frame -> match -> greedy NMS top-3 on the device -> poseRefine of the
    three hypotheses (max 10 ICP iterations) in one batched call.  Inputs: the frame, bank and render of the recorded
    driver run (tests/golden/driver_trace.npz, bank_allScales_full_{a,b}.npz).  Pose error against the ICP oracle with the
    same iteration cap (PARITY UNPINNED: the reference's ICP arithmetic is Open3D's, see oracle/icp_oracle.py)."""
    g = os.path.join(ROOT, "tests", "golden")
    tr = np.load(os.path.join(g, "driver_trace.npz"))
    from oracle import golden
    packed, _ = golden.allscales_full_bank()
    nat = lib.NativeDetector(tr["T"].tolist(), device=local)
    nat.load_bank(packed, 4)
    nat.set_boxes(np.full((int(packed["class_begin"][-1]), 2), 70, np.int32))  # the driver's info files: 70 x 70 boxes
    icp = lib.NativeIcp(local)
    rgb, depth, render = tr["rgb"], tr["depth"], tr["render"]
    K, Km, R, t = tr["rf0_sceneK"], tr["rf0_modelK"], tr["rf0_modelR"], tr["rf0_modelT"].reshape(3)
    thr = float(tr["threshold"])

    def once(max_it=10):
        nat.upload_images(rgb, depth)
        nat.enqueue(thr)
        nat.enqueue_post(0.5, 3)
        top, nrec = nat.complete_post()
        n = len(top)
        if n == 0:
            return top, None
        xy = [[int(m["x"]), int(m["y"])] for m in top]
        return top, icp.process_batch(depth, [render] * n, K, np.stack([Km] * n), np.stack([R] * n), np.stack([t] * n), xy, max_it)

    for _ in range(3):
        top, res = once()
    n_it = 30
    t0 = time.perf_counter()
    for _ in range(n_it):
        top, res = once()
    dt = time.perf_counter() - t0
    out = {"frames_per_s": n_it / dt, "ms_per_frame": dt / n_it * 1e3, "hypotheses": int(len(top)), "max_iterations": 10,
           "top": [[int(m["x"]), int(m["y"]), int(m["template_id"]), float(m["similarity"])] for m in top],
           "note": "lm_upload_images + lm_enqueue + lm_enqueue_post (NMS IoU 0.5, top 3) + lm_icp_process_batch; host buffers in, "
                   "poses out; ICP parity unpinned (Open3D)"}
    try:
        from oracle import icp_oracle
        errs = []
        for i, m in enumerate(top):
            o = icp_oracle.pose_refine(depth, render, K, Km, R, t, int(m["x"]), int(m["y"]), max_iter=10)
            if o["R"] is None:
                continue
            errs.append(max(float(np.linalg.norm(res[0][i] - o["R"]) / np.linalg.norm(o["R"])),
                            float(np.linalg.norm(res[1][i] - o["t"].reshape(3)) / np.linalg.norm(o["t"]))))
        out["pose_rel_error_vs_icp_oracle_max"] = max(errs) if errs else None
        out["fitness"] = [float(v) for v in res[2]]
    except Exception as e:  # informative only
        out["pose_rel_error_vs_icp_oracle_max"] = repr(e)
    nat.close()
    return out


def metric_name(args):
    return "frames/sec @%dx%d, %d-template bank, Detector::match after quantization" % (
        args.width, args.height, args.templates * max(args.objects, 1))


def workload_config(args, n):
    return {"workload": "obj_01-like synthetic bank, %d object(s) x %d templates (views x 35 variants), %d features/modality at L0, "
                        "T=[4,8], %dx%d quantized RGB-D frames, threshold %g, 8 planted templates per frame"
                        % (args.objects, args.templates, args.features, args.width, args.height, args.threshold),
            "templates": args.templates * args.objects, "objects": args.objects, "frame": [args.width, args.height],
            "threshold": args.threshold,
            "parallelism": "template-shard x%d (%s)" % (n, args.shards), "lanes": args.lanes,
            "exchange": "none" if n == 1 else ("fused into the exact refinement kernel (peer stores over NVLink + collector kernel)"
                                               if args.exchange == "fused" else "nccl all-gather of result blocks"),
            "l2": "ring of %d distinct frames (%.0f MB of label images > 126 MB L2); bank and linear memories are "
                  "L2-resident by design" % (args.ring, args.ring * (args.width * args.height * 2 * 1.25) / 1e6)}


_REAL_STDOUT = None


def emit(line):
    """The driver expects exactly ONE line on stdout: the JSON.  Libraries (NCCL prints its version
    banner to stdout) are kept away from it by pointing fd 1 at stderr for the whole run."""
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (line + "\n").encode())


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    if args.lanes <= 0:
        args.lanes = 3 if world == 1 else 6
    lib = importlib.import_module("6dpose_b200._lib")
    bank, frames = make_workload(args, args.ring)
    packed = bank.pack(bank.class_ids(), 4)
    nats = []
    layout = lib.SHARD_INTERLEAVED if args.shards == "interleaved" else lib.SHARD_CONTIGUOUS
    for _ in range(max(1, args.lanes)):
        n_ = lib.NativeDetector(T_PYR, device=local)
        n_.load_bank(packed, 4)
        n_.select(None, rank, world, layout)
        nats.append(n_)
    nat = nats[0]

    # frame ring resident in HBM (torch owns the memory; the library borrows the pointers)
    rows = [args.height, args.height // 2]
    cols = [args.width, args.width // 2]
    ring = []
    for q in frames:
        ts = [torch.from_numpy(np.ascontiguousarray(q[l][m])).cuda() for l in range(2) for m in range(2)]
        ring.append((ts, [t.data_ptr() for t in ts]))
    stream = torch.cuda.ExternalStream(nat.stream(), device=local)
    lane_streams = [torch.cuda.ExternalStream(n_.stream(), device=local) for n_ in nats]

    for n_ in nats:  # everything lazy (feature addresses for this frame size, work lists, buffers) now: no rank's
        n_.bind_quantized_device(ring[0][1], rows, cols)  # first frame lags the others' behind the barrier below
        n_.prepare()
    # records a shard may keep per frame (the fused exchange's blocks are fixed-size; N=1 grows its block on demand)
    cap = 16384 if args.templates * args.objects * args.width * args.height <= 4000 * 640 * 480 else 1 << 17
    blk_bytes = 16 + 16 * cap
    fused = world > 1 and args.exchange == "fused"
    res = gathered = None
    if fused:
        # exchange fused into the refinement kernels: peer stores into every rank's exchange buffer (CUDA IPC mappings over
        # NVLink) + a collector kernel; the process group only carries the IPC handles, once
        for n_ in nats:
            handles = [None] * world
            dist.all_gather_object(handles, n_.peer_export(world, cap))
            n_.peer_connect(rank, world, handles)
        dist.barrier()
    elif world > 1:
        # baseline exchange: torch-owned result block = the send buffer of one NCCL all-gather per frame
        res = torch.zeros(blk_bytes, dtype=torch.uint8, device="cuda")
        nat.set_result_buffer(res.data_ptr(), cap)
        gathered = torch.zeros(world * blk_bytes, dtype=torch.uint8, device="cuda")

    bind_args = [lib.NativeDetector.bind_args(ptrs, rows, cols) for _, ptrs in ring]  # ctypes arrays built once

    def step(i):
        n_ = nats[i % len(nats)] if (fused or world == 1) else nat
        n_.bind_quantized_device_args(bind_args[i % len(ring)])
        n_.enqueue(args.threshold)
        if world > 1 and not fused:
            with torch.cuda.stream(stream):
                dist.all_gather_into_tensor(gathered, res)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def complete_all():
        for n_ in nats:
            n_.complete()

    def join_lanes():
        # the timing stream (lane 0) waits for the other lanes' work issued so far
        for ls in lane_streams[1:]:
            ev = torch.cuda.Event()
            ev.record(ls)
            stream.wait_event(ev)

    sampler = ClockSampler(local)   # clocks / throttle reasons from the warm-up to the end of the timed region
    sampler.start()
    for i in range(max(args.warmup, 3) * len(nats)):
        step(i)
    complete_all()
    barrier()

    # ---- timed region: K steps, device resident --------------------------------------------------
    launches0 = sum(n_.launch_count() for n_ in nats)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for i in range(args.steps):
        step(args.warmup + i)
    join_lanes()
    e1.record(stream)
    complete_all()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = sum(n_.launch_count() for n_ in nats) - launches0
    clocks = sampler.stop()
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        lt = torch.tensor([launches], device="cuda")
        dist.all_reduce(lt)
        launches = int(lt.item())
    fps = args.steps / (ms / 1e3)

    def finished(n_, host):
        """The match list of the last frame `n_` completed, as lm_finish hands it to a caller.  host: every rank's result
        block after the NCCL all-gather, or None when the records sit in the handle's own block."""
        if host is not None:
            blocks = host.numpy().reshape(world, blk_bytes)
            rec = np.concatenate([blocks[r, 16:16 + 16 * int(blocks[r, :4].view(np.int32)[0])].view(lib.RECORD_DTYPE)
                                  for r in range(world)])
        else:
            rec = n_.fetch_records()
        return n_.finish(rec)

    if args.dump_outputs:
        if rank == 0:
            last = args.warmup + args.steps - 1
            dump_outputs(args.dump_outputs, finished(nats[last % len(nats)] if (fused or world == 1) else nat,
                                                     gathered.cpu() if (world > 1 and not fused) else None))
        barrier()

    # ---- result check: the frames at both ends of the timed region, through every lane (same calls as the timed loop:
    # bind -> enqueue -> complete), against the oracle's list.  A mismatch fails the run.
    parity = {"checked": False, "ok": None, "frames": 0}
    if not args.no_parity:
        ok_all = True
        check_ids = sorted({(args.warmup) % len(ring), (args.warmup + args.steps - 1) % len(ring)})
        for fi in check_ids:
            want = oracle_expected(args, packed, frames[fi], world)
            for n_ in (nats if (fused or world == 1) else nats[:1]):
                n_.bind_quantized_device(ring[fi][1], rows, cols)
                n_.enqueue(args.threshold)
            if world > 1 and not fused:
                with torch.cuda.stream(stream):
                    dist.all_gather_into_tensor(gathered, res)
                    host = gathered.to("cpu", non_blocking=False)
            for k_, n_ in enumerate(nats if (fused or world == 1) else nats[:1]):
                n_.complete()
                got = finished(n_, host if (world > 1 and not fused) else None)
                good = same_matches(got, want)
                if not good:
                    sys.stderr.write("PARITY MISMATCH rank %d lane %d frame %d: got %d matches, oracle %d\n" % (rank, k_, fi, len(got), len(want)))
                ok_all = ok_all and good
                parity["frames"] += 1
        parity["checked"], parity["ok"] = True, bool(ok_all)
        if world > 1:
            t = torch.tensor([1 if ok_all else 0], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            parity["ok"] = bool(int(t.item()))
    barrier()

    # ---- per-kernel durations over K more steps (CUDA events on the launching stream) ------------
    all_lanes, nats = nats, nats[:1]     # one lane: stage durations without overlap
    nat.set_timing(min(args.steps, 256))
    if fused and len(all_lanes) > 1:
        barrier()
    for i in range(min(args.steps, 256)):
        step(args.warmup + i)
    nat.complete()
    stage = nat.stage_times_us()
    nat.set_timing(0)
    # counters of the SAME frames (algorithmic bytes are data dependent): one more pass, completed frame by
    # frame, averaged like the stage durations
    acc = {}
    n_cnt = min(args.steps, 256)
    for i in range(n_cnt):
        step(args.warmup + i)
        nat.complete()
        for k_, v_ in nat.counters().items():
            acc[k_] = acc.get(k_, 0) + v_
    counters = {k_: (v_ // n_cnt if k_ != "templates" else v_ // n_cnt) for k_, v_ in acc.items()}
    nats = all_lanes
    barrier()

    # ---- e2e: host buffers through the C-ABI match call ------------------------------------------
    host_frames = []
    for q in frames[:min(len(frames), 64)]:
        hq = [[torch.from_numpy(np.ascontiguousarray(q[l][m])).pin_memory().numpy() for m in range(2)] for l in range(2)]
        host_frames.append(hq)
    h2d = sum(a.nbytes for lvl in host_frames[0] for a in lvl)

    def e2e_step(i):
        q = host_frames[i % len(host_frames)]
        if world == 1 or fused:
            return nat.match_quantized(q, args.threshold)   # the blocking C-ABI call, host buffers in and out
        nat.upload_quantized(q)
        nat.enqueue(args.threshold)
        with torch.cuda.stream(stream):
            dist.all_gather_into_tensor(gathered, res)   # fixed-size result blocks, one NCCL all-gather
            host = gathered.to("cpu", non_blocking=False)
        nat.complete()
        blocks = host.numpy().reshape(world, blk_bytes)
        parts = []
        for r in range(world):
            n = int(blocks[r, :4].view(np.int32)[0])
            parts.append(blocks[r, 16:16 + 16 * n].view(lib.RECORD_DTYPE))
        return nat.finish(np.concatenate(parts))

    for i in range(3):
        out = e2e_step(i)
    barrier()
    n_e2e = min(args.steps, 100)
    if not args.no_parity:
        # first and last frame of the e2e passes, through the same blocking call
        ok_e2e = True
        for fi in sorted({0, (n_e2e - 1) % len(host_frames)}):
            got = e2e_step(fi)
            good = same_matches(got, oracle_expected(args, packed, frames[fi], world))
            if not good:
                sys.stderr.write("PARITY MISMATCH (e2e) rank %d frame %d\n" % (rank, fi))
            ok_e2e = ok_e2e and good
            parity["frames"] += 1
        if world > 1:
            t = torch.tensor([1 if ok_e2e else 0], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            ok_e2e = bool(int(t.item()))
        parity["ok"] = bool(parity["ok"] and ok_e2e)
        barrier()
    # the blocking call is host-latency bound (sync wake-ups, ctypes): 3 passes of n_e2e steps, the MEDIAN pass is
    # reported so that one scheduler hiccup on a shared host does not decide the number
    passes = []
    for rep in range(3):
        barrier()
        t0 = time.perf_counter()
        d2h = 0
        for i in range(n_e2e):
            out = e2e_step(i)
            d2h += 16 + 16 * nat.counters()["kept"]
        torch.cuda.synchronize()
        passes.append(time.perf_counter() - t0)
    dt = sorted(passes)[1]
    if world > 1:
        t = torch.tensor([dt], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    e2e_fps = n_e2e / dt

    # the drivers' next step (NMS at IoU 0.5, first three survivors) fused behind the match: lm_match_top
    top3 = None
    if world == 1 or fused:
        for i in range(3):
            nat.match_top(host_frames[i % len(host_frames)], args.threshold, 0.5, 3)
        barrier()
        t0 = time.perf_counter()
        for i in range(n_e2e):
            nat.match_top(host_frames[i % len(host_frames)], args.threshold, 0.5, 3)
        dtt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dtt], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dtt = float(t.item())
        top3 = {"value": n_e2e / dtt, "unit": "frames/s",
                "note": "lm_match_top: match + greedy NMS (IoU 0.5) + top-3 on the device, 60 bytes back"}

    # the same blocking call from several host threads, one handle (stream) per thread: what a caller serving
    # several cameras gets; reported beside e2e, not instead of it
    conc = None
    if len(nats) > 1 and (world == 1 or fused):
        import threading

        def caller(n_, k, cnt):
            for i in range(cnt):
                n_.match_quantized(host_frames[(k + i * len(nats)) % len(host_frames)], args.threshold)

        def run_callers(cnt):
            th = [threading.Thread(target=caller, args=(n_, k, cnt)) for k, n_ in enumerate(nats)]
            t0 = time.perf_counter()
            for t_ in th:
                t_.start()
            for t_ in th:
                t_.join()
            return time.perf_counter() - t0

        run_callers(3)
        barrier()
        dtc = run_callers(n_e2e)
        if world > 1:
            t = torch.tensor([dtc], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dtc = float(t.item())
        conc = {"threads": len(nats), "value": n_e2e * len(nats) / dtc, "unit": "frames/s",
                "note": "blocking lm_match_quantized from %d host threads, one handle each" % len(nats)}
    if fused:
        barrier()
        for n_ in nats:
            n_.peer_disconnect()
        barrier()

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        if parity["checked"] and not parity["ok"]:
            raise SystemExit(1)
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6650 GB/s"
    scan_us, refine_us = stage["coarse_scan"], stage["refine"]
    scan_gbs = counters["scan_bytes"] / (scan_us * 1e-6) / 1e9 if scan_us > 0 else 0.0
    refine_gbs = counters["refine_bytes"] / (refine_us * 1e-6) / 1e9 if refine_us > 0 else 0.0
    dominant = "k_coarse_scan" if scan_us >= refine_us else "k_refine"
    ach = scan_gbs if dominant == "k_coarse_scan" else refine_gbs
    # DRAM bytes per launch of the dominant kernel, from the committed `ncu --set full` capture of this workload
    # (profiles/ncu_traffic.json; valid for the default single-GPU workload only)
    traffic, traffic_src = None, None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_r02_traffic.json")))
        default_wl = (args.templates, args.features, args.width, args.height, args.threshold) == (3115, 150, 640, 480, 75.0)
        key = "k_coarse_packed" if dominant == "k_coarse_scan" else "k_refine_filter_w"
        if world == 1 and default_wl and key in tr["kernels"]:
            traffic = tr["kernels"][key]["dram_bytes"]
            traffic_src = tr["source"]
    except (OSError, KeyError, ValueError):
        pass
    # what actually binds each kernel: on-chip pipes from the committed `ncu --set full` capture of this workload
    # (profiles/ncu_r02_summary.json, reduced by tools/ncu_summary.py); the algorithmic-bytes figure above it is the
    # BASELINE.json metric (effective bandwidth), not a physical roofline
    on_chip, binding = {}, None
    try:
        ns = json.load(open(os.path.join(ROOT, "profiles", "ncu_r02_summary.json")))
        pick = {"l1_data_pipe_pct": "l1tex__data_pipe_lsu_wavefronts.avg.pct_of_peak_sustained_elapsed",
                "l2_pct": "lts__throughput.avg.pct_of_peak_sustained_elapsed",
                "alu_pipe_pct": "sm__pipe_alu_cycles_active.avg.pct_of_peak_sustained_elapsed",
                "issue_pct": "smsp__issue_active.avg.pct_of_peak_sustained_active",
                "dram_pct": "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed",
                "warps_active_pct": "sm__warps_active.avg.pct_of_peak_sustained_active",
                "l1_bytes": "l1tex__t_bytes.sum", "l2_bytes": "lts__t_bytes.sum", "us_under_ncu": "gpu__time_duration.sum"}
        for kk in ns["kernels"]:
            name = kk["kernel"].split("(")[0].replace("void ", "")
            on_chip[name] = {a: kk[b] for a, b in pick.items() if b in kk}
            on_chip[name]["top_stalls"] = kk.get("top_stalls_warps_per_issue")
        binding = ns.get("binding")
    except (OSError, KeyError, ValueError):
        pass
    roofline = {
        "bound": "hbm", "kernel": dominant, "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm,
        "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
        "note": "effective bandwidth over ALGORITHMIC bytes (one response byte per feature x position; SURVEY 8d) "
                "of this rank's shard -- the BASELINE.json metric.  The kernels no longer move those bytes (bit-planes in "
                "shared memory / L1, an exact filter in front of the refinement), so `frac` exceeds 1 and is NOT headroom: "
                "see `binding` and `on_chip` for what limits each kernel",
        "binding": binding, "on_chip": on_chip,
        "kernels": {
            "k_linear_memories": {"us": stage["linear_memories"]},
            "k_coarse_scan": {"us": scan_us, "alg_bytes": counters["scan_bytes"], "gbs": scan_gbs, "frac": scan_gbs / hbm},
            "k_scan_counts": {"us": stage["offsets"],
                              "note": "the offset scan runs in the last CTA of the coarse scan (inside k_coarse_scan.us) "
                                      "unless the bank needs k_coarse_bytes; this is the gap between the two events"},
            "k_refine": {"us": refine_us, "alg_bytes": counters["refine_bytes"], "gbs": refine_gbs, "frac": refine_gbs / hbm,
                         "parts_us": {"k_refine_prep (candidate list + H-planes)": stage["refine_prep"],
                                      "k_refine_filter (bit-sliced upper bound)": stage["refine_filter"],
                                      "k_refine<split> (exact, survivors)": stage["refine_exact"]},
                         "filter_dropped_alg_bytes": counters.get("filter_dropped_bytes"),
                         "filter_plane_bytes_read": counters.get("filter_bytes_read"),
                         "exact_lm_bytes_read": counters.get("refine_bytes_read")},
            "stages_total_us": stage["total"],
        },
    }
    out = {
        "metric": metric_name(args),
        "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u8/u16", "data": "synthetic", "config": workload_config(args, world),
        "clocks": clocks,
        "e2e": {"value": e2e_fps, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h // max(n_e2e, 1),
                "steps": n_e2e, "passes_s": passes, "concurrent_callers": conc, "match_top3": top3, "api": "lm_match_quantized (C-ABI), pinned host label images -> matches"},
        "gpu_launches": launches,
        "parity_checked": bool(parity["checked"] and parity["ok"]),
        "parity": dict(parity, against="CPU oracle (oracle/lm_oracle.cpp) on the frames at both ends of the timed region, every lane, "
                                       "and on the first / last frame of the e2e passes; match lists compared field by field, float ==",
                       ),
        "roofline": roofline,
        "counters": counters, "counters_note": "per-frame averages over the frames of the stage-timing pass",
    }
    if world == 1 and not args.no_extras:
        for name, fn in (("real_data", lambda: real_data_arm(lib, torch, local)),
                         ("threshold_sweep", lambda: threshold_sweep(lib, torch, local, args, packed, ring, rows, cols)),
                         ("pose_pipeline", lambda: pose_pipeline(lib, local))):
            try:
                out[name] = fn()
            except Exception as e:  # informative blocks: never lose the headline line over them
                out[name] = {"error": repr(e)}
    if world == 1 and not args.no_extras:
        # quantization front-end (upstream of the metric): raw 640x480 RGB-D -> label pyramids, GPU kernels
        # (incl. the 1.5 MB H2D of the raw frame) vs the cv2 calls the reference makes; identical outputs
        synth = importlib.import_module("6dpose_b200.synth")
        fe = importlib.import_module("6dpose_b200.frontend")
        rgb, dep = synth.synth_rgbd(args.width, args.height, seed=5)
        rgb_p = torch.from_numpy(rgb).pin_memory().numpy()
        dep_p = torch.from_numpy(dep.view(np.int16)).pin_memory().numpy().view(np.uint16)
        for _ in range(3):
            nat.upload_images(rgb_p, dep_p)
        t0 = time.perf_counter()
        for _ in range(50):
            nat.upload_images(rgb_p, dep_p)
        gpu_ms = (time.perf_counter() - t0) / 50 * 1e3
        fe.quantize_pyramid([rgb, dep], 2)
        t0 = time.perf_counter()
        for _ in range(5):
            fe.quantize_pyramid([rgb, dep], 2)
        cv2_ms = (time.perf_counter() - t0) / 5 * 1e3
        t0 = time.perf_counter()
        for _ in range(20):
            mi = nat.match_images(rgb_p, dep_p, None, args.threshold)
        mi_ms = (time.perf_counter() - t0) / 20 * 1e3
        out["frontend"] = {"gpu_ms_per_frame": gpu_ms, "cv2_ms_per_frame": cv2_ms, "match_images_synth_rgbd_ms_per_frame": mi_ms,
                           "note": "lm_upload_images (H2D of raw RGB-D + 9 kernels + sync) vs 6dpose_b200/frontend.py (cv2); "
                                   "match_images_synth_rgbd = lm_match_images on a structured synthetic RGB-D image WITHOUT planted "
                                   "templates (few candidates): a front-end figure, not comparable with e2e (see pose_pipeline / "
                                   "real_data for whole-frame figures on the reference's fixture)"}
    if world == 1 and not args.no_extras:
        # poseRefine (BASELINE.json config 2): the drivers refine the first three NMS survivors; here as one batched
        # call on the reference's own ICP fixture (tests/golden/icp_case1.npz = test/case1/pose/*), host buffers
        try:
            gold = np.load(os.path.join(ROOT, "tests", "golden", "icp_case1.npz"))
            icp = lib.NativeIcp(local)
            nh = 3  # three hypotheses of the fixture's converging case (fitness 1, several Gauss-Newton iterations)
            xy = [[int(v) for v in gold["xy_shift_0"]]] * nh
            a = dict(scene_depth=gold["scene_shift_0"], model_depths=[gold["model"]] * nh, sceneK=gold["K"],
                     modelKs=np.stack([gold["K"]] * nh), Rs=np.stack([gold["R"]] * nh),
                     ts=np.stack([gold["t"].reshape(3)] * nh), detect_xy=xy)
            for _ in range(3):
                icp.process_batch(**a)
            t0 = time.perf_counter()
            for _ in range(20):
                Ro, to, res = icp.process_batch(**a)
            icp_ms = (time.perf_counter() - t0) / 20 * 1e3
            st = icp.last_stats()
            out["icp"] = {"hypotheses_per_call": nh, "ms_per_call": icp_ms, "hypotheses_per_s": nh / icp_ms * 1e3,
                          "points": st["points"], "iterations_last": st["iterations"], "fitness": [float(r) for r in res],
                          "note": "lm_icp_process_batch (host depth images in, poses out) on the reference's pose fixture; "
                                  "parity vs the ICP oracle is held to 1e-4 in tests/test_gpu_icp.py (unpinned: Open3D)"}
        except Exception as e:  # informative only
            out["icp"] = {"error": repr(e)}
    if not args.no_cpu_baseline and world == 1:
        # the CPU arm runs in its own process (torch's bundled OpenMP runtime in this one throttles the oracle's
        # thread pool): same workload, same code path as `bench.py --impl reference`
        cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", str(max(args.cpu_frames, 1) * 4),
               "--templates", str(args.templates), "--features", str(args.features), "--width", str(args.width),
               "--height", str(args.height), "--threshold", str(args.threshold), "--seed", str(args.seed)]
        env = dict(os.environ)
        env.pop("OMP_NUM_THREADS", None)
        try:
            ref = json.loads(subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env).stdout.strip().split("\n")[-1])
            out["cpu_baseline"] = ref["cpu_baseline"]
            if "icp_cpu" in ref and isinstance(out.get("icp"), dict):
                out["icp"]["cpu_oracle"] = ref["icp_cpu"]
        except Exception as e:  # the baseline is informative; never lose the GPU line over it
            out["cpu_baseline"] = {"value": None, "unit": "frames/s", "cores": 0, "kind": "port", "sample": "failed: %r" % (e,)}
    emit(json.dumps(out))
    if dist is not None:
        dist.destroy_process_group()
    if parity["checked"] and not parity["ok"]:
        raise SystemExit("bench.py: results differ from the oracle (see stderr)")


if __name__ == "__main__":
    main()
