"""Template-extraction throughput: host Detector.addTemplate (cv2 + numpy) against Detector.addTemplates (GPU).

Views are seeded warps of the reference's training fixture (tests/golden/train_case1.npz, 640x480: rotation, scale
and shift; synth.warp_views).  The host path is timed per view on a subset; the GPU path end to end (the call is
blocking: it returns after the device has finished and the templates are in the bank) on each batch size, after a
warm-up.  The outputs of both paths are compared on the subset.  Prints one JSON line with the card's name and power
limit read in the same run.

    python tools/train_bench.py [--batches 256 2048] [--host-views 20] [--detector default|nf150] [--profile] [--out F]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return q[0], q[1]
    except (OSError, subprocess.SubprocessError, IndexError):
        return "unknown", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[256, 2048])
    ap.add_argument("--host-views", type=int, default=20)
    ap.add_argument("--detector", choices=["default", "nf150"], default="default")
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--profile", action="store_true", help="per-kernel device time (torch.profiler) of one extra batch of 256")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    pkg = importlib.import_module("6dpose_b200")
    synth = importlib.import_module("6dpose_b200.synth")
    det_args = () if args.detector == "default" else (150, [4, 8])
    g = np.load(os.path.join(ROOT, "tests", "golden", "train_case1.npz"))
    n = max(args.batches + [args.host_views])
    views = synth.warp_views(g["rgb"], g["dep"], g["mask"], n, seed=11)
    srcs = [[r, d] for r, d, _ in views]
    masks = [m for _, _, m in views]

    sub = args.host_views
    host = pkg.Detector(*det_args)
    t0 = time.perf_counter()
    host_ids = [host.addTemplate(srcs[i], "obj", masks[i]) for i in range(sub)]
    host_s = (time.perf_counter() - t0) / sub

    gpu = pkg.Detector(*det_args)
    gpu.addTemplates(srcs[:32], "warmup", masks[:32])
    gpu_ids = gpu.addTemplates(srcs[:sub], "obj", masks[:sub])
    pa, pb = host.bank.pack(["obj"], 2 * host.pyramid_levels), gpu.bank.pack(["obj"], 2 * gpu.pyramid_levels)
    identical = host_ids == gpu_ids and all(np.array_equal(pa[k], pb[k]) for k in pa)

    rows = []
    for b in args.batches:
        times = []
        for r in range(args.repeat):
            det = pkg.Detector(*det_args)
            det._native = gpu._native   # one device handle: no per-repeat handle creation in the window
            t0 = time.perf_counter()
            ids = det.addTemplates(srcs[:b], "obj", masks[:b])
            times.append(time.perf_counter() - t0)
        rows.append(dict(views=b, seconds=min(times), seconds_all=[round(t, 4) for t in times], views_per_s=b / min(times),
                         extracted=int(sum(i >= 0 for i in ids))))

    kernels = None
    if args.profile:
        import torch
        from torch.profiler import ProfilerActivity, profile
        det = pkg.Detector(*det_args)
        det._native = gpu._native
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            det.addTemplates(srcs[:256], "obj", masks[:256])
            torch.cuda.synchronize()
        acc = {}
        for e in prof.events():
            if e.device_type == torch.autograd.DeviceType.CUDA:
                name = e.name.split("(")[0].split("<")[0]
                if name.startswith("void "):
                    name = name[5:]
                acc[name] = acc.get(name, 0.0) + e.device_time
        kernels = {k: round(v / 256, 2) for k, v in sorted(acc.items(), key=lambda kv: -kv[1])}  # us per view

    name, power = card()
    out = dict(metric="template_extraction", card=name, power_limit=power, detector=args.detector, image="640x480",
               host_views=sub, host_s_per_view=host_s, host_views_per_s=1.0 / host_s, outputs_identical=bool(identical),
               host_ids_ok=int(sum(i >= 0 for i in host_ids)), gpu=rows, kernel_us_per_view=kernels)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    return 0 if identical else 1


if __name__ == "__main__":
    sys.exit(main())
