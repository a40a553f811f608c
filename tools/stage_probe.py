#!/usr/bin/env python
"""Per-stage device times and counters of the match path on the bench workload (or the reference's fixture frame with the
full allScales bank), filter on / off.  Development probe: prints one JSON line per configuration.

  python tools/stage_probe.py [--templates 3115] [--frames 32] [--real] [--threshold 75]
"""
import argparse
import importlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--templates", type=int, default=3115)
    ap.add_argument("--frames", type=int, default=32)
    ap.add_argument("--threshold", type=float, default=75.0)
    ap.add_argument("--width", type=int, default=640)
    ap.add_argument("--height", type=int, default=480)
    ap.add_argument("--real", action="store_true", help="fixture frame + full allScales bank (tests/golden)")
    ap.add_argument("--filters", default="1,0")
    args = ap.parse_args()
    lib = importlib.import_module("6dpose_b200._lib")
    synth = importlib.import_module("6dpose_b200.synth")
    if args.real:
        from oracle import golden
        packed, T = golden.allscales_full_bank()
        fr = np.load(os.path.join(golden.GOLD, "frames_case1.npz"))
        frames = [[[fr["full_l%d_m%d" % (l, m)] for m in range(2)] for l in range(2)]]
    else:
        T = [4, 8]
        bank = synth.synth_bank(args.templates, num_features=150, levels=2, seed=1234, variants=35)
        packed = bank.pack(bank.class_ids(), 4)
        frames = [synth.synth_frame(args.width, args.height, levels=2, seed=1000 + i, bank=bank, plant=8, T=T)[0]
                  for i in range(min(args.frames, 16))]
    for flt in args.filters.split(","):
        os.environ["LINEMOD_B200_FILTER"] = flt
        nat = lib.NativeDetector(T)
        nat.load_bank(packed, 4)
        for q in frames[:2]:
            nat.match_quantized(q, args.threshold)
        nat.set_timing(args.frames)
        acc = {}
        for i in range(args.frames):
            nat.upload_quantized(frames[i % len(frames)])
            nat.run(args.threshold)
            for k, v in nat.counters().items():
                acc[k] = acc.get(k, 0) + v
        st = nat.stage_times_us()
        nat.set_timing(0)
        print(json.dumps({"filter": flt, "stage_us": {k: round(v, 1) for k, v in st.items()},
                          "counters_per_frame": {k: v // args.frames for k, v in acc.items()}}))
        nat.close()


if __name__ == "__main__":
    main()
