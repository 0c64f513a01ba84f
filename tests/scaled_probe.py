"""Probe (not a pytest file): the libjpeg pixel model's scaled decode (b2j_batch_set_scale) on the synthetic batches of
configs 1 and 4.

For each config one batch is decoded with b2j_batch_decode_steps in the libjpeg model, the scales alternating
(1, 2, 4, 8, 1, 2, 4, 8, ...), and the median IDCT/colour-stage milliseconds of every run are printed. Then
b2j_decode_host_ex in RGB24 on config 1, host buffers to host buffers, alternating scales 1 and 2 (wall time of the whole
call; the outputs are one pinned arena). Every run's pixels of the first images are checked against the numpy model.
The card's name and power limit are printed with the numbers.
usage: python tests/scaled_probe.py [--steps K] [--warmup W] [--rounds R] [--configs 1,4] [--scales 1,2,4,8]
                                    [--host-scales 1,2] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

import ocljpegdecoder_b200 as b2j  # noqa: E402
import synth  # noqa: E402


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True)
    return out.stdout.strip() if out.returncode == 0 else "unknown"


def check_pixels(orc, files, outs, scale, k):
    """outs[i]: RGB24 pixels of files[i] at 1/scale; the first k against the numpy model."""
    from oracle import GATE_EXTENDED
    import libjpeg_model
    for i in range(k):
        assert np.array_equal(outs[i], libjpeg_model.decode_oracle(orc, files[i], GATE_EXTENDED, scale)), (scale, i)


def device_runs(batch, scales, rounds, steps, warmup):
    batch.set_pixel_model(b2j.PIXELS_LIBJPEG)
    batch.set_output_format(b2j.OUT_RGB24)
    runs = []
    for r in range(rounds):
        for s in scales:
            batch.set_scale(s)
            batch.decode_steps(warmup)
            per, total = batch.decode_steps(steps)
            assert not batch.status().any()
            med = lambda f: float(np.median([getattr(p, f) for p in per]))   # noqa: E731
            runs.append(dict(scale=s, round=r, idct_ms=med("idct_ms"), total_ms=med("total_ms"), window_ms_per_step=total / steps))
            print("  scale %d round %d: %s" % (s, r, json.dumps({k: round(v, 4) for k, v in runs[-1].items() if k.endswith("ms") or "step" in k})),
                  flush=True)
    batch.set_scale(1)
    return runs


def host_runs(dec, files, c, scales, rounds, orc):
    n = len(files)
    full = c["width"] * c["height"] * 3
    arena = b2j.PinnedBuffer(n * full)
    runs = []
    try:
        for r in range(rounds + 1):   # round 0 warms the pools and the pinned staging
            for s in scales:
                w, h = -(-c["width"] // s), -(-c["height"] // s)
                outs = [arena.address + i * w * h * 3 for i in range(n)]
                t0 = time.perf_counter()
                _, st = dec.decode_host_ex(files, outs=outs, out_format=b2j.OUT_RGB24, pixel_model=b2j.PIXELS_LIBJPEG, scale=s)
                ms = 1e3 * (time.perf_counter() - t0)
                assert not st.any()
                if r == 0:
                    check_pixels(orc, files, [arena.array[i * w * h * 3:(i + 1) * w * h * 3].reshape(h, w, 3) for i in range(2)], s, 2)
                    continue
                runs.append(dict(scale=s, round=r, ms=ms, pixel_bytes=n * w * h * 3))
                print("  host to host RGB24 scale %d round %d: %.2f ms (%d pixel bytes)" % (s, r, ms, n * w * h * 3), flush=True)
    finally:
        arena.close()
    return runs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--configs", default="1,4")
    ap.add_argument("--scales", default="1,2,4,8")
    ap.add_argument("--host-scales", default="1,2")
    ap.add_argument("--out")
    args = ap.parse_args()
    from oracle import Oracle
    orc = Oracle()
    scales = [int(s) for s in args.scales.split(",")]
    res = dict(card=card(), steps=args.steps, rounds=args.rounds, configs={})
    print("card:", res["card"], flush=True)
    dec = b2j.Decoder(0)
    for cfg in [int(c) for c in args.configs.split(",")]:
        c = synth.CONFIGS[cfg]
        files = synth.config_batch(cfg, c["count"])
        print("config %d: %d x %dx%d %s" % (cfg, c["count"], c["width"], c["height"], c["subsampling"]), flush=True)
        batch = dec.batch(files)
        batch.upload()
        runs = device_runs(batch, scales, args.rounds, args.steps, args.warmup)
        for s in scales:
            batch.set_scale(s)
            batch.decode()
            k = min(2, len(files))   # config 3 is one image
            check_pixels(orc, files, [batch.pixels(i) for i in range(k)], s, k)
        batch.close()
        entry = dict(images=c["count"], width=c["width"], height=c["height"], device=runs)
        if cfg == 1 and args.host_scales:
            entry["host"] = host_runs(dec, files, c, [int(s) for s in args.host_scales.split(",")], args.rounds, orc)
        res["configs"][cfg] = entry
    dec.close()
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
