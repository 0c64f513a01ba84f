"""Probe (not a pytest file): the libjpeg pixel model's grayscale output (B2J_OUT_GRAY8, k_idct_gray) against RGB24 on the
synthetic batches of configs 1 and 4.

For each config one batch is decoded with b2j_batch_decode_steps in the libjpeg model, alternating (RGB24, GRAY8) at each
scale (1: RGB24, GRAY8, 2: RGB24, GRAY8, then the next round), and the median IDCT/colour-stage and step milliseconds of
every run are printed. Then b2j_decode_host_ex on config 1 at scale 1, host buffers to host buffers, alternating RGB24 and
GRAY8 (wall time of the whole call; the outputs are one pinned arena). The pixels of the first images are checked against
the numpy model in every format and scale. The card's name and power limit are printed with the numbers.
usage: python tests/gray_probe.py [--steps K] [--warmup W] [--rounds R] [--configs 1,4] [--scales 1,2] [--out FILE]"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

import ocljpegdecoder_b200 as b2j  # noqa: E402
import synth  # noqa: E402
from scaled_probe import card  # noqa: E402

FORMATS = {"rgb24": b2j.OUT_RGB24, "gray8": b2j.OUT_GRAY8}


def check_pixels(orc, files, outs, fmt, scale):
    """outs[i]: pixels of files[i] in fmt at 1/scale, against the numpy model."""
    from oracle import GATE_EXTENDED
    import libjpeg_gray_model
    import libjpeg_model
    model = libjpeg_gray_model.decode_oracle_gray if fmt == b2j.OUT_GRAY8 else libjpeg_model.decode_oracle
    for i, o in enumerate(outs):
        assert np.array_equal(o, model(orc, files[i], GATE_EXTENDED, scale)), (fmt, scale, i)


def device_runs(batch, scales, rounds, steps, warmup):
    batch.set_pixel_model(b2j.PIXELS_LIBJPEG)
    runs = []
    for r in range(rounds):
        for s in scales:
            for name, fmt in FORMATS.items():
                batch.set_scale(s)
                batch.set_output_format(fmt)
                batch.decode_steps(warmup)
                per, total = batch.decode_steps(steps)
                assert not batch.status().any()
                med = lambda f: float(np.median([getattr(p, f) for p in per]))   # noqa: E731
                runs.append(dict(format=name, scale=s, round=r, idct_ms=med("idct_ms"), total_ms=med("total_ms"),
                                 window_ms_per_step=total / steps, kernel_launches=batch.info().kernel_launches))
                print("  %s scale %d round %d: %s" % (name, s, r, json.dumps({k: round(v, 4) for k, v in runs[-1].items() if k.endswith("ms") or "step" in k})),
                      flush=True)
    batch.set_scale(1)
    return runs


def host_runs(dec, files, c, rounds, orc):
    n = len(files)
    w, h = c["width"], c["height"]
    arena = b2j.PinnedBuffer(n * w * h * 3)
    runs = []
    try:
        for r in range(rounds + 1):   # round 0 warms the pools and the pinned staging
            for name, fmt in FORMATS.items():
                bpp = 1 if fmt == b2j.OUT_GRAY8 else 3
                outs = [arena.address + i * w * h * bpp for i in range(n)]
                t0 = time.perf_counter()
                _, st = dec.decode_host_ex(files, outs=outs, out_format=fmt, pixel_model=b2j.PIXELS_LIBJPEG)
                ms = 1e3 * (time.perf_counter() - t0)
                assert not st.any()
                if r == 0:
                    shape = (h, w) if bpp == 1 else (h, w, 3)
                    check_pixels(orc, files, [arena.array[i * w * h * bpp:(i + 1) * w * h * bpp].reshape(shape) for i in range(2)], fmt, 1)
                    continue
                runs.append(dict(format=name, round=r, ms=ms, pixel_bytes=n * w * h * bpp))
                print("  host to host %s round %d: %.2f ms (%d pixel bytes)" % (name, r, ms, n * w * h * bpp), flush=True)
    finally:
        arena.close()
    return runs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--configs", default="1,4")
    ap.add_argument("--scales", default="1,2")
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
            for fmt in FORMATS.values():
                batch.set_scale(s)
                batch.set_output_format(fmt)
                batch.decode()
                k = min(2, len(files))
                check_pixels(orc, files, [batch.pixels(i) for i in range(k)], fmt, s)
        batch.close()
        entry = dict(images=c["count"], width=c["width"], height=c["height"], device=runs)
        if cfg == 1:
            entry["host"] = host_runs(dec, files, c, args.rounds, orc)
        res["configs"][cfg] = entry
    dec.close()
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
