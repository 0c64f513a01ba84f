"""Probe (not a pytest file): what a crop window per image (b2j_batch_set_crops) saves on the synthetic batches of configs
1 and 4.

For each config one batch is decoded with b2j_batch_decode_steps in the libjpeg model, in RGB24 and GRAY8 at scales 1
and 2, with the crops alternating on the one batch between none, a centre crop of half the area and seeded
RandomResizedCrop boxes (torchvision's defaults: scale (0.08, 1), ratio (3/4, 4/3)); the median IDCT/colour-stage and step
milliseconds of every run are printed with the output bytes and the MCUs transformed. Then
b2j_decode_host_ex / b2j_decode_host_crop in RGB24 on config 1, host buffers to host buffers, without and with the random
boxes, alternating (wall time of the whole call; the outputs are one pinned arena). The first images' crops are checked
against slices of the uncropped decode. The card's name and power limit are printed with the numbers.
usage: python tests/crop_probe.py [--steps K] [--warmup W] [--rounds R] [--configs 1,4] [--out FILE]"""
import argparse
import json
import math
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

SETTINGS = [(fmt, s) for fmt in ("OUT_RGB24", "OUT_GRAY8") for s in (1, 2)]


def random_resized_boxes(frames, seed):
    """torchvision's RandomResizedCrop.get_params (scale (0.08, 1), ratio (3/4, 4/3)), seeded, per (w, h)."""
    rng = np.random.default_rng(seed)
    out = []
    for w, h in frames:
        area = w * h
        for _ in range(10):
            a = area * rng.uniform(0.08, 1.0)
            r = math.exp(rng.uniform(math.log(3 / 4), math.log(4 / 3)))
            cw, ch = int(round(math.sqrt(a * r))), int(round(math.sqrt(a / r)))
            if 0 < cw <= w and 0 < ch <= h:
                out.append((int(rng.integers(0, w - cw + 1)), int(rng.integers(0, h - ch + 1)), cw, ch))
                break
        else:   # torchvision's fallback; with these ratios and a frame of ratio 3/4..4/3 it is the whole frame
            cw, ch = w, h
            out.append(((w - cw) // 2, (h - ch) // 2, cw, ch))
    return out


def centre_boxes(frames):
    """Half the area: sides / sqrt(2), centred."""
    out = []
    for w, h in frames:
        cw, ch = max(1, round(w / math.sqrt(2))), max(1, round(h / math.sqrt(2)))
        out.append(((w - cw) // 2, (h - ch) // 2, cw, ch))
    return out


def mcus_of(batch, boxes, scale, halo):
    """MCUs the crop tile list transforms (the window's plus `halo` around them), against the image's."""
    got = whole = 0
    for i, d in enumerate(batch.descs):
        if boxes is None:
            got += d.mcu_count
        else:
            x, y, w, h = boxes[i]
            mw, mh = d.mcu_width // scale, d.mcu_height // scale
            c = min((x + w - 1) // mw + halo, d.mcu_count_w - 1) - max(x // mw - halo, 0) + 1
            r = min((y + h - 1) // mh + halo, d.mcu_count_h - 1) - max(y // mh - halo, 0) + 1
            got += c * r
        whole += d.mcu_count
    return got, whole


def device_runs(batch, rounds, steps, warmup):
    runs = []
    for r in range(rounds):
        for fmt_name, scale in SETTINGS:
            batch.set_output_format(getattr(b2j, fmt_name))
            batch.set_scale(scale)
            frames = [batch.crop_frame(i) for i in range(batch.n)]
            crops = {"none": None, "centre_half": centre_boxes(frames), "random_resized": random_resized_boxes(frames, 7)}
            for cname, boxes in crops.items():
                batch.set_crops(boxes)
                batch.decode_steps(warmup)
                per, total = batch.decode_steps(steps)
                assert not batch.status().any()
                med = lambda f: float(np.median([getattr(p, f) for p in per]))   # noqa: E731
                out_bytes = sum(batch.pixels_device(i)[1] for i in range(batch.n))
                halo = 0 if fmt_name == "OUT_GRAY8" or scale == 8 else 1
                mcus, whole = mcus_of(batch, boxes, scale, halo)
                runs.append(dict(format=fmt_name, scale=scale, crops=cname, round=r, idct_ms=med("idct_ms"), total_ms=med("total_ms"),
                                 window_ms_per_step=total / steps, output_bytes=out_bytes, mcus_transformed=mcus, mcus_whole=whole))
                print("  %s 1/%d %s round %d: %s" % (fmt_name, scale, cname, r, json.dumps(
                    {k: (round(v, 4) if isinstance(v, float) else v) for k, v in runs[-1].items() if k not in ("format", "scale", "crops", "round")})),
                    flush=True)
                if r == 0:
                    check(batch, boxes, min(3, batch.n))
    batch.set_crops(None)
    return runs


def check(batch, boxes, k):
    """The first k images of the last decode against slices of an uncropped decode."""
    got = [batch.pixels(i) for i in range(k)]
    if boxes is None:
        return
    batch.set_crops(None)
    batch.decode()
    for i in range(k):
        x, y, w, h = boxes[i]
        assert np.array_equal(got[i], batch.pixels(i)[y:y + h, x:x + w]), i
    batch.set_crops(boxes)


def host_runs(dec, files, c, rounds):
    n = len(files)
    w, h = c["width"], c["height"]
    boxes = random_resized_boxes([b2j.crop_frame(b2j.parse_header(f)[1]) for f in files], 11)
    arena = b2j.PinnedBuffer(n * w * h * 3)
    runs = []
    try:
        for r in range(rounds + 1):   # round 0 warms the pools and the pinned staging
            for cname in ("none", "random_resized"):
                crops = None if cname == "none" else boxes
                sizes = [w * h * 3 if crops is None else bx[2] * bx[3] * 3 for bx in (crops or [None] * n)]
                offs = np.cumsum([0] + sizes)
                outs = [arena.address + int(o) for o in offs[:-1]]
                t0 = time.perf_counter()
                _, st = dec.decode_host_ex(files, outs=outs, out_format=b2j.OUT_RGB24, pixel_model=b2j.PIXELS_LIBJPEG, crops=crops)
                ms = 1e3 * (time.perf_counter() - t0)
                assert not st.any()
                if r == 0:
                    continue
                runs.append(dict(crops=cname, round=r, ms=ms, d2h_bytes=int(offs[-1])))
                print("  host to host RGB24 %s round %d: %.2f ms, %d bytes back" % (cname, r, ms, offs[-1]), flush=True)
    finally:
        arena.close()
    return runs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--configs", default="1,4")
    ap.add_argument("--out")
    args = ap.parse_args()
    res = dict(card=card(), steps=args.steps, rounds=args.rounds, configs={})
    print("card:", res["card"], flush=True)
    dec = b2j.Decoder(0)
    for cfg in [int(c) for c in args.configs.split(",")]:
        c = synth.CONFIGS[cfg]
        files = synth.config_batch(cfg, c["count"])
        print("config %d: %d x %dx%d %s" % (cfg, c["count"], c["width"], c["height"], c["subsampling"]), flush=True)
        batch = dec.batch(files)
        batch.upload()
        batch.set_pixel_model(b2j.PIXELS_LIBJPEG)
        entry = dict(images=c["count"], width=c["width"], height=c["height"], device=device_runs(batch, args.rounds, args.steps, args.warmup))
        batch.close()
        if cfg == 1:
            entry["host"] = host_runs(dec, files, c, args.rounds)
        res["configs"][cfg] = entry
    dec.close()
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
