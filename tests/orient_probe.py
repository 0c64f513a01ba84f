"""Probe (not a pytest file): the cost of EXIF orientation (b2j_batch_set_orientations, k_orient) on the synthetic batches
of configs 1 and 4.

For each config one batch is decoded with b2j_batch_decode_steps in three settings -- the libjpeg model in RGB24 and in
GRAY8, the reference model in BGRA -- with the orientation codes alternating between all 1, all 6 and half 6 (every
other image), and the median IDCT/colour-stage (which includes the orientation pass) and step milliseconds of every run
are printed. Then k_orient alone, with every code 6: its device time per step from torch.profiler, the bytes it moves
(each oriented image read once and written once) and their share of the HGX B200 data sheet's 7.7 TB/s. Last,
b2j_decode_host_ex in RGB24 on config 1, host buffers to host buffers, with exif_orientation 0 and 1 alternating, on the
config's files with an Exif APP1 of orientation 6 put behind SOI (wall time of the whole call; the outputs are one pinned
arena). Every oriented result of the first images is checked against the transform of the unoriented decode. The card's
name and power limit are printed with the numbers.
usage: python tests/orient_probe.py [--steps K] [--warmup W] [--rounds R] [--configs 1,4] [--out FILE]"""
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
from test_orientation_parse import exif_app1, orient, with_segments  # noqa: E402

SETTINGS = {"libjpeg_rgb24": (b2j.PIXELS_LIBJPEG, b2j.OUT_RGB24), "libjpeg_gray8": (b2j.PIXELS_LIBJPEG, b2j.OUT_GRAY8),
            "reference_bgra": (b2j.PIXELS_REFERENCE, b2j.OUT_BGRA)}
PEAK_BYTES_PER_S = 7.7e12


def code_sets(n):
    return {"all1": None, "all6": np.full(n, 6, np.uint8), "half6": np.array([6 if i % 2 else 1 for i in range(n)], np.uint8)}


def check(batch, codes, k):
    """The first k images of a decode with `codes` against the transform of an unoriented decode."""
    batch.set_orientations(None)
    batch.decode()
    plain = [batch.pixels(i) for i in range(k)]
    batch.set_orientations(codes)
    batch.decode()
    for i in range(k):
        c = 1 if codes is None else int(codes[i])
        p = plain[i]
        want = np.stack([orient(q, c) for q in p]) if batch.out_format == b2j.OUT_RGB_PLANAR else orient(p, c)
        assert np.array_equal(batch.pixels(i), want), (batch.out_format, c, i)


def device_runs(batch, rounds, steps, warmup):
    runs = []
    sets = code_sets(batch.n)
    for r in range(rounds):
        for name, (model, fmt) in SETTINGS.items():
            batch.set_pixel_model(model)
            batch.set_output_format(fmt)
            for cname, codes in sets.items():
                batch.set_orientations(codes)
                batch.decode_steps(warmup)
                per, total = batch.decode_steps(steps)
                assert not batch.status().any()
                med = lambda f: float(np.median([getattr(p, f) for p in per]))   # noqa: E731
                runs.append(dict(setting=name, codes=cname, round=r, idct_ms=med("idct_ms"), total_ms=med("total_ms"),
                                 window_ms_per_step=total / steps, kernel_launches=batch.info().kernel_launches))
                print("  %s %s round %d: %s" % (name, cname, r, json.dumps({k: round(v, 4) for k, v in runs[-1].items() if k.endswith("ms") or "step" in k})),
                      flush=True)
    for name, (model, fmt) in SETTINGS.items():
        batch.set_pixel_model(model)
        batch.set_output_format(fmt)
        for codes in sets.values():
            check(batch, codes, min(3, batch.n))
    batch.set_orientations(None)
    return runs


def kernel_time(batch, out_dir, steps):
    """Per setting: k_orient's device milliseconds per step with every code 6 (torch.profiler), its bytes and share of peak."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    res = {}
    for name, (model, fmt) in SETTINGS.items():
        batch.set_pixel_model(model)
        batch.set_output_format(fmt)
        batch.set_orientations(np.full(batch.n, 6, np.uint8))
        batch.decode_steps(2)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            batch.decode_steps(steps)
        us = [e.time_range.elapsed_us() for e in prof.events() if "k_orient" in e.name]
        assert len(us) == steps, (name, len(us))
        ms = float(np.median(us)) / 1e3
        moved = 2 * sum(batch.pixels_device(i)[1] for i in range(batch.n))
        res[name] = dict(k_orient_ms=ms, bytes=moved, gb_per_s=moved / ms / 1e6, share_of_7_7_tb_s=moved / (ms * 1e-3) / PEAK_BYTES_PER_S)
        print("  k_orient %s: %s" % (name, json.dumps({k: round(v, 4) for k, v in res[name].items()})), flush=True)
        if out_dir:
            prof.export_chrome_trace(os.path.join(out_dir, "orient_%s.json" % name))
    batch.set_orientations(None)
    return res


def host_runs(dec, files, c, rounds):
    n = len(files)
    w, h = c["width"], c["height"]
    tagged = [with_segments(f, exif_app1(6)) for f in files]
    arena = b2j.PinnedBuffer(n * w * h * 3)
    runs = []
    try:
        for r in range(rounds + 1):   # round 0 warms the pools and the pinned staging
            for on in (0, 1):
                outs = [arena.address + i * w * h * 3 for i in range(n)]
                t0 = time.perf_counter()
                _, st = dec.decode_host_ex(tagged, outs=outs, out_format=b2j.OUT_RGB24, pixel_model=b2j.PIXELS_LIBJPEG, exif_orientation=bool(on))
                ms = 1e3 * (time.perf_counter() - t0)
                assert not st.any()
                if r == 0:
                    continue
                runs.append(dict(exif_orientation=on, round=r, ms=ms))
                print("  host to host RGB24 exif_orientation=%d round %d: %.2f ms" % (on, r, ms), flush=True)
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
    out_dir = os.path.dirname(os.path.abspath(args.out)) if args.out else None
    dec = b2j.Decoder(0)
    for cfg in [int(c) for c in args.configs.split(",")]:
        c = synth.CONFIGS[cfg]
        files = synth.config_batch(cfg, c["count"])
        print("config %d: %d x %dx%d %s" % (cfg, c["count"], c["width"], c["height"], c["subsampling"]), flush=True)
        batch = dec.batch(files)
        batch.upload()
        entry = dict(images=c["count"], width=c["width"], height=c["height"], device=device_runs(batch, args.rounds, args.steps, args.warmup))
        entry["k_orient"] = kernel_time(batch, out_dir, args.steps)
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
