"""Probe (not a pytest file): device time of both pixel models on the synthetic batches of configs 1 and 4.

For each config one batch is decoded with b2j_batch_decode_steps, the two models alternating (reference, libjpeg,
reference, libjpeg), and the median per-stage milliseconds of every run are printed with the traffic the libjpeg model
adds (the sample plane is written by k_idct_libjpeg and read back by k_upsample_libjpeg: at least 128 bytes per block),
the card's name and its power limit. A separate profiled run per model (torch.profiler, CUDA activities) splits the device
time of one step by kernel. The libjpeg model's pixels of the first images are checked against the numpy model.
usage: python tests/libjpeg_probe.py [--steps K] [--warmup W] [--configs 1,4] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

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


def run(batch, model, steps, warmup):
    batch.set_pixel_model(model)
    batch.decode_steps(warmup)
    per, total = batch.decode_steps(steps)
    med = lambda f: float(np.median([getattr(p, f) for p in per]))   # noqa: E731
    assert not batch.status().any()
    return dict(prepass_ms=med("prepass_ms"), huffman_ms=med("huffman_ms"), idct_ms=med("idct_ms"), total_ms=med("total_ms"),
                window_ms_per_step=total / steps)


def kernel_split(batch, model, steps):
    """Device milliseconds per step of every kernel, from a profiled run of its own (tracing is kept out of the timed runs)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    batch.set_pixel_model(model)
    batch.decode_steps(2)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        batch.decode_steps(steps)
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        t = e.cuda_time_total if t is None else t
        if "b2j::" in e.key and t > 0:
            name = e.key.split("b2j::", 1)[1].split("(", 1)[0]
            out[name] = out.get(name, 0.0) + t / 1e3 / steps
    return {k: round(v, 4) for k, v in sorted(out.items(), key=lambda kv: -kv[1])}


def check_pixels(batch, files, k):
    from oracle import GATE_EXTENDED, Oracle
    import libjpeg_model
    orc = Oracle()
    batch.set_pixel_model(b2j.PIXELS_LIBJPEG)
    batch.set_output_format(b2j.OUT_RGB24)
    batch.decode()
    for i in range(k):
        assert np.array_equal(batch.pixels(i), libjpeg_model.decode_oracle(orc, files[i], GATE_EXTENDED)), i
    batch.set_output_format(b2j.OUT_BGRA)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--configs", default="1,4")
    ap.add_argument("--out")
    args = ap.parse_args()
    res = dict(card=card(), steps=args.steps, configs={})
    dec = b2j.Decoder(0)
    for cfg in [int(c) for c in args.configs.split(",")]:
        c = synth.CONFIGS[cfg]
        files = synth.config_batch(cfg, c["count"])
        batch = dec.batch(files)
        batch.upload()
        info = batch.info()
        runs = []
        for model in (b2j.PIXELS_REFERENCE, b2j.PIXELS_LIBJPEG, b2j.PIXELS_REFERENCE, b2j.PIXELS_LIBJPEG):
            r = run(batch, model, args.steps, args.warmup)
            r["model"] = "libjpeg" if model else "reference"
            runs.append(r)
            print("config %d %-9s %s" % (cfg, r["model"], json.dumps({k: round(v, 4) for k, v in r.items() if k != "model"})), flush=True)
        split = {}
        for model in (b2j.PIXELS_REFERENCE, b2j.PIXELS_LIBJPEG):
            name = "libjpeg" if model else "reference"
            try:
                split[name] = kernel_split(batch, model, 5)
            except Exception as e:   # the split is extra evidence: without a working profiler it is "not measured"
                split[name] = "not measured: %r" % (e,)
            print("config %d %-9s kernel ms per step: %s" % (cfg, name, split[name]), flush=True)
        check_pixels(batch, files, 4)
        res["configs"][cfg] = dict(images=c["count"], width=c["width"], height=c["height"], subsampling=c["subsampling"],
                                   total_blocks=info.total_blocks, sample_plane_bytes=64 * info.total_blocks,
                                   extra_traffic_bytes=128 * info.total_blocks, runs=runs, kernel_ms_per_step=split)
        batch.close()
    dec.close()
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
