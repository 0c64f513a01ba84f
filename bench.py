#!/usr/bin/env python
"""bench.py -- benchmark of the B200-native baseline-JPEG decode path, one JSON line per run.

    python bench.py --gpus N --steps K --warmup W [--config C]     # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...        # the reference's CPU path, host cores

--config selects a BASELINE.json workload (default 1, the one the headline metric is quoted on):
    1  256 x 1920x1080 4:2:0 q90, restart interval 16 MCUs      per GPU (weak scaling: distinct images per rank)
    2  64 x 3840x2160 4:4:4 q95, no restart markers              per GPU (weak)
    3  one 7680x4320 4:2:2 q85 image, no restart markers         per GPU (weak: N distinct images on N GPUs)
    4  8192 x 500x375 4:2:0 q75, no restart markers              in total, sharded by compressed bytes over the
                                                                 ranks (strong scaling, sharding.shard_by_bytes)
A "step" is one pass of the hot path (pre-pass -> entropy decode -> IDCT/colour) over the rank's batch.

  value      whole-job MPix/s with the compressed batch already resident in HBM; K steps timed with
             CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks.
  e2e        same metric through b2j_decode_host(): host JPEG bytes in, host (pinned) BGRA out; header
             parsing, staging, H2D, decode and D2H are all inside the timed region.
  roofline   dominant stage: algorithmic bytes per launch / its mean duration (CUDA events inside the timed
             region) against the measured HBM copy bandwidth in MEASURED_PEAKS.json; frac_pipeline is the
             whole step (the north-star fraction, SURVEY.md 8d).
  parity     outside the timed region: the batch's coefficients and pixels against the unmodified reference
             (oracle/_ref) where it decodes the file, else against the non-strict oracle port.
  cpu_baseline  the reference CPU path on the host cores of this box, bounded sample. The parity check, this
             leg and --impl reference are the only places oracle/ is executed by this file.

--dump-outputs DIR writes what the last timed step computed (see dump_outputs) so that two builds can be compared
output for output: the inputs are synthetic and seeded, identical from run to run for the same arguments.
"""
import argparse
import hashlib
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True      # the benchmark leaves the tree as it found it (which may be read-only)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

FALLBACK_HBM_GBS = 6650.0

# index -> (tests/synth.py config, images per rank or in total, scaling, metric, workload)
WORKLOADS = {
    1: dict(count=256, scaling="weak", metric="MPix/s decoded (1080p 4:2:0 q90 batch)",
            workload="256 synthetic 1920x1080 4:2:0 baseline q90 JPEGs, restart interval 16 MCUs (BASELINE configs[1])"),
    2: dict(count=64, scaling="weak", metric="MPix/s decoded (4K 4:4:4 q95 batch, no restart markers)",
            workload="64 synthetic 3840x2160 4:4:4 baseline q95 JPEGs, no restart markers (BASELINE configs[2])"),
    3: dict(count=1, scaling="weak", metric="MPix/s decoded (one 8K 4:2:2 q85 image per GPU)",
            workload="one synthetic 7680x4320 4:2:2 baseline q85 JPEG per GPU, no restart markers (BASELINE configs[3])"),
    4: dict(count=8192, scaling="strong", metric="MPix/s decoded (8192 x 500x375 4:2:0 q75, sharded by image)",
            workload="8192 synthetic 500x375 4:2:0 baseline q75 JPEGs, no restart markers, sharded over the GPUs (BASELINE configs[4])"),
}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def common_config(cfg):
    """The `config` object: identical in both arms (the driver compares them)."""
    w = WORKLOADS[cfg]
    return {"workload": w["workload"], "baseline_config": cfg,
            "images": w["count"], "images_are": "per GPU" if w["scaling"] == "weak" else "in total"}


# ----------------------------------------------------------------------------------------------
# CPU side (reference arm / cpu_baseline / parity digests): runs before any CUDA context exists (fork-safe).
_W = {}


def _cpu_worker_init(files):
    from oracle import Oracle, Reference, reference_available
    _W["ref"] = Reference() if reference_available() else None
    _W["orc"] = Oracle()
    _W["files"] = files


def _cpu_decode_chunk(idx):
    """Decodes files[i] for i in idx; returns [(pixels or 0, huffman seconds, idct+colour seconds)]."""
    out = []
    for i in idx:
        data = _W["files"][i]
        if _W["ref"] is not None:
            ok, info, _, _, ts = _W["ref"].decode(data, skip_gate=_W["skip"], want_pixels=True)
            out.append(((info.width * info.height if ok else 0), ts[0], ts[1]))
        else:
            t0 = time.perf_counter()
            rc, img, _, _ = _W["orc"].decode(data)   # strict mode: fails where the reference would
            out.append(((img.width * img.height if rc == 0 else 0), time.perf_counter() - t0, 0.0))
    return out


def _cpu_digest_chunk(idx):
    """Parity digests: for files[i], (kind, coef sha256, pixel sha256) from the reference where it decodes the
    file, else from the oracle port in its non-strict mode (the intended behaviour, DESIGN.md)."""
    out = []
    for i in idx:
        data = _W["files"][i]
        kind, coef, bgra = None, None, None
        if _W["ref"] is not None:
            ok, _, coef, bgra, _ = _W["ref"].decode(data, skip_gate=_W["skip"], want_pixels=True)
            kind = "reference" if ok else None
        if kind is None:
            _W["orc"].set_strict(False)
            rc, _, coef, bgra = _W["orc"].decode(data)
            _W["orc"].set_strict(True)
            kind = "oracle" if rc == 0 else "failed"
        if kind == "failed":
            out.append((kind, "", ""))
        else:
            out.append((kind, hashlib.sha256(coef.tobytes()).hexdigest(), hashlib.sha256(bgra.tobytes()).hexdigest()))
    return out


class CpuPool:
    def __init__(self, files, cores, skip_gate):
        import multiprocessing as mp
        self.cores = cores
        self.n = len(files)
        _W["skip"] = skip_gate
        self.pool = mp.get_context("fork").Pool(cores, initializer=_cpu_worker_init, initargs=(files,))

    def _chunks(self, idx, per_core=1):
        """Contiguous index chunks, `per_core` per worker at least 4 long where the list allows it."""
        n_chunks = max(1, min(len(idx) // 4 or 1, self.cores * per_core))
        size = (len(idx) + n_chunks - 1) // n_chunks
        return [idx[k:k + size] for k in range(0, len(idx), size)]

    def decode(self, idx):
        """One pass over files[idx] on all workers: (MPix/s wall, wall s, per-file results in order)."""
        t0 = time.perf_counter()
        parts = self.pool.map(_cpu_decode_chunk, self._chunks(idx, 2), chunksize=1)
        dt = time.perf_counter() - t0
        res = [r for p in parts for r in p]
        return sum(r[0] for r in res) / dt / 1e6, dt, res

    def digests(self, idx):
        parts = self.pool.map(_cpu_digest_chunk, self._chunks(idx, 4), chunksize=1)
        return [r for p in parts for r in p]

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_kind():
    from oracle import reference_available
    return "reference" if reference_available() else "port"


def usable_for_cpu(pool, idx):
    """The reference loses an RSTn whose FF is the last byte of one of its 2 KiB reads (decoder.cpp:118-131,
    DESIGN.md) and then aborts the image: about 1 in 5 of the 1080p RI=16 images. Such images are left out of
    the CPU timing (an aborted decode would flatter it). One screening pass, which also warms the workers."""
    _, _, res = pool.decode(idx)
    good = [i for i, r in zip(idx, res) if r[0]]
    return good, len(idx) - len(good)


def cpu_sample_size(cfg, n_files):
    """How many files of the batch one CPU pass decodes -- the same in the reference arm and in the cpu_baseline leg:
    the whole 256-image batch of config 1, about 1.2 GPix (a second or two on 16 cores) of the larger ones."""
    import synth
    npix = synth.CONFIGS[cfg]["width"] * synth.CONFIGS[cfg]["height"]
    return n_files if cfg == 1 else max(1, min(n_files, int(1.2e9 // npix)))


def build_oracle_only():
    import subprocess
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "all"], stdout=sys.stderr)


def reference_arm(args, rank, world):
    """The reference's own CPU path (oracle/_ref, else the oracle port) on every host core, on the same config:
    every step decodes every reference-decodable file of the rank-0 batch (bounded for the large configs)."""
    if rank != 0:
        return 0
    import synth
    build_oracle_only()          # the checker only: libb2j.so is neither built nor loaded by this arm
    w = WORKLOADS[args.config]
    cores = os.cpu_count() or 1
    files = synth.config_batch(args.config, w["count"])
    npix = synth.CONFIGS[args.config]["width"] * synth.CONFIGS[args.config]["height"]
    take = cpu_sample_size(args.config, len(files))
    pool = CpuPool(files, cores, skip_gate=(args.config == 3))
    good, bad = usable_for_cpu(pool, list(range(take)))
    for _ in range(args.warmup):
        pool.decode(good[:max(cores, 1)])
    t_total, pix_total, t_h, t_m = 0.0, 0.0, 0.0, 0.0
    for _ in range(args.steps):
        mp, dt, res = pool.decode(good)
        t_total += dt
        pix_total += mp * dt * 1e6
        t_h += sum(r[1] for r in res)
        t_m += sum(r[2] for r in res)
    pool.close()
    value = pix_total / t_total / 1e6
    sample = ("every step: the %d files of the first %d of the batch that the reference decodes (it aborts on %d, lost RSTn at a "
              "2 KiB read boundary), one process per host core, contiguous chunks" % (len(good), take, bad))
    line = {
        "impl": "reference", "metric": w["metric"], "value": round(value, 3), "unit": "MPix/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * t_total / args.steps, 3),
        "higher_is_better": True, "scaling": w["scaling"], "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": common_config(args.config),
        "cpu_baseline": {"value": round(value, 3), "unit": "MPix/s", "cores": cores, "kind": cpu_kind(), "sample": sample,
                         "stage_timer_mpix_s": round(pix_total / (t_h + t_m) * cores / 1e6, 3) if (t_h + t_m) > 0 else None,
                         "huffman_share": round(t_h / (t_h + t_m), 3) if (t_h + t_m) > 0 else None},
        "e2e": {"value": round(value, 3), "unit": "MPix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ----------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed regions run."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.stop_flag = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:   # NVML missing: report nothing rather than guess
            self.err = str(e)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag.is_set():
            try:
                util = nv.nvmlDeviceGetUtilizationRates(self.h).gpu
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((mhz, util))
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "NVML unavailable"}
        busy = [m for m, u in self.samples if u > 0] or [m for m, _ in self.samples]
        return {"sm_mhz": int(statistics.median(busy)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def measured_traffic(cfg, kernel):
    """DRAM bytes per launch of `kernel` from the newest committed ncu capture of this config, or (None, None)."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                d = json.load(f)
            key = kernel if cfg == 1 else "cfg%d:%s" % (cfg, kernel)
            if key in d:
                return int(d[key]), "committed ncu --set full capture (profiles/%s), not measured in this run" % name
        except Exception:
            pass
    return None, None


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy bandwidth)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md, MEASURED_PEAKS.json absent)"


def rank_files(cfg, rank, world, dist):
    """The JPEGs this rank decodes, and how many images the whole job holds."""
    import synth
    from ocljpegdecoder_b200 import sharding
    w = WORKLOADS[cfg]
    if w["scaling"] == "weak":
        return synth.config_batch(cfg, w["count"], first=rank * w["count"]), w["count"] * world, None
    # strong scaling: one image list, cut into contiguous slices of similar compressed size
    n = w["count"]
    lo, hi = sharding.shard_range(n, rank, world)
    mine = dict(zip(range(lo, hi), synth.config_batch(cfg, hi - lo, first=lo)))
    if world == 1:
        return [mine[i] for i in range(n)], n, [(0, n)]
    sizes = [None] * world
    dist.all_gather_object(sizes, [len(mine[i]) for i in range(lo, hi)])
    flat = [s for part in sizes for s in part]
    cuts = sharding.shard_by_bytes(flat, world)
    a, b = cuts[rank]
    missing = [i for i in range(a, b) if i not in mine]
    for i in missing:          # the few images next to a slice border that moved
        mine[i] = synth.config_jpeg(cfg, i)
    return [mine[i] for i in range(a, b)], n, cuts


def parity_indices(cfg, n, world):
    """Which images of the rank's batch are compared with the reference outside the timed region."""
    if cfg == 1:
        return list(range(n)) if world == 1 else list(range(0, n, 8))      # all 256 on one GPU
    if cfg == 2:
        return list(range(0, n, 8)) if n >= 8 else list(range(n))          # >= 10 % of the 4K batch
    if cfg == 3:
        return list(range(n))
    step = 8 if world == 1 else 32
    return list(range(0, n, step))                                          # >= 10 % of the small images


def check_parity(batch, idx, digests):
    """Compares images idx of the decoded batch with the CPU digests. Returns the `parity` object."""
    import numpy as np
    from concurrent.futures import ThreadPoolExecutor
    out = {"images": len(idx), "vs_reference": 0, "vs_oracle": 0, "coef_mismatches": 0, "pixel_mismatch_frac": 0.0,
           "max_abs": 0, "images_differing": 0}

    def sha(a):
        return hashlib.sha256(a.tobytes()).hexdigest()
    # the device reads are serial (one expansion buffer per batch), the hashing runs behind them on threads
    with ThreadPoolExecutor(min(16, os.cpu_count() or 1)) as tp:
        jobs = [(tp.submit(sha, batch.coefs(i)), tp.submit(sha, batch.pixels(i))) for i in idx]
        got = [(a.result(), b.result()) for a, b in jobs]
    bad, npix, nbadpix = [], 0, 0
    for i, (kind, cs, ps), (hc, hp) in zip(idx, digests, got):
        if kind == "failed":
            out["images"] -= 1
            continue
        out["vs_reference" if kind == "reference" else "vs_oracle"] += 1
        npix += batch.descs[i].width * batch.descs[i].height
        if hc != cs or hp != ps:
            bad.append(i)
    if bad:
        # slow path, only ever taken on a failure: count what differs
        from oracle import Oracle
        orc = Oracle()
        orc.set_strict(False)
        for i in bad:
            rc, _, coef, bgra = orc.decode(batch.files[i])
            if rc != 0:
                continue
            out["coef_mismatches"] += int((coef != batch.coefs(i)).sum())
            d = np.abs(bgra.astype(np.int16) - batch.pixels(i).astype(np.int16)).max(axis=2)
            nbadpix += int((d > 0).sum())
            out["max_abs"] = max(out["max_abs"], int(d.max()))
        out["images_differing"] = len(bad)
        out["pixel_mismatch_frac"] = nbadpix / max(npix, 1)
    return out


DUMP_VALUES = 4 << 20      # values per dumped array and job: 16 MiB of pixels and 32 MiB of coefficients


def dump_outputs(out_dir, batch, rank, world):
    """Writes the batch's outputs as a caller reads them after the last timed step, flat and image after image: the
    BGRA pixels (uint8 [H, W, 4] per image) to pixels.npy as float32 and the coefficient tap (int32 [blocks, 64] per
    image) to coefs.npy as float64 (with 16-bit quantisers a coefficient can exceed what float32 holds exactly). An
    image whose output is larger than its share of DUMP_VALUES contributes a fixed sample: flat indices drawn by numpy's
    default_rng seeded with (image index, array number), sorted. With several ranks every rank writes its own files
    (suffix _rank<r>) and the share shrinks with the rank count."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = max(1, DUMP_VALUES // (world * batch.n))
    suffix = "_rank%d" % rank if world > 1 else ""
    for k, (name, read, dtype) in enumerate((("pixels", batch.pixels, np.float32), ("coefs", batch.coefs, np.float64))):
        parts = []
        for i in range(batch.n):
            a = read(i).reshape(-1)
            if a.size > share:
                a = a[np.sort(np.random.default_rng((i, k)).integers(0, a.size, share))]
            parts.append(a.astype(dtype))
        np.save(os.path.join(out_dir, name + suffix + ".npy"), np.concatenate(parts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b2j", choices=["b2j", "reference"])
    ap.add_argument("--config", type=int, default=1, choices=sorted(WORKLOADS))
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--cpu-sample", type=int, default=0, help="images in the cpu_baseline sample (0 = about 8 per core)")
    ap.add_argument("--no-parity", action="store_true", help="skip the comparison with the reference (measurement scripts)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the pixels and coefficients of the last timed step to DIR/pixels.npy and DIR/coefs.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b2j" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return reference_arm(args, rank, world)

    import numpy as np
    import synth
    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    cfg = args.config
    w = WORKLOADS[cfg]

    # Strong scaling exchanges the compressed sizes of the images before the slices are final: a short-lived gloo
    # group does that on the host. The NCCL group is created after the CPU pools have forked (no CUDA before a fork).
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if w["scaling"] == "strong":
            dist.init_process_group("gloo")

    # ---- inputs, the CPU baseline and the parity digests: all before CUDA is touched (the pools fork)
    t0 = time.time()
    files, n_job, cuts = rank_files(cfg, rank, world, dist)
    if world > 1 and w["scaling"] == "strong":
        dist.destroy_process_group()
    log("[rank %d] config %d: %d JPEGs, %.1f MB, %.1f s" % (rank, cfg, len(files), sum(map(len, files)) / 1e6, time.time() - t0))
    cpu, digests, pidx = None, None, []
    cores = os.cpu_count() or 1
    pool_cores = cores if world == 1 else max(1, cores // world)
    if not args.no_parity or (rank == 0 and world == 1):
        pool = CpuPool(files, pool_cores, skip_gate=(cfg == 3))
        if rank == 0 and world == 1:
            npix = synth.CONFIGS[cfg]["width"] * synth.CONFIGS[cfg]["height"]
            n_cpu = args.cpu_sample or cpu_sample_size(cfg, len(files))
            good, bad = usable_for_cpu(pool, list(range(n_cpu)))        # also warms the workers
            mp_all, dt_all, res = max((pool.decode(good) for _ in range(2)), key=lambda r: r[0])   # the better of two passes
            th, tm = sum(r[1] for r in res), sum(r[2] for r in res)
            cpu = {"value": round(mp_all, 3), "unit": "MPix/s", "cores": cores, "kind": cpu_kind(),
                   "sample": "%d of the %d images (the sample of the reference arm), one process per host core, better of two passes, %.2f s wall; "
                             "the reference aborts on %d of the first %d (lost RSTn at a 2 KiB read boundary), those are excluded" % (len(good), len(files), dt_all, bad, n_cpu),
                   "one_core_mpix_s": round(len(good) * npix / (th + tm) / 1e6, 3) if (th + tm) > 0 else None,
                   "stage_timer_mpix_s": round(len(good) * npix / (th + tm) * cores / 1e6, 3) if (th + tm) > 0 else None,
                   "huffman_share": round(th / (th + tm), 3) if (th + tm) > 0 else None}
            log("[cpu] %s" % cpu)
        if not args.no_parity:
            t0 = time.time()
            pidx = parity_indices(cfg, len(files), world)
            digests = pool.digests(pidx)
            log("[rank %d] parity digests of %d images on %d cores: %.1f s" % (rank, len(pidx), pool_cores, time.time() - t0))
        pool.close()

    import torch
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    if rank != 0:
        ge.build()
    import ocljpegdecoder_b200 as b2j

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    dec = b2j.Decoder(local_rank)
    batch = dec.batch(files)
    info = batch.info()
    batch.upload()
    batch.sync()

    sampler = ClockSampler(local_rank)
    sampler.start()

    # ---- device-resident timing: W warm-up steps, then exactly K steps
    batch.decode_steps(args.warmup)
    barrier()
    per, total_ms = batch.decode_steps(args.steps)
    barrier()
    st = batch.status()
    assert not st.any(), "decode status not clean: %s" % st[st != 0][:8]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, batch, rank, world)
    ms_per_step = allmax(total_ms) / args.steps
    pix_job = allsum(float(info.total_pixels))
    value = pix_job / (ms_per_step * 1e-3) / 1e6
    stage = {k: statistics.mean(getattr(p, k) for p in per) for k in ("prepass_ms", "huffman_ms", "idct_ms", "total_ms")}
    sync_stats = batch.sync_stats().tolist() if cfg != 1 else None

    # ---- parity of this batch against the reference, outside the timed region
    parity = None
    if digests is not None:
        parity = check_parity(batch, pidx, digests)
        for k in ("images", "vs_reference", "vs_oracle", "coef_mismatches", "images_differing"):
            parity[k] = int(allsum(float(parity[k])))
        parity["max_abs"] = int(allmax(float(parity["max_abs"])))
        parity["pixel_mismatch_frac"] = allmax(parity["pixel_mismatch_frac"])
        parity["of_batch"] = "%d of the %d images of the job" % (parity["images"], n_job)
        parity["note"] = ("coefficients (int32 tap) and BGRA pixels, SHA-256 per image against oracle/_ref (the unmodified reference) "
                          "where it decodes the file, else against the oracle port in non-strict mode")

    # ---- end to end through the public host API: JPEG bytes in host memory -> BGRA in pinned host memory
    e2e = None
    if not args.no_e2e:
        c = synth.CONFIGS[cfg]
        img_bytes = c["height"] * c["width"] * 4
        flat = torch.empty((len(files) * img_bytes,), dtype=torch.uint8, pin_memory=True)     # one pinned allocation
        outs = [flat[i * img_bytes:(i + 1) * img_bytes].view(c["height"], c["width"], 4).numpy() for i in range(len(files))]
        # the ctypes argument arrays are built once, outside the timed region: the timed call is the C entry point
        call4 = b2j.HostArgs(files, outs=outs, out_format=b2j.OUT_BGRA)
        dec.decode_host_args(call4)                      # warm-up (allocations, page faults)
        dec.decode_host_args(call4)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            _, st2 = dec.decode_host_args(call4)
        barrier()
        e2e_s = allmax((time.perf_counter() - t0) / args.e2e_steps)
        assert not st2.any()
        e2e = {"value": round(pix_job / e2e_s / 1e6, 1), "unit": "MPix/s", "h2d_bytes_per_step": int(allsum(float(info.h2d_bytes))),
               "d2h_bytes_per_step": int(allsum(float(info.pixel_bytes))), "ms_per_step": round(e2e_s * 1e3, 3),
               "api": "b2j_decode_host_ex (= b2j_decode_host with the defaults): parse + stage (host threads) + H2D + decode + D2H into pinned host buffers, the reference's BGRA"}
        # the same call with RGB24 output (b2j_decode_host_ex): 25 % fewer bytes over PCIe, which is what bounds e2e
        rgb_bytes = img_bytes // 4 * 3
        outs3 = [flat[i * rgb_bytes:(i + 1) * rgb_bytes].view(c["height"], c["width"], 3).numpy() for i in range(len(files))]
        call3 = b2j.HostArgs(files, outs=outs3, out_format=b2j.OUT_RGB24)
        dec.decode_host_args(call3)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            _, st3 = dec.decode_host_args(call3)
        barrier()
        e2e3_s = allmax((time.perf_counter() - t0) / args.e2e_steps)
        assert not st3.any()
        e2e["rgb24"] = {"value": round(pix_job / e2e3_s / 1e6, 1), "unit": "MPix/s", "ms_per_step": round(e2e3_s * 1e3, 3),
                        "d2h_bytes_per_step": int(allsum(float(info.pixel_bytes))) // 4 * 3,
                        "api": "b2j_decode_host_ex(out_format = B2J_OUT_RGB24): same pixels, three bytes each"}

    sampler.stop_flag.set()
    sampler.join(timeout=2)
    alg_job = allsum(float(info.algorithmic_bytes))
    launches = int(allsum(float(info.kernel_launches))) * args.steps

    if rank == 0:
        peak, peak_src = measured_peak()
        # stages and their algorithmic bytes per step of THIS rank (DESIGN.md "Roofline arithmetic"):
        #   entropy stage  : scan bytes read + int16 coefficient plane written  = C + 128*B
        #   IDCT/colour    : coefficient plane read + BGRA written              = 128*B + 4*W*H
        entropy_kernel = "k_huff_decode" if cfg == 1 else "entropy stage (k_sync_* + k_huff_decode<SYNC>)"
        kb = {"huffman_ms": (entropy_kernel, info.scan_bytes + info.coef_plane_bytes),
              "idct_ms": ("k_idct_csc", info.coef_plane_bytes + info.pixel_bytes)}
        dom = max(kb, key=lambda k: stage[k])
        achieved = kb[dom][1] / (stage[dom] * 1e-3) / 1e9
        pipe = info.algorithmic_bytes / (stage["total_ms"] * 1e-3) / 1e9
        traffic, traffic_src = measured_traffic(cfg, kb[dom][0])
        config = common_config(cfg)
        line = {
            "metric": w["metric"], "value": round(value, 1), "unit": "MPix/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms_per_step, 4), "higher_is_better": True, "scaling": w["scaling"],
            "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": config,
            "detail": {"images_this_rank": len(files), "scan_bytes_this_rank": info.scan_bytes, "blocks_this_rank": info.total_blocks,
                       "algorithmic_bytes_per_step_this_rank": info.algorithmic_bytes, "algorithmic_bytes_per_step_job": int(alg_job),
                       "l2": "no explicit flush: every step streams %.2f GB per GPU (>> 126 MB L2)" % (info.algorithmic_bytes / 1e9),
                       "parallelism": "images sharded by rank, no collective" + ("; slices by compressed bytes: %s" % cuts if cuts and world > 1 else ""),
                       "sync_stats": sync_stats},
            "roofline": {"bound": "hbm", "kernel": kb[dom][0], "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                         "frac": round(achieved / peak, 4), "frac_pipeline": round(pipe / peak, 4),
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "bytes_per_launch": kb[dom][1], "launch_ms": round(stage[dom], 4),
                         "pipeline": {"achieved": round(pipe, 1), "frac": round(pipe / peak, 4),
                                      "note": "all kernels of a step (pre-pass, entropy decode, IDCT+colour): (C + 2*128*B + 4*W*H) / step time, SURVEY.md 8(d); rank 0"},
                         "stage_ms": {k: round(v, 4) for k, v in stage.items()},
                         "huffman_gbit_s": round(info.scan_bytes * 8 / (stage["huffman_ms"] * 1e-3) / 1e9, 1)},
            "parity": parity,
            "cpu_baseline": cpu,
            "e2e": e2e,
            "gpu_launches": launches,
            "clocks": sampler.summary(),
        }
        print(json.dumps(line), flush=True)
    batch.close()
    dec.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
