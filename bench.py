#!/usr/bin/env python
"""bench.py -- fpng hot-path benchmark (encode MP/s on synthetic batches) for the B200-native implementation.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c3|c4|c1] [--kind g1|g0|g2]
                    [--dump-outputs DIR]

One "step" = one pass of the encode hot path over one batch of synthetic images (device-resident for `value`,
host-resident pinned buffers through the C ABI for `e2e`).  Prints ONE JSON line on rank 0.  See DESIGN.md section
"Measurement" for the definition of every field.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import imagegen  # noqa: E402

MP = 1e6

# BASELINE.json configs.  `images` is the per-GPU batch (weak scaling: every rank encodes this many images).
WORKLOADS = {
    "c1": dict(name="C1 1 x 512x512 RGBA, 1-pass", w=512, h=512, chans=4, images=1, flags=0),
    "c2": dict(name="C2 256 x 1920x1080 RGB, 1-pass", w=1920, h=1080, chans=3, images=256, flags=0),
    "c3": dict(name="C3 128/GPU x 3840x2160 RGBA (green->alpha), 1-pass", w=3840, h=2160, chans=4, images=128, flags=0),
    "c4": dict(name="C4 128/GPU x 2048x2048 RGB, 2-pass (FPNG_ENCODE_SLOWER)", w=2048, h=2048, chans=3, images=128, flags=1),
    # not a BASELINE config: the reference's own test image shape (example.png, 687 x 1012 RGB): 2061-byte scanlines, no alignment at all
    "odd": dict(name="ODD 512 x 687x1012 RGB (unaligned 2061-byte scanlines), 1-pass", w=687, h=1012, chans=3, images=512, flags=0),
}
N_UNIQUE_NOISE = 16


def workload_image(wl, kind: str, i: int) -> np.ndarray:
    """Image i of the synthetic batch (numpy twin of make_device_batch; used for the CPU arms and parity checks)."""
    w, h, c = wl["w"], wl["h"], wl["chans"]
    if kind == "g0":
        return imagegen.gradient(w, h, c, i)
    if kind == "g2":
        return imagegen.random_bytes(w, h, c, i % N_UNIQUE_NOISE)
    base = imagegen.gradient(w, h, c, i).astype(np.int16)
    rs = np.random.RandomState(1234 + (i % N_UNIQUE_NOISE))
    noise = rs.randint(-3, 4, size=base.shape).astype(np.int16)
    return ((base + noise) & 255).astype(np.uint8)


def make_device_batch(wl, kind: str, n: int, device, first_index: int = 0):
    """Builds the batch on the GPU: G0 gradient per image index + one of 16 host-generated noise fields."""
    import torch

    w, h, c = wl["w"], wl["h"], wl["chans"]
    x = torch.arange(w, device=device, dtype=torch.int32)[None, :]
    y = torch.arange(h, device=device, dtype=torch.int32)[:, None]
    r = ((255 * x) // max(w - 1, 1) + 0 * y).to(torch.int16)
    g = ((255 * y) // max(h - 1, 1) + 0 * x).to(torch.int16)
    batch = torch.empty((n, h, w, c), dtype=torch.uint8, device=device)
    noises = None
    if kind == "g1":
        u = min(N_UNIQUE_NOISE, n)
        host = np.stack([np.random.RandomState(1234 + j).randint(-3, 4, size=(h, w, c)).astype(np.int16) for j in range(u)])
        noises = torch.from_numpy(host).to(device)
    elif kind == "g2":
        u = min(N_UNIQUE_NOISE, n)
        host = np.stack([imagegen.random_bytes(w, h, c, j) for j in range(u)])
        noises = torch.from_numpy(host).to(device)
    for k in range(n):
        i = first_index + k
        if kind == "g2":
            batch[k] = noises[i % N_UNIQUE_NOISE]
            continue
        b = ((x + y + i) & 255).to(torch.int16)
        planes = [r, g, b] + ([g] if c == 4 else [])
        img = torch.stack(planes, dim=-1)
        if kind == "g1":
            img = img + noises[i % N_UNIQUE_NOISE]
        batch[k] = (img & 255).to(torch.uint8)
    return batch


DUMP_BYTES = 64 << 20


def dump_outputs(dump_dir: str, out, sizes):
    """Writes what the last timed encode step returned to its caller, as float arrays a later build's dump can be compared with:
    sizes.npy (float64, every file's size) and files.npy (float32 [k, m]: the bytes of the k files files_index.npy names, chosen
    with a fixed seed, -1 past a file's end).  A file longer than its share of the 64 MB is sampled at positions drawn with a fixed
    seed, always including its last 16 bytes (Adler-32, IDAT CRC-32 and IEND depend on every byte before them); files_positions.npy
    (float64) says where."""
    n = out.shape[0]
    sz = sizes.cpu().numpy().astype(np.int64) & 0xFFFFFFFF
    rs = np.random.RandomState(0)
    pick = np.sort(rs.choice(n, size=min(n, 4), replace=False))
    cap = (DUMP_BYTES - (1 << 20)) // (12 * len(pick))       # 4 bytes in files.npy + 8 in files_positions.npy per sampled byte
    rows, pos = [], []
    for i in pick:
        size = int(sz[i])
        p = np.arange(size) if size <= cap else \
            np.union1d(np.sort(rs.choice(size - 16, size=cap - 16, replace=False)), np.arange(size - 16, size))
        rows.append(out[i].cpu().numpy()[p])
        pos.append(p)
    m = max(len(p) for p in pos)
    files = np.full((len(pick), m), -1, np.float32)
    where = np.full((len(pick), m), -1, np.float64)
    for k, (r, p) in enumerate(zip(rows, pos)):
        files[k, :len(r)] = r
        where[k, :len(p)] = p
    os.makedirs(dump_dir, exist_ok=True)
    np.save(os.path.join(dump_dir, "sizes.npy"), sz.astype(np.float64))
    np.save(os.path.join(dump_dir, "files.npy"), files)
    np.save(os.path.join(dump_dir, "files_positions.npy"), where)
    np.save(os.path.join(dump_dir, "files_index.npy"), pick.astype(np.float64))


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe): the sampler runs
    from before the warm-up, every sample is time-stamped, and only samples inside [t0, t1] are summarised."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.rows = []          # (timestamp, sm MHz, max sm MHz, [4 throttle reasons]) parsed as nvidia-smi prints them
        self.thread = None

    def _reader(self):
        import datetime
        for line in self.proc.stdout:
            f = [t.strip() for t in line.split(",")]
            if len(f) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                self.rows.append((ts, float(f[1]), float(f[2]), f[4:8]))
            except ValueError:
                continue

    def start(self):
        import threading
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, bufsize=1)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._reader, daemon=True)
        self.thread.start()

    def wait_ready(self, timeout: float = 15.0):
        """nvidia-smi needs up to a few seconds for its first sample on a fresh box: do not start the timed region before it."""
        t = time.time()
        while self.proc is not None and not self.rows and time.time() - t < timeout and self.proc.poll() is None:
            time.sleep(0.01)

    def stop(self, t0: float, t1: float):
        """t0/t1: time.time() bounds of the timed region."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t = time.time()
        while (not self.rows or self.rows[-1][0] < t1) and time.time() - t < 0.5 and self.proc.poll() is None:
            time.sleep(0.01)        # one more sample past the end of the region
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        if self.thread is not None:
            self.thread.join(timeout=2)
        rows = list(self.rows)
        inside = [r for r in rows if t0 - 0.02 <= r[0] <= t1 + 0.02]
        note = "samples inside the timed region"
        if not inside:   # timed region shorter than the sampling period: take the closest samples under the same load
            inside = sorted(rows, key=lambda r: abs(r[0] - 0.5 * (t0 + t1)))[:3]
            note = "timed region shorter than the sampling period; nearest samples (warm-up/timed loop)"
        reasons = set()
        for r in inside:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median([r[1] for r in inside]) if inside else None,
                "sm_max_mhz": max([r[2] for r in inside]) if inside else None,
                "samples": len(inside), "reasons": sorted(reasons), "note": note}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def host_cores() -> int:
    """Usable host threads: scheduler affinity capped by the cgroup CPU quota (the box may expose more CPUs than it grants)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    return max(1, n)


def _timed_pool(work_once, cores: int, seconds: float):
    """Runs work_once(k) repeatedly on `cores` threads until `seconds` elapse; returns (calls completed, elapsed)."""
    from concurrent.futures import ThreadPoolExecutor

    deadline = time.perf_counter() + seconds
    counts = [0] * cores

    def loop(k):
        while time.perf_counter() < deadline:
            work_once(k)
            counts[k] += 1

    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=cores) as ex:
        list(ex.map(loop, range(cores)))
    return sum(counts), time.perf_counter() - t0


def cpu_reference_run(wl, kind: str, seconds: float, steps: int = 1):
    """Times the UNMODIFIED reference encoder (oracle/_ref; the oracle port if it is not built) on all usable host threads,
    each encoding whole images of the workload sample until `seconds` elapse.  Returns (MP/s per step, cores, sample, kind)."""
    from oracle.pyoracle import Oracle, Ref

    cores = host_cores()
    w, h, c, flags = wl["w"], wl["h"], wl["chans"], wl["flags"]
    use_ref = Ref.available()
    enc = Ref() if use_ref else Oracle()
    imgs = [np.ascontiguousarray(workload_image(wl, kind, i)) for i in range(min(cores, 16, wl["images"]))]

    def once(k):
        img = imgs[k % len(imgs)]
        if use_ref:
            enc.encode_discard(img, w, h, c, flags, 1)
        else:
            enc.encode(img, w, h, c, flags)

    vals, total = [], 0
    for _ in range(steps):
        calls, dt = _timed_pool(once, cores, seconds)
        total += calls
        vals.append(calls * w * h / MP / dt)
    sample = f"{cores} threads, whole-image encodes of the first {len(imgs)} workload images ({kind}) for {seconds:.1f}s per step ({total} encodes)"
    return vals, cores, sample, ("reference" if use_ref else "port")


def cpu_reference_decode_run(wl, kind: str, seconds: float):
    """Reference decoder (fpng_decode_memory) on all usable host threads over reference-written files of the workload sample."""
    from oracle.pyoracle import Oracle, Ref

    cores = host_cores()
    w, h, c, flags = wl["w"], wl["h"], wl["chans"], wl["flags"]
    use_ref = Ref.available()
    dec = Ref() if use_ref else Oracle()
    files = [dec.encode(workload_image(wl, kind, i), w, h, c, flags) for i in range(min(cores, 8, wl["images"]))]

    def once(k):
        f = files[k % len(files)]
        if use_ref:
            dec.decode_discard(f, c, 1)
        else:
            dec.decode(f, c)

    calls, dt = _timed_pool(once, cores, seconds)
    return calls * w * h / MP / dt, cores, f"{cores} threads, {calls} decodes of {len(files)} reference-written workload files in {seconds:.1f}s", \
        ("reference" if use_ref else "port")


def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    total = max(args.steps + args.warmup, 1)
    per_step = max(0.5, min(8.0, 60.0 / total))
    vals, cores, sample, kind = cpu_reference_run(wl, args.kind, per_step, steps=args.warmup + args.steps)
    timed = vals[args.warmup:] or vals
    v = float(statistics.mean(timed))
    pixels_per_step = None
    line = {
        "impl": "reference", "metric": "encode_megapixels_per_sec", "value": v, "unit": "MP/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_step * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": wl["name"], "kind": args.kind, "images_per_gpu": args.images or wl["images"], "w": wl["w"], "h": wl["h"],
                   "chans": wl["chans"], "flags": wl["flags"], "where": "host CPU, reference fpng.cpp SSE4.1/PCLMUL build"},
        "cpu_baseline": {"value": v, "unit": "MP/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit_line(line)
    return 0


def run_ours(args, wl):
    import torch
    import torch.distributed as dist

    import fpng_b200
    from fpng_b200._lib import lib
    import ctypes as C

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this implementation has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    fpng_b200.fpng_init(local)
    L = lib()
    # multi-rank runs: keep this rank's host threads and pinned staging on the GPU's own NUMA node (e2e legs are PCIe-bound)
    numa_node = L.fpngb_bind_host_thread_to_device_numa() if world > 1 else -1
    if args.encoder != "default":
        L.fpngb_debug_use_fused(1 if args.encoder == "fused" else 0)
        L.fpngb_debug_crc_overlap(1 if args.encoder == "two_kernel" else 0)
        L.fpngb_debug_pack_crc(0 if args.encoder == "two_kernel_file_crc" else 1)
    L.fpngb_profile_enable.argtypes = [C.c_int]
    L.fpngb_profile_read.argtypes = [C.POINTER(C.c_float), C.c_int]

    w, h, c, flags, n = wl["w"], wl["h"], wl["chans"], wl["flags"], args.images or wl["images"]
    sampler = ClockSampler(local)      # started early: nvidia-smi's first sample can take seconds on a fresh box
    sampler.start()
    batch = make_device_batch(wl, args.kind, n, dev, first_index=rank * n)
    stride = (fpng_b200.max_encoded_size(w, h, c) + 15) // 16 * 16
    out = torch.empty((n, stride), dtype=torch.uint8, device=dev)
    sizes = torch.empty((n,), dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream(dev)

    def step():
        fpng_b200.encode_batch_device(batch, flags, out=out, sizes=sizes, stream=stream.cuda_stream)

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize(dev)

    # parity spot check against the reference/oracle on image 0 of this rank (outside the timed region)
    fsz = int(sizes[0].item()) & 0xFFFFFFFF
    got0 = bytes(out[0, :fsz].cpu().numpy())
    parity = None
    if rank == 0:
        from oracle.pyoracle import Oracle
        parity = got0 == Oracle().encode(workload_image(wl, args.kind, 0), w, h, c, flags)

    sampler.wait_ready()
    for _ in range(3):        # the GPU is under load again when the timed region starts
        step()
    L.fpngb_profile_enable(1)
    launches0 = fpng_b200.launch_count()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    wall0 = time.time()
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    torch.cuda.synchronize(dev)
    wall1 = time.time()
    if world > 1:
        dist.barrier()
    clocks = sampler.stop(wall0, wall1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out, sizes)
    launches = fpng_b200.launch_count() - launches0
    ms = e0.elapsed_time(e1)
    prof = (C.c_float * 9)()
    L.fpngb_profile_read(prof, 9)
    L.fpngb_profile_enable(0)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    per_rank_ms = None
    if world > 1:
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        per_rank_ms = [float(x.item()) / args.steps for x in allt]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    total_pixels = world * n * w * h * args.steps
    value = total_pixels / MP / (ms / 1e3)

    out_bytes = int((sizes.to(torch.int64) & 0xFFFFFFFF).sum().item())
    in_bytes = n * w * h * c
    names = ["hist", "huffman", "scan", "offsets", "fused", "finish", "pack", "adler", "crc"]
    kern = {k: float(v) for k, v in zip(names, prof)}
    peak, peak_src = measured_peak()
    fused_path = kern["fused"] > 0
    algo = {"hist": in_bytes, "huffman": 0, "scan": in_bytes, "offsets": 0, "fused": in_bytes + out_bytes, "finish": 0,
            "pack": 0 if fused_path else in_bytes + out_bytes, "adler": 0,
            # default encoder: the pack kernel computes the scanline CRCs, kernels_ms.crc is the small combine kernel (no file bytes read)
            "crc": out_bytes if (fused_path or args.encoder == "two_kernel_file_crc") else 0}
    dominant = max(kern, key=lambda k: kern[k])

    # DRAM traffic per launch from the committed `ncu --set full` capture of the same workload (profiles/traffic.json,
    # written by profiles/extract_ncu.py), scaled from the capture's image count to this launch; null when no capture exists
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            traffic_db = json.load(f)
    except Exception:
        traffic_db = {}

    def traffic_of(k):
        t = traffic_db.get(f"{args.workload}/{args.kind}/{k}")
        return t["dram_bytes_per_launch"] * n / t["images_in_capture"] if t else None

    def roof(k):
        gbs = algo[k] / 1e9 / (kern[k] / 1e3) if kern[k] > 0 else 0.0
        return {"kernel": k, "bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak, "traffic": traffic_of(k),
                "traffic_source": "static: dram__bytes_read.sum + dram__bytes_write.sum of the committed ncu --set full capture (profiles/traffic.json), scaled by images per launch; not measured in this run",
                "ms_per_launch": kern[k], "algorithmic_bytes_per_launch": algo[k], "peak_source": peak_src}

    line = {
        "metric": "encode_megapixels_per_sec", "value": value, "unit": "MP/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": wl["name"], "kind": args.kind, "images_per_gpu": n, "w": w, "h": h, "chans": c, "flags": flags,
                   "l2": "inputs larger than L2 (%.0f MB per step)" % (in_bytes / 1e6) if in_bytes > 126e6 else "input smaller than L2: L2-warm",
                   "out_over_in": out_bytes / in_bytes, "parity_image0_vs_oracle": parity,
                   "g1_noise": "gradient + uniform integer noise in [-3, 3] from numpy RandomState(1234 + i % 16).randint (MT19937; SURVEY 8d words it as std::mt19937(1234 + i): same engine, different integer mapping, 16 distinct noise fields per batch); both arms use this generator"},
        "clocks": clocks, "gpu_launches": int(launches), "per_rank_ms_per_step": per_rank_ms,
        "scaling_note": None if world == 1 else "weak scaling, no data-path collective: every rank encodes its own 128-image shard; --gpus 1 defaults to C2 "
                        "(BASELINE config 2), --gpus N>1 to C3 (config 3): the same-workload N=1 value is the `same_workload_as_multi_gpu` key of the `--gpus 1` line (or `--gpus 1 --workload c3`)",
        "kernels_ms": kern, "roofline": roof(dominant), "roofline_scan": roof("fused" if fused_path else "scan"),
        "encoder": "single-pass fused kernel (encode_fused.cu: filter + match + code emission + bit placement in one read of the pixels)" if fused_path
                   else "two-kernel scan + pack" + (" (IDAT CRC by the file-reading kernel)" if args.encoder == "two_kernel_file_crc" else
                                                   " (scanline CRCs computed by the pack kernel on the staged code words; kernels_ms.crc is the combine kernel)"),
        "kernels_ms_sum": float(sum(kern.values())),
        "whole_step": {"algorithmic_gbs": (in_bytes + out_bytes) / 1e9 / (ms / args.steps / 1e3),
                       "frac_of_peak": (in_bytes + out_bytes) / 1e9 / (ms / args.steps / 1e3) / peak},
    }

    # ---- decode leg: the rank's own encoded files, device resident (container walk on the host, outside the timed region)
    if not args.no_decode:
        sz_host = (sizes.cpu().numpy().astype(np.int64) & 0xFFFFFFFF)
        files = [bytes(out[i, : int(sz_host[i])].cpu().numpy()) for i in range(n)]
        dec_input = "this rank's GPU-encoded files, device resident"
        # BASELINE config 5 decodes REFERENCE-written files: write them with the unmodified reference encoder (oracle/_ref)
        # on the host threads, outside every timed region; they must equal the GPU-written files byte for byte.
        from oracle.pyoracle import Ref
        if Ref.available() and not args.own_files:
            from concurrent.futures import ThreadPoolExecutor
            rref = Ref()
            host_batch = batch.cpu().numpy()
            with ThreadPoolExecutor(max_workers=max(1, host_cores() // max(1, world))) as ex:
                ref_files = list(ex.map(lambda i: rref.encode(host_batch[i], w, h, c, flags), range(n)))
            same = sum(a == b for a, b in zip(files, ref_files))
            files = ref_files
            dec_input = f"reference-written files (unmodified reference encoder, oracle/_ref), device resident; {same}/{n} byte-identical to the GPU-written files"
            del host_batch
        files_dev, fstride, fsizes, fofs, flens, ww, hh, cc = fpng_b200.pack_files_for_device(files, dev)
        px = torch.empty((n, h, w, c), dtype=torch.uint8, device=dev)
        status = torch.empty((n,), dtype=torch.int32, device=dev)

        def dstep():
            fpng_b200.decode_batch_device(files_dev, fsizes, fofs, flens, w, h, c, c, out=px, status=status, stream=stream.cuda_stream)

        for _ in range(3):
            dstep()
        torch.cuda.synchronize(dev)
        dec_ok = bool((status == 0).all().item()) and bool(torch.equal(px, batch))
        dsteps = max(1, min(args.steps, 10))
        if world > 1:
            dist.barrier()
        d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        d0.record(stream)
        for _ in range(dsteps):
            dstep()
        d1.record(stream)
        torch.cuda.synchronize(dev)
        td = torch.tensor([d0.elapsed_time(d1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(td, op=dist.ReduceOp.MAX)
        dms = float(td.item()) / dsteps
        dec_bytes = out_bytes + n * w * h * c
        # per-kernel device times of one more decode call (CUDA events between the launches)
        L.fpngb_decode_profile_enable.argtypes = [C.c_int]
        L.fpngb_decode_profile_read.argtypes = [C.POINTER(C.c_float), C.c_int]
        L.fpngb_decode_profile_enable(1)
        L.fpngb_debug_decode_repairs.restype = C.c_ulonglong
        L.fpngb_debug_decode_repairs.argtypes = [C.c_int]
        L.fpngb_debug_decode_repairs(1)
        dstep()
        torch.cuda.synchronize(dev)
        repairs = int(L.fpngb_debug_decode_repairs(1))
        dprof = (C.c_float * 6)()
        have_dprof = L.fpngb_decode_profile_read(dprof, 6)
        L.fpngb_decode_profile_enable(0)
        line["decode"] = {"value": world * n * w * h / MP / (dms / 1e3), "unit": "MP/s", "ms_per_step": dms, "steps": dsteps,
                          "pixels_match_input": dec_ok, "algorithmic_gbs": dec_bytes / 1e9 / (dms / 1e3),
                          "frac_of_peak": dec_bytes / 1e9 / (dms / 1e3) / peak,
                          "input": dec_input,
                          "link_repairs_per_call": repairs,     # subsequences whose speculative start was wrong (decoded again by the link pass)
                          "kernels_ms": dict(zip(["prepare", "scan", "link", "write", "stored", "unfilter"], [float(v) for v in dprof])) if have_dprof else None}
        # end to end through the C ABI with host buffers: files (pinned) -> H2D -> kernels -> D2H pixels (pinned)
        hfiles = torch.zeros((n, fstride), dtype=torch.uint8).pin_memory()
        hfiles.copy_(files_dev.cpu())
        hpx = torch.empty((n, h * w * c), dtype=torch.uint8).pin_memory()
        ptrs = [hfiles.data_ptr() + i * fstride for i in range(n)]

        def de2e():
            rc, ww2, hh2, cc2, stt = fpng_b200.decode_batch_host(ptrs, fsizes, c, hpx, h * w * c)
            if rc or (stt != 0).any():
                raise RuntimeError("fpngb_decode_batch_host failed")

        de2e()
        if world > 1:
            dist.barrier()
        ksteps = max(1, min(args.steps, 3))
        t0 = time.perf_counter()
        for _ in range(ksteps):
            de2e()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        line["decode"]["e2e"] = {"value": world * n * w * h * ksteps / MP / float(tt.item()), "unit": "MP/s",
                                 "h2d_bytes_per_step": int(fsizes.astype(np.int64).sum()), "d2h_bytes_per_step": n * w * h * c + 4 * n,
                                 "api": "fpngb_decode_batch_host (C ABI, pinned host buffers, blocking)",
                                 "pixels_match_input": bool(torch.equal(hpx.view(n, h, w, c), batch.cpu()))}
        del files_dev, px, hfiles, hpx

    # ---- the ONE gather of the encoded buffers (north_star) through the C ABI (fpngb_gather_encoded_device: sizes
    # all-gather + peer-window push over NVLink + 4-byte completion all-reduce).  Three numbers: the gather alone, and the
    # whole job "encode + gather to rank 0" timed barrier to barrier (value_with_gather), plus the all-gather form.
    if world > 1:
        import hashlib
        from fpng_b200 import dist as fd
        fd.init_comm()
        window_bytes = world * n * stride
        fd.gather_setup(window_bytes, n)
        _, _, _, p2p = fd.comm_info()
        ptrs = fd.gather_encoded_device(out, sizes, dst_rank=0, stream=stream.cuda_stream)
        torch.cuda.synchronize(dev)
        dist.barrier()
        # verify on hardware what rank 0 received: sha256 of the first and last file of every rank's shard against the
        # oracle's encoding of those images (rank 0 regenerates them), plus every size against the senders' own sizes
        gather_ok = None
        all_sz = [torch.zeros((n,), dtype=torch.int32, device=dev) for _ in range(world)]
        dist.all_gather(all_sz, sizes)
        if rank == 0:
            from oracle.pyoracle import Oracle
            orc = Oracle()
            win, offs, alls = fd.gathered_views(*ptrs, window_bytes, world, n, dev)
            offs_h = offs.cpu().numpy(); alls_h = alls.cpu().numpy().astype(np.int64) & 0xFFFFFFFF
            gather_ok = (int(offs_h[-1]) >> 63) == 0
            for r in range(world):
                gather_ok = gather_ok and bool(np.array_equal(alls_h[r * n:(r + 1) * n], all_sz[r].cpu().numpy().astype(np.int64) & 0xFFFFFFFF))
                for i in (0, n - 1):
                    o0, sz = int(offs_h[r * n + i]), int(alls_h[r * n + i])
                    got = hashlib.sha256(win[o0:o0 + sz].cpu().numpy().tobytes()).hexdigest()
                    exp = hashlib.sha256(orc.encode(workload_image(wl, args.kind, r * n + i), w, h, c, flags)).hexdigest()
                    gather_ok = gather_ok and got == exp
        tb = torch.tensor([float(out_bytes)], dtype=torch.float64, device=dev)
        dist.all_reduce(tb)
        total_bytes = float(tb.item())

        def timed(fn, reps):
            dist.barrier(); torch.cuda.synchronize(dev)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            for _ in range(reps):
                fn()
            b.record(stream)
            torch.cuda.synchronize(dev)
            dist.barrier()
            tt = torch.tensor([a.elapsed_time(b) / reps], dtype=torch.float64, device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt.item())

        greps = max(1, min(args.steps, 10))
        g_ms = timed(lambda: fd.gather_encoded_device(out, sizes, dst_rank=0, stream=stream.cuda_stream), greps)
        ag_ms = timed(lambda: fd.gather_encoded_device(out, sizes, dst_rank=-1, stream=stream.cuda_stream), greps)

        def step_with_gather():
            step()
            fd.gather_encoded_device(out, sizes, dst_rank=0, stream=stream.cuda_stream)

        sg_ms = timed(step_with_gather, greps)
        line["gather"] = {"ms": g_ms, "bytes_total": total_bytes, "to_rank": 0, "path": "peer-window push over NVLink (CUDA IPC)" if p2p else "NCCL grouped send/recv fallback",
                          "gbs_into_rank0": (total_bytes - total_bytes / world) / 1e9 / (g_ms / 1e3),
                          "nvlink_ingress_reference_gbs": 770.0, "frac_of_nvlink_ingress": (total_bytes - total_bytes / world) / 1e9 / (g_ms / 1e3) / 770.0,
                          "allgather_ms": ag_ms, "allgather_gbs_into_each_rank": (total_bytes - total_bytes / world) / 1e9 / (ag_ms / 1e3),
                          "bytes_verified_on_rank0": gather_ok,
                          "what": "fpngb_gather_encoded_device (C ABI): ncclAllGather(sizes) + offsets kernel + every rank stores its files into rank 0's window + 4-byte all-reduce; no host sync"}
        line["value_with_gather"] = {"value": world * n * w * h / MP / (sg_ms / 1e3), "unit": "MP/s", "ms_per_step": sg_ms, "steps": greps,
                                     "what": "encode of every rank's shard + the gather of all encoded files to rank 0, barrier to barrier, max over ranks",
                                     "limiter": "rank 0's NVLink ingress (one receiver)" if g_ms > 0.5 * (ms / args.steps) else "encode kernels"}
        fd.destroy_comm()

    # ---- end to end through the C ABI with host (pinned) buffers: H2D + kernels + D2H inside the timed region
    n_e2e = min(n, args.e2e_images) if args.e2e_images else n
    hin = torch.empty((n_e2e, h, w, c), dtype=torch.uint8).pin_memory()
    hin.copy_(batch[:n_e2e].cpu())
    hout = torch.empty((n_e2e, stride), dtype=torch.uint8).pin_memory()
    hsizes = np.zeros(n_e2e, dtype=np.uint32)

    def e2e_step():
        rc = L.fpngb_encode_batch_host(hin.data_ptr(), h * w * c, n_e2e, w, h, c, flags, hout.data_ptr(), stride, hsizes.ctypes.data_as(C.c_void_p))
        if rc:
            raise RuntimeError(f"fpngb_encode_batch_host failed: {rc}")

    e2e_step()
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    e2e_steps = max(1, min(args.steps, 5))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dt = float(t.item())
    e2e_ok = bytes(hout[0, : int(hsizes[0])].numpy()) == got0
    line["e2e"] = {"value": world * n_e2e * w * h * e2e_steps / MP / dt, "unit": "MP/s", "h2d_bytes_per_step": n_e2e * w * h * c,
                   "d2h_bytes_per_step": int(hsizes.astype(np.int64).sum()) + 4 * n_e2e, "images_per_step": n_e2e, "steps": e2e_steps,
                   "api": "fpngb_encode_batch_host (C ABI, pinned host buffers, blocking)", "timer": "host wall clock around the blocking calls",
                   "numa_node_bound": numa_node,
                   "per_rank_gbs": {"h2d": n_e2e * w * h * c * e2e_steps / 1e9 / dt, "d2h": int(hsizes.astype(np.int64).sum()) * e2e_steps / 1e9 / dt},
                   "matches_device_path": bool(e2e_ok)}

    # ---- N = 1 under `--workload auto` (the driver's call): also time the workload the N > 1 runs use (C3, the same per-GPU batch),
    # so that the N > 1 lines can be read against a same-workload single-GPU number of the same round.  Last GPU leg of the run and
    # self-contained: a failure here only replaces the key by its error text.
    if world == 1 and getattr(args, "auto_workload", False) and not args.images and args.encoder == "default":
        try:
            wl3 = WORKLOADS["c3"]
            w3, h3, ch3, fl3, n3 = wl3["w"], wl3["h"], wl3["chans"], wl3["flags"], wl3["images"]
            b3 = make_device_batch(wl3, args.kind, n3, dev)
            stride3 = (fpng_b200.max_encoded_size(w3, h3, ch3) + 15) // 16 * 16
            out3 = torch.empty((n3, stride3), dtype=torch.uint8, device=dev)
            sizes3 = torch.empty((n3,), dtype=torch.int32, device=dev)

            def step3():
                fpng_b200.encode_batch_device(b3, fl3, out=out3, sizes=sizes3, stream=stream.cuda_stream)

            for _ in range(3):
                step3()
            torch.cuda.synchronize(dev)
            steps3 = max(1, min(args.steps, 10))
            ev_a, ev_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev_a.record(stream)
            for _ in range(steps3):
                step3()
            ev_b.record(stream)
            torch.cuda.synchronize(dev)
            ms3 = ev_a.elapsed_time(ev_b) / steps3
            fsz3 = int(sizes3[0].item()) & 0xFFFFFFFF
            from oracle.pyoracle import Oracle as _Oracle3
            par3 = bytes(out3[0, :fsz3].cpu().numpy()) == _Oracle3().encode(workload_image(wl3, args.kind, 0), w3, h3, ch3, fl3)
            line["same_workload_as_multi_gpu"] = {
                "workload": wl3["name"], "kind": args.kind, "images": n3, "value": n3 * w3 * h3 / MP / (ms3 / 1e3), "unit": "MP/s",
                "ms_per_step": ms3, "steps": steps3, "parity_image0_vs_oracle": bool(par3),
                "what": "device-resident encode of the per-GPU batch that `--gpus N > 1` runs on every rank (weak scaling: N x this value is the "
                        "ideal N-GPU `value`); the headline `value` of this line is C2, BASELINE config 2"}
            del b3, out3, sizes3
        except Exception as e:                                    # noqa: BLE001 -- never let the extra leg cost the line
            line["same_workload_as_multi_gpu"] = {"error": repr(e)[:300]}

    if rank == 0 and world == 1 and not args.no_cpu:
        vals, cores, sample, kind = cpu_reference_run(wl, args.kind, args.cpu_seconds)
        line["cpu_baseline"] = {"value": float(vals[0]), "unit": "MP/s", "cores": cores, "kind": kind, "sample": sample}
        if "decode" in line:
            dv, dcores, dsample, dkind = cpu_reference_decode_run(wl, args.kind, max(2.0, args.cpu_seconds / 3))
            line["decode"]["cpu_baseline"] = {"value": float(dv), "unit": "MP/s", "cores": dcores, "kind": dkind, "sample": dsample}
    if rank == 0:
        emit_line(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


_REAL_STDOUT = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries (NCCL with NCCL_DEBUG=VERSION, torchrun banners) also write to
    fd 1, so keep a private copy of the real stdout for the JSON line and point fd 1 at stderr for everything else."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit_line(line: dict):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="auto", choices=["auto"] + sorted(WORKLOADS),
                    help="auto: C2 (BASELINE config 2, the 1-GPU configuration) at --gpus 1, C3 (config 3, the north-star 8-GPU configuration) at --gpus > 1")
    ap.add_argument("--kind", default="g1", choices=["g0", "g1", "g2"])
    ap.add_argument("--images", type=int, default=0, help="images per GPU (default: the workload's)")
    ap.add_argument("--e2e-images", type=int, default=0, help="images per e2e step (0 = the whole per-GPU batch)")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-decode", action="store_true")
    ap.add_argument("--encoder", default="default", choices=["default", "two_kernel", "two_kernel_serial", "two_kernel_file_crc", "fused"],
                    help="default: the library's choice; two_kernel: scan+pack with the chunked CRC overlap; two_kernel_serial: scan+pack, serial; two_kernel_file_crc: scan+pack, IDAT CRC by the file-reading kernel instead of the pack kernel; fused: single-pass encoder")
    ap.add_argument("--own-files", action="store_true", help="decode leg: use the GPU-written files instead of reference-written ones")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the encoded files of the last step (sizes and a fixed sample of files) as .npy to DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU encoder's outputs; --impl reference has none")
    args.auto_workload = args.workload == "auto"
    if args.workload == "auto":
        args.workload = "c2" if max(args.gpus, int(os.environ.get("WORLD_SIZE", "1"))) <= 1 else "c3"
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        return run_reference(args, wl)
    return run_ours(args, wl)


if __name__ == "__main__":
    sys.exit(main())
