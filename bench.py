#!/usr/bin/env python3
"""Headline benchmark: MPix/s of guetzli::Process(RGB) (bit-exact JPEG) on B200.

    python bench.py --gpus N --steps K --warmup W          # this repo (CUDA, sm_100a)
    python bench.py --impl reference --gpus N ...          # reference CPU arm (oracle/_ref)
    python bench.py --mode tiled --workload gradnoise8k_q95 --gpus N   # ONE image over N GPUs

Default (batch) mode: a "step" = `--batch` full Process() calls per GPU, each on its own
host thread + CUDA stream (BASELINE.json configs[1]: 1920x1080 sRGB noise, --quality 95,
unless --workload says otherwise).  Multi-GPU = independent images sharded over ranks (weak
scaling, no data-path collective; torch.distributed only for the barrier and the
max-over-ranks time).  The same run also reports the latency of ONE image alone on the GPU
(SURVEY.md §8(d)'s per-call definition) and, unless --no-tiled-leg, one 8K image tiled over
all N ranks through the NCCL strip mode (BASELINE configs[3], strong scaling).
Prints ONE JSON line on rank 0.  See DESIGN.md "Measurement".
"""
import argparse
import hashlib
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

HAVE_CUDA = True

# cpu_px_s: single-core reference rate used only to SIZE the bounded CPU sample
# (BASELINE.md §2 / tests/golden/golden_large.json); the rate reported is measured.
WORKLOADS = {
    # BASELINE.json configs[1] -- the single-GPU configuration the metric is quoted on
    "noise1080p_q95": dict(gen="noise", h=1080, w=1920, seed=1234, quality=95, cpu_px_s=2500.0,
                           golden="noise1080p_s1234_q95"),
    "gradnoise4k_q90": dict(gen="gradnoise", h=2160, w=3840, seed=4321, quality=90, cpu_px_s=6500.0,
                            golden="gradnoise4k_s4321_q90"),
    "gradnoise8k_q95": dict(gen="gradnoise", h=4320, w=7680, seed=8192, quality=95, cpu_px_s=5000.0,
                            golden="gradnoise8k_s8192_q95"),
    "gradnoise1024_q84": dict(gen="gradnoise", h=1024, w=1024, seed=1000, quality=84, cpu_px_s=11000.0,
                              golden="gradnoise1024_s1000_q84"),
    "gradnoise512_q90": dict(gen="gradnoise", h=512, w=512, seed=4321, quality=90, cpu_px_s=7400.0),
    "noise512_q95": dict(gen="noise", h=512, w=512, seed=1234, quality=95, cpu_px_s=2500.0),
    "gradnoise256_q90": dict(gen="gradnoise", h=256, w=256, seed=4321, quality=90, cpu_px_s=7400.0),
}

# Algorithmic bytes per launched element (pixel of one plane, or 8x8 block) of each kernel:
# compulsory reads + writes of that stage (DESIGN.md §5).
ALG_BYTES = {
    # TMA-staged fused chain (fused_kernels.cuh); elements as counted by the launchers in pipeline.cu
    "tma_blur_x": 8, "tma_blur_y": 8, "opsin_fused": 24, "lf_fused_y": 16, "mf_fused_y": 56.0 / 3, "hf_fused": 84,
    "malta_sums": 16, "noise_fused_y": 20, "mask_pre": 28, "mask_y_combine": 40, "final_fused": 8,
    # staged chain (GB200_COMPARE=staged) and the other per-iteration kernels
    "malta_channel": 28, "blur_x": 8, "blur_y": 8, "sub_planes": 12, "opsin_px": 36, "split_mf_hf": 44, "split_hf_uhf": 68,
    "malta_pre": 12, "malta_acc_hf": 8, "malta_acc_lf": 12, "noise_pre": 12, "noise_asym_acc": 20,
    "mask_diff_pre": 40, "combine_sqrt": 44, "diffmap_mix": 12, "render_blocks": 1152,
    "block_max": 260, "jpeg_unit_bits": 128, "jpeg_emit": 140, "jpeg_hist_acc": 128, "jpeg_hist": 128, "linearize_rgb": 15, "quantize_coeffs": 4, "fdct_blocks": 576,
}
# Kernels that make up one ButteraugliComparator::Compare (a7+a9+a10); their summed time
# is compared with the compulsory 50 B/px of SURVEY.md §8(d).
COMPARE_KERNELS = {
    "tma_blur_x", "tma_blur_y", "opsin_fused", "lf_fused_y", "mf_fused_y", "hf_fused", "malta_sums", "noise_fused_y",
    "mask_pre", "mask_y_combine", "final_fused",
    "render_blocks", "blur_x", "blur_y", "opsin_px", "sub_planes", "split_mf_hf", "split_hf_uhf", "malta_channel",
    "noise_pre", "noise_asym_acc", "mask_diff_pre", "combine_sqrt", "diffmap_mix", "block_max", "partial_max",
}
COMPARE_FLOP_PER_PX = 2500.0  # SURVEY.md §8(d): un-fused FP32 instructions per pixel per Compare (no FMA)

# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu
# --set full captures (profiles/), bytes; None until captured.
NCU_TRAFFIC = {
    # profiles/r02_ncu_fused.csv (noise1080p, per launch: dram read + write)
    "hf_fused": 74.76e6 + 47.16e6, "mf_fused_y": 58.22e6 + 12.7e6, "mask_y_combine": 74.77e6 + 3.22e6,
    "malta_sums": 49.82e6 + 3.18e6, "opsin_fused": 24.96e6 + 0.08e6, "lf_fused_y": 49.82e6 + 10.12e6,
    "noise_fused_y": 33.26e6, "final_fused": 8.32e6, "mask_pre": 41.48e6 + 0.33e6,
    # profiles/r01_final2_ncu_full.csv / r01_ncu_full_malta_blur.csv (staged chain)
    "malta_channel": 49.8e6 + 1.7e6 + 24.9e6,
    "blur_x": 8.33e6, "blur_y": 8.32e6,
}


def make_image(spec, index=0):
    from guetzli_b200 import synth
    seed = spec["seed"] + index
    if spec["gen"] == "noise":
        return synth.noise(spec["h"], spec["w"], seed)
    return synth.gradnoise(spec["h"], spec["w"], seed)


def usable_cores():
    """Host threads this process may really use: affinity mask and cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    how = f"sched_getaffinity={n}"
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    q = int(math.floor(int(txt[0]) / int(txt[1])))
                    how += f", cgroup cpu.max={txt[0]}/{txt[1]}"
                    n = max(1, min(n, q))
            else:
                quota = int(txt[0])
                period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if quota > 0:
                    how += f", cfs_quota={quota}/{period}"
                    n = max(1, min(n, quota // period))
            break
        except (OSError, ValueError, IndexError):
            continue
    return n, how


def cpu_sample_spec(wl, seconds):
    """A crop-sized image of the same generator that one reference core encodes in about
    `seconds` (the CPU cost is proportional to the pixel count for a given content)."""
    side = int(math.sqrt(max(1.0, wl["cpu_px_s"] * seconds)))
    side = max(96, min(side, min(wl["h"], wl["w"]), 768)) // 32 * 32
    return dict(gen=wl["gen"], h=side, w=side, seed=wl["seed"])


class DeviceTimer:
    """CUDA events on torch's current stream (the library's own streams are drained by the
    blocking calls before stop()).  Without a GPU -- only when GUETZLI_B200_LIB points the
    harness at the CPU port for a plumbing rehearsal -- falls back to the host clock."""

    def __init__(self):
        import torch
        self.cuda = torch.cuda.is_available()
        if self.cuda:
            self.e0, self.e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def start(self):
        if self.cuda:
            self.e0.record()
        else:
            self.t0 = time.perf_counter()

    def stop(self):
        if self.cuda:
            import torch
            self.e1.record()
            torch.cuda.synchronize()
            return self.e0.elapsed_time(self.e1) / 1e3
        return time.perf_counter() - self.t0


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "200"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[5:9]):
                if v.strip().lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------
# reference arm
def _ref_worker(args):
    spec, quality, index = args
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import reflib
    rgb = make_image(spec, index)
    ok, jpeg, _, _, secs = reflib.process_rgb(rgb, quality, trace=False)
    if not ok:
        raise RuntimeError("reference Process() failed")
    return secs


def run_reference(args, wl, name, emit):
    """Reference arm: the unmodified reference (oracle/_ref) on the host cores this process
    may use, one single-threaded Process() per core (the reference's own parallelism idiom,
    tests/golden_test.sh:25).  Each step = one bounded crop-sized sample of the workload's
    generator per core, sized so that the whole --steps/--warmup run ends within minutes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    import reflib
    if not reflib.available():
        emit({"impl": "reference", "unavailable": "oracle/_ref/libguetzli_ref.so not built"})
        return
    cores, how = usable_cores()
    cores = max(1, min(cores, 64))
    per_step = max(3.0, min(40.0, 200.0 / max(1, args.steps + args.warmup)))
    spec = cpu_sample_spec(wl, per_step)
    px = spec["h"] * spec["w"]
    ctx = mp.get_context("spawn")
    per_core = []
    with ctx.Pool(cores) as pool:
        for _ in range(args.warmup):
            pool.map(_ref_worker, [(spec, wl["quality"], r) for r in range(cores)])
        t0 = time.perf_counter()
        for _ in range(args.steps):
            per_core += pool.map(_ref_worker, [(spec, wl["quality"], r) for r in range(cores)])
        dt = time.perf_counter() - t0
    value = cores * args.steps * px / dt / 1e6
    sample = (f"{spec['gen']}({spec['h']},{spec['w']},seed {spec['seed']}+core) q{wl['quality']}: crop-sized image of the "
              f"workload's generator, one per core per step ({how})")
    line = {
        "impl": "reference", "metric": "MPix/s (bit-exact JPEG, guetzli::Process)", "value": value,
        "unit": "MPix/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32/f64+int16 (CPU)", "data": "synthetic",
        "config": {"workload": name, "sample": sample},
        "cpu_baseline": {"value": value, "unit": "MPix/s", "cores": cores, "kind": "reference", "sample": sample,
                         "per_core_mpix_s": px / float(np.mean(per_core)) / 1e6,
                         "full_size_cached": cached_reference_timing(wl)},
        "e2e": {"value": value, "unit": "MPix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def cached_reference_timing(wl):
    """Full-size timing of the unmodified reference on this workload's image, measured once on
    one core of the build container (tests/golden/golden_large.json, BASELINE.md §3 step 5)."""
    key = wl.get("golden")
    path = os.path.join(ROOT, "tests", "golden", "golden_large.json")
    if not key or not os.path.exists(path):
        return None
    g = json.load(open(path)).get(key)
    if not g:
        return None
    return {"seconds_one_core": g["ref_seconds_here"], "mpix_s": g["shape"][0] * g["shape"][1] / g["ref_seconds_here"] / 1e6,
            "input_sha256": g["input_sha256"], "jpeg_sha256": g["jpeg_sha256"], "where": "build container, 1 core"}


# --------------------------------------------------------------------------------------
def golden_sha(wl):
    c = cached_reference_timing(wl)
    return c["jpeg_sha256"] if c else None


def run_tiled(args, wl, name, gb, dist, rank, world, local, steps, warmup):
    """ONE image over all ranks (gb200_process_rgb_tiled, NCCL strip mode); world == 1 runs the
    plain single-GPU call.  -> dict (rank 0) with MPix/s and the library's own timers."""
    import torch
    from guetzli_b200 import distributed as gdist
    if HAVE_CUDA:
        torch.cuda.set_device(local)  # this may run on a helper thread
    rgb = make_image(wl)
    h, w, _ = rgb.shape
    params = gb.Params(butteraugli_target=gb.butteraugli_score_for_quality(wl["quality"]))
    if world > 1:
        box = [gb.dist_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        gb.dist_init(box[0], rank, world, local)

    def once():
        st = gb.ProcessStats()
        if world > 1:
            ok, jpeg = gb.process_tiled(params, st, rgb, w, h)
        else:
            ok, jpeg = gb.process(params, st, rgb, w, h, device=local)
        if not ok:
            raise RuntimeError("tiled Process failed: " + gb.last_error())
        return st, jpeg

    for _ in range(warmup):
        once()
    gdist.barrier(dist, cuda=HAVE_CUDA)
    tm = DeviceTimer()
    tm.start()
    shas = set()
    st = jpeg = None
    for _ in range(steps):
        st, jpeg = once()
        shas.add(hashlib.sha256(jpeg).hexdigest())
    dt_local = tm.stop()
    gdist.barrier(dist, cuda=HAVE_CUDA)
    dt = gdist.max_over_ranks(dist, dt_local, device=f"cuda:{local}" if HAVE_CUDA else None)
    want = golden_sha(wl)
    out = {"workload": name, "n_gpus": world, "steps": steps, "warmup": warmup, "value": steps * h * w / dt / 1e6,
           "unit": "MPix/s", "ms_per_image": dt / steps * 1e3, "scaling": "strong",
           "collective": "NCCL in-place all-gather of per-block results (library communicator)" if world > 1 else "none",
           "output_sha256": sorted(shas)[0], "deterministic": len(shas) == 1,
           "matches_reference_golden": (sorted(shas)[0] == want) if want else None,
           "timers_ms_rank0": {k: round(st.device[k], 1) for k in
                               ("ms_total", "ms_device_setup", "ms_compare", "ms_zeroing", "ms_jpeg", "ms_sort", "ms_walk")},
           "gpu_launches_rank0": st.device["gpu_launches"], "h2d_bytes_rank0": st.device["h2d_bytes"],
           "d2h_bytes_rank0": st.device["d2h_bytes"],
           "iterations": st.counters["number of iterations"]}
    if world > 1:
        gb.dist_shutdown()
    return out, jpeg


def dump_outputs(path, jpegs, rank, world, budget=64 << 20):
    """What the timed path returned in its last step: every JPEG file as DIR/jpeg_<image>.npy, its
    bytes as float32, at most `budget` bytes over all ranks.  A JPEG larger than its share is stored
    as a fixed sample of its bytes (positions drawn with seed 0, in increasing order, the same for
    equal file sizes); DIR/sizes_rank<r>.npy holds the full sizes of rank r's files."""
    os.makedirs(path, exist_ok=True)
    share = max(1, (budget - 4096 * world) // 4 // (world * len(jpegs)))
    for i, data in jpegs.items():
        a = np.frombuffer(data, dtype=np.uint8)
        if a.size > share:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, share, replace=False))]
        np.save(os.path.join(path, "jpeg_%03d.npy" % i), a.astype(np.float32))
    np.save(os.path.join(path, "sizes_rank%d.npy" % rank), np.array([len(d) for d in jpegs.values()], dtype=np.float64))


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries print there too (NCCL's version banner
    when NCCL_DEBUG is set on the box, warnings of child processes): everything this process and
    its libraries write to fd 1 goes to stderr instead; the line is written to the real stdout."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


def main():
    real_stdout = claim_stdout()

    def emit(line):
        real_stdout.write(json.dumps(line) + "\n")
        real_stdout.flush()

    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="noise1080p_q95", choices=sorted(WORKLOADS))
    ap.add_argument("--mode", default="batch", choices=["batch", "tiled"],
                    help="batch: independent images per GPU (weak scaling); tiled: ONE image over all GPUs (strong)")
    ap.add_argument("--batch", type=int, default=16,
                    help="images per GPU per step, encoded concurrently (one host thread + CUDA stream each)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-tiled-leg", action="store_true",
                    help="skip the extra 8K image tiled over all ranks at the end of a batch-mode run")
    ap.add_argument("--tiled-leg-workload", default="gradnoise8k_q95", choices=sorted(WORKLOADS))
    ap.add_argument("--tiled-leg-timeout", type=float, default=900.0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the JPEGs of the last step to DIR as .npy (float32) files")
    args = ap.parse_args()
    wl = WORKLOADS[args.workload]

    if args.impl == "reference":
        run_reference(args, wl, args.workload, emit)
        return

    from concurrent.futures import ThreadPoolExecutor
    from guetzli_b200 import distributed as gdist
    import torch
    rank, world, local, dist = gdist.setup("nccl" if torch.cuda.is_available() else "gloo")
    import guetzli_b200 as gb
    lib = gb.load_library()
    global HAVE_CUDA
    HAVE_CUDA = torch.cuda.is_available()
    rehearsal = lib.gb200_backend_name() != b"cuda-sm_100a"
    if lib.gb200_device_count() < 1 or (not HAVE_CUDA and not rehearsal):
        raise SystemExit("bench.py: no CUDA device; the product has no CPU fallback")
    if HAVE_CUDA:
        torch.cuda.set_device(local)

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_kind = json.load(open(peaks_path))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_kind = 6650.0, "fallback (B200_PROFILING.md)"

    if args.mode == "tiled":
        sampler = ClockSampler(local)
        sampler.start()
        n0, a0, b0 = gb.counters()
        res, jpeg = run_tiled(args, wl, args.workload, gb, dist, rank, world, local, args.steps, args.warmup)
        n1, a1, b1 = gb.counters()
        clocks = sampler.stop()
        if args.dump_outputs and rank == 0:  # every rank holds the same file
            dump_outputs(args.dump_outputs, {0: jpeg}, 0, 1)
        if dist is not None:
            dist.destroy_process_group()
        if rank != 0:
            return
        line = {"metric": "MPix/s (bit-exact JPEG, guetzli::Process)", "value": res["value"], "unit": "MPix/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_image"],
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32 (+f64 sub-expressions), int16/int32", "data": "synthetic",
                "config": {"workload": args.workload, "mode": "tiled: one image, row strips over the ranks",
                           "l2_policy": "one image's work planes exceed L2"},
                "clocks": clocks,
                "e2e": {"value": res["value"], "unit": "MPix/s", "ms_per_step": res["ms_per_image"],
                        "h2d_bytes_per_step": int((a1 - a0) / max(1, args.steps + args.warmup)),
                        "d2h_bytes_per_step": int((b1 - b0) / max(1, args.steps + args.warmup)),
                        "note": "the tiled call takes HOST buffers: value and e2e are the same measurement"},
                "gpu_launches": int((n1 - n0) * args.steps / max(1, args.steps + args.warmup)), "tiled": res}
        emit(line)
        return

    M = args.batch
    # weak scaling: rank r encodes images r*M .. r*M+M-1 of the generator, every step
    images = [make_image(wl, rank * M + j) for j in range(M)]
    h, w, _ = images[0].shape
    params = gb.Params(butteraugli_target=gb.butteraugli_score_for_quality(wl["quality"]))
    px = h * w
    pool = ThreadPoolExecutor(M)
    shas = [set() for _ in range(M)]
    last = {}  # image index -> JPEG of the latest timed step

    def encode_host(j):  # reference-facing call: host buffer in, JPEG bytes out
        st = gb.ProcessStats()
        ok, jpeg = gb.process(params, st, images[j], w, h, device=local)
        if not ok:
            raise RuntimeError(f"gb200_process_rgb failed on image {j}: {gb.last_error()}")
        shas[j].add(hashlib.sha256(jpeg).hexdigest())
        return st

    # M resident contexts, reused by every step (memory does not depend on --steps)
    resident = []

    def encode_resident(j):  # image already uploaded; the whole job (incl. the one-time kernels) is redone
        st = gb.ProcessStats()
        resident[j].reset()
        ok, jpeg = resident[j].process(params, st)
        if not ok:
            raise RuntimeError(f"gb200_image_process failed on image {j}: {gb.last_error()}")
        shas[j].add(hashlib.sha256(jpeg).hexdigest())
        last[rank * M + j] = jpeg
        return st

    for _ in range(args.warmup):
        list(pool.map(encode_host, range(M)))

    # ---- value: images already resident in HBM when the timed region starts ----
    resident.extend(gb.DeviceImage(images[j], device=local, prepare=False) for j in range(M))
    sampler = ClockSampler(local)
    gdist.barrier(dist, cuda=HAVE_CUDA)
    sampler.start()
    n0, _, _ = gb.counters()
    tm = DeviceTimer()
    tm.start()
    stats_list = []
    for step in range(args.steps):
        stats_list = list(pool.map(encode_resident, range(M)))
    dt_local = tm.stop()
    gdist.barrier(dist, cuda=HAVE_CUDA)
    clocks = sampler.stop()
    n1, _, _ = gb.counters()
    dt = gdist.max_over_ranks(dist, dt_local, device=f"cuda:{local}" if HAVE_CUDA else None)
    launches = n1 - n0
    for img in resident:
        img.close()
    resident.clear()
    value = world * args.steps * M * px / dt / 1e6
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(sorted(last.items())), rank, world)

    # ---- e2e: same job through the reference-facing call with HOST buffers ----
    gdist.barrier(dist, cuda=HAVE_CUDA)
    _, a0, b0 = gb.counters()
    tm = DeviceTimer()
    tm.start()
    for _ in range(args.steps):
        list(pool.map(encode_host, range(M)))
    dt_local = tm.stop()
    gdist.barrier(dist, cuda=HAVE_CUDA)
    _, a1, b1 = gb.counters()
    dt_e2e = gdist.max_over_ranks(dist, dt_local, device=f"cuda:{local}" if HAVE_CUDA else None)
    e2e_value = world * args.steps * M * px / dt_e2e / 1e6
    h2d, d2h = (a1 - a0) / args.steps, (b1 - b0) / args.steps
    if not all(len(x) == 1 for x in shas):
        raise RuntimeError("non-deterministic output")

    # ---- ONE image alone on the GPU: latency (SURVEY §8(d)) + per-kernel CUDA-event times ----
    kernels, gpu_ms, prof_st, single = [], 0.0, None, None
    if rank == 0:
        import ctypes as C
        t0 = time.perf_counter()
        st1 = encode_host(0)
        t_single = time.perf_counter() - t0
        single = {"ms": t_single * 1e3, "mpix_s": px / t_single / 1e6,
                  "what": "one gb200_process_rgb call (host buffers) with the GPU otherwise idle",
                  "breakdown_ms": {k: round(st1.device[k], 1) for k in
                                   ("ms_total", "ms_compare", "ms_zeroing", "ms_jpeg", "ms_sort", "ms_walk")},
                  "order_partial": st1.device["order_partial"], "order_exact": st1.device["order_exact"],
                  "gpu_launches": st1.device["gpu_launches"], "h2d_bytes": st1.device["h2d_bytes"],
                  "d2h_bytes": st1.device["d2h_bytes"], "compares": st1.device["compares"]}
        lib.gb200_profile_reset()
        lib.gb200_profile_enable(1)
        prof_st = encode_host(0)
        lib.gb200_profile_enable(0)
        cap = 96
        names = ((C.c_char * 48) * cap)()
        kl = (C.c_long * cap)()
        kms = (C.c_double * cap)()
        kel = (C.c_double * cap)()
        nk = lib.gb200_profile_get(names, kl, kms, kel, cap)
        for i in range(min(nk, cap)):
            kernels.append({"name": names[i].value.decode(), "launches": kl[i], "ms": kms[i], "elements": kel[i]})
        kernels.sort(key=lambda k: -k["ms"])
        gpu_ms = sum(k["ms"] for k in kernels)

    # ---- extra leg: ONE 8K image tiled over all ranks (strong scaling, NCCL) ----
    tiled, hung = None, False
    if not args.no_tiled_leg:
        box = {}

        def leg():
            try:
                box["res"] = run_tiled(args, WORKLOADS[args.tiled_leg_workload], args.tiled_leg_workload, gb, dist,
                                       rank, world, local, steps=1, warmup=0)[0]
            except Exception as e:  # the main line must survive a failure of the extra leg
                box["res"] = {"error": f"{type(e).__name__}: {e}"}

        t = threading.Thread(target=leg, daemon=True)
        t.start()
        t.join(timeout=args.tiled_leg_timeout)
        hung = t.is_alive()  # a hung collective cannot be joined: print what we have and leave
        tiled = box.get("res", {"error": f"tiled leg did not finish within {args.tiled_leg_timeout} s"})
    if dist is not None and not hung:
        gdist.barrier(dist, cuda=HAVE_CUDA)
        dist.destroy_process_group()
    if rank != 0:
        if hung:
            os._exit(0)
        return

    roofline = None
    ranked = [k for k in kernels if k["name"] in ALG_BYTES and k["launches"] > 1]
    compares = max(1, prof_st.device["compares"]) if prof_st else 1
    cmp_ms = sum(k["ms"] for k in kernels if k["name"] in COMPARE_KERNELS)
    if ranked:
        top = ranked[0]
        bpe = ALG_BYTES[top["name"]]
        achieved = bpe * top["elements"] / (top["ms"] * 1e-3) / 1e9
        us_per_compare = cmp_ms * 1e3 / compares
        roofline = {"bound": "hbm", "kernel": top["name"], "achieved": achieved, "peak": peak,
                    "unit": "GB/s", "frac": achieved / peak, "traffic": NCU_TRAFFIC.get(top["name"]),
                    "peak_source": peak_kind, "avg_launch_us": top["ms"] / max(1, top["launches"]) * 1e3,
                    "share_of_gpu_time": top["ms"] / gpu_ms if gpu_ms else None,
                    "alg_bytes_per_element": bpe,
                    "measured_on": "one extra image encoded alone (single stream) after the timed region",
                    # the whole Compare chain against SURVEY §8(d)'s compulsory traffic and issue floor
                    "compare_chain": {
                        "us_per_compare": us_per_compare, "compares": compares,
                        "compulsory_bytes_per_px": 50,
                        "hbm_frac": 50.0 * px / (us_per_compare * 1e-6) / 1e9 / peak if us_per_compare else None,
                        "fp32_issue_frac": (COMPARE_FLOP_PER_PX * px / (us_per_compare * 1e-6)) /
                                           (148 * 128 * (clocks.get("sm_max_mhz") or 1965.0) * 1e6) if us_per_compare else None,
                        "note": "event times include ~2-5 us of event overhead per launch"}}
    st = stats_list[-1]
    line = {
        "metric": "MPix/s (bit-exact JPEG, guetzli::Process)", "value": value, "unit": "MPix/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 (+f64 sub-expressions), int16/int32", "data": "synthetic",
        "config": {"workload": args.workload, "batch_per_gpu": M,
                   "image": f"{wl['gen']}({h},{w},seed {wl['seed']}+rank*{M}+j), j<{M}",
                   "quality": wl["quality"], "input_sha256_rank0_img0": hashlib.sha256(images[0].tobytes()).hexdigest(),
                   "output_sha256_rank0_img0": sorted(shas[0])[0],
                   "output_matches_reference_golden": (sorted(shas[0])[0] == golden_sha(wl)) if golden_sha(wl) else None,
                   "iterations_img_last": st.counters["number of iterations"],
                   "sharding": f"{world} GPU(s) x {M} independent images per step, one host thread + stream each",
                   "l2_policy": "working set of one step (>= 16 images x their float planes) exceeds L2"},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "MPix/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": dt_e2e / args.steps * 1e3},
        "gpu_launches": int(launches),
        "roofline": roofline,
        "single_image": single,
        # the library's wall timers of the images of the last timed step (mean over the batch): where a
        # Process() call spends its time when `batch_per_gpu` of them share the GPU and the host cores
        "batch_breakdown_ms": {k: round(float(np.mean([s.device[k] for s in stats_list])), 1) for k in
                               ("ms_total", "ms_compare", "ms_zeroing", "ms_jpeg", "ms_sort", "ms_walk")},
        "single_image_gpu_kernel_ms": round(gpu_ms, 2),
        "top_kernels": [{"name": k["name"], "ms": round(k["ms"], 2), "launches": k["launches"]} for k in kernels[:30]],
        "tiled": tiled,
    }
    if world == 1 and not args.no_cpu_baseline:
        import reflib
        if reflib.available():
            spec = cpu_sample_spec(wl, 15.0)
            rgb = make_image(spec)
            ok, jpeg, _, counters, secs = reflib.process_rgb(rgb, wl["quality"], trace=False)
            if not ok:
                raise RuntimeError("reference Process() failed on the CPU sample")
            line["cpu_baseline"] = {
                "value": spec["h"] * spec["w"] / secs / 1e6, "unit": "MPix/s", "cores": 1, "kind": "reference",
                "sample": f"{spec['gen']}({spec['h']},{spec['w']},seed {spec['seed']}) q{wl['quality']}, "
                          f"{secs:.1f} s, {counters[0]} iterations (crop-sized image of the same generator)",
                "full_size_cached": cached_reference_timing(wl)}
    if rehearsal:
        line["rehearsal_cpu_port"] = True  # plumbing check only, not a measurement
    emit(line)
    if hung:
        os._exit(0)


if __name__ == "__main__":
    main()
