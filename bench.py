#!/usr/bin/env python
"""bench.py — megapixels/s decoded (JPEG XL VarDCT d1.0) on N B200s; CPU baseline beside it.

A "step" is one pass of the decode hot path over one batch of independent frames per GPU
(weak scaling: every rank decodes its own batch; there is no data-path collective — groups and
frames are independent, SURVEY.md §8e). `value` is timed with the encoded frames already
resident in HBM and the decoded planes left in HBM; `e2e` goes through the public API with host
bytes in and planar f32 pixels copied back to pinned host memory every step.

  python bench.py --gpus 1 --steps 5 --warmup 3
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference      # CPU arm: the oracle (port of jxl-oxide's generic path)
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

# Several decoder contexts (CUDA streams) run concurrently; with the default 8 hardware work queues
# streams alias and a long entropy kernel delays other streams' launches.
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

GOLDEN = os.path.join(ROOT, "tests", "golden")


# ----------------------------------------------------------------------------------------------
# workloads
SYNTH_TOOL = os.path.join(ROOT, "tools", "_build_synth_enc")
_synth_dir = None


def build_synth_tool():
    """Compiles tools/synth_enc.cc (build() does this, so that the benchmark can run from a read-only tree)."""
    src = os.path.join(ROOT, "tools", "synth_enc.cc")
    if os.path.exists(SYNTH_TOOL) and os.path.getmtime(SYNTH_TOOL) >= os.path.getmtime(src):
        return
    host = os.path.join(ROOT, "jxl_oxide_b200", "csrc", "host")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-o", SYNTH_TOOL, src] +
                          [os.path.join(host, f) for f in ("entropy.cc", "frame_syntax.cc", "modular_syntax.cc", "headers.cc")])


def synth_frame(w, h, seed, distance=1.0, extra=()):
    """Synthetic encoded frame from tools/synth_enc.cc: the same bytes for the same arguments. Frames are cached for the
    life of the process in a temporary directory, not in the tree."""
    global _synth_dir
    build_synth_tool()
    if _synth_dir is None:
        _synth_dir = tempfile.TemporaryDirectory(prefix="jxlb_synth_")
    tag = "".join(extra).replace("-", "")
    path = os.path.join(_synth_dir.name, f"synth_{w}x{h}_d{distance}_s{seed}{tag}.jxl")
    if not os.path.exists(path):
        subprocess.check_call([SYNTH_TOOL, "--width", str(w), "--height", str(h), "--seed", str(seed), "--distance", str(distance),
                               "-o", path] + list(extra), stderr=subprocess.DEVNULL)
    with open(path, "rb") as f:
        return f.read()


def load_workload(name, nframes=16):
    """Returns (description, list of encoded frames (bytes) for ONE step on ONE GPU, (w, h) per frame)."""
    if name == "mosaic8k":
        with open(os.path.join(GOLDEN, "benchmark-data", "starrail.d1-e6.jxl"), "rb") as f:
            tile = f.read()
        desc = ("8K-equivalent (33.18 MP/step/GPU): 3x3 mosaic of a real libjxl VarDCT d1.0 2560x1440 frame "
                "(starrail.d1-e6.jxl, Gaborish + EPF), decoded as 9 independent frames")
        return desc, [tile] * 9, (2560, 1440)
    if name in ("synth8k", "synth4k", "synth8k_d2"):
        w, h = (3840, 2160) if name == "synth4k" else (7680, 4320)
        d2 = name == "synth8k_d2"  # BASELINE config #3: d2.0, the full filter chain (EPF 3 iterations: steps 0, 1, 2)
        frames = []
        for seed in (1, 2, 3, 4):
            frames.append(synth_frame(w, h, seed, distance=2.0, extra=("--epf-iters", "3")) if d2 else synth_frame(w, h, seed))
        frames = [frames[i % len(frames)] for i in range(max(1, nframes))]
        bpp = sum(len(f) for f in frames) * 8.0 / (w * h * len(frames))
        desc = (f"{w}x{h} VarDCT d{'2.0' if d2 else '1.0'} synthetic encoded frames (tools/synth_enc.cc seeds 1-4, {bpp:.2f} bit/px, "
                f"libjxl-like: WP-coded LF, mixed varblocks 8x8..64x64, Gaborish + EPF {3 if d2 else 2} iters), "
                f"{len(frames)} independent frames per step")
        return desc, frames, (w, h)
    if name == "synthmod4k":  # BASELINE config #4: Modular lossless, RCT + default Squeeze + weighted predictor
        w, h = 3840, 2160
        frames = [synth_frame(w, h, seed, extra=("--modular",)) for seed in (1, 2, 3, 4)]
        frames = [frames[i % len(frames)] for i in range(max(1, nframes))]
        bpp = sum(len(f) for f in frames) * 8.0 / (w * h * len(frames))
        desc = (f"{w}x{h} Modular lossless RGB 8-bit synthetic frames (tools/synth_enc.cc --modular, seeds 1-4, {bpp:.2f} bit/px: "
                "YCoCg RCT, default Squeeze schedule, weighted predictor under a WP-error context chain, 135 pass groups + 4 LF "
                f"groups), {len(frames)} independent frames per step")
        return desc, frames, (w, h)
    if name.startswith("file:"):
        with open(name[5:], "rb") as f:
            data = f.read()
        import oracle_lib
        img = oracle_lib.OracleImage(data, output_colour=2, threads=os.cpu_count())
        return f"file {name[5:]}", [data], (img.width, img.height)
    raise SystemExit(f"unknown workload {name}")


# ----------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons during the timed region, from ONE long-running `nvidia-smi -lms 200` process
    (the profiling recipe's clocks line) - starting a new nvidia-smi per sample re-initialises NVML each time and
    perturbs the run it is supposed to observe."""

    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu_index, uuid=None):
        # `uuid` ("GPU-...") identifies the CUDA device whatever CUDA_VISIBLE_DEVICES remaps; else the index is used
        self.gpu = uuid or gpu_index
        self.index = gpu_index
        self.proc = None
        self.lines = []
        self.reader = None

    def _start_nvml(self):
        """In-process NVML (what nvidia-smi itself reads): one init, then cheap polls every 200 ms."""
        import pynvml
        pynvml.nvmlInit()
        try:
            h = (pynvml.nvmlDeviceGetHandleByUUID(self.gpu) if isinstance(self.gpu, str)
                 else pynvml.nvmlDeviceGetHandleByIndex(self.gpu))
        except Exception:
            if not isinstance(self.gpu, str):
                raise
            self.gpu = self.index  # the UUID did not resolve: fall back to the CUDA ordinal
            h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
        pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)  # raises when unsupported
        bits = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}
        self.nvml_samples, self.nvml_reasons, self.nvml_max, self.nvml_util = [], set(), None, []
        self._halt = threading.Event()

        def poll():
            while not self._halt.is_set():
                try:
                    self.nvml_samples.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                    self.nvml_max = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
                    self.nvml_util.append(float(pynvml.nvmlDeviceGetUtilizationRates(h).gpu))
                    mask = int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                    for n, b in bits.items():
                        if mask & b:
                            self.nvml_reasons.add(n)
                except Exception:
                    pass
                self._halt.wait(0.2)
        self.nvml_thread = threading.Thread(target=poll, daemon=True)
        self.nvml_thread.start()

    def start(self):
        self.nvml_thread = None
        try:
            self._start_nvml()
            return
        except Exception:
            self.nvml_thread = None
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["stdbuf", "-oL", "nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return

        def pump():
            try:
                for line in self.proc.stdout:
                    self.lines.append(line)
            except Exception:
                pass
        self.reader = threading.Thread(target=pump, daemon=True)
        self.reader.start()

    def stop(self):
        if self.nvml_thread is not None:
            self._halt.set()
            self.nvml_thread.join(timeout=5)
            if self.nvml_samples:
                return {"sm_mhz": float(np.median(self.nvml_samples)), "sm_max_mhz": self.nvml_max,
                        "reasons": sorted(self.nvml_reasons), "samples": len(self.nvml_samples),
                        "gpu_busy_pct_mean": (float(np.mean(self.nvml_util)) if self.nvml_util else None),
                        "how": "NVML polled every 200 ms during the timed region"}
        if self.proc is not None:
            try:
                self.proc.terminate()  # the exact process started above
                self.proc.wait(timeout=5)
            except Exception:
                pass
            if self.reader is not None:
                self.reader.join(timeout=5)
        mode = "nvidia-smi -lms 200 during the timed region"
        if not self.lines:  # nothing arrived through the pipe: one query right after the region instead
            mode = "single nvidia-smi query right after the timed region"
            try:
                q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                     "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
                self.lines = [subprocess.run(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                             capture_output=True, text=True, timeout=10).stdout]
            except Exception:
                self.lines = []
        samples, reasons, max_mhz = [], set(), None
        for line in self.lines:
            out = [x.strip() for x in line.strip().split(",")]
            try:
                samples.append(float(out[0]))
                max_mhz = float(out[1])
            except (ValueError, IndexError):
                continue
            for n, v in zip(self.NAMES, out[2:]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        med = float(np.median(samples)) if samples else None
        return {"sm_mhz": med, "sm_max_mhz": max_mhz, "reasons": sorted(reasons), "samples": len(samples), "how": mode}


def algorithmic_bytes(kernel, w, h, stream_bytes):
    """Algorithmic HBM bytes of ONE frame for a kernel family (DESIGN.md 'Kernels')."""
    px = w * h
    lf = ((w + 7) // 8) * ((h + 7) // 8)
    table = {
        "modular_decode": stream_bytes * 0.12 + lf * 3 * 4 + lf * 4 + (px / 4096) * 8,  # LF + HfMetadata streams
        "decode_hf": stream_bytes * 0.88 + px * 12,       # HF sections read, 3 x i32 coefficients written
        "build_block_info": lf * 4 * 4,
        "hf_block_ctx": lf * 6 * 4,                        # type, multiplier, 3 quantised LF read, 1 word written
        "hf_dequant_cfl": px * 24,
        "hf_transform": px * 24 + lf * 12,
        "filters_fused": px * 24,                          # Gaborish + EPF + colour in one pass
        "gaborish": px * 24,                               # 3 launches x 8 B/px
        "epf_step": px * 24,
        "xyb_to_rgb": px * 24,
        "lf_dequant": lf * 24, "lf_cfl": lf * 24, "lf_smooth": lf * 24,
    }
    return table.get(kernel)


KERNELS = ["modular_decode", "build_block_info", "hf_block_ctx", "decode_hf", "lf_dequant", "lf_cfl", "lf_smooth", "hf_dequant_cfl",
           "hf_transform", "filters_fused", "gaborish", "epf_step", "xyb_to_rgb", "copy_rect", "squeeze_inverse", "rct_inverse",
           "int_to_float", "modular_xyb", "palette_inverse_simple"]


def gpu_local_cpus(device_index):
    """CPUs local to the GPU's PCIe root (sysfs); empty when the topology cannot be read."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(device_index).pci_bus_id
        dom = getattr(torch.cuda.get_device_properties(device_index), "pci_domain_id", 0)
        devid = getattr(torch.cuda.get_device_properties(device_index), "pci_device_id", 0)
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{devid:02x}.0/local_cpulist"
        out = []
        for part in open(path).read().strip().split(","):
            a, _, b = part.partition("-")
            out.extend(range(int(a), int(b or a) + 1))
        return out
    except Exception:
        return []


# HF coefficient schedule of the timed run: fixed, never probed inside the bench. 128 = one THREAD per stream (32 streams per
# warp): a frame's 510 streams then take 16 warps for ~42 ms instead of 510 one-lane warps for ~14 ms. With ~26 frames
# in their heavy stage the one-lane form alone asks for more warp slots than the GPU has (26 x 510 > 148 x 64) and starves
# the pixel kernels; measured whole-job (profiles/r02_progress.md section 6): 185-197 frames/s against 116-167.
# jxlb_decode (one frame, latency matters) keeps the 16-warp form.
HF_STREAMS_PER_CTA = 128
HF_LATENCY_SCHEDULE = 16
CHAIN = ["hf_dequant_cfl", "hf_transform", "filters_fused", "gaborish", "epf_step", "xyb_to_rgb"]
# Modular frames: the HBM-bound part is everything after the entropy decode (inverse Squeeze, RCT, sample conversion)
MODULAR_CHAIN = ["squeeze_inverse", "rct_inverse", "int_to_float", "copy_rect", "modular_xyb", "palette_inverse_simple"]
ENTROPY = ["modular_decode", "build_block_info", "decode_hf"]


def run_ours(args, rank, world, local_rank):
    import torch
    import jxl_oxide_b200 as J
    from jxl_oxide_b200 import build as jb
    if not os.path.exists(J.LIB_PATH):
        jb.build()
    torch.cuda.set_device(local_rank)
    cpus = gpu_local_cpus(local_rank)
    if cpus:
        try:
            os.sched_setaffinity(0, cpus)  # this process (and the pinned buffers it touches first) next to its GPU
        except Exception:
            cpus = []
    env_knob = os.environ.get("JXLB_HF_LANES")
    hf_lanes = int(env_knob) if env_knob is not None else (HF_STREAMS_PER_CTA if args.hf_lanes == "auto" else int(args.hf_lanes))
    desc, frames, (w, h) = load_workload(args.workload, args.frames_per_step)
    px_per_frame = w * h
    workers = args.contexts or (64 if "mod" in args.workload else 96)
    heavy = args.heavy_frames or 26  # + 6 batch streams = the device's 32 hardware queues
    args.contexts, args.heavy_frames = workers, heavy
    pipe = J.Pipeline(local_rank, workers=workers, heavy_frames=heavy, hf_streams_per_cta=hf_lanes, batch_streams=args.batch_streams)
    # encoded frames resident in HBM ("inputs already resident"): one preloaded slot per distinct frame
    distinct = {}
    slots = []
    for f in frames:
        if id(f) not in distinct:
            distinct[id(f)] = len(distinct)
            pipe.preload(distinct[id(f)], f)
        slots.append(distinct[id(f)])

    def run_steps(mode, nsteps):
        """`nsteps` passes over the batch, frames flowing through the pipeline without a barrier between steps
        (the contract's barriers sit on both sides of the K timed steps)."""
        total = nsteps * len(frames)
        sent = 0
        got = 0
        checksum = 0
        # keep the queue a few steps deep at most: submission is cheap, but host buffers of submitted e2e jobs are not
        depth = max(2 * pipe.workers(), 64)
        while got < total:
            while sent < total and sent - got < depth:
                k = sent % len(frames)
                if mode == "value":
                    pipe.submit(slot=slots[k])
                elif mode == "e2e":
                    pipe.submit(data=frames[k], mode=J.Pipeline.OUT_PLANAR_F32)   # host bytes in, planar f32 to pinned host
                else:
                    pipe.submit(data=frames[k], mode=J.Pipeline.OUT_U8)           # host bytes in, interleaved u8 to pinned host
                sent += 1
            if mode == "value":
                pipe.wait()
            else:
                _, addr, nbytes = pipe.wait(want_output=True)
                checksum ^= nbytes  # the pixels are in host memory here; hand the buffer back to the ring
                pipe.release_output(addr)
            got += 1
        return checksum

    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(mode, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run_steps(mode, steps)
        torch.cuda.synchronize()
        e1.record()
        e1.synchronize()
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms], device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    run_steps("value", max(1, args.warmup))
    launches0 = pipe.launch_count()
    try:
        dev_uuid = "GPU-" + str(torch.cuda.get_device_properties(local_rank).uuid)
    except Exception:
        dev_uuid = None
    sampler = ClockSampler(local_rank, dev_uuid)
    sampler.start()
    ms = timed("value", args.steps)
    clocks = sampler.stop()
    launches = pipe.launch_count() - launches0
    run_steps("e2e", 1)
    ms_e2e = timed("e2e", args.steps)
    run_steps("u8", 1)
    ms_e2e_u8 = timed("u8", args.steps)

    # per-kernel device time (CUDA events on each worker's stream) of one extra step under full load, then of one frame
    # alone on the GPU. Profiling is off during the timed steps: an event pair per launch costs stream concurrency.
    decs = [pipe.decoder(i) for i in range(pipe.workers())]
    for d in decs:
        d.set_profile(True)
        d.profile_reset()
    run_steps("value", 1)
    prof = {}
    for k in KERNELS:
        n = sum(d.profile(k)[0] for d in decs)
        t = sum(d.profile(k)[1] for d in decs)
        if n:
            prof[k] = {"launches": n, "ms": t}
    for d in decs:
        d.profile_reset()
    solo_reps = 3
    for _ in range(solo_reps):
        pipe.submit(slot=slots[0])
        pipe.wait()
    solo = {}
    for k in KERNELS:
        n = sum(d.profile(k)[0] for d in decs)
        t = sum(d.profile(k)[1] for d in decs)
        if n:
            solo[k] = t / solo_reps
    for d in decs:
        d.set_profile(False)
    # the same HF streams under the single-frame (latency) schedule, one frame alone
    hf_latency_ms = None
    if "decode_hf" in solo and hf_lanes != HF_LATENCY_SCHEDULE:
        for d in decs:
            d._L.jxlb_set_hf_streams_per_cta(d._h, HF_LATENCY_SCHEDULE)
            d.set_profile(True)
            d.profile_reset()
        for _ in range(2):
            pipe.submit(slot=slots[0])
            pipe.wait()
        n = sum(d.profile("decode_hf")[0] for d in decs)
        if n:
            hf_latency_ms = sum(d.profile("decode_hf")[1] for d in decs) / n
        for d in decs:
            d.set_profile(False)
            d._L.jxlb_set_hf_streams_per_cta(d._h, hf_lanes)

    total_px = px_per_frame * len(frames) * world
    gather = None
    if args.gather != "none":
        gather = run_gather(args, torch, dist, J, local_rank, world, rank, frames, total_px, barrier, hf_lanes)
    value = total_px / (ms / args.steps / 1e3) / 1e6
    e2e_value = total_px / (ms_e2e / args.steps / 1e3) / 1e6
    e2e_u8_value = total_px / (ms_e2e_u8 / args.steps / 1e3) / 1e6
    u8_bytes = px_per_frame * 3
    if args.dump_outputs and rank == 0:
        dump_outputs(pipe, slots, w, h, args.dump_outputs)
    pipe.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("hbm_gbs", 6650.0)
    peak_source = "MEASURED_PEAKS.json hbm_gbs (burst copy bandwidth)" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    # The dominant HBM-bound work: the pixel chain coefficients -> RGB planes (SURVEY 8d: 24.3 B/px when fully fused).
    # One "launch" = the chain's kernels for one frame; duration = the sum of their CUDA-event times.
    modular = "mod" in args.workload
    chain = MODULAR_CHAIN if modular else CHAIN
    # Modular: 4 B/sample of decoded residuals read + 4 B/sample of f32 output written, three channels, when Squeeze, RCT
    # and the sample conversion are fully fused (SURVEY 8d)
    chain_bytes = px_per_frame * (24.0 if modular else 24.3)
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        if tj.get("workload") == args.workload:
            traffic = tj.get("chain_dram_bytes_per_frame")
    except Exception:
        pass
    roofline = None
    chain_solo_ms = sum(solo.get(k, 0.0) for k in chain)
    chain_load_ms = sum(prof[k]["ms"] for k in chain if k in prof) / max(1, len(frames))
    if chain_solo_ms > 0:
        ach = chain_bytes / (chain_solo_ms / 1e3) / 1e9
        roofline = {"kernel": "+".join(k for k in chain if k in solo), "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s",
                    "frac": ach / peak, "traffic": traffic, "peak_source": peak_source,
                    "bytes_per_launch": chain_bytes, "avg_launch_ms": chain_solo_ms,
                    "per_kernel_ms": {k: round(solo[k], 4) for k in chain if k in solo},
                    "measured": "CUDA events around the chain's launches, one frame alone on the GPU (mean of 3)",
                    "under_load": {"avg_launch_ms": chain_load_ms, "achieved": chain_bytes / (chain_load_ms / 1e3) / 1e9 if chain_load_ms else None,
                                   "note": "same kernels during one step with every worker busy: event times include waiting "
                                           "for SMs held by other frames' kernels"},
                    "bound_note": None if modular else
                                  ("reported against the HBM roof as the contract asks; the chain itself is fp32-issue bound: the bit-exact "
                                   "(un-fused) filter + colour formula needs ~330 fp32 instructions per pixel = 0.29 ms per 8K frame at "
                                   "148 SMs x 128 lanes x 1.97 GHz, 2.4x the 0.12 ms of the 24.3 B/px at HBM peak (DESIGN.md section 4)"),
                    "algorithmic_bytes": ("24 B/px x pixels: 3 x 4 B decoded residuals read, 3 x 4 B f32 samples written (Squeeze, RCT and "
                                          "sample conversion fully fused)") if modular else
                                         "24.3 B/px x pixels: 12 B coefficients + 0.33 B LF/meta read, 12 B RGB written (fully fused chain)"}
    entropy = None
    try:
        sym = json.load(open(os.path.join(ROOT, "profiles", "r02_symbols.json"))).get(args.workload)
    except Exception:
        sym = None
    ent_solo = {k: round(solo[k], 3) for k in ENTROPY if k in solo}
    if ent_solo:
        entropy = {"bound": "latency", "ms_per_frame_solo": ent_solo,
                   "ms_per_frame_under_load": {k: round(prof[k]["ms"] / len(frames), 3) for k in ENTROPY if k in prof},
                   "note": "serial ANS / context chains (one per LF-group stream, one per 256x256 group): reported as "
                           "symbols/s, not against the HBM roofline"}
        if hf_latency_ms is not None:
            entropy["decode_hf_ms_solo_latency_schedule"] = round(hf_latency_ms, 3)
            entropy["hf_schedules"] = ("timed run: one thread per stream (hf_streams_per_cta=%d); latency schedule: one warp per "
                                       "stream, %d per CTA (what jxlb_decode uses)" % (hf_lanes, HF_LATENCY_SCHEDULE))
        if sym and "decode_hf" in solo:
            entropy["hf_symbols_per_frame"] = sym.get("hf_symbols")
            entropy["hf_symbols_per_s_solo"] = sym.get("hf_symbols", 0) / (solo["decode_hf"] / 1e3)
            entropy["hf_symbols_per_s_whole_job"] = sym.get("hf_symbols", 0) * len(frames) * world / (ms / args.steps / 1e3)
        if sym and "modular_decode" in solo:
            n = sym.get("lf_samples") or sym.get("modular_samples") or 0
            entropy["modular_samples_per_frame"] = n
            entropy["modular_samples_per_s_solo"] = n / (solo["modular_decode"] / 1e3)
            entropy["modular_samples_per_s_whole_job"] = n * len(frames) * world / (ms / args.steps / 1e3)
        if sym:
            entropy["symbol_counts"] = "profiles/r02_symbols.json (" + str(sym.get("how")) + ")"
    # the CPU leg runs beside the 1-GPU line only (rank 0, N = 1); the driver's reference arm covers the other N
    cpu = cpu_baseline(args, frames, px_per_frame) if (not args.no_cpu_baseline and world == 1) else None
    line = {
        "metric": METRIC.get(args.workload, "Megapixels/s decoded"), "value": value, "unit": "MP/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32" if "mod" not in args.workload else "i32",
        "data": "synthetic" if "synth" in args.workload else "real-file mosaic",
        "config": {"workload": desc, "frames_per_step_per_gpu": len(frames), "pipeline_workers_per_gpu": pipe_workers(args),
                   "heavy_frames_per_gpu": args.heavy_frames, "lf_batch_streams": args.batch_streams,
                   "cache": "inputs+planes per step (>= 33 MP x 24 B) exceed L2 (126 MB); no explicit L2 flush",
                   "step_barrier": "before and after the K timed steps; frames flow through the in-library pipeline",
                   "hf_streams_per_cta": hf_lanes, "cpu_affinity": "GPU-local CPUs" if cpus else "unchanged"},
        "e2e": {"value": e2e_value, "unit": "MP/s", "h2d_bytes_per_step": int(sum(len(f) for f in frames)),
                "d2h_bytes_per_step": int(px_per_frame * 12 * len(frames)), "ms_per_step": ms_e2e / args.steps,
                "path": "jxlb_pipeline_submit(host bytes) -> planar f32 in pinned host memory (jxlb_pipeline_wait)"},
        "e2e_u8": {"value": e2e_u8_value, "unit": "MP/s", "h2d_bytes_per_step": int(sum(len(f) for f in frames)),
                   "d2h_bytes_per_step": int(u8_bytes) * len(frames), "ms_per_step": ms_e2e_u8 / args.steps,
                   "note": "same call path, output = interleaved 8-bit RGB packed on the device (ImageStream::write_to_buffer::<u8>); "
                           "reported beside e2e, not instead of it"},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "entropy": entropy,
        "kernel_ms_per_step_summed_over_streams": {k: round(v["ms"], 3) for k, v in prof.items()},
        "kernel_ms_per_frame_solo": {k: round(v, 3) for k, v in solo.items()}, "cpu_baseline": cpu,
    }
    if gather is not None:
        line["gather"] = gather
    print(json.dumps(line))


def dump_outputs(pipe, slots, w, h, out_dir):
    """--dump-outputs: the planar f32 frame (channels, h, w) a caller of the timed path receives, for every frame of one
    step, as out_dir/frame_<k>.npy. The timed steps leave their frames in HBM and release them, so the step is decoded
    once more through the same pipeline with each frame copied to host memory; the inputs and the decode are
    deterministic, so these are the last timed step's outputs. Every frame is sampled at the same seeded pixel positions,
    keeping the files within DUMP_BYTES in all."""
    os.makedirs(out_dir, exist_ok=True)
    for k, slot in enumerate(slots):
        pipe.submit(slot=slot, mode=pipe.OUT_PLANAR_F32, tag=k)
    pos = None
    while pipe.in_flight:
        k, addr, nbytes = pipe.wait(want_output=True)
        try:
            planes = np.ctypeslib.as_array((ctypes.c_float * (nbytes // 4)).from_address(addr)).reshape(-1, w * h)
            if pos is None:
                pos = dump_positions(w * h, planes.shape[0], len(slots))
            np.save(os.path.join(out_dir, f"frame_{k:03d}.npy"), planes[:, pos])
        finally:
            pipe.release_output(addr)


DUMP_BYTES = 48 << 20


def dump_positions(npx, channels, nframes):
    """Sorted pixel indices of the --dump-outputs sample: all of a frame when it fits, else a seeded subset."""
    n = min(npx, DUMP_BYTES // (nframes * channels * 4))
    return np.sort(np.random.default_rng(0).choice(npx, size=n, replace=False))


def pipe_workers(args):
    return args.contexts


METRIC = {"synth8k": "Megapixels/s decoded (8K VarDCT d1.0)", "synth4k": "Megapixels/s decoded (4K VarDCT d1.0)",
          "synth8k_d2": "Megapixels/s decoded (8K VarDCT d2.0, EPF 3 iterations)",
          "synthmod4k": "Megapixels/s decoded (4K Modular lossless, Squeeze + weighted predictor)",
          "mosaic8k": "Megapixels/s decoded (8K VarDCT d1.0)"}


def run_gather(args, torch, dist, J, local_rank, world, rank, frames, total_px, barrier, hf_lanes):
    """BASELINE config #5's delivery: every frame is packed on its GPU (interleaved u8 / u16: 3-6 B/px instead of the
    12 B/px of f32 planes) straight into a device tensor by the frame pipeline (out_mode 4 / 5) and gathered to rank 0
    over NCCL, one `gather` per round of world_size frames (jxl_oxide_b200.sharding.gather_frames). The rounds are
    fed as the frames come out of the pipeline, so the gather of round r overlaps the decode of the later frames."""
    from jxl_oxide_b200 import sharding
    tdt = torch.uint8 if args.gather == "u8" else torch.uint16
    pipe = J.Pipeline(local_rank, workers=args.contexts, heavy_frames=args.heavy_frames, hf_streams_per_cta=hf_lanes,
                      batch_streams=args.batch_streams)
    distinct, slots = {}, []
    for f in frames:
        if id(f) not in distinct:
            distinct[id(f)] = len(distinct)
            pipe.preload(distinct[id(f)], f)
        slots.append(distinct[id(f)])
    d0 = J.Decoder(local_rank)
    d0.decode(frames[0])
    shape = tuple(d0.frame_to_buffer(0, np.uint8).shape)
    d0.close()
    bufs = [[torch.empty(shape, dtype=tdt, device=f"cuda:{local_rank}") for _ in frames] for _ in range(2)]
    state = {"step": 0}

    def decode_step(with_gather):
        cur = bufs[state["step"] & 1]
        state["step"] += 1
        done = set()
        for k in range(len(frames)):
            pipe.submit(slot=slots[k], out=cur[k], tag=k)

        def getter(k):
            def g():
                while k not in done:
                    done.add(pipe.wait())
                return cur[k]
            return g
        if with_gather:
            got = sharding.gather_frames([getter(k) for k in range(len(frames))], len(frames) * world, dst=0)
        else:
            got = None
        pipe.drain()
        return got

    got = decode_step(True)
    barrier()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    for _ in range(args.steps):
        got = decode_step(True)
    torch.cuda.synchronize()
    g1.record()
    g1.synchronize()
    tg = torch.tensor([g0.elapsed_time(g1)], device="cuda")
    if dist is not None:
        dist.all_reduce(tg, op=dist.ReduceOp.MAX)
    ms_g = float(tg.item())
    # decode + pack without the collective: what the gather adds
    barrier()
    d0e, d1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    d0e.record()
    for _ in range(args.steps):
        decode_step(False)
    torch.cuda.synchronize()
    d1e.record()
    d1e.synchronize()
    td = torch.tensor([d0e.elapsed_time(d1e)], device="cuda")
    if dist is not None:
        dist.all_reduce(td, op=dist.ReduceOp.MAX)
    ms_d = float(td.item())
    nbytes = int(bufs[0][0].numel() * bufs[0][0].element_size())
    pipe.close()
    return {"value": total_px / (ms_g / args.steps / 1e3) / 1e6, "unit": "MP/s", "ms_per_step": ms_g / args.steps,
            "decode_pack_only": {"value": total_px / (ms_d / args.steps / 1e3) / 1e6, "ms_per_step": ms_d / args.steps},
            "format": f"{args.gather} interleaved RGB, packed on the device by the pipeline (out_mode 4/5)",
            "bytes_to_rank0_per_step": nbytes * len(frames) * (world - 1),
            "nvlink_gb_s_into_rank0": nbytes * len(frames) * (world - 1) / (ms_g / args.steps / 1e3) / 1e9,
            "collective": "torch.distributed gather (nccl), one per round of world_size frames, overlapped with the decode of later frames"
                          if world > 1 else "none (1 rank)",
            "frames_at_rank0": (len([g for g in got if g is not None]) if got is not None else 0) if rank == 0 else None}


def cpu_throughput(frames, px_per_frame, steps, warm=1):
    """The CPU restatement at its best on this host: frame-level parallelism (what the reference's CLI does across
    keyframes, jxl-oxide-cli/src/decode.rs:293-301) on top of the per-frame thread pool. The restatement's intra-frame
    scaling flattens after a few threads (measured: 1.5x at 8 threads), so the cores are split into P concurrent
    frames x T threads each. One step = P frames of the workload, each decoded once (bytes -> planar f32)."""
    import oracle_lib
    oracle_lib.build()
    cores = os.cpu_count() or 1
    t_per_frame = 4 if cores >= 4 else cores
    par = max(1, cores // t_per_frame)
    try:  # keep P concurrent decodes (~64 B of planes per pixel each) within half of the free host memory
        import psutil
        par = max(1, min(par, int(psutil.virtual_memory().available * 0.5 // (px_per_frame * 64))))
    except Exception:
        par = min(par, 16)
    sample = [frames[i % len(frames)] for i in range(par)]

    def one_step():
        errs = []

        def work(f):
            try:
                oracle_lib.OracleImage(f, threads=t_per_frame).close()
            except Exception as e:  # noqa: BLE001
                errs.append(e)
        ts = [threading.Thread(target=work, args=(f,)) for f in sample]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        if errs:
            raise errs[0]
    for _ in range(warm):
        one_step()
    t0 = time.time()
    for _ in range(steps):
        one_step()
    dt = (time.time() - t0) / steps
    value = px_per_frame * par / dt / 1e6
    return value, dt, {"value": value, "unit": "MP/s", "cores": par * t_per_frame, "kind": "port",
                       "sample": f"{par} frame(s) of the step's workload decoded concurrently, {t_per_frame} threads each "
                                 f"({cores} host cores), decode chain only (bytes -> planar f32); CPU restatement of "
                                 "jxl-oxide's generic path (not jxl-oxide itself: no Rust toolchain)"}


def cpu_baseline(args, frames, px_per_frame, steps=1):
    return cpu_throughput(frames, px_per_frame, steps)[2]


def run_reference(args, rank, world):
    if rank != 0:
        return
    desc, frames, (w, h) = load_workload(args.workload, args.frames_per_step)
    value, dt, cpu = cpu_throughput(frames, w * h, max(1, args.steps), warm=max(1, min(args.warmup, 1)))
    print(json.dumps({
        "impl": "reference", "metric": METRIC.get(args.workload, "Megapixels/s decoded"), "value": value, "unit": "MP/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic" if "synth" in args.workload else "real-file mosaic",
        "config": {"workload": desc, "note": "CPU restatement of jxl-oxide's generic render path, all host cores: "
                                              "concurrent frames x per-frame thread pool"},
        "cpu_baseline": cpu,
        "e2e": {"value": value, "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="synth8k", help="synth8k | synth4k | mosaic8k | file:PATH")
    ap.add_argument("--contexts", type=int, default=0, help="pipeline workers = frames in flight per GPU (0: 96, Modular workloads 64)")
    ap.add_argument("--heavy-frames", type=int, default=0,
                    help="heavy slots (HBM slab + CUDA stream) per GPU (0: 20, Modular workloads 26)")
    ap.add_argument("--batch-streams", type=int, default=6, help="CUDA streams of the LF batch service")
    ap.add_argument("--frames-per-step", type=int, default=96, help="independent frames decoded per step per GPU")
    ap.add_argument("--cpu-sample-frames", type=int, default=1)
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU leg (experiments only)")
    ap.add_argument("--gather", default="none", choices=["none", "u8", "u16"],
                    help="also time decode + device-side packing + NCCL gather of every frame to rank 0 (BASELINE config #5)")
    ap.add_argument("--hf-lanes", default="auto", choices=["auto", "0", "8", "16", "32", "64", "128"],
                    help="HF coefficient schedule = streams per CTA: 0 (= 4) / 8 / 16 one warp per stream, 32 / 64 / 128 one "
                         "thread per stream; auto = the fixed default (HF_STREAMS_PER_CTA). JXLB_HF_LANES in the environment "
                         "overrides.")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the frames of one step as DIR/frame_<k>.npy: planar f32 "
                         "(channels, samples), the same seeded sample of pixels in every frame, at most %d MiB in all"
                         % (DUMP_BYTES >> 20))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
