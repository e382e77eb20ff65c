#!/usr/bin/env python
"""bench.py -- bone-poses/s of the batched seek + decompress_tracks hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--workload c2|c3|c5|c4] [--impl reference]

One "step" = one pass of the hot path over the whole request batch of the workload:
    c2 (default, BASELINE.json configs[1]): 10 000 clips x 100 bones x 60 samples, variable bit rate + range reduction,
        600 000 requests = every clip x every (s + u) / 30 s, u ~ U[0, 1)  -> 60 M bone-poses per step per GPU
    c3: 1 000 clips x 540 bones, 60 000 requests        c5: 125 000 clips x 30 bones x 32 samples per GPU, one random time per clip
    c4: scalar float1f 4096 tracks x 1024 samples replicated x64, 65 536 requests (unit: track-samples/s)
Inputs are SYNTHETIC clips compressed by the reference compressor (oracle/_ref, outside every timed region); when that
library is absent the committed golden clip of the same shape is replicated at distinct addresses instead (config.clips says which).

Default arm: the CUDA product through the C ABI (acl_b200). `value` = whole-job bone-poses/s with inputs resident in HBM,
`e2e` = the same through aclb200_decompress_tracks_host with pinned HOST buffers (H2D of the requests + D2H of every pose inside
the timed region). `--impl reference` times the reference's own CPU implementation (oracle/_ref: acl::decompression_context with the
benchmark settings of tools/acl_decompressor/sources/benchmark.cpp:94-101) on all host threads for the same workload.
Multi-GPU (torchrun, one rank per GPU): clips shard by rank with no data-path collective (weak scaling); NCCL carries only the
barrier and the max-over-ranks of the device time.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
ROUND = 2       # profiles/traffic_*.json of another round are reported as stale

WORKLOADS = {
    # name: (kind, clips per GPU, bones, samples, description)
    "c2": ("transform", 10000, 100, 60, "C2: 10k clips x 100 bones x 60 samples, variable bit rate + range reduction, 600k requests (every clip x every (s+u)/30)"),
    "c3": ("transform", 1000, 540, 60, "C3: 1k clips x 540 bones x 60 samples, quatf_drop_w_variable + segmenting, 60k requests"),
    "c5": ("transform", 125000, 30, 32, "C5: 125k clips per GPU x 30 bones x 32 samples, one random sample_time per clip"),
    "c4": ("scalar", 64, 4096, 1024, "C4: scalar float1f 4096 tracks x 1024 samples replicated x64, 65536 requests"),
}
GOLDEN_FALLBACK = {"c2": "c2_100bones", "c3": "paragon_like", "c5": "c5_30x32", "c4": "float1_c4_small"}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ------------------------------------------------------------------------------------------------------------------
# workload synthesis (never timed)
# ------------------------------------------------------------------------------------------------------------------
def make_workload(name: str, rank: int, clips_override: int | None, world: int = 1, replicated: bool = False):
    """`replicated`: the committed golden clip even when the reference compressor is available (the request list is the same)."""
    kind, num_clips, bones, samples, description = WORKLOADS[name]
    if clips_override:
        num_clips = clips_override
    from oracle import ref
    distinct = ref.available() and not replicated
    if kind == "transform":
        if distinct:
            spec = ref.TransformSpec(num_tracks=bones, num_samples=samples, seed={"c2": 2000, "c3": 3000, "c5": 5000}[name] + rank * num_clips)
            if name == "c3":
                spec.scale_default_pct, spec.scale_constant_pct = 95, 0       # 5 % animated scale (SURVEY 8d)
            t0 = time.time()
            # the ranks of one box share its host cores
            buffer, offsets, sizes = ref.compress_transform_batch(spec, num_clips, num_threads=max(1, (os.cpu_count() or 1) // max(world, 1)))
            log(f"[bench] rank {rank}: compressed {num_clips} clips with the reference in {time.time() - t0:.1f} s ({buffer.size / 1e6:.1f} MB)")
        else:
            buffer, offsets, sizes = replicate_golden(GOLDEN_FALLBACK[name], num_clips)
        rng = np.random.default_rng({"c2": 7, "c3": 7, "c5": 11}[name] + rank)
        if name == "c5":
            req_clip = np.arange(num_clips, dtype=np.uint32)
            req_time = (rng.random(num_clips) * ((samples - 1) / 30.0)).astype(np.float32)
        else:
            req_clip = np.repeat(np.arange(num_clips, dtype=np.uint32), samples)
            s = np.tile(np.arange(samples, dtype=np.float64), num_clips)
            req_time = ((s + rng.random(s.size)) / 30.0).astype(np.float32)
        num_tracks = bones
    else:
        if distinct:
            blob = ref.compress_scalar(ref.ScalarSpec(num_tracks=bones, num_samples=samples, seed=42, track_type=ref.TRACK_FLOAT1F, constant_pct=12, precision=0.001))
            buffer, offsets, sizes = replicate_blob(blob, num_clips)
        else:
            buffer, offsets, sizes = replicate_golden(GOLDEN_FALLBACK[name], num_clips)
            header = buffer[int(offsets[0]):int(offsets[0]) + 32].view(np.uint32)
            bones, samples = int(header[4]), int(header[5])
        rng = np.random.default_rng(42 + rank)
        req_clip = np.repeat(np.arange(num_clips, dtype=np.uint32), samples)
        s = np.tile(np.arange(samples, dtype=np.float64), num_clips)
        req_time = ((s + rng.random(s.size)) / 30.0).astype(np.float32)
        num_tracks = bones
    return dict(kind=kind, name=name, description=description, buffer=buffer, offsets=offsets, sizes=sizes, req_clip=req_clip,
                req_time=req_time, num_tracks=num_tracks, num_clips=num_clips, distinct=distinct and kind == "transform")


def replicate_blob(blob: np.ndarray, copies: int):
    stride = (blob.size + 63) & ~63
    raw = np.zeros(stride * copies + 128, dtype=np.uint8)
    shift = (-raw.ctypes.data) % 64
    buffer = raw[shift:shift + stride * copies + 64]
    for i in range(copies):
        buffer[i * stride:i * stride + blob.size] = blob
    return buffer, (np.arange(copies, dtype=np.uint64) * stride), np.full(copies, blob.size, dtype=np.uint32)


def replicate_golden(golden_name: str, copies: int):
    from tests import clips
    return replicate_blob(clips.load_blob(golden_name), copies)


# ------------------------------------------------------------------------------------------------------------------
# algorithmic bytes of one launch (SURVEY.md 8d: the reference's own decomp_touched_bytes, de-duplicated over the batch,
# plus 40 B per bone-pose written)
# ------------------------------------------------------------------------------------------------------------------
def gather_u32(buffer: np.ndarray, byte_offsets: np.ndarray) -> np.ndarray:
    idx = byte_offsets.astype(np.int64)[:, None] + np.arange(4, dtype=np.int64)[None, :]
    return buffer[idx].copy().view(np.uint32)[:, 0]


def algorithmic_bytes_transform(w) -> dict:
    buffer, offsets = w["buffer"], w["offsets"].astype(np.int64)
    req_clip, req_time = w["req_clip"].astype(np.int64), w["req_time"]
    f = lambda rel: gather_u32(buffer, offsets + rel).astype(np.int64)
    num_tracks, num_samples, misc = f(16), f(20), f(28)
    rate = gather_u32(buffer, offsets + 24).view(np.float32).astype(np.float64)
    nseg, nvar = f(32), f(36)
    nar, nat, nas = f(40), f(44), f(48)
    ncr, nct, ncs = f(52), f(56), f(60)
    seg_headers = f(68)
    has_scale = misc & 1
    rot_fmt = (misc >> 4) & 15
    trans_var, scale_var = (misc >> 3) & 1, (misc >> 2) & 1
    stripped = (misc >> 10) & 1
    hsize = np.where(stripped == 1, 20, 16)
    entries = (num_tracks + 15) // 16
    clip_bytes = 84 + np.where(nseg > 1, 4 * (nseg + 1), 0) + 4 * entries * np.where(has_scale == 1, 3, 2)
    clip_bytes = clip_bytes + np.where(rot_fmt == 0, 16, 12) * ncr + 12 * (nct + np.where(has_scale == 1, ncs, 0))
    clip_bytes = clip_bytes + np.where(rot_fmt == 3, 24 * nar, 0) + np.where(trans_var == 1, 24 * nat, 0) + np.where((has_scale == 1) & (scale_var == 1), 24 * nas, 0)
    seg_meta = hsize + nvar + np.where(nseg > 1, 6 * nvar, 0)

    # key frames touched by each request (clamp policy, no stripping: what the bench workloads contain)
    t = np.clip(req_time.astype(np.float64), 0.0, None)
    last = num_samples[req_clip] - 1
    k0 = np.minimum(np.floor(t * rate[req_clip]).astype(np.int64), last)
    k1 = np.minimum(k0 + 1, last)
    max_samples = int(num_samples.max()) + 1
    keys = np.unique(np.concatenate([req_clip * max_samples + k0, req_clip * max_samples + k1]))
    key_clip, key_frame = keys // max_samples, keys % max_samples

    # segment of each touched key frame and its pose size
    max_seg = int(nseg.max())
    starts = np.zeros((len(offsets), max_seg + 1), dtype=np.int64)
    pose_bits = np.zeros((len(offsets), max_seg), dtype=np.int64)
    for s in range(max_seg):
        valid = nseg > s
        pose_bits[valid, s] = gather_u32(buffer, offsets[valid] + 32 + seg_headers[valid] + s * hsize[valid])
        multi = valid & (nseg > 1)
        starts[multi, s] = gather_u32(buffer, offsets[multi] + 84 + 4 * s)
    starts[np.arange(len(offsets)), nseg] = np.iinfo(np.int64).max // 2
    for s in range(max_seg + 1):
        starts[nseg < s, s] = np.iinfo(np.int64).max // 2
    key_seg = (starts[key_clip] <= key_frame[:, None]).sum(axis=1) - 1
    key_seg = np.clip(key_seg, 0, None)
    key_bytes = (pose_bits[key_clip, key_seg] + 7) // 8
    touched_clips = np.unique(req_clip)
    touched_segments = np.unique(key_clip * (max_seg + 1) + key_seg)

    in_bytes = int(clip_bytes[touched_clips].sum() + seg_meta[touched_segments // (max_seg + 1)].sum() + key_bytes.sum())
    out_bytes = int((num_tracks[req_clip] * 40).sum())
    return dict(in_bytes=in_bytes, out_bytes=out_bytes, total=in_bytes + out_bytes, units=int(num_tracks[req_clip].sum()))


def algorithmic_bytes_scalar(w) -> dict:
    from tests import clips  # noqa: F401  (only for the lane constants elsewhere)
    buffer, offsets = w["buffer"], w["offsets"].astype(np.int64)
    req_clip, req_time = w["req_clip"].astype(np.int64), w["req_time"]
    o = int(offsets[0])
    hdr = buffer[o:o + 52].view(np.uint32)
    track_type, num_tracks, num_samples = int(buffer[o + 15]), int(hdr[4]), int(hdr[5])
    bits_per_frame, metadata = int(hdr[8]), int(hdr[9])
    comps = track_type + 1 if track_type <= 3 else 4
    rates = buffer[o + 32 + metadata:o + 32 + metadata + num_tracks]
    table = np.array([0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 32])
    bits = table[rates]
    per_clip = 52 + num_tracks + 4 * comps * int((bits == 0).sum()) + 8 * comps * int(((bits != 0) & (bits != 32)).sum())
    k0 = np.minimum(np.floor(np.clip(req_time.astype(np.float64), 0, None) * 30.0).astype(np.int64), num_samples - 1)
    k1 = np.minimum(k0 + 1, num_samples - 1)
    keys = np.unique(np.concatenate([req_clip * (num_samples + 1) + k0, req_clip * (num_samples + 1) + k1]))
    in_bytes = per_clip * len(np.unique(req_clip)) + len(keys) * ((bits_per_frame + 7) // 8)
    out_bytes = len(req_clip) * num_tracks * comps * 4
    return dict(in_bytes=int(in_bytes), out_bytes=int(out_bytes), total=int(in_bytes + out_bytes), units=len(req_clip) * num_tracks)


# ------------------------------------------------------------------------------------------------------------------
# clocks under load
# ------------------------------------------------------------------------------------------------------------------
MATH_DESCRIPTION = {
    "exact": "exact: every float bit-identical to the reference's SSE path (IEEE mul/add/sqrt/div in its order, never fused)",
    "fast": "fast: integer / format decode, translations and scales bit-exact; rotations use hardware sqrt / rsqrt and fused multiply-adds after "
            "the exact W-reconstruction input, <= 1e-5 absolute vs the reference (north star gate; measured < 2e-6, tests/test_gpu_parity.py::test_fast_math_within_tolerance)",
}


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region: an NVML polling thread (1 ms period, samples stamped with the host
    clock and filtered to the region), falling back to `nvidia-smi -lms` when the NVML binding is missing."""
    QUERY = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, device_index: int):
        self.device_index = device_index
        self.proc = None
        self.lines: list[str] = []
        self.nvml = None
        self.samples: list[tuple[float, int, int]] = []
        self.running = False
        self.window = (0.0, float("inf"))

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            index = int(visible.split(",")[self.device_index]) if visible and visible.replace(",", "").isdigit() else self.device_index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = int(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self.running = True
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.device_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll(self):
        nvml = self.nvml
        reasons_fn = getattr(nvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(nvml, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while self.running:
            try:
                self.samples.append((time.perf_counter(), int(nvml.nvmlDeviceGetClockInfo(self.handle, nvml.NVML_CLOCK_SM)), int(reasons_fn(self.handle))))
            except Exception:
                pass
            time.sleep(0.001)

    def mark(self, begin: float, end: float):
        """Host clock stamps (time.perf_counter) bracketing the timed region."""
        self.window = (begin, end)

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.nvml is not None:
            self.running = False
            self.thread.join(timeout=1)
            nvml = self.nvml
            inside = [s for s in self.samples if self.window[0] <= s[0] <= self.window[1]]
            if not inside:
                return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": ["no samples"]}
            masks = {"hw_slowdown": getattr(nvml, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                     "hw_thermal_slowdown": getattr(nvml, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                     "sw_thermal_slowdown": getattr(nvml, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                     "sw_power_cap": getattr(nvml, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
            reasons = sorted(label for label, mask in masks.items() if any(s[2] & mask for s in inside))
            return {"sm_mhz": float(np.median([s[1] for s in inside])), "sm_max_mhz": float(self.sm_max), "reasons": reasons,
                    "samples": len(inside), "source": "nvml, 1 ms polling inside the timed region"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, sm_max, reasons = [], [], set()
        for line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); sm_max.append(float(parts[2]))
            except ValueError:
                continue
            for label, value in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if value.lower().startswith("active"):
                    reasons.add(label)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(sm_max)), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline (oracle/_ref on the host cores)
# ------------------------------------------------------------------------------------------------------------------
def host_blobs(w):
    return [w["buffer"][int(o):int(o) + int(s)] for o, s in zip(w["offsets"], w["sizes"])]


def cpu_reference_pass(w, blobs, sample_requests: int, threads: int, repeats: int):
    """Seconds for ONE pass of the reference CPU decoder over the first `sample_requests` requests (fastest of `repeats`)."""
    from oracle import ref
    return ref.bench(blobs, w["req_clip"][:sample_requests], w["req_time"][:sample_requests], w["num_tracks"], threads, repeats,
                     scalar=(w["kind"] == "scalar"))


def bounded_sample(w, threads: int, seconds: float = 4.0) -> int:
    # ~45 M bone-poses/s/core (BASELINE.md probe) -> keep one pass around `seconds`
    per_request = max(w["num_tracks"], 1)
    budget = int(seconds * 45e6 * max(threads, 1) / per_request)
    return int(min(len(w["req_clip"]), max(budget, 1000)))


# ------------------------------------------------------------------------------------------------------------------
def bind_to_gpu_numa_node(local_rank: int) -> dict:
    """Pins this rank's host threads to the CPUs of its GPU's NUMA node BEFORE any pinned host buffer is allocated (first touch then
    places the pages next to the GPU's PCIe root). Without it the ranks of an 8 GPU box share one node's memory controllers and
    the D2H copies of the e2e path collapse (round 1: 0.54 G bone-poses/s per GPU at N=8 against 1.32 alone)."""
    info = {"numa_node": None, "cpus": None}
    try:
        import pynvml
        pynvml.nvmlInit()
        visible = os.environ.get("CUDA_VISIBLE_DEVICES")
        index = int(visible.split(",")[local_rank]) if visible and visible.replace(",", "").isdigit() else local_rank
        bus_id = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(index)).busId
        bus_id = (bus_id.decode() if isinstance(bus_id, bytes) else bus_id).lower()
        if len(bus_id.split(":")[0]) == 8:
            bus_id = bus_id[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus_id}/numa_node").read())
        if node < 0:
            return info
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & set(os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
            info = {"numa_node": node, "cpus": len(allowed)}
    except Exception as error:      # no NVML / sysfs: keep the default placement, say so
        info["error"] = str(error)[:80]
    return info


def workload_config(args, w, world: int, num_requests: int, pose_bytes: int, blob_bytes: int) -> dict:
    """The `config` both arms print (the driver compares them key for key)."""
    is_transform = w["kind"] == "transform"
    return {"workload": w["description"], "clips": "distinct" if w["distinct"] else "replicated", "clips_per_gpu": w["num_clips"],
            "requests_per_step_per_gpu": num_requests, "bones": w["num_tracks"], "layout": args.layout,
            "l2": f"inputs larger than L2: {blob_bytes / 1e6:.0f} MB compressed + {num_requests * pose_bytes / 1e6:.0f} MB of poses per step vs 126 MB L2",
            "math": MATH_DESCRIPTION[args.math if is_transform else "exact"], "parallelism": f"clip-sharded x{world}, no data-path collective"}


DUMP_BYTES = 32 << 20      # --dump-outputs budget, shared by the ranks
DUMP_SEED = 0


def dump_outputs(directory: str, d_out, num_requests: int, max_tracks: int, bone_bytes: int, rank: int, world: int) -> None:
    """Writes the poses of a fixed, seeded sample of this rank's requests (all of them when they fit its DUMP_BYTES / world share) in request order:
    float32 [requests][max_tracks][bone_bytes / 4], the layout the caller's output buffer holds."""
    import torch
    lanes = bone_bytes // 4
    poses = d_out.view(torch.float32).view(num_requests, max_tracks, lanes)
    keep = min(num_requests, max(1, DUMP_BYTES // world // (max_tracks * bone_bytes)))
    if keep < num_requests:
        pick = np.sort(np.random.default_rng(DUMP_SEED).choice(num_requests, size=keep, replace=False))
        poses = poses.index_select(0, torch.from_numpy(pick).to(poses.device))
    os.makedirs(directory, exist_ok=True)
    name = "poses.npy" if world == 1 else f"poses.rank{rank}.npy"
    np.save(os.path.join(directory, name), poses.cpu().numpy())
    log(f"[bench] wrote {keep} of {num_requests} requests' poses to {os.path.join(directory, name)}")


def time_launches(torch, launch, stream, steps: int, warmup: int, barrier, sampler=None):
    """W untimed + K timed launches bracketed by barrier + synchronize; returns (elapsed ms of the K steps, median launch ms)."""
    for _ in range(warmup):
        launch()
    barrier()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    per_launch = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    barrier()
    host_begin = time.perf_counter()
    start.record(stream)
    for a, b in per_launch:
        a.record(stream)
        launch()
        b.record(stream)
    stop.record(stream)
    barrier()
    if sampler is not None:
        sampler.mark(host_begin, time.perf_counter())
    return start.elapsed_time(stop), float(np.median([a.elapsed_time(b) for a, b in per_launch]))


def measured_traffic(workload: str):
    """DRAM bytes per launch of the dominant kernel from THIS round's ncu --set full capture (profiles/traffic_<workload>.json, written
    by tools/ncu_summary.py next to the summary it came from); a file of another round is reported as stale, never silently."""
    path = os.path.join(ROOT, "profiles", f"traffic_{workload}.json")
    if not os.path.exists(path):
        return None, "no ncu capture of this workload"
    d = json.load(open(path))
    if d.get("round") != ROUND:
        return None, f"stale: captured in round {d.get('round', 1)} ({d.get('kernel', '?')}), not re-measured"
    return d.get("dram_bytes_per_launch"), d.get("source", "ncu --set full")


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed launches of every timed loop (headline, other math mode, e2e, extra workloads, routed C5 job); the per workload "
                         "clock records poll NVML every 1 ms, so a fast workload needs enough steps to span a few ms or it reports no samples")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=list(WORKLOADS))
    ap.add_argument("--clips", type=int, default=None, help="override the number of clips per GPU (debugging)")
    ap.add_argument("--layout", default="qvv40", choices=["qvv40", "qvv48"])
    ap.add_argument("--math", default="exact", choices=["exact", "fast"],
                    help="exact (default, the API default and the bit-exact contract): bit-identical to the reference. fast: hardware sqrt/rsqrt + fused "
                         "multiply-adds on rotations (<= 1e-5 of the reference, the north star's float gate; translations / scales and every integer "
                         "stage stay bit-exact). The other mode is timed too and reported next to it.")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--gather", action="store_true", help="N > 1: also time decode + NCCL all-gather of the poses (SURVEY 8e, optional consumer-side gather)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra blocks (other workloads at N = 1, the routed C5 job at N > 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the poses the last timed step produced (a fixed sample of the requests, at most "
                         f"{DUMP_BYTES >> 20} MB over all ranks) as DIR/poses.npy (poses.rank<r>.npy with N > 1), float32 [requests][tracks][lanes], to compare two builds output for output")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    unit = "bone-poses/s" if WORKLOADS[args.workload][0] == "transform" else "track-samples/s"
    metric = "bone_poses_per_sec" if unit == "bone-poses/s" else "track_samples_per_sec"

    if args.impl == "reference":
        if rank != 0:
            return
        from oracle import ref
        w = make_workload(args.workload, 0, args.clips)
        blobs = host_blobs(w)
        threads = ref.usable_threads() if ref.available() else 1
        sample = bounded_sample(w, threads)
        for _ in range(args.warmup):
            cpu_reference_pass(w, blobs, sample, threads, 1)
        # the pass times itself between "every thread is ready" and "every thread has joined" (oracle/ref_tool.cpp): thread start-up is not
        # charged to the reference; a thread's context stays bound to its clip and is re-initialised only when the clip changes
        elapsed = 0.0
        for _ in range(args.steps):
            elapsed += cpu_reference_pass(w, blobs, sample, threads, 1)
        units = sample * w["num_tracks"]
        value = units * args.steps / elapsed
        single = sample_single_thread(w, blobs)
        bone_bytes = (40 if args.layout == "qvv40" else 48) if w["kind"] == "transform" else 4
        print(json.dumps({
            "impl": "reference", "metric": metric, "value": value, "unit": unit, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * elapsed / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": workload_config(args, w, 1, len(w["req_clip"]), w["num_tracks"] * bone_bytes, int(w["sizes"].astype(np.int64).sum())),
            "cpu_baseline": {"value": value, "unit": unit, "cores": threads, "kind": "reference", "single_thread_value": single,
                             "sample": f"{sample} of {len(w['req_clip'])} requests per step, acl::decompression_context<benchmark settings> (one context per clip, "
                                       f"re-seek per request) on {threads} host threads (affinity / cgroup quota; hardware_concurrency = {os.cpu_count()})"},
            "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return

    import torch
    import acl_b200 as ab

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback")
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa_node(local_rank)
    distributed = world > 1
    if distributed:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    w = make_workload(args.workload, rank, args.clips, world)
    is_transform = w["kind"] == "transform"
    ctx = ab.Context(local_rank)
    upload_begin = time.perf_counter()
    clipset = ctx.upload_packed(w["buffer"], w["offsets"], w["sizes"])
    upload_seconds = time.perf_counter() - upload_begin
    requests = ab.make_requests(w["req_clip"], w["req_time"])
    num_requests = len(requests)
    layout = ab.LAYOUT_QVV40 if args.layout == "qvv40" else ab.LAYOUT_QVV48
    math_mode = ab.MATH_FAST if args.math == "fast" and is_transform else ab.MATH_EXACT
    options = ab.Options(output_layout=layout, math_mode=math_mode)
    bone_bytes = (40 if layout == ab.LAYOUT_QVV40 else 48) if is_transform else 4 * clipset.components
    pose_bytes = clipset.max_tracks * bone_bytes
    d_requests = torch.from_numpy(requests.view(np.uint8)).cuda()
    # zeroed when dumped: lanes the layout leaves unwritten must not carry whatever the allocator held
    d_out = (torch.zeros if args.dump_outputs else torch.empty)(num_requests * pose_bytes, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream()

    def launch():
        if is_transform:
            ctx.decompress_tracks(clipset, d_requests, num_requests, options, d_out, stream)
        else:
            ctx.scalar_decompress_tracks(clipset, d_requests, num_requests, options, d_out, stream)

    alg = algorithmic_bytes_transform(w) if is_transform else algorithmic_bytes_scalar(w)
    units_per_step = alg["units"]

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    from acl_b200.sharding import JobReducer
    reducer = JobReducer(device="cuda")
    sampler = ClockSampler(local_rank)
    sampler.start()             # before the warm-up: NVML initialisation must not eat the (milliseconds long) timed region
    launches_before = ctx.launch_count
    rank_ms, kernel_ms = time_launches(torch, launch, stream, args.steps, args.warmup, barrier, sampler)
    clocks = sampler.stop()
    if args.dump_outputs:       # before the other arithmetic mode and the e2e path overwrite the buffer
        dump_outputs(args.dump_outputs, d_out, num_requests, clipset.max_tracks, bone_bytes, rank, world)
    gpu_launches = ctx.launch_count - launches_before - args.warmup
    elapsed_ms = reducer.max(rank_ms)                                   # slowest rank
    value = reducer.sum(units_per_step * args.steps) / (elapsed_ms * 1e-3)   # every rank's units
    per_rank_ms = [rank_ms / args.steps]
    if distributed:
        gathered_ms = [None] * world
        dist.all_gather_object(gathered_ms, rank_ms / args.steps)
        per_rank_ms = [float(v) for v in gathered_ms]

    # ---- the other arithmetic mode, same launches, reported next to the headline ----
    other_math = None
    if is_transform:
        other_mode = ab.MATH_EXACT if math_mode == ab.MATH_FAST else ab.MATH_FAST
        other_options = ab.Options(output_layout=layout, math_mode=other_mode)
        other_ms, other_kernel_ms = time_launches(torch, lambda: ctx.decompress_tracks(clipset, d_requests, num_requests, other_options, d_out, stream),
                                                  stream, args.steps, args.warmup, barrier)
        other_ms = reducer.max(other_ms)
        other_math = {"math": "exact" if other_mode == ab.MATH_EXACT else "fast", "value": reducer.sum(units_per_step * args.steps) / (other_ms * 1e-3),
                      "unit": unit, "ms_per_step": other_ms / args.steps, "kernel_ms": other_kernel_ms}

    # ---- optional: every rank ends up with every pose (one NCCL all-gather after the decode; not part of the decode path) ----
    gather = None
    if distributed and args.gather:
        gathered = torch.empty(world * d_out.numel(), dtype=torch.uint8, device="cuda")

        def decode_and_gather():
            launch()
            dist.all_gather_into_tensor(gathered, d_out)
        gather_ms, _ = time_launches(torch, decode_and_gather, stream, args.steps, 2, barrier)
        gather_ms = reducer.max(gather_ms)
        gather = {"value": reducer.sum(units_per_step * args.steps) / (gather_ms * 1e-3), "unit": unit,
                  "bytes_gathered_per_step_per_gpu": int(world * d_out.numel()), "collective": "ncclAllGather of the pose buffers"}
        del gathered

    # ---- e2e: host buffers through aclb200_decompress_tracks_host (H2D of the requests, decode, D2H of every pose, all inside the timed region) ----
    e2e = None
    if not args.no_e2e:
        h_requests = torch.from_numpy(requests.view(np.uint8).copy()).pin_memory()
        h_out = torch.empty(num_requests * pose_bytes, dtype=torch.uint8).pin_memory()
        req_np = h_requests.numpy().view(ab.api.REQUEST_DTYPE)
        out_np = h_out.numpy()
        e2e_steps = args.steps
        for _ in range(2):
            ctx.decompress_tracks_host(clipset, req_np, options, out_np)     # warm-up (allocates the device scratch)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            ctx.decompress_tracks_host(clipset, req_np, options, out_np)
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        per_rank_gbs = num_requests * pose_bytes * e2e_steps / e2e_s / 1e9
        e2e_s = reducer.max(e2e_s)
        e2e = {"value": reducer.sum(units_per_step * e2e_steps) / e2e_s, "unit": unit, "h2d_bytes_per_step": int(requests.nbytes),
               "d2h_bytes_per_step": int(num_requests * pose_bytes), "steps": e2e_steps, "d2h_gbs_this_rank": per_rank_gbs, "host_numa": numa,
               "note": "PCIe bound: every pose crosses to the host (at N = 1 about 1.3-1.4 G bone-poses/s whatever the kernel does); "
                       "device-resident consumers are the use case"}
        del h_out

    # ---- N > 1: BASELINE.json configs[4] as ONE routed job ----
    c5_sharded = None
    if distributed and not args.no_extra:
        c5_sharded = routed_c5_job(args, torch, dist, ab, ctx, rank, local_rank, world, reducer, barrier, layout)

    if rank != 0:
        if distributed:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant (only) kernel ----
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy read+write)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    written_per_step = alg["out_bytes"] * bone_bytes // 40 if is_transform else alg["out_bytes"]
    achieved = (alg["in_bytes"] + alg["out_bytes"]) / (kernel_ms * 1e-3) / 1e9
    traffic, traffic_source = measured_traffic(args.workload)
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_source,
                "kernel": "transform_tracks_pipeline_kernel" if is_transform else "scalar_tracks_pipeline_kernel",
                "kernel_ms": kernel_ms, "algorithmic_bytes_in": alg["in_bytes"], "algorithmic_bytes_out": alg["out_bytes"],
                "bytes_written": int(written_per_step), "peak_source": peak_src, "math": args.math if is_transform else "exact"}

    # ---- CPU baseline (reported, not the target) ----
    cpu_baseline = None
    if not args.no_cpu_baseline and world == 1:
        from oracle import ref
        if ref.available():
            blobs = host_blobs(w)
            threads = ref.usable_threads()
            sample = bounded_sample(w, threads)
            seconds = cpu_reference_pass(w, blobs, sample, threads, 3)
            cpu_baseline = {"value": sample * w["num_tracks"] / seconds, "unit": unit, "cores": threads, "kind": "reference",
                            "single_thread_value": sample_single_thread(w, blobs),
                            "sample": f"{sample} of {num_requests} requests, fastest of 3 passes, acl::decompression_context<benchmark settings> (one context per clip, "
                                      f"re-seek per request) on {threads} host threads (affinity / cgroup quota; hardware_concurrency = {os.cpu_count()})"}
        else:
            from oracle import port
            blobs = host_blobs(w)
            sample = min(num_requests, 20000)
            seconds = port.bench_transform(blobs, w["req_clip"][:sample], w["req_time"][:sample], w["num_tracks"])
            cpu_baseline = {"value": sample * w["num_tracks"] / seconds, "unit": unit, "cores": 1, "kind": "port",
                            "sample": f"{sample} of {num_requests} requests, plain-C port, 1 thread"}

    # ---- the other BASELINE.json configs on this GPU (N = 1 only: value + roofline fraction + clocks per workload) ----
    workloads = None
    if world == 1 and not args.no_extra and args.workload == "c2" and args.clips is None:
        del d_out
        workloads = {}
        for name in ("c3", "c5", "c4"):
            workloads[name] = extra_workload(name, torch, ab, ctx, local_rank, peak, barrier, args.steps)
        if w["distinct"]:
            try:
                workloads["error_metric"] = error_metric_workload(torch, ab, ctx, w, clipset, local_rank, peak, barrier, args.steps)
            except Exception as failure:      # an extra block must not take the headline line down with it; it is reported, not hidden
                workloads["error_metric"] = {"failed": f"{type(failure).__name__}: {failure}"}

    result = {
        "metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": workload_config(args, w, world, num_requests, pose_bytes, int(clipset.blob_bytes)),
        "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "other_math": other_math, "gather": gather, "gpu_launches": int(gpu_launches), "clocks": clocks,
        "per_rank_ms_per_step": per_rank_ms,
        "upload": {"ms": upload_seconds * 1e3, "compressed_mb": clipset.blob_bytes / 1e6, "mb_per_s": clipset.blob_bytes / 1e6 / upload_seconds,
                   "what": "aclb200_upload_clips_packed: validation + transcode into the HBM image (host threads) + H2D, once per clip set, never inside a timed region"},
        "workloads": workloads, "c5_sharded": c5_sharded,
    }
    print(json.dumps(result))
    if distributed:
        dist.destroy_process_group()


def sample_single_thread(w, blobs) -> float:
    """The reference on ONE host thread (compare BASELINE.md: about 50 M bone-poses/s/core on the survey box)."""
    sample = min(len(w["req_clip"]), max(1000, int(1.5 * 45e6 / max(w["num_tracks"], 1))))
    seconds = cpu_reference_pass(w, blobs, sample, 1, 2)
    return sample * w["num_tracks"] / seconds


def extra_workload(name: str, torch, ab, ctx, local_rank: int, peak: float, barrier, steps: int) -> dict:
    """One of the other configs on the same GPU: `steps` timed launches with their own clock record."""
    w = make_workload(name, 0, None)
    is_transform = w["kind"] == "transform"
    clipset = ctx.upload_packed(w["buffer"], w["offsets"], w["sizes"])
    requests = ab.make_requests(w["req_clip"], w["req_time"])
    n = len(requests)
    options = ab.Options(output_layout=ab.LAYOUT_QVV40, math_mode=ab.MATH_EXACT)
    bone_bytes = 40 if is_transform else 4 * clipset.components
    d_requests = torch.from_numpy(requests.view(np.uint8)).cuda()
    d_out = torch.empty(n * clipset.max_tracks * bone_bytes, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream()

    def launch():
        if is_transform:
            ctx.decompress_tracks(clipset, d_requests, n, options, d_out, stream)
        else:
            ctx.scalar_decompress_tracks(clipset, d_requests, n, options, d_out, stream)
    alg = algorithmic_bytes_transform(w) if is_transform else algorithmic_bytes_scalar(w)
    sampler = ClockSampler(local_rank)
    sampler.start()
    elapsed_ms, kernel_ms = time_launches(torch, launch, stream, steps, 3, barrier, sampler)
    clocks = sampler.stop()
    achieved = alg["total"] / (kernel_ms * 1e-3) / 1e9
    out = {"workload": w["description"], "value": alg["units"] * steps / (elapsed_ms * 1e-3), "unit": "bone-poses/s" if is_transform else "track-samples/s",
           "steps": steps, "kernel_ms": kernel_ms, "math": "exact", "roofline": {"achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                                                                                "algorithmic_bytes_in": alg["in_bytes"], "algorithmic_bytes_out": alg["out_bytes"]},
           "clocks": clocks}
    clipset.release()
    return out


def error_metric_workload(torch, ab, ctx, w, clipset, local_rank: int, peak: float, barrier, steps: int, num_clips: int = 4096) -> dict:
    """SURVEY 8(f1): acl::calculate_compression_error (decode every sample of a clip, object space, qvvf_transform_error_metric against the
    raw poses, worst track) for the first `num_clips` clips of the C2 clip set in ONE call, poses never leaving the GPU. Unit: bone-poses
    MEASURED per second. The CPU figure next to it is the unmodified reference's calculate_compression_error on a bounded sample."""
    from oracle import ref
    num_clips = min(num_clips, w["num_clips"])
    spec = ref.TransformSpec(num_tracks=w["num_tracks"], num_samples=60, seed=2000)
    t0 = time.time()
    raw, parents, shells = ref.sample_raw_transform_batch(spec, num_clips)
    log(f"[bench] error metric: raw poses of {num_clips} clips in {time.time() - t0:.1f} s ({raw.nbytes / 1e6:.0f} MB)")
    num_samples, num_tracks = raw.shape[1], raw.shape[2]
    jobs = np.zeros(num_clips, dtype=ab.ERROR_JOB_DTYPE)
    jobs["clip"] = np.arange(num_clips)
    jobs["num_samples"] = num_samples
    jobs["sample_rate"] = spec.sample_rate
    jobs["duration"] = ref.finite_duration(num_samples, spec.sample_rate)
    jobs["num_tracks"] = num_tracks
    jobs["first_raw_pose"] = np.arange(num_clips, dtype=np.uint64) * num_samples
    d_raw = torch.from_numpy(raw.reshape(-1)).cuda()
    d_parents = torch.from_numpy(parents.view(np.int32)).cuda()
    d_shells = torch.from_numpy(shells).cuda()
    d_errors = torch.zeros(num_clips * 4, dtype=torch.int32, device="cuda")
    # what tools/acl_compressor measures with: debug_transform_decompression_settings, bind pose = identity
    options = ab.Options(normalization=ab.NORMALIZE_ALWAYS, per_track_rounding=1, multiple_rotation_formats=1, default_modes=(ab.DEFAULT_CONSTANT,) * 3,
                         constant_defaults=[0, 0, 0, 1, 0, 0, 0, 0, 1, 1, 1, 0])
    stream = torch.cuda.current_stream()

    def launch():
        ctx.calculate_compression_error(clipset, jobs, d_raw, d_parents, d_shells, options, d_errors, stream=stream)
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches_before = ctx.launch_count
    launch()
    launches_per_call = ctx.launch_count - launches_before
    torch.cuda.synchronize()
    elapsed_ms, call_ms = time_launches(torch, launch, stream, steps, 3, barrier, sampler)
    clocks = sampler.stop()
    errors = d_errors.cpu().numpy().view(ab.TRACK_ERROR_DTYPE)

    units = num_clips * num_samples * num_tracks
    compressed = int(w["sizes"][:num_clips].astype(np.int64).sum())
    alg_in = compressed + raw.nbytes + parents.nbytes + shells.nbytes
    alg_out = 16 * num_clips
    achieved = (alg_in + alg_out) / (call_ms * 1e-3) / 1e9

    # the unmodified reference on the host threads, a bounded sample of the same clips; its worst tracks must be the GPU's
    threads = ref.usable_threads()
    sample = int(min(num_clips, max(threads * 8, 64)))
    blobs = host_blobs(w)[:sample]
    seconds, cpu_errors = ref.bench_transform_error(spec, blobs, threads)
    single_sample = int(min(sample, 64))
    single_seconds, _ = ref.bench_transform_error(spec, blobs[:single_sample], 1)
    worst = float(np.max(np.abs(errors["error"][:sample] - cpu_errors["error"])))
    same_track = float(np.mean(errors["index"][:sample] == cpu_errors["index"]))
    del d_raw
    return {"workload": f"8(f1): calculate_compression_error of {num_clips} clips x {num_tracks} bones x {num_samples} samples in one call "
                        "(decode every sample + object space + qvvf_transform_error_metric + worst track per clip)",
            "value": units * steps / (elapsed_ms * 1e-3), "unit": "bone-poses measured/s", "steps": steps, "call_ms": call_ms, "launches_per_call": int(launches_per_call),
            "roofline": {"achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "algorithmic_bytes_in": int(alg_in),
                         "algorithmic_bytes_out": int(alg_out),
                         "note": "algorithmic = compressed clips + raw poses (48 B per bone-pose) in, 16 B per clip out; the decoded poses are an intermediate "
                                 "(written and read back once through L2 / HBM: about 2 x 48 B per bone-pose on top)"},
            "cpu_baseline": {"value": sample * num_samples * num_tracks / seconds, "unit": "bone-poses measured/s", "cores": threads, "kind": "reference",
                             "single_thread_value": single_sample * num_samples * num_tracks / single_seconds,
                             "sample": f"{sample} of {num_clips} clips, acl::calculate_compression_error(debug settings, qvvf_transform_error_metric) on {threads} host threads"},
            "parity_vs_cpu_sample": {"max_abs_error_difference": worst, "same_worst_track_fraction": same_track, "gate": 5e-5},
            "flags_set": int(np.count_nonzero(errors["flags"])), "clocks": clocks}


def routed_c5_job(args, torch, dist, ab, ctx, rank, local_rank, world, reducer, barrier, layout) -> dict:
    """BASELINE.json configs[4]: ONE global list of world x 125 000 (clip, random t) requests over world x 125 000 small clips.
    Every rank compresses a contiguous range of the clips; `partition_clips` then balances the ranges by compressed bytes and the
    clips that change owner travel with one NCCL all_to_all over NVLink (the batch split); `route_requests` hands every rank the
    requests of its clips (host side bucket: every rank holds the global list); decode; poses stay on the GPU that made them."""
    from acl_b200 import sharding
    w = make_workload("c5", rank, args.clips, world)
    per_rank = w["num_clips"]
    sizes_mine = w["sizes"].astype(np.int64)
    all_sizes = [None] * world
    dist.all_gather_object(all_sizes, sizes_mine)
    sizes = np.concatenate(all_sizes)
    generated = [(r * per_rank, (r + 1) * per_rank) for r in range(world)]
    owner, local_index, bounds = sharding.partition_clips(sizes, world)
    plan = sharding.exchange_plan(generated, bounds, sizes)
    # this rank's clips back to back, without the generator's alignment padding
    packed = np.concatenate([w["buffer"][int(o):int(o) + int(s)] for o, s in zip(w["offsets"], w["sizes"])])
    t0 = time.perf_counter()
    mine = sharding.redistribute_clips(torch.from_numpy(packed).cuda(), rank, plan)
    torch.cuda.synchronize()
    exchange_s = time.perf_counter() - t0
    moved = sum(plan[rank][dst][2] for dst in range(world) if dst != rank)
    lo, hi = bounds[rank]
    my_sizes = sizes[lo:hi].astype(np.uint32)
    # clips must sit at 16 byte aligned addresses for the upload's readers: re-pack with 64 byte strides
    strides = (my_sizes.astype(np.int64) + 63) & ~63
    my_offsets = np.concatenate([[0], np.cumsum(strides)[:-1]]).astype(np.uint64)
    host_flat = mine.cpu().numpy()
    raw = np.zeros(int(strides.sum()) + 128, dtype=np.uint8)
    shift = (-raw.ctypes.data) % 64
    buffer = raw[shift:shift + int(strides.sum()) + 64]
    src = np.concatenate([[0], np.cumsum(my_sizes.astype(np.int64))])
    for i in range(len(my_sizes)):
        buffer[int(my_offsets[i]):int(my_offsets[i]) + int(my_sizes[i])] = host_flat[src[i]:src[i + 1]]
    clipset = ctx.upload_packed(buffer, my_offsets, my_sizes)

    # the global request list: every clip once, in random order, random time (same list on every rank)
    rng = np.random.default_rng(11)
    total_clips = world * per_rank
    req_clip = rng.permutation(total_clips).astype(np.uint32)
    req_time = (rng.random(total_clips) * (31 / 30.0)).astype(np.float32)
    positions, local_clip, times = sharding.route_requests(req_clip, req_time, owner, local_index, rank)
    requests = ab.make_requests(local_clip, times)
    n = len(requests)
    options = ab.Options(output_layout=layout, math_mode=ab.MATH_EXACT)
    bone_bytes = 40 if layout == ab.LAYOUT_QVV40 else 48
    d_requests = torch.from_numpy(requests.view(np.uint8)).cuda()
    d_out = torch.empty(max(n, 1) * clipset.max_tracks * bone_bytes, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream()
    sampler = ClockSampler(local_rank)
    sampler.start()
    steps = args.steps
    rank_ms, kernel_ms = time_launches(torch, lambda: ctx.decompress_tracks(clipset, d_requests, n, options, d_out, stream), stream, steps, 5, barrier, sampler)
    clocks = sampler.stop()
    elapsed_ms = reducer.max(rank_ms)
    units = n * 30
    value = reducer.sum(units * steps) / (elapsed_ms * 1e-3)
    per_rank = [None] * world
    dist.all_gather_object(per_rank, {"requests": n, "clips": int(hi - lo), "ms_per_step": rank_ms / steps, "bytes_sent": int(moved)})
    clipset.release()
    return {"workload": f"C5 routed: {total_clips} clips x 30 bones x 32 samples over {world} GPUs, one global list of {total_clips} (clip, random t) requests",
            "value": value, "unit": "bone-poses/s", "steps": steps, "ms_per_step": elapsed_ms / steps, "math": "exact",
            "split": "partition_clips by compressed bytes; clips that change owner: one ncclAllToAll (all_to_all_single over NVLink); requests: host side bucket "
                     "(route_requests on the global list every rank holds)",
            "clip_exchange_ms": reducer.max(exchange_s * 1e3), "per_rank": per_rank, "clocks_rank0": clocks,
            "data_path_collective": "none (poses stay sharded)"}


if __name__ == "__main__":
    main()
