"""GPU parity of the BENCHMARKED workloads, exhaustively: the exact request lists `bench.py` times (BASELINE.json configs C2, C3, C5 at
full size, same seeds) over distinct committed clips the reference compressed with bench.py's seeds, laid out round-robin so that a
decoder reading another clip's bytes cannot produce the expected bits, and C4 as a 4096 track scalar clip replicated x64 (the shape
bench.py measures, with fewer samples). The lists are decoded in one launch through the C ABI and EVERY request is compared with what
the unmodified reference decoded for it (acl::decompression_context<benchmark settings>::seek + decompress_tracks into a
debug_track_writer style pose, oracle/ref_tool.cpp aclref_bench_transform / aclref_bench_scalar), stored as one digest per slice of the
list (tests/golden/make_reference_checks.py). Where the compiled reference is present (oracle/_ref), the distinct clips bench.py then
times (it compresses them itself) are decoded and compared with the reference live as well.
Mirrors what the reference's own validation walks (tools/acl_compressor/sources/validate_tracks.cpp:92-260,328-511).

Bar: ACLB200_MATH_EXACT bit-identical on every defined lane; ACLB200_MATH_FAST rotations <= 1e-5 absolute, translations and
scales bit-identical.
"""
import numpy as np
import pytest

from tests import clips

pytestmark = pytest.mark.gpu

LANES = clips.DEFINED_LANES
FAST_MATH_TOLERANCE = 1e-5
# (workload, requests per slice): the list is compared with the reference slice by slice, one stored digest per slice
TRANSFORM_WORKLOADS = [("c2", 60000), ("c3", 6000), ("c5", 125000)]
C4_SLICE_REQUESTS = 4096
# committed clips of each workload's shape: the first is bench.py's clip 0 (same recipe and seed), the others its next seeds. C3 has
# one: a 540 bone clip is about 146 kB.
BENCH_CLIPS = {"c2": ["c2_100bones", "bench_c2_2001", "bench_c2_2002"], "c3": ["paragon_like"],
               "c5": ["c5_30x32"] + [f"bench_c5_{seed}" for seed in range(5001, 5008)], "c4": ["bench_c4_4096x4"]}


@pytest.fixture(scope="module")
def env():
    import torch
    import acl_b200 as ab
    return dict(torch=torch, ab=ab, ctx=ab.Context(0))


def _blobs(w):
    return [w["buffer"][int(o):int(o) + int(s)] for o, s in zip(w["offsets"], w["sizes"])]


def workload(name, clips_override=None):
    """bench.py's workload `name` (its request list) over the committed clips of BENCH_CLIPS[name], clip i being clip i % K of them."""
    import bench
    blobs = [clips.load_blob(n) for n in BENCH_CLIPS[name]]
    if name == "c4":
        # bench.py's C4 request list, built for the committed clip's sample count (every clip x every (s + u) / 30)
        num_clips = clips_override or bench.WORKLOADS["c4"][1]
        tracks, samples = (int(v) for v in blobs[0][16:24].view(np.uint32))
        rng = np.random.default_rng(42)
        s = np.tile(np.arange(samples, dtype=np.float64), num_clips)
        w = dict(kind="scalar", num_clips=num_clips, num_tracks=tracks, req_clip=np.repeat(np.arange(num_clips, dtype=np.uint32), samples),
                 req_time=((s + rng.random(s.size)) / 30.0).astype(np.float32))
    else:
        w = bench.make_workload(name, 0, clips_override, replicated=True)
    order = np.arange(w["num_clips"]) % len(blobs)
    strides = np.array([(blobs[i].size + 63) & ~63 for i in order], dtype=np.int64)
    offsets = np.concatenate([[0], np.cumsum(strides)[:-1]]).astype(np.uint64)
    raw = np.zeros(int(strides.sum()) + 128, dtype=np.uint8)
    shift = (-raw.ctypes.data) % 64
    buffer = raw[shift:shift + int(strides.sum()) + 64]
    for offset, i in zip(offsets, order):
        buffer[int(offset):int(offset) + blobs[i].size] = blobs[i]
    w.update(buffer=buffer, offsets=offsets, sizes=np.array([blobs[i].size for i in order], dtype=np.uint32))
    return w


def _slice_digests(rows, slice_requests: int) -> list[int]:
    """rows: [requests][tracks][lanes] on the device; one digest per `slice_requests` consecutive requests."""
    return [clips.digest(rows[begin:begin + slice_requests].contiguous().cpu().numpy()) for begin in range(0, rows.shape[0], slice_requests)]


def _first_difference(w, rows, begin: int, end: int) -> str:
    """The first request of [begin, end) whose decoded bits differ from the oracle's (itself pinned bit for bit to the reference)."""
    from oracle import port
    blobs = _blobs(w)
    scalar = w["kind"] == "scalar"
    settings = port.SettingsBuilder(per_track_rounding=False) if scalar else port.settings_for_kind(0)
    for r in range(begin, end):
        clip, t = int(w["req_clip"][r]), float(w["req_time"][r])
        want = port.scalar_decompress(blobs[clip], settings, t)[:, 0] if scalar else port.transform_decompress_tracks(blobs[clip], settings, t)[:, LANES]
        got = rows[r].cpu().numpy()[:want.shape[0]]
        if not clips.bit_equal(got, want):
            index = tuple(int(i) for i in np.argwhere(got.view(np.uint32) != want.view(np.uint32))[0])
            return f"request {r} (clip {clip}, t={t}) at {index}: got {got[index]} want {want[index]}"
    return "every request of the slice matches the oracle: the digest or the oracle is off"


def _compare_slices(w, rows, want: np.ndarray, slice_requests: int, label: str):
    got = _slice_digests(rows, slice_requests)
    assert len(got) == len(want), label
    bad = [i for i, (g, x) in enumerate(zip(got, want)) if g != x]
    if bad:
        begin = bad[0] * slice_requests
        raise AssertionError(f"{label}: {len(bad)} of {len(want)} slices differ from the reference; "
                             f"{_first_difference(w, rows, begin, min(begin + slice_requests, rows.shape[0]))}")


def _decode_transform(env, w, clipset):
    """Decodes the whole request list in ONE launch per arithmetic mode (the launch bench.py times). Returns (40 byte layout rows, worst
    fast-math rotation error): fast math is held to exact, which the callers hold to the reference."""
    torch, ab, ctx = env["torch"], env["ab"], env["ctx"]
    n_req, tracks = len(w["req_clip"]), clipset.max_tracks
    requests = ab.make_requests(w["req_clip"], w["req_time"])
    d_requests = torch.from_numpy(requests.view(np.uint8)).cuda()
    d_exact = torch.full((n_req, tracks, 12), float("nan"), dtype=torch.float32, device="cuda")
    ctx.decompress_tracks(clipset, d_requests, n_req, ab.Options(output_layout=ab.LAYOUT_QVV48, math_mode=ab.MATH_EXACT), d_exact)
    d_fast = torch.full((n_req, tracks, 12), float("nan"), dtype=torch.float32, device="cuda")
    ctx.decompress_tracks(clipset, d_requests, n_req, ab.Options(output_layout=ab.LAYOUT_QVV48, math_mode=ab.MATH_FAST), d_fast)
    # the 40 byte layout the bench measures carries the same bits
    d_40 = torch.full((n_req, tracks, 10), float("nan"), dtype=torch.float32, device="cuda")
    ctx.decompress_tracks(clipset, d_requests, n_req, ab.Options(output_layout=ab.LAYOUT_QVV40, math_mode=ab.MATH_EXACT), d_40)
    torch.cuda.synchronize()
    assert torch.equal(d_40.view(torch.int32), d_exact[:, :, LANES].contiguous().view(torch.int32))
    worst_fast = float((d_fast[:, :, :4] - d_exact[:, :, :4]).abs().max())
    vector_lanes = torch.tensor([4, 5, 6, 8, 9, 10], device="cuda")
    assert torch.equal(d_fast.index_select(2, vector_lanes).view(torch.int32), d_exact.index_select(2, vector_lanes).view(torch.int32))
    assert worst_fast <= FAST_MATH_TOLERANCE, worst_fast
    return d_40, worst_fast


def _compare_live(env, w, rows, slice_requests: int, label: str):
    """Every request against the compiled reference, slice by slice."""
    from oracle import ref
    torch = env["torch"]
    blobs = _blobs(w)
    for begin in range(0, rows.shape[0], slice_requests):
        end = min(begin + slice_requests, rows.shape[0])
        want = torch.from_numpy(np.ascontiguousarray(ref.decode_requests(blobs, w["req_clip"][begin:end], w["req_time"][begin:end], w["num_tracks"])[:, :, LANES])).cuda()
        if not torch.equal(rows[begin:end].view(torch.int32), want.view(torch.int32)):
            raise AssertionError(f"{label} (live): {_first_difference(w, rows, begin, end)}")


@pytest.mark.parametrize("name, slice_requests", TRANSFORM_WORKLOADS)
def test_bench_workload_every_request_vs_reference(env, name, slice_requests):
    import bench
    from oracle import ref
    w = workload(name)
    clipset = env["ctx"].upload_packed(w["buffer"], w["offsets"], w["sizes"], check_hash=True)
    assert clipset.max_tracks == w["num_tracks"]
    rows, worst_fast = _decode_transform(env, w, clipset)
    _compare_slices(w, rows, clips.reference_checks(f"bench_workload/{name}"), slice_requests, name)
    print(f"{name}: {rows.shape[0]} requests x {w['num_tracks']} bones bit-identical to the reference; fast math worst rotation error {worst_fast:.2e}")
    del rows
    clipset.release()
    if ref.available():
        live = bench.make_workload(name, 0, None)
        assert live["distinct"]
        clipset = env["ctx"].upload_packed(live["buffer"], live["offsets"], live["sizes"], check_hash=True)
        rows, _ = _decode_transform(env, live, clipset)
        _compare_live(env, live, rows, slice_requests, name)
        clipset.release()


def test_bench_workload_c4_every_request_vs_reference(env):
    """C4: a 4096 track scalar float1f clip replicated x64, every request of bench.py's C4 list for its sample count."""
    torch, ab, ctx = env["torch"], env["ab"], env["ctx"]
    w = workload("c4")
    clipset = ctx.upload_packed(w["buffer"], w["offsets"], w["sizes"], check_hash=True)
    n_req, tracks = len(w["req_clip"]), clipset.max_tracks
    assert tracks == 4096 and clipset.components == 1
    requests = ab.make_requests(w["req_clip"], w["req_time"])
    d_requests = torch.from_numpy(requests.view(np.uint8)).cuda()
    d_out = torch.full((n_req, tracks), float("nan"), dtype=torch.float32, device="cuda")
    ctx.scalar_decompress_tracks(clipset, d_requests, n_req, ab.Options(), d_out)
    torch.cuda.synchronize()
    _compare_slices(w, d_out, clips.reference_checks("bench_workload/c4"), C4_SLICE_REQUESTS, "c4")
    clipset.release()


# ------------------------------------------------------------------------------------------------------------------
# v02_00_00 clips: the raw bit rate marker is 32 instead of 31 (animated_track_cache.transform.h:523), scalar tracks use the 19 entry
# bit rate table (decompression.scalar.h:259-263), the wrap flag does not exist (compressed_tracks.impl.h:127-134). The compressor
# here only writes the latest version: the fixtures are golden blobs re-labelled on the host (version field, markers / table
# indices re-mapped so that the payload means the same, hash recomputed) and decoded by the unmodified reference (it accepted exactly these bytes,
# hash checked, and its outputs are stored as digests).
# ------------------------------------------------------------------------------------------------------------------
def _fnv1a32(data: np.ndarray) -> int:
    acc = 2166136261
    for byte in data.tobytes():
        acc = ((acc ^ byte) * 16777619) & 0xFFFFFFFF
    return acc


def _as_version_7(blob: np.ndarray):
    """Returns (re-labelled blob, number of raw / re-mapped entries), or None when the clip cannot be expressed in v02_00_00."""
    b = blob.copy()
    u32 = lambda off: int(b[off:off + 4].view(np.uint32)[0])
    size = u32(0)
    track_type, misc = int(b[15]), u32(28)
    touched = 0
    if track_type == 12:
        if (misc >> 10) & 1 or (misc >> 30) & 1:
            return None                                  # stripped key frames / wrap optimised loops do not exist in v02_00_00
        num_segments, num_variable = u32(32), u32(36)
        headers = 32 + u32(32 + 36)
        for s in range(num_segments):
            data = 32 + u32(headers + 16 * s + 12)
            fmt = b[data:data + num_variable]
            touched += int((fmt == 31).sum())
            fmt[fmt == 31] = 32
    else:
        v10 = [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 32]
        v7 = [0, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 32]
        num_tracks = u32(16)
        meta = 32 + u32(32 + 4)
        rates = b[meta:meta + num_tracks]
        bits = [v10[r] for r in rates]
        if any(x not in v7 for x in bits):
            return None
        rates[:] = [v7.index(x) for x in bits]
        touched = num_tracks
    b[12:14] = np.array([7], dtype=np.uint16).view(np.uint8)
    b[4:8] = np.array([_fnv1a32(b[8:size])], dtype=np.uint32).view(np.uint8)
    return b, touched


def v02_00_00_times(spec):
    return [float(t) for t in clips.sample_times(spec)]


@pytest.mark.parametrize("name", ["noisy_raw", "mixed_scale", "c1_30bones", "full_formats"])
def test_v02_00_00_transform_clip_vs_reference(env, name):
    torch, ab, ctx = env["torch"], env["ab"], env["ctx"]
    made = _as_version_7(clips.load_blob(name))
    assert made is not None
    blob, raw_entries = made
    want = clips.reference_checks(f"v02_00_00/{name}")
    assert clips.digest(blob) == want[0], "not the re-labelled clip the reference accepted"
    blob = clips.ref.aligned_blob(blob)
    if name == "noisy_raw":
        assert raw_entries > 0, "this clip is here for its raw bit rate sub-tracks"
    clipset = ctx.upload([blob], check_hash=True)
    spec = clips.TRANSFORM_SPECS[name]
    times = v02_00_00_times(spec)
    requests = ab.make_requests(np.zeros(len(times), np.uint32), np.array(times, np.float32))
    d_requests = torch.from_numpy(requests.view(np.uint8)).cuda()
    d_out = torch.full((len(times), clipset.max_tracks, 12), float("nan"), dtype=torch.float32, device="cuda")
    # debug settings: every format, version `any`, rotations always normalised
    options = ab.Options(normalization=ab.NORMALIZE_ALWAYS, per_track_rounding=1, multiple_rotation_formats=1,
                         default_modes=(ab.DEFAULT_CONSTANT, ab.DEFAULT_CONSTANT, ab.DEFAULT_LEGACY))
    ctx.decompress_tracks(clipset, d_requests, len(times), options, d_out)
    torch.cuda.synchronize()
    got = d_out.cpu().numpy()
    for i, t in enumerate(times):
        assert clips.digest(got[i][:, LANES]) == want[1 + i], (name, t)
    clipset.release()


@pytest.mark.parametrize("name", ["float1", "float3", "vector4"])
def test_v02_00_00_scalar_clip_vs_reference(env, name):
    torch, ab, ctx = env["torch"], env["ab"], env["ctx"]
    made = _as_version_7(clips.load_blob(name))
    if made is None:
        pytest.skip("this clip uses bit rates the v02_00_00 table does not have")
    want = clips.reference_checks(f"v02_00_00/{name}")
    assert clips.digest(made[0]) == want[0], "not the re-labelled clip the reference accepted"
    blob = clips.ref.aligned_blob(made[0])
    clipset = ctx.upload([blob], check_hash=True)
    spec = clips.SCALAR_SPECS[name]
    times = v02_00_00_times(spec)
    requests = ab.make_requests(np.zeros(len(times), np.uint32), np.array(times, np.float32))
    d_requests = torch.from_numpy(requests.view(np.uint8)).cuda()
    d_out = torch.full((len(times), clipset.max_tracks, clipset.components), float("nan"), dtype=torch.float32, device="cuda")
    ctx.scalar_decompress_tracks(clipset, d_requests, len(times), ab.Options(), d_out)
    torch.cuda.synchronize()
    got = d_out.cpu().numpy()
    for i, t in enumerate(times):
        assert clips.digest(got[i]) == want[1 + i], (name, t)
    clipset.release()


def routed_c5_requests(num_clips):
    rng = np.random.default_rng(11)
    return rng.permutation(num_clips).astype(np.uint32), (rng.random(num_clips) * (31 / 30.0)).astype(np.float32)


def test_routed_c5_job_matches_reference_per_shard(env):
    """bench.py's routed C5 job (SURVEY 8e) on one GPU: the clip table is split with partition_clips, every shard becomes its own clip
    set, the global request list is bucketed with route_requests, each shard decodes its requests, and every pose is compared with
    the reference decoding the ORIGINAL (global) request (one stored digest per request). The 3000 clips cycle through 8 distinct ones, so
    a request routed to the wrong clip decodes other bits. What N ranks do, shard after shard."""
    from acl_b200 import sharding
    torch, ab, ctx = env["torch"], env["ab"], env["ctx"]
    w = workload("c5", 3000)
    sizes = w["sizes"].astype(np.int64)
    blobs = _blobs(w)
    world = 3
    owner, local_index, bounds = sharding.partition_clips(sizes, world)
    req_clip, req_time = routed_c5_requests(len(blobs))
    want = clips.reference_checks("routed_c5")
    assert len(want) == len(req_clip)
    seen = 0
    for rank in range(world):
        lo, hi = bounds[rank]
        clipset = ctx.upload(blobs[lo:hi], check_hash=True)
        positions, local_clip, times = sharding.route_requests(req_clip, req_time, owner, local_index, rank)
        requests = ab.make_requests(local_clip, times)
        d_requests = torch.from_numpy(requests.view(np.uint8)).cuda()
        d_out = torch.zeros((len(requests), 30, 12), dtype=torch.float32, device="cuda")
        ctx.decompress_tracks(clipset, d_requests, len(requests), ab.Options(), d_out)
        torch.cuda.synchronize()
        got = d_out.cpu().numpy()
        for row, position in enumerate(positions):
            assert clips.digest(got[row][:, LANES]) == want[position], (rank, int(position))
        seen += len(positions)
        clipset.release()
    assert seen == len(req_clip)
