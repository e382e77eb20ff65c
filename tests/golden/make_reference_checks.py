"""Regenerates tests/golden/reference_checks.npz, the database clips tests/golden/database_{c2_100bones,looping,single_segment}.acl.bin and the
bench shaped clips tests/golden/bench_*.acl.bin (tests/test_gpu_bench_workloads.py BENCH_CLIPS):
what the UNMODIFIED reference computes for the comparisons the tests make, so that they run without it. Run where
oracle/_ref/libaclref.so exists:

    python tests/golden/make_reference_checks.py

Outputs the tests compare bit for bit are stored as digests (tests/clips.py digest) of the reference's float32 outputs, one per group
of calls; the tests build the same groups of calls (the *_cases functions they export) and digest the port's or the GPU's outputs.
"""
from __future__ import annotations

import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))

from oracle import ref  # noqa: E402
from tests import clips  # noqa: E402
from tests import test_gpu_bench_workloads as W  # noqa: E402
from tests import test_oracle_vs_reference as O  # noqa: E402

LANES = clips.DEFINED_LANES


def write_or_check(name: str, blob: np.ndarray) -> None:
    path = clips.golden_path(name, "acl.bin")
    if os.path.exists(path):
        assert np.array_equal(blob, clips.load_blob(name)), f"{path} is not what the reference compresses"
    else:
        with open(path, "wb") as f:
            f.write(blob.tobytes())


def oracle_checks(out: dict) -> None:
    for name in O.ALL_POLICIES:
        blob = clips.load_blob(name)
        policies, constant_defaults, variable_defaults, groups = O.all_policies_cases(name)
        out[f"all_policies/{name}"] = [clips.digest(*[ref.decompress_tracks(blob, t, rounding, looping, kind, writer, policies, constant_defaults,
                                                                            variable_defaults, out=pre.copy())[:, LANES] for t, pre in calls])
                                       for (kind, writer, rounding, looping), calls in groups]
    for name in O.SINGLE_TRACK:
        blob = clips.load_blob(name)
        out[f"single_track/{name}"] = [clips.digest(*[ref.decompress_track(blob, t, bone, rounding, settings=kind)[:, LANES] for t, bone in calls])
                                       for (kind, rounding), calls in O.single_track_cases(name)]
    for name, spec in clips.SCALAR_SPECS.items():
        blob = clips.load_blob(name)
        nc = min(spec.track_type + 1, 4)
        policies, groups = O.scalar_cases(name)
        out[f"scalars/{name}"] = [clips.digest(*[ref.scalar_decompress(blob, t, rounding, looping, kind, track_index=track, per_track_rounding=policies)[:, :nc]
                                                 for t, track in calls]) for (kind, rounding, looping), calls in groups]
    for name, medium, low in O.DATABASE_CASES:
        blob = ref.compress_transform_database(clips.TRANSFORM_SPECS[name], medium, low)
        write_or_check(f"database_{name}", blob)
        out[f"database/{name}"] = [clips.digest(*[ref.decompress_tracks_without_database(blob, t, rounding, looping)[:, LANES] for t in times])
                                   for (looping, rounding), times in O.database_cases(name)]


def bench_clips() -> None:
    """bench.py's recipes (make_workload) at their next seeds; C4's 4096 track clip with 4 samples instead of 1024."""
    for seed in (2001, 2002):
        write_or_check(f"bench_c2_{seed}", ref.compress_transform(ref.TransformSpec(num_tracks=100, num_samples=60, seed=seed)))
    for seed in range(5001, 5008):
        write_or_check(f"bench_c5_{seed}", ref.compress_transform(ref.TransformSpec(num_tracks=30, num_samples=32, seed=seed)))
    write_or_check("bench_c4_4096x4", ref.compress_scalar(ref.ScalarSpec(num_tracks=4096, num_samples=4, seed=42, track_type=ref.TRACK_FLOAT1F,
                                                                         constant_pct=12, precision=0.001)))


def gpu_workload_checks(out: dict) -> None:
    bench_clips()
    threads = ref.usable_threads()
    for name, slice_requests in W.TRANSFORM_WORKLOADS + [("c4", W.C4_SLICE_REQUESTS)]:
        w = W.workload(name)
        blobs = W._blobs(w)
        scalar = w["kind"] == "scalar"
        digests = []
        for begin in range(0, len(w["req_clip"]), slice_requests):
            end = begin + slice_requests
            want = ref.decode_requests(blobs, w["req_clip"][begin:end], w["req_time"][begin:end], w["num_tracks"], threads, scalar=scalar)
            digests.append(clips.digest(want[:, :, 0] if scalar else want[:, :, LANES]))
        out[f"bench_workload/{name}"] = digests
        print("bench workload", name, len(w["req_clip"]), "requests")
    for name in ("noisy_raw", "mixed_scale", "c1_30bones", "full_formats", "float1", "float3", "vector4"):
        made = W._as_version_7(clips.load_blob(name))
        if made is None:
            continue
        blob = ref.aligned_blob(made[0])
        assert ref.lib().aclref_is_valid(blob.ctypes.data, 1) == 0, f"the reference refuses the re-labelled {name}"
        spec = clips.TRANSFORM_SPECS.get(name) or clips.SCALAR_SPECS[name]
        if name in clips.TRANSFORM_SPECS:
            want = [ref.decompress_tracks(blob, t, settings=ref.SETTINGS_DEBUG, writer=ref.WRITER_LEGACY)[:, LANES] for t in W.v02_00_00_times(spec)]
        else:
            nc = min(spec.track_type + 1, 4)
            want = [ref.scalar_decompress(blob, t)[:, :nc] for t in W.v02_00_00_times(spec)]
        out[f"v02_00_00/{name}"] = [clips.digest(made[0])] + [clips.digest(x) for x in want]
    w = W.workload("c5", 3000)
    req_clip, req_time = W.routed_c5_requests(len(w["req_clip"]))
    want = ref.decode_requests(W._blobs(w), req_clip, req_time, 30)
    out["routed_c5"] = [clips.digest(pose[:, LANES]) for pose in want]


def main() -> None:
    out: dict = {}
    oracle_checks(out)
    gpu_workload_checks(out)
    np.savez_compressed(clips.REFERENCE_CHECKS, **{k: np.array(v, dtype=np.uint64) for k, v in out.items()})
    print(f"{clips.REFERENCE_CHECKS}: {len(out)} comparisons, {os.path.getsize(clips.REFERENCE_CHECKS) / 1e3:.0f} kB")


if __name__ == "__main__":
    main()
