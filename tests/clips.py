"""Named synthetic clips shared by the parity tests.

Every entry is a recipe for oracle/ref.py (the reference compressor). The compressed blobs and the reference's own
outputs for them are committed under tests/golden/ (tests/golden/make_golden.py), so the tests never need
/root/reference at run time; when oracle/_ref/libaclref.so is present the tests ALSO regenerate the blobs live and
check they match the committed ones byte for byte.

The matrix mirrors the reference's regression configs (test_data/configs/*.sjson: variable / raw / mixed formats,
key frame stripping) and the edge cases its validation walks (tools/acl_compressor/sources/validate_tracks.cpp:92-260).
"""
from __future__ import annotations

import hashlib
import os

import numpy as np

from oracle import ref

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

T = ref.TransformSpec
S = ref.ScalarSpec

TRANSFORM_SPECS: dict[str, ref.TransformSpec] = {
    # BASELINE.json configs at reduced clip counts
    "c1_30bones": T(num_tracks=30, num_samples=60, seed=1000),
    "c2_100bones": T(num_tracks=100, num_samples=60, seed=2000),
    "c5_30x32": T(num_tracks=30, num_samples=32, seed=5000),
    # every sub-track kind, scale, constant-in-segment bit rates, raw bit rates
    "mixed_scale": T(num_tracks=57, num_samples=75, seed=7, rot_default_pct=10, rot_constant_pct=30, trans_default_pct=20,
                     trans_constant_pct=40, scale_default_pct=60, scale_constant_pct=20, partial_activity_pct=30, noisy_pct=10),
    "single_segment": T(num_tracks=33, num_samples=20, seed=9, rot_constant_pct=30, trans_constant_pct=40, scale_default_pct=50,
                        scale_constant_pct=20),
    "noisy_raw": T(num_tracks=40, num_samples=90, seed=11, noisy_pct=30, trans_constant_pct=50),
    # wrap optimised loops, stripped key frames (one and many segments)
    "looping": T(num_tracks=40, num_samples=61, seed=12, looping_content=1, trans_constant_pct=50),
    "stripped_loop": T(num_tracks=40, num_samples=120, seed=13, strip_proportion=0.4, trans_constant_pct=50, looping_content=1),
    "stripped_single": T(num_tracks=40, num_samples=25, seed=17, strip_proportion=0.5, trans_constant_pct=50),
    # full precision and mixed formats
    "full_formats": T(num_tracks=21, num_samples=50, seed=14, strip_trivial=0, rotation_format=ref.QUATF_FULL,
                      translation_format=ref.VECTOR3F_FULL, scale_format=ref.VECTOR3F_FULL, scale_default_pct=50, rot_constant_pct=20),
    "drop_w_full": T(num_tracks=21, num_samples=50, seed=15, strip_trivial=0, rotation_format=ref.QUATF_DROP_W_FULL,
                     translation_format=ref.VECTOR3F_VARIABLE, scale_format=ref.VECTOR3F_FULL, scale_default_pct=50, rot_constant_pct=20),
    "mixed_formats": T(num_tracks=21, num_samples=50, seed=16, strip_trivial=0, rotation_format=ref.QUATF_DROP_W_VARIABLE,
                       translation_format=ref.VECTOR3F_FULL, scale_format=ref.VECTOR3F_VARIABLE, scale_default_pct=50, rot_constant_pct=20),
    # degenerate sizes
    "one_sample": T(num_tracks=5, num_samples=1, seed=18),
    "two_samples": T(num_tracks=5, num_samples=2, seed=19),
    "one_bone": T(num_tracks=1, num_samples=40, seed=20, trans_constant_pct=0),
    "all_default": T(num_tracks=16, num_samples=40, seed=21, rot_default_pct=100, trans_default_pct=100),
    "ragged_17": T(num_tracks=17, num_samples=47, seed=22, rot_constant_pct=25, trans_constant_pct=25, scale_default_pct=40, scale_constant_pct=30),
    "paragon_like": T(num_tracks=540, num_samples=60, seed=3000, scale_default_pct=95, scale_constant_pct=0),
    # rotations around half a turn: W crosses 0, where quat_from_positive_w4 is ill-conditioned (1 ulp on x moves W by ulp / W)
    "half_turn": T(num_tracks=64, num_samples=60, seed=23, rotation_offset=3.0, trans_constant_pct=60),
}

SCALAR_SPECS: dict[str, ref.ScalarSpec] = {
    "float1": S(num_tracks=67, num_samples=100, seed=42, track_type=ref.TRACK_FLOAT1F, constant_pct=20, noisy_pct=15),
    "float2": S(num_tracks=31, num_samples=40, seed=43, track_type=ref.TRACK_FLOAT2F, constant_pct=20, noisy_pct=15),
    "float3": S(num_tracks=31, num_samples=40, seed=44, track_type=ref.TRACK_FLOAT3F, constant_pct=20, noisy_pct=15),
    "float4": S(num_tracks=31, num_samples=40, seed=45, track_type=ref.TRACK_FLOAT4F, constant_pct=20, noisy_pct=15),
    "vector4": S(num_tracks=31, num_samples=40, seed=46, track_type=ref.TRACK_VECTOR4F, constant_pct=20, noisy_pct=15),
    "float1_one_sample": S(num_tracks=9, num_samples=1, seed=47, track_type=ref.TRACK_FLOAT1F, constant_pct=20),
    "float1_c4_small": S(num_tracks=512, num_samples=64, seed=48, track_type=ref.TRACK_FLOAT1F, constant_pct=12),
}

# the float lanes that are defined by the reference: rotation xyzw, translation xyz, scale xyz of a [.., 12] row
# (translation.w / scale.w are "TODO: Fill in W", animated_track_cache.transform.h:964)
DEFINED_LANES = [0, 1, 2, 3, 4, 5, 6, 8, 9, 10]


def golden_path(name: str, suffix: str) -> str:
    return os.path.join(GOLDEN_DIR, f"{name}.{suffix}")


def load_blob(name: str) -> np.ndarray:
    """The committed reference-compressed clip, 64 byte aligned with tail slack."""
    with open(golden_path(name, "acl.bin"), "rb") as f:
        return ref.aligned_blob(f.read())


def sample_times(spec) -> np.ndarray:
    """Times the parity tests walk: every flavour of seek (before 0, exact key frames, mid frames, past the end)."""
    duration = max(spec.num_samples - 1, 0) / spec.sample_rate
    base = np.linspace(0.0, duration, 9)
    extra = np.array([-0.2, duration + 1.0, 0.3333, duration * 0.999, duration * 0.5 + 1e-3], dtype=np.float64)
    key_frame = np.array([k / spec.sample_rate for k in (1, 7, 19, 20, 21) if k < spec.num_samples], dtype=np.float64)
    return np.concatenate([base, extra, key_frame]).astype(np.float32)


def bit_equal(a: np.ndarray, b: np.ndarray) -> bool:
    return np.array_equal(np.ascontiguousarray(a, dtype=np.float32).view(np.uint32), np.ascontiguousarray(b, dtype=np.float32).view(np.uint32))


def digest(*arrays: np.ndarray) -> int:
    """64 bit BLAKE2b of the bytes of `arrays` (floats as float32), in order: two digests are equal exactly when every bit is (a
    chance collision aside), so a stored digest of the reference's output stands for the output in a bit for bit comparison."""
    h = hashlib.blake2b(digest_size=8)
    for a in arrays:
        a = np.asarray(a)
        h.update(np.ascontiguousarray(a, dtype=np.float32 if a.dtype.kind == "f" else a.dtype).tobytes())
    return int.from_bytes(h.digest(), "little")


REFERENCE_CHECKS = os.path.join(GOLDEN_DIR, "reference_checks.npz")


def reference_checks(key: str) -> np.ndarray:
    """What the reference computed for the comparison `key` (tests/golden/make_reference_checks.py)."""
    with np.load(REFERENCE_CHECKS) as stored:
        return stored[key]
