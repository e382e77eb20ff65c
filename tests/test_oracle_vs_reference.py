"""Pins the oracle (oracle/acl_oracle.c, the plain-C restatement) against the reference.

Everything is compared bit for bit with what the UNMODIFIED reference produced for the committed clips (tests/golden/): golden
vectors, and for the sweeps over every policy, digests of the reference's outputs (tests/golden/make_reference_checks.py). The port
repeats the reference's float operations in the same order. Only test_golden_blobs_are_reproducible needs the compiled reference
(oracle/_ref/libaclref.so): it checks that the reference's compressor still writes the committed clips.
"""
import numpy as np
import pytest

from tests import clips
from oracle import port as P
from oracle import ref

LANES = clips.DEFINED_LANES


def _settings(kind, **kw):
    return P.settings_for_kind(kind, **kw)


@pytest.mark.parametrize("name", list(clips.TRANSFORM_SPECS))
def test_port_matches_golden_poses(oracle_port, name):
    blob = clips.load_blob(name)
    assert oracle_port.validate(blob, check_hash=True) == 0
    g = np.load(clips.golden_path(name, "golden.npz"))
    for ci, (kind, rounding) in enumerate(g["combos"]):
        s = _settings(int(kind))
        for ti, t in enumerate(g["times"]):
            got = oracle_port.transform_decompress_tracks(blob, s, float(t), int(rounding))[:, LANES]
            assert clips.bit_equal(got, g["poses"][ci, ti]), (name, kind, rounding, t)


@pytest.mark.parametrize("name", list(clips.TRANSFORM_SPECS))
def test_port_matches_golden_single_track(oracle_port, name):
    blob = clips.load_blob(name)
    g = np.load(clips.golden_path(name, "golden.npz"))
    s = _settings(1)
    for ri, rounding in enumerate((0, 3)):
        for ti, t in enumerate(g["times"]):
            for bi, bone in enumerate(g["bones"]):
                got = oracle_port.transform_decompress_track(blob, s, float(t), int(bone), rounding)[int(bone), LANES]
                assert clips.bit_equal(got, g["single"][ri, ti, bi]), (name, rounding, t, bone)


@pytest.mark.parametrize("name", list(clips.TRANSFORM_SPECS))
def test_port_matches_golden_seek_integers(oracle_port, name):
    blob = clips.load_blob(name)
    g = np.load(clips.golden_path(name, "golden.npz"))
    s = _settings(1)
    for row in g["seek"]:
        looping, rounding = int(row[0]), int(row[1])
        t = float(np.uint32(row[2]).view(np.float32))
        st = oracle_port.transform_seek(blob, s, t, rounding, looping)
        got = [np.float32(st.sample_time).view(np.uint32), np.float32(st.interpolation_alpha).view(np.uint32),
               st.key_frame_bit_offsets[0], st.key_frame_bit_offsets[1], st.animated_offsets[0], st.animated_offsets[1],
               st.format_offsets[0], st.format_offsets[1], st.range_offsets[0], st.range_offsets[1],
               st.uses_single_segment, st.looping_policy]
        if st.sample_time < 0:      # empty clip: the reference leaves the context untouched
            continue
        assert [int(x) for x in got] == [int(x) for x in row[3:]], (name, looping, rounding, t)


@pytest.mark.parametrize("name", list(clips.SCALAR_SPECS))
def test_port_matches_golden_scalars(oracle_port, name):
    blob = clips.load_blob(name)
    assert oracle_port.validate(blob, check_hash=True) == 0
    g = np.load(clips.golden_path(name, "golden.npz"))
    nc = g["values"].shape[-1]
    s = P.SettingsBuilder(per_track_rounding=False)
    for rounding in range(4):
        for looping in range(3):
            for ti, t in enumerate(g["times"]):
                got = oracle_port.scalar_decompress(blob, s, float(t), rounding, looping)[:, :nc]
                assert clips.bit_equal(got, g["values"][rounding, looping, ti]), (name, rounding, looping, t)


# ---- the reference's outputs over every policy, stored as digests (tests/golden/make_reference_checks.py) ----

@pytest.mark.parametrize("name", list(clips.TRANSFORM_SPECS))
def test_golden_blobs_are_reproducible(reference, name):
    live = reference.compress_transform(clips.TRANSFORM_SPECS[name])
    assert np.array_equal(live, clips.load_blob(name)), "the reference no longer produces the committed blob"


ALL_POLICIES = ["mixed_scale", "stripped_loop", "single_segment", "full_formats", "noisy_raw", "looping"]


def _kinds(spec):
    is_full = spec.rotation_format == ref.QUATF_FULL
    default_ok = spec.rotation_format == ref.QUATF_DROP_W_VARIABLE and spec.translation_format == ref.VECTOR3F_VARIABLE
    return [1, 3, 4] + ([0] if default_ok else []) + ([5] if is_full else [])


def all_policies_cases(name):
    """Per track rounding policies, default values, and the calls in groups of one (kind, writer, rounding, looping) each:
    ((kind, writer, rounding, looping), [(t, pose the writer starts from), ...])."""
    spec = clips.TRANSFORM_SPECS[name]
    n = spec.num_tracks
    rng = np.random.default_rng(1234)
    policies = rng.integers(0, 4, size=n).astype(np.uint8)
    constant_defaults = rng.normal(size=12).astype(np.float32)
    variable_defaults = rng.normal(size=(n, 12)).astype(np.float32)
    groups = []
    for kind in _kinds(spec):
        for writer in range(4):
            for rounding in ((0, 1, 2, 3, 4) if kind == 1 else (0, 1, 2, 3)):
                for looping in (0, 1, 2):
                    calls = [(float(t), rng.normal(size=(n, 12)).astype(np.float32)) for t in clips.sample_times(spec)[::2]]
                    groups.append(((kind, writer, rounding, looping), calls))
    return policies, constant_defaults, variable_defaults, groups


@pytest.mark.parametrize("name", ALL_POLICIES)
def test_port_matches_live_reference_all_policies(oracle_port, name):
    blob = clips.load_blob(name)
    policies, constant_defaults, variable_defaults, groups = all_policies_cases(name)
    want = clips.reference_checks(f"all_policies/{name}")
    assert len(want) == len(groups)
    for ((kind, writer, rounding, looping), calls), expected in zip(groups, want):
        s = _settings(kind, default_modes=P.writer_modes(writer), constant_defaults=constant_defaults,
                      variable_defaults=variable_defaults, per_track_policies=policies)
        got = [oracle_port.transform_decompress_tracks(blob, s, t, rounding, looping, out=pre.copy())[:, LANES] for t, pre in calls]
        assert clips.digest(*got) == expected, (name, kind, writer, rounding, looping)


SINGLE_TRACK = ["mixed_scale", "full_formats", "single_segment"]


def single_track_cases(name):
    """((kind, rounding), [(t, bone), ...]) groups."""
    spec = clips.TRANSFORM_SPECS[name]
    return [((kind, rounding), [(float(t), bone) for t in clips.sample_times(spec)[::3] for bone in range(0, spec.num_tracks, 3)])
            for kind in _kinds(spec) for rounding in (0, 1, 2, 3)]


@pytest.mark.parametrize("name", SINGLE_TRACK)
def test_port_matches_live_reference_single_track(oracle_port, name):
    blob = clips.load_blob(name)
    groups = single_track_cases(name)
    want = clips.reference_checks(f"single_track/{name}")
    assert len(want) == len(groups)
    for ((kind, rounding), calls), expected in zip(groups, want):
        s = _settings(kind)
        got = [oracle_port.transform_decompress_track(blob, s, t, bone, rounding)[:, LANES] for t, bone in calls]
        assert clips.digest(*got) == expected, (name, kind, rounding)


def scalar_cases(name):
    """Per track rounding policies and ((kind, rounding, looping), [(t, track or -1 for every track), ...]) groups."""
    spec = clips.SCALAR_SPECS[name]
    n = spec.num_tracks
    policies = np.random.default_rng(1).integers(0, 4, size=n).astype(np.uint8)
    groups = []
    for kind in (0, 1):
        for rounding in ((0, 1, 2, 3) if kind == 0 else (0, 1, 2, 3, 4)):
            for looping in (0, 1, 2):
                groups.append(((kind, rounding, looping), [(float(t), track) for t in clips.sample_times(spec)[::2] for track in (-1, 0, n // 2, n - 1)]))
    return policies, groups


@pytest.mark.parametrize("name", list(clips.SCALAR_SPECS))
def test_port_matches_live_reference_scalars(oracle_port, name):
    spec = clips.SCALAR_SPECS[name]
    blob = clips.load_blob(name)
    nc = min(spec.track_type + 1, 4)
    policies, groups = scalar_cases(name)
    settings = {0: P.SettingsBuilder(per_track_rounding=False), 1: P.SettingsBuilder(per_track_rounding=True, per_track_policies=policies)}
    want = clips.reference_checks(f"scalars/{name}")
    assert len(want) == len(groups)
    for ((kind, rounding, looping), calls), expected in zip(groups, want):
        got = [oracle_port.scalar_decompress(blob, settings[kind], t, rounding, looping, track=track)[:, :nc] for t, track in calls]
        assert clips.digest(*got) == expected, (name, kind, rounding, looping)


def test_interpolation_golden_table(oracle_port):
    """Known-answer rows in the spirit of the reference's tests/sources/core/test_interpolation_utils.cpp:33-409: key frame pairs
    and alphas of find_linear_interpolation_samples_with_sample_rate, observed through seek() on a single-segment clip."""
    blob = clips.load_blob("single_segment")          # 20 samples @ 30 Hz
    s = _settings(1)
    bits = oracle_port.transform_seek(blob, s, 1.0 / 30.0, 0, 0).key_frame_bit_offsets[0]      # == animated_pose_bit_size
    cases = [
        # (time, rounding, looping, key frame 0, key frame 1, alpha)
        (0.0, 0, 0, 0, 1, 0.0),
        (1.0 / 30.0, 0, 0, 1, 2, 0.0),
        (19.0 / 30.0, 0, 0, 19, 19, 0.0),
        (0.5 / 30.0, 1, 0, 0, 1, 0.0),      # floor
        (0.5 / 30.0, 2, 0, 0, 1, 1.0),      # ceil
        (0.75 / 30.0, 3, 0, 0, 1, 1.0),     # nearest
        (0.25 / 30.0, 3, 0, 0, 1, 0.0),
        (19.5 / 30.0, 0, 1, 19, 0, None),   # wrap: interpolates back to the first sample
        (20.0 / 30.0, 0, 1, 0, 0, 0.0),     # wrap: the repeated first sample with full weight
    ]
    for t, rounding, looping, k0, k1, alpha in cases:
        st = oracle_port.transform_seek(blob, s, float(np.float32(t)), rounding, looping)
        assert st.key_frame_bit_offsets[0] == k0 * bits and st.key_frame_bit_offsets[1] == k1 * bits, (t, rounding, looping)
        if alpha is not None:
            assert st.interpolation_alpha == alpha, (t, rounding, looping, st.interpolation_alpha)
        else:
            assert 0.0 < st.interpolation_alpha < 1.0


def test_validate_rejects_bad_buffers(oracle_port):
    blob = clips.load_blob("c1_30bones")
    assert oracle_port.validate(blob, True) == 0
    bad = blob.copy(); bad[8] ^= 0xFF                       # tag
    assert oracle_port.validate(clips.ref.aligned_blob(bad), False) != 0
    bad = blob.copy(); bad[12] = 3                          # version below v02_00_00
    assert oracle_port.validate(clips.ref.aligned_blob(bad), False) != 0
    bad = blob.copy(); bad[200] ^= 0x01                     # payload bit flip -> hash mismatch only
    assert oracle_port.validate(clips.ref.aligned_blob(bad), False) == 0
    assert oracle_port.validate(clips.ref.aligned_blob(bad), True) != 0
    bad = blob.copy(); bad[29] |= 0x01                      # has_database without a database header: corrupt
    assert oracle_port.validate(clips.ref.aligned_blob(bad), False) != 0


DATABASE_CASES = [("c1_30bones", 0.0, 0.5), ("c2_100bones", 0.25, 0.5), ("mixed_scale", 0.3, 0.3), ("looping", 0.0, 0.75), ("single_segment", 0.5, 0.25)]


def database_cases(name):
    """((looping, rounding), [t, ...]) groups."""
    times = [float(t) for t in clips.sample_times(clips.TRANSFORM_SPECS[name])]
    return [((looping, rounding), times) for looping in (0, 1, 2) for rounding in (0, 1, 2, 3)]


@pytest.mark.parametrize("name,medium,low", DATABASE_CASES)
def test_port_decodes_database_clips_like_a_context_without_its_database(oracle_port, name, medium, low):
    """SURVEY 8(f2), first step: a clip bound to a streaming database (acl::build_database moved its movable key frames out) decodes from the
    key frames that stay resident, exactly like decompression_context<settings with database support>::initialize(tracks) with no database
    bound (decompress.impl.h:67-83, decompression.transform.h:262-265). Bit for bit, every rounding and looping policy. The clip is the one
    acl::build_database made with these proportions (tests/golden/database_<name>.acl.bin); where the compiled reference is present, it
    must still build that clip byte for byte."""
    blob = clips.load_blob(f"database_{name}")
    if ref.available():
        assert np.array_equal(ref.compress_transform_database(clips.TRANSFORM_SPECS[name], medium, low), blob), "acl::build_database no longer makes this clip"
    assert (int(blob[28:32].view(np.uint32)[0]) >> 8) & 1 == 1
    assert blob.size < clips.load_blob(name).size               # key frames really left the clip
    assert oracle_port.validate(blob, True) == 0
    settings = _settings(1)
    groups = database_cases(name)
    want = clips.reference_checks(f"database/{name}")
    assert len(want) == len(groups)
    for ((looping, rounding), times), expected in zip(groups, want):
        got = [oracle_port.transform_decompress_tracks(blob, settings, t, rounding, looping)[:, LANES] for t in times]
        assert clips.digest(*got) == expected, (name, looping, rounding)


@pytest.mark.parametrize("golden_name", ["database_c1_30bones", "database_mixed_scale"])
def test_port_matches_golden_database_clips(oracle_port, golden_name):
    """The committed database clips (tests/golden/make_golden.py) and what the reference decoded from them without their database."""
    blob = clips.load_blob(golden_name)
    assert oracle_port.validate(blob, True) == 0
    g = np.load(clips.golden_path(golden_name, "golden.npz"))
    settings = _settings(1)
    for rounding in range(4):
        for ti, t in enumerate(g["times"]):
            got = oracle_port.transform_decompress_tracks(blob, settings, float(t), rounding)[:, LANES]
            assert clips.bit_equal(got, g["poses"][rounding, ti]), (golden_name, rounding, float(t))
