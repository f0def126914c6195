"""CPU tests (-m "not gpu"): the oracle against the golden vectors minted from the reference's own
source, and the restatement against digests of what the serialised reference build returned on the
same inputs (tests/golden/reference_serial.json)."""
import json
import os
import zlib

import numpy as np
import pytest

import pyoracle
from densesurfelmapping_b200 import synth
from densesurfelmapping_b200.elements import SEED_DTYPE, SURFEL_DTYPE
from util import bits_equal_nan

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def canon(a):
    """field-by-field bytes (struct padding excluded) with every NaN canonicalised: NaN payload/sign
    and padding bytes are not part of the contract."""
    parts = []
    for f in a.dtype.names:
        v = np.ascontiguousarray(a[f]).copy()
        if v.dtype.kind == "f":
            v[np.isnan(v)] = np.float32(np.nan)
        parts.append(v.tobytes())
    return b"".join(parts)


def crc(x):
    return zlib.crc32(x if isinstance(x, (bytes, bytearray)) else np.ascontiguousarray(x).tobytes()) & 0xFFFFFFFF


def assert_records_equal(a, b, what):
    assert len(a) == len(b), what
    for f in a.dtype.names:
        if a.dtype[f].kind == "f":
            bad = np.nonzero(~bits_equal_nan(a[f], b[f]))[0]
        else:
            bad = np.nonzero(a[f] != b[f])[0]
        assert len(bad) == 0, f"{what}.{f} differs at {bad[:6]}"


def oracles(cam):
    out = [("restatement", pyoracle.Restatement(cam))]
    if pyoracle.have_reference():
        out.append(("reference_serial", pyoracle.RefSerial(cam)))
    return out


def test_golden_vga_two_pass():
    """BASELINE config 1: every oracle reproduces the committed golden vectors bit for bit."""
    z = np.load(os.path.join(GOLD, "vga_two_pass.npz"))
    cam = synth.VGA
    g, d = synth.make_frame(cam, 0)
    assert crc(g) == int(z["gray_crc"]) and crc(d) == int(z["depth_crc"]), "synthetic generator drifted from the golden inputs"
    pose = synth.identity_pose()
    for name, o in oracles(cam):
        _, new0 = o.fuse(0, g, d, pose, np.zeros(0, SURFEL_DTYPE))
        assert (o.labels() == z["labels0"].astype(np.int32)).all(), name
        assert_records_equal(o.seeds(), z["seeds0"].view(SEED_DTYPE).reshape(-1), name + " seeds0")
        assert_records_equal(new0, z["new0"].view(SURFEL_DTYPE).reshape(-1), name + " new0")
        loc1, new1 = o.fuse(1, g, d, pose, new0)
        assert (o.labels() == z["labels1"].astype(np.int32)).all(), name
        assert_records_equal(o.seeds(), z["seeds1"].view(SEED_DTYPE).reshape(-1), name + " seeds1")
        assert_records_equal(loc1, z["local1"].view(SURFEL_DTYPE).reshape(-1), name + " local1")
        assert_records_equal(new1, z["new1"].view(SURFEL_DTYPE).reshape(-1), name + " new1")
        assert (loc1["update_times"] == 2).sum() > 1000  # the pure-fuse pass really fused


@pytest.mark.parametrize("key,camname,flat", [("kitti", "kitti", False), ("kitti_flat", "kitti", True), ("vga_flat", "vga", True),
                                              ("hd", "hd", False)])
def test_golden_stream_checksums(key, camname, flat):
    """Larger frames: CRC32 of labels / seeds / surfels over a short stream with a carried pool."""
    sums = json.load(open(os.path.join(GOLD, "checksums.json")))[key]
    cam = synth.CAMERAS[camname]
    o = pyoracle.Restatement(cam)
    pool = np.zeros(0, SURFEL_DTYPE)
    for rec in sums:
        t = rec["frame"]
        pose = synth.pose_stream(t)
        g, d = synth.make_frame(cam, t, pose, flat=flat)
        assert crc(g) == rec["gray_crc"] and crc(d) == rec["depth_crc"]
        loc, new = o.fuse(t // 2, g, d, pose, pool)
        assert crc(o.labels()) == rec["labels_crc"], f"{key} frame {t} labels"
        assert crc(canon(o.seeds())) == rec["seeds_crc"], f"{key} frame {t} seeds"
        assert crc(canon(loc)) == rec["local_crc"] and crc(canon(new)) == rec["new_crc"], f"{key} frame {t} surfels"
        assert len(new) == rec["n_new"]
        keep = loc[loc["update_times"] > 0] if len(loc) else loc
        pool = np.concatenate([keep, new])


def reference_digests(key):
    """CRC32 digests of what the serialised reference build (oracle/_ref/libdsm_ref_serial*.so) returned on the
    inputs of the test `key`; minted by tests/golden/make_golden.py."""
    return json.load(open(os.path.join(GOLD, "reference_serial.json")))[key]


def digest_stream(o, frames):
    """fuse_initialize_map over (ref_idx, gray, depth, pose) frames, the pool carried as SurfelMap carries it; per
    frame the CRC32 of labels, seeds, local and new surfels (NaN-canonical bytes) and the surfel counts."""
    pool, out = np.zeros(0, SURFEL_DTYPE), []
    for ref, g, d, pose in frames:
        loc, new = o.fuse(ref, g, d, pose, pool)
        out.append(dict(labels_crc=crc(o.labels()), seeds_crc=crc(canon(o.seeds())), local_crc=crc(canon(loc)),
                        new_crc=crc(canon(new)), n_local=int(len(loc)), n_new=int(len(new))))
        pool = np.concatenate([loc[loc["update_times"] > 0] if len(loc) else loc, new])
    return out


def assert_digests_equal(got, want, what):
    assert len(got) == len(want), what
    for t, (g, w) in enumerate(zip(got, want)):
        bad = sorted(k for k in w if g[k] != w[k])
        assert not bad, f"{what} frame {t}: {bad} differ from the reference"


SMALL_CAM = synth.Camera(324, 242, 260.0, 260.0, 161.5, 120.5, 0.5, 30.0)
RGBD_CAM = synth.Camera(324, 242, 260.0, 260.0, 161.5, 120.5, 0.3, 5.0)
ODD_SHAPES = [(64, 48), (97, 66), (130, 83), (244, 100), (160, 124)]


def small_frames():
    return [(t, *synth.make_frame(SMALL_CAM, 50 + t, synth.pose_stream(t)), synth.pose_stream(t)) for t in range(3)]


def rgbd_frames():
    out = []
    for t in range(3):
        pose = synth.pose_stream(t)
        g, d = synth.make_frame(RGBD_CAM, 60 + t, pose)
        out.append((t, g, (d * np.float32(0.15)).astype(np.float32), pose))  # metres of an indoor scene
    return out


def odd_shape_camera(w, h):
    return synth.Camera(w, h, 0.8 * w, 0.8 * w, (w - 1) / 2.0, (h - 1) / 2.0, 0.5, 30.0)


def odd_shape_frames(cam):
    """a carried pool and a reference-index jump (kills unstable surfels)"""
    return [(ref, *synth.make_frame(cam, 900 + t, synth.pose_stream(t), flat=(t == 1)), synth.pose_stream(t))
            for t, ref in enumerate([0, 1, 9])]


def random_images():
    """60 random 64x48 frames inside the input domain (depth 0 or >= 0.02 m): uniform noise, binary
    salt-and-pepper, smooth ramps, with and without holes, some with many exact depth ties."""
    yy, xx = np.mgrid[0:48, 0:64]
    for seed in range(60):
        rng = np.random.RandomState(seed)
        mode = seed % 3
        if mode == 0:
            gray = rng.randint(0, 256, (48, 64)).astype(np.uint8)
        elif mode == 1:
            gray = (rng.randint(0, 2, (48, 64)) * 255).astype(np.uint8)
        else:
            gray = ((xx * 3 + yy * 2 + rng.randint(0, 4, (48, 64))) % 256).astype(np.uint8)
        depth = rng.uniform(0.02, 25.0, (48, 64)).astype(np.float32)
        if seed % 2:
            depth[rng.rand(48, 64) < 0.4] = 0
        if seed % 5 == 0:
            depth = np.round(depth)  # many exact ties
        yield gray, depth


RANDOM_IMAGE_CAM = synth.Camera(64, 48, 60.0, 60.0, 31.5, 23.5, 0.5, 30.0)


def digest_superpixels(o):
    out = []
    for gray, depth in random_images():
        lab, seeds = o.superpixels(gray, depth)
        out.append(dict(labels_crc=crc(lab), seeds_crc=crc(canon(seeds))))
    return out


def test_restatement_equals_reference_serial_small():
    """A small odd-shaped frame (W%8 == 4, H%8 == 2) with a pool: byte-identical modulo NaN payload."""
    assert_digests_equal(digest_stream(pyoracle.Restatement(SMALL_CAM), small_frames()), reference_digests("small"), "small")


def test_restatement_equals_reference_serial_with_the_rgbd_constant_set():
    """The reference's second constant set (fusion_functions.h:17-21, HUBER_RANGE 0.05 ...): the restatement with
    run-time constants against the reference source compiled with those #defines, on an indoor-range stream; and the
    two sets must really differ on that data (otherwise the test would not notice a dropped constant)."""
    frames = rgbd_frames()
    got = digest_stream(pyoracle.Restatement(RGBD_CAM, pyoracle.CONSTANTS_RGBD), frames)
    assert_digests_equal(got, reference_digests("rgbd"), "rgbd")
    drive = digest_stream(pyoracle.Restatement(RGBD_CAM), frames)  # drive set on the same frames
    assert any(a[k] != b[k] for a, b in zip(drive, got) for k in ("labels_crc", "new_crc", "n_new"))


def test_every_seed_keeps_its_centre_pixel():
    """Why the update_seeds early `return` (fusion_functions.cpp:516-517) can never fire for a valid
    shape: the pixel at (8sx+4, 8sy+4) has exactly one candidate seed, so every seed always owns it."""
    cam = synth.VGA
    o = pyoracle.Restatement(cam)
    g, d = synth.make_frame(cam, 3)
    lab, _ = o.superpixels(g, d)
    spw = cam.width // 8
    for s in range(0, o.S, 37):
        sx, sy = s % spw, s // spw
        assert lab[8 * sy + 4, 8 * sx + 4] == s
    o.lib.dsmor_debug_abort_events.restype = int
    assert o.lib.dsmor_debug_abort_events(0) == 0


def test_quirks_documented_in_survey_appendix_a():
    cam = synth.VGA
    o = pyoracle.Restatement(cam)
    g, d = synth.make_frame(cam, 0)
    lab, seeds = o.superpixels(g, d)
    assert lab.min() >= 0 and lab.max() < o.S
    # rejected seeds keep zero normal / view_cos (H6-i) and are never initialised
    rej = (seeds["norm_x"] == 0) & (seeds["norm_y"] == 0) & (seeds["norm_z"] == 0)
    assert rej.any() and (seeds["view_cos"][rej] == 0).all() and (seeds["size"][rej] == 0).all()
    _, new = o.fuse(0, g, d, synth.identity_pose(), np.zeros(0, SURFEL_DTYPE))
    ok = ~rej & (seeds["mean_depth"] != 0) & ~(seeds["view_cos"] < 0.1)
    assert len(new) == int(ok.sum())
    assert (new["update_times"] == 1).all() and (new["last_update"] == 0).all()
    # unsupported shapes are rejected rather than reading out of bounds (H6-ii)
    import ctypes
    lib = pyoracle._lib("libdsm_oracle.so")
    lib.dsmor_create.restype = ctypes.c_void_p
    lib.dsmor_create.argtypes = [ctypes.c_int, ctypes.c_int] + [ctypes.c_float] * 6
    assert lib.dsmor_create(645, 480, 1.0, 1.0, 1.0, 1.0, 30.0, 0.5) is None


@pytest.mark.parametrize("w,h", ODD_SHAPES)
def test_restatement_equals_reference_serial_on_odd_shapes(w, h):
    """Every supported remainder combination (W%8, H%8 in 0..4), tiny frames, a carried pool and a
    reference-index jump (kills unstable surfels): restatement == serialised reference, byte for byte."""
    cam = odd_shape_camera(w, h)
    got = digest_stream(pyoracle.Restatement(cam), odd_shape_frames(cam))
    assert_digests_equal(got, reference_digests(f"odd_{w}x{h}"), f"{w}x{h}")


def test_restatement_equals_reference_serial_on_random_images():
    """The 60 random 64x48 frames of random_images(): labels and seeds byte-identical."""
    got = digest_superpixels(pyoracle.Restatement(RANDOM_IMAGE_CAM))
    assert_digests_equal(got, reference_digests("random_images"), "random image")
