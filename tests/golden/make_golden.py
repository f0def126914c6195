"""Mints the committed golden vectors from the reference's own source, compiled by oracle/Makefile into
oracle/_ref/ (set REF_ROOT to the reference's checkout when running make).  Run where that source is present:
python tests/golden/make_golden.py [file ...]   (no argument: every file)

vga_two_pass.npz     : BASELINE config 1 — one synthetic 640x480 frame, identity pose, empty pool
                       (pure initialise), then the same frame again against the surfels it produced
                       (pure fuse).  Full labels (u16), seeds (60-byte records), surfels (44-byte records).
checksums.json       : CRC32 of labels / seeds / surfels for larger frames (KITTI 1226x370 stream of 3,
                       flat KITTI, HD 1280x720) so that the oracle can be re-pinned anywhere cheaply.
reference_serial.json: CRC32 digests of the serialised reference (both constant sets) on the inputs of the
                       restatement-vs-reference tests of tests/test_oracle.py.
reference_map.json   : what the reference's SurfelMap node did on the drives of tests/test_refmap.py: the
  + reference_map_warp.npz   drift-free window after every frame, digests of its maps and published clouds,
                       and a fixed sample of the surfels a loop closure warped.
"""
import json
import os
import sys
import tempfile
import zlib

import numpy as np
from scipy.spatial.transform import Rotation

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.dirname(HERE))  # tests/: the inputs of the tests the digests pin
import pyoracle  # noqa: E402
from densesurfelmapping_b200 import synth  # noqa: E402
from densesurfelmapping_b200.elements import SURFEL_DTYPE  # noqa: E402


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


def stream_checksums(cam, n, flat):
    rs = pyoracle.RefSerial(cam)
    pool = np.zeros(0, SURFEL_DTYPE)
    out = []
    for t in range(n):
        pose = synth.pose_stream(t)
        g, d = synth.make_frame(cam, t, pose, flat=flat)
        loc, new = rs.fuse(t // 2, g, d, pose, pool)
        out.append(dict(frame=t, gray_crc=crc(g), depth_crc=crc(d), labels_crc=crc(rs.labels()),
                        seeds_crc=crc(canon(rs.seeds())), local_crc=crc(canon(loc)), new_crc=crc(canon(new)),
                        n_local=int(len(loc)), n_new=int(len(new)), n_fused=int((loc["update_times"] > 1).sum()) if len(loc) else 0,
                        n_killed=int((loc["update_times"] == 0).sum()) if len(loc) else 0))
        keep = loc[loc["update_times"] > 0] if len(loc) else loc
        pool = np.concatenate([keep, new])
    return out


def vga_two_pass():
    cam = synth.VGA
    g, d = synth.make_frame(cam, 0)
    pose = synth.identity_pose()
    rs = pyoracle.RefSerial(cam)
    _, new0 = rs.fuse(0, g, d, pose, np.zeros(0, SURFEL_DTYPE))
    labels0, seeds0 = rs.labels(), rs.seeds()
    loc1, new1 = rs.fuse(1, g, d, pose, new0)
    labels1, seeds1 = rs.labels(), rs.seeds()
    np.savez_compressed(os.path.join(HERE, "vga_two_pass.npz"), gray_crc=crc(g), depth_crc=crc(d),
                        labels0=labels0.astype(np.uint16), seeds0=seeds0.view(np.uint8), new0=new0.view(np.uint8),
                        labels1=labels1.astype(np.uint16), seeds1=seeds1.view(np.uint8), local1=loc1.view(np.uint8), new1=new1.view(np.uint8))


def checksums():
    sums = {"kitti": stream_checksums(synth.KITTI, 3, False), "kitti_flat": stream_checksums(synth.KITTI, 2, True),
            "hd": stream_checksums(synth.HD, 2, False), "vga_flat": stream_checksums(synth.VGA, 2, True)}
    json.dump(sums, open(os.path.join(HERE, "checksums.json"), "w"), indent=1)


def reference_serial():
    import test_oracle as t
    out = {"small": t.digest_stream(pyoracle.RefSerial(t.SMALL_CAM), t.small_frames()),
           "rgbd": t.digest_stream(pyoracle.RefSerialRGBD(t.RGBD_CAM), t.rgbd_frames()),
           "random_images": t.digest_superpixels(pyoracle.RefSerial(t.RANDOM_IMAGE_CAM))}
    for w, h in t.ODD_SHAPES:
        cam = t.odd_shape_camera(w, h)
        out[f"odd_{w}x{h}"] = t.digest_stream(pyoracle.RefSerial(cam), t.odd_shape_frames(cam))
    json.dump(out, open(os.path.join(HERE, "reference_serial.json"), "w"), separators=(",", ":"))


def reference_map():
    import test_refmap as t
    from test_output_formats import random_surfels
    cam, digest, out = t.CAM, t.digest, {}
    orc = pyoracle.RefSerial(cam)
    # fuse_map on a pool the test carries itself (set_local before every frame)
    m, pool, rec = pyoracle.RefMap(cam), np.zeros(0, SURFEL_DTYPE), []
    for k in range(4):
        pose = synth.pose_stream(k)
        gray, depth = synth.make_frame(cam, 50 + k, pose)
        m.set_local(pool)
        m.fuse_map(gray, depth, pose, k + (7 if k == 3 else 0))
        pool = m.local()
        rec.append(digest(pool))
    out["fuse_map_poststep"] = rec
    a = np.deg2rad(2.0)
    Wm = np.eye(4)
    Wm[:3, :3] = [[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]]
    Wm[:3, 3] = [0.5, -0.1, 0.25]
    m.set_local(random_surfels(5000, 3))
    m.warp_active(np.ascontiguousarray(Wm.T.astype(np.float32).reshape(16)))
    out["warp_active"] = digest(m.local())
    out["mesh_vertices"] = digest(m.mesh_vertices(random_surfels(4000, 11)))
    m.close()
    # a 1-pose drift-free window: retired keyframes, the published clouds, the saved cloud and mesh
    m = pyoracle.RefMap(cam, drift_free_poses=1)
    g = {"drive": t.drive(m, 5), "num_poses": m.num_poses()}
    local = m.local()
    g["local"] = digest(local)
    g["attached"] = [digest(m.attached(p)) for p in range(m.num_poses())]
    g["inactive"] = digest(m.inactive_points())
    m.publish_clouds(m.num_poses() - 1)
    g["published"] = {k: crc(m.published(k)) for k in ("active_pointcloud", "inactive_pointcloud", "pointcloud")}
    g["published"]["neighbor_pointcloud_local_part"] = crc(m.published("neighbor_pointcloud")[:len(pyoracle.cloud_points(local, 1))])
    with tempfile.TemporaryDirectory() as tmp:
        g["published"]["save_cloud"] = crc(m.save_cloud(os.path.join(tmp, "x.pcd")))
        m.save_mesh(os.path.join(tmp, "x.ply"))
        g["save_mesh"] = digest(open(os.path.join(tmp, "x.ply"), "rb").read())
    out["drift_free_1"] = g
    m.close()
    # a loop edge 4-0 brings keyframe 0 back into a 2-pose window
    m = pyoracle.RefMap(cam, drift_free_poses=2)
    g = {"drive": t.drive(m, 5)}
    g["local_before"], g["inactive_before"] = digest(m.local()), digest(m.inactive_points())
    path = [pyoracle.pose_to_ros7(synth.pose_stream(k)) for k in range(5)]
    m.frame(100.5, None, None, pyoracle.pose_to_ros7(synth.pose_stream(5)), False, 4, path7=np.array(path), loops=[4, 0])
    g["window_before"] = m.local_pose_indexs()
    m.move_add_surfels(4)
    g["window_after"] = m.local_pose_indexs()
    g["attached_0_after"] = len(m.attached(0))
    g["attached_after"] = {str(p): digest(m.attached(p)) for p in g["window_before"] if p not in g["window_after"]}
    g["local_after"], g["inactive_after"] = digest(m.local()), digest(m.inactive_points())
    out["insertion"] = g
    m.close()
    # a corrected loop path on the pose feed warps the active surfels
    m = pyoracle.RefMap(cam, drift_free_poses=10)
    g = {"drive": t.drive(m, 4)}
    g["local_before"] = digest(m.local())
    path = [pyoracle.pose_to_ros7(synth.pose_stream(k)) for k in range(4)]
    a = np.deg2rad(1.5)
    C = np.eye(4)
    C[:3, :3] = [[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]]
    C[:3, 3] = [0.3, 0.0, -0.2]
    corrected = []
    for p7 in path:
        T = C @ t.ros7_to_matrix(p7)
        corrected.append(np.concatenate([T[:3, 3], Rotation.from_matrix(T[:3, :3]).as_quat()]))
    m.frame(100.4, None, None, pyoracle.pose_to_ros7(synth.pose_stream(4)), True, 3, path7=np.array(corrected))
    after = m.local()
    g["n_after"] = len(after)
    idx = np.sort(np.random.RandomState(0).choice(len(after), min(len(after), 256), replace=False)).astype(np.int32)
    np.savez_compressed(os.path.join(HERE, "reference_map_warp.npz"), index=idx, after=after[idx].view(np.uint8))
    out["loop_closure"] = g
    m.close()
    # the drive the device-resident map follows on the GPU
    m = pyoracle.RefMap(cam, drift_free_poses=2)
    g = {"drive": [], "local": [], "n_inactive": []}

    def record_state(k):  # called by drive() before every frame: the state after the previous one
        if k:
            g["local"].append(digest(m.local()))
            g["n_inactive"].append(len(m.inactive_points()))
        return [4, 0] if k == 5 else ()
    g["drive"] = t.drive(m, 7, loops_at=record_state)
    record_state(7)
    out["device_drive"] = g
    m.close()
    json.dump(out, open(os.path.join(HERE, "reference_map.json"), "w"), separators=(",", ":"))


WRITERS = {"vga_two_pass.npz": vga_two_pass, "checksums.json": checksums, "reference_serial.json": reference_serial,
           "reference_map.json": reference_map}


def main(names):
    assert pyoracle.have_reference() and pyoracle.have_refmap(), "needs oracle/_ref/libdsm_ref_serial.so and libdsm_refmap.so (make -C oracle)"
    for name in names or WRITERS:
        WRITERS[name]()
    print("golden written:", os.listdir(HERE))


if __name__ == "__main__":
    main(sys.argv[1:])
