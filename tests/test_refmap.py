"""The reference's whole SurfelMap (surfel_map.cpp, compiled in place by oracle/ref_map_driver.cpp) against the restated
SurfelMap members this repo's tests lean on -- fuse_map's post-step, the active-surfel warp, move_add_surfels' removal
and insertion, the cloud builders -- and against the PRODUCT's PLY-mesh writer and hexagon generator (host code in the C
ABI).  What the reference node did on each input is stored in tests/golden/reference_map.json (the drift-free window it
chose after every frame, CRC32 digests of its state and outputs) and reference_map_warp.npz, minted by
tests/golden/make_golden.py; NodeReplay rebuilds the node's map from the restated members and those windows, and its
digests must equal the reference's byte for byte.  GPU: the device-resident map against the same replay.  Two tests need
the libraries compiled from the reference's own source (oracle/_ref/libdsm_refmap*.so) and skip without them."""
import json
import os
import subprocess
import zlib

import numpy as np
import pytest

import pyoracle
from densesurfelmapping_b200 import capi, synth
from densesurfelmapping_b200.elements import SURFEL_DTYPE
from test_output_formats import random_surfels
from util import oracle_for

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CAM = synth.Camera(320, 240, 262.5, 262.5, 159.5, 119.5, 0.5, 30.0)  # quarter-VGA keeps the CPU suite short


def golden(key):
    return json.load(open(os.path.join(GOLD, "reference_map.json")))[key]


def crc(a):
    return zlib.crc32(a if isinstance(a, (bytes, bytearray)) else np.ascontiguousarray(a).tobytes()) & 0xFFFFFFFF


def digest(a):
    return {"n": int(len(a)), "crc": crc(a)}


def drive(m, n_frames, keyframe_every=1, seed0=1000, loops_at=None):
    """n frames of the synthetic drive through the node callbacks; every frame references the newest keyframe.
    Returns the reference index and the node's drift-free window of every frame."""
    path, last_kf, record = [], 0, []
    for t in range(n_frames):
        pose = synth.pose_stream(t)
        gray, depth = synth.make_frame(CAM, seed0 + t, pose)
        p7 = pyoracle.pose_to_ros7(pose)
        is_kf = (t % keyframe_every) == 0
        ref = last_kf if t else 0
        m.frame(100.0 + 0.1 * t, gray, depth, p7, is_kf, ref, path7=np.array(path).reshape(-1, 7),
                loops=loops_at(t) if loops_at else ())
        record.append([ref, m.local_pose_indexs()])
        if is_kf or t == 0:
            path.append(p7)
            last_kf = m.num_poses() - 1
    return record


def ros7_to_matrix(p7):
    from scipy.spatial.transform import Rotation
    T = np.eye(4)
    T[:3, :3] = Rotation.from_quat(p7[3:7]).as_matrix()
    T[:3, 3] = p7[:3]
    return T


def rebase(p7_first):
    """The node re-bases the world with K = idea * T_first^-1 (surfel_map.cpp:214-232)."""
    idea = np.zeros((4, 4))
    idea[0, 0], idea[1, 2], idea[2, 1], idea[3, 3] = 1.0, 1.0, -1.0, 1.0
    return idea @ np.linalg.inv(ros7_to_matrix(p7_first))


class NodeReplay:
    """The reference node's map -- local_surfels, attached_surfels per pose, inactive_pointcloud -- rebuilt from the
    restated members: move() is move_add_surfels for the window the node chose (removal of the poses that left it
    first, then the poses that came back are appended), fuse() is fuse_map on a frame of drive() in the node's
    re-based world frame (hot path + post-step)."""

    def __init__(self, seed0=1000):
        self.orc = oracle_for(CAM)
        self.seed0 = seed0
        self.local = np.zeros(0, SURFEL_DTYPE)
        self.attached = {}  # pose -> retired surfels, in the order the poses were retired
        self.window = []
        self.K = rebase(pyoracle.pose_to_ros7(synth.pose_stream(0)))

    def move(self, window):
        for p in [q for q in self.window if q not in window]:
            self.local, self.attached[p] = pyoracle.retire(self.local, p)
        for p in [q for q in window if q not in self.window and q in self.attached]:
            self.local = np.concatenate([self.local, self.attached.pop(p)])
        self.window = list(window)

    def fuse(self, t, ref_index):
        pose = synth.pose_stream(t)
        gray, depth = synth.make_frame(CAM, self.seed0 + t, pose)
        fuse_pose = (self.K @ ros7_to_matrix(pyoracle.pose_to_ros7(pose))).astype(np.float32)  # what synchronize_msgs hands to fuse_map
        lo, no = self.orc.fuse(ref_index, gray, depth, np.ascontiguousarray(fuse_pose.T.reshape(16)), self.local)
        self.local = pyoracle.fuse_map_poststep(lo, no)
        return gray, depth, fuse_pose

    def run(self, record):
        for t, (ref, window) in enumerate(record):
            self.move(window)
            self.fuse(t, ref)
        return self

    def attached_to(self, pose):
        return self.attached.get(pose, np.zeros(0, SURFEL_DTYPE))

    def inactive(self):
        return np.concatenate([np.zeros((0, 4), np.float32)] + [pyoracle.cloud_points(a, -(2 ** 31)) for a in self.attached.values()])


def test_fuse_map_poststep_is_pinned():
    """SurfelMap::fuse_map (surfel_map.cpp:1060-1113) == reference hot path + the restated post-step."""
    orc = oracle_for(CAM)
    pool = np.zeros(0, SURFEL_DTYPE)
    for t, want_ref in enumerate(golden("fuse_map_poststep")):
        pose = synth.pose_stream(t)
        gray, depth = synth.make_frame(CAM, 50 + t, pose)
        ref = t + (7 if t == 3 else 0)  # the jump kills unstable surfels: slot recycling AND swap-with-back both run
        lo, no = orc.fuse(ref, gray, depth, pose, pool)
        want = pyoracle.fuse_map_poststep(lo, no)
        assert digest(want) == want_ref, f"frame {t}"
        pool = want
    assert (lo["update_times"] == 0).sum() > 0


def test_warp_active_is_pinned():
    pool = random_surfels(5000, 3)
    a = np.deg2rad(2.0)
    Wm = np.eye(4)
    Wm[:3, :3] = [[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]]
    Wm[:3, 3] = [0.5, -0.1, 0.25]
    w = np.ascontiguousarray(Wm.T.astype(np.float32).reshape(16))
    assert digest(pyoracle.warp_active(pool, w)) == golden("warp_active")


def test_move_add_surfels_and_cloud_builders_are_pinned():
    """A drive with a 1-pose drift-free window: keyframes leave the window, their surfels move to attached_surfels /
    inactive_pointcloud (surfel_map.cpp:1479-1497).  Checked member by member against the restatements."""
    g = golden("drift_free_1")
    r = NodeReplay().run(g["drive"])
    assert g["num_poses"] == 5
    before = r.local
    assert digest(before) == g["local"]
    keep = set(r.window)
    # 1. everything that left the window is attached to its pose, in pool order, and nowhere else
    n_att = 0
    for p in range(g["num_poses"]):
        att = r.attached_to(p)
        assert digest(att) == g["attached"][p], f"pose {p}"
        n_att += len(att)
        if len(att):
            assert p not in keep and (att["last_update"] == p).all() and (att["update_times"] > 0).all()
    assert n_att > 0, "the drive never retired a keyframe"
    inactive = r.inactive()
    assert len(inactive) == n_att and digest(inactive) == g["inactive"]
    assert not np.isin(before["last_update"][before["update_times"] > 0], [p for p in range(5) if p not in keep]).any()
    # 2. the cloud builders over the current state
    pub = g["published"]
    assert crc(pyoracle.cloud_points(before, 5)) == pub["active_pointcloud"]
    assert crc(inactive) == pub["inactive_pointcloud"]
    assert crc(np.concatenate([pyoracle.cloud_points(before, 5), inactive])) == pub["pointcloud"]
    assert crc(pyoracle.cloud_points(before, 1)) == pub["neighbor_pointcloud_local_part"]  # update_times != 0 (:1291-1300)
    assert crc(np.concatenate([pyoracle.cloud_points(before, 5), inactive])) == pub["save_cloud"]


def test_move_add_surfels_insertion_is_an_append():
    """A loop edge brings an old keyframe back into the drift-free window: its attached_surfels are appended to
    local_surfels in order and leave the inactive cloud (surfel_map.cpp:1526-1590) -- the semantics of
    dsm_pool_append / dsm_inactive_reactivate."""
    g = golden("insertion")
    r = NodeReplay().run(g["drive"])
    att0, local_before, inactive_before = r.attached_to(0), r.local, r.inactive()
    assert digest(local_before) == g["local_before"] and digest(inactive_before) == g["inactive_before"]
    assert len(att0) > 0 and 0 not in r.window
    window_before = g["window_before"]  # after a pose feed with the loop edge 4-0, before move_add_surfels(4)
    assert window_before == r.window
    window_after = g["window_after"]
    assert 0 in window_after and g["attached_0_after"] == 0
    # the same call retires whatever left the window rooted at pose 4 (removal runs before insertion)
    want_local, retired = local_before, []
    for p in [q for q in window_before if q not in window_after]:
        want_local, out = pyoracle.retire(want_local, p)
        assert digest(out) == g["attached_after"][str(p)], f"pose {p}"
        retired.append(out)
    assert digest(np.concatenate([want_local, att0])) == g["local_after"]
    # pose 0 was the first segment of the inactive cloud: the rest moved down unchanged, new segments follow
    assert crc(inactive_before[:len(att0)]) == crc(pyoracle.cloud_points(att0, -(2 ** 31)))
    want_inactive = np.concatenate([inactive_before[len(att0):]] + [pyoracle.cloud_points(o, -(2 ** 31)) for o in retired])
    assert digest(want_inactive) == g["inactive_after"]


def test_loop_closure_warps_the_active_surfels():
    """A corrected loop path arrives on the pose feed: orb_results_input -> warp_surfels (surfel_map.cpp:795-824) moves
    every active surfel by W = T_loop * T_cam^-1 of the oldest local keyframe.  Checks the restated warp (and the W
    the product's dsm_pool_transform is handed) against the node's own state, in the node's re-based world frame, on a
    fixed sample of the warped surfels."""
    g = golden("loop_closure")
    r = NodeReplay().run(g["drive"])
    before = r.local
    assert digest(before) == g["local_before"]
    z = np.load(os.path.join(GOLD, "reference_map_warp.npz"))
    idx, after = z["index"], z["after"].view(SURFEL_DTYPE).reshape(-1)
    assert g["n_after"] == len(before) and len(idx) == len(after) > 100
    path = [pyoracle.pose_to_ros7(synth.pose_stream(t)) for t in range(4)]
    a = np.deg2rad(1.5)
    C = np.eye(4)   # the correction the loop closure applies to every keyframe
    C[:3, :3] = [[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]]
    C[:3, 3] = [0.3, 0.0, -0.2]
    K = rebase(path[0])
    Wm = K @ C @ np.linalg.inv(K)  # in the re-based frame
    w = np.ascontiguousarray(Wm.T.astype(np.float32).reshape(16))
    want = pyoracle.warp_active(before, w)[idx]
    e = pyoracle.surfel_errors(after, want)
    assert e["pos"] < 2e-5 and e["nrm"] < 2e-5 and e["int_mismatch"] == 0, e
    moved = np.abs(after["px"] - before["px"][idx]).max()
    assert moved > 0.05, "the loop correction did not move anything"


def test_product_mesh_writer_equals_reference_save_mesh(tmp_path):
    """dsm_write_ply_mesh / dsm_mesh_vertices (product, host code) against SurfelMap::save_mesh / push_a_surfel of the
    reference: byte-identical file, bit-identical vertices."""
    s = random_surfels(4000, 11)
    assert digest(capi.mesh_vertices(s)) == golden("mesh_vertices")
    assert digest(pyoracle.mesh_vertices(s)) == golden("mesh_vertices")
    g = golden("drift_free_1")
    r = NodeReplay().run(g["drive"])
    local = r.local
    surfels = np.concatenate([r.attached_to(p) for p in range(g["num_poses"])] + [local[local["update_times"] >= 5]])
    assert len(surfels) > 100
    our_file = tmp_path / "ours.ply"
    capi.write_ply_mesh(str(our_file), surfels)
    assert digest(our_file.read_bytes()) == g["save_mesh"]
    assert digest(pyoracle.ply_mesh_text(surfels).encode()) == g["save_mesh"]


def test_three_line_patch_compiles_against_the_reference_source():
    """libdsm_refmap_b200.so is the reference's surfel_map.cpp, unmodified, with dsm::FusionFunctions in place of
    FusionFunctions (include path only): it exists, exports the driver, and takes the hot path from the C ABI."""
    if not pyoracle.have_refmap(b200=True):
        pytest.skip("libdsm_refmap_b200.so not built (needs the reference's source)")
    path = os.path.join(pyoracle.REFDIR, "libdsm_refmap_b200.so")
    und = subprocess.run(["nm", "-D", "--undefined-only", path], capture_output=True, text=True).stdout
    assert " dsm_create" in und and " dsm_fuse_frame" in und
    dfn = subprocess.run(["nm", "-D", "--defined-only", path], capture_output=True, text=True).stdout
    assert "dsmmap_frame" in dfn and "generate_super_pixels" not in dfn  # no CPU hot path inside


@pytest.mark.gpu
def test_reference_node_over_the_product_matches_the_reference_node():
    """The drop-in claim end to end: the same 6-frame drive through the reference's SurfelMap with its own CPU
    FusionFunctions and with the product library underneath.  Maps agree as sets within the surfel tolerance."""
    from test_gpu_resident import match_as_sets
    if not pyoracle.have_refmap(b200=True):
        pytest.skip("libdsm_refmap_b200.so not built (needs the reference's source)")
    a, b = pyoracle.RefMap(CAM, drift_free_poses=2), pyoracle.RefMap(CAM, drift_free_poses=2, b200=True)
    drive(a, 6)
    drive(b, 6)
    assert a.num_poses() == b.num_poses() and a.local_pose_indexs() == b.local_pose_indexs()
    la, lb = a.local(), b.local()
    assert abs(len(la) - len(lb)) <= max(2, len(la) // 500)
    if len(la) == len(lb):
        match_as_sets(lb, la, tol=1e-3)
    for p in range(a.num_poses()):
        assert abs(len(a.attached(p)) - len(b.attached(p))) <= max(2, len(a.attached(p)) // 200)
    a.close()
    b.close()


@pytest.mark.gpu
def test_device_resident_map_tracks_the_reference_node():
    """System level, INTEGRATION.md steps 2+3: the reference node ran a drive on the CPU (its windows and digests are
    golden data, its map is rebuilt by NodeReplay and pinned to those digests); the same frames go through the product
    with local_surfels AND attached_surfels resident on the device, replaying the node's own window decisions (which
    keyframes leave / re-enter; a loop edge 4-0 brings keyframe 0 back at frame 5).  After every frame the device's
    local pool and inactive store equal the node's local_surfels / inactive_pointcloud as sets, within the surfel
    tolerance."""
    from test_gpu_resident import match_as_sets
    g = golden("device_drive")
    r = NodeReplay()
    ctx = capi.Context(CAM, max_batch=2, max_local_surfels=60000)
    ctx.pool_upload(np.zeros(0, SURFEL_DTYPE))
    ctx.inactive_reserve(200000)
    window_prev, stored = [], set()
    for t, ((ref_index, window), want_digest, want_inactive) in enumerate(zip(g["drive"], g["local"], g["n_inactive"])):
        r.move(window)
        gray, depth, fuse_pose = r.fuse(t, ref_index)
        want = r.local
        assert digest(want) == want_digest, f"frame {t}: the replay left the reference node's map"
        assert len(r.inactive()) == want_inactive
        for p in [q for q in window_prev if q not in window]:          # move_add_surfels: removal first ...
            if ctx.inactive_retire(p) > 0:
                stored.add(p)
        for p in [q for q in window if q not in window_prev and q in stored]:   # ... then insertion
            ctx.inactive_reactivate(p)
            stored.discard(p)
        window_prev = window
        ctx.fuse_frame_resident(ref_index, gray, depth, np.ascontiguousarray(fuse_pose.T.reshape(16)))
        got = ctx.pool_download()
        got = got[got["update_times"] > 0]
        assert abs(len(got) - len(want)) <= max(2, len(want) // 300), f"frame {t}: {len(got)} vs {len(want)} local surfels"
        if len(got) == len(want):
            match_as_sets(got, want, tol=1e-3)
        n_in = ctx.inactive_size()[0]
        assert abs(n_in - want_inactive) <= max(2, n_in // 300), f"frame {t}: inactive {n_in}"
    assert ctx.inactive_size()[0] > 0, "the drive never retired a keyframe"
    ctx.close()
