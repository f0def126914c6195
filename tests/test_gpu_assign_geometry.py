"""Assign pass on frame shapes whose edges cut its CTAs in different places.  A CTA of the assign pass covers one
seed-row band (pixel rows 8k-4 .. 8k+3) and a run of 128 columns starting at 128a - 4, so what matters is where
W + 4 and H + 4 fall: exactly on a run or band boundary, a few pixels past it, or in the middle.  After every assign
and every seed update the labels and the clustering state must equal the restatement's."""
import numpy as np
import pytest

from densesurfelmapping_b200 import synth
from densesurfelmapping_b200.elements import SURFEL_DTYPE
from util import bits_equal_nan

pytestmark = pytest.mark.gpu

# (W, H): W + 4 = 32 / 128 / 256 (whole runs), 264 / 272 (one / two threads in the last run), 1230 / 1245 (wide);
# H + 4 = 28 / 380 (last band half full), 32 / 40 (whole bands), 374 (last band 6 rows).  W % 8 and H % 8 stay <= 4.
SHAPES = [(28, 28), (124, 36), (252, 24), (260, 376), (268, 370), (1226, 28), (1241, 36)]


@pytest.fixture(scope="module")
def capi():
    from densesurfelmapping_b200 import capi as m
    m.load_library()
    return m


@pytest.mark.parametrize("flat", [False, True], ids=["noisy", "flat"])
@pytest.mark.parametrize("shape", SHAPES, ids=[f"{w}x{h}" for w, h in SHAPES])
def test_assign_stage_by_stage(capi, shape, flat):
    import pyoracle
    W, H = shape
    cam = synth.Camera(W, H, 0.8 * W, 0.8 * W, (W - 1) / 2, (H - 1) / 2, 0.5, 30.0)
    gray, depth = synth.make_frame(cam, W + H, flat=flat)
    ro = pyoracle.Restatement(cam)
    ctx = capi.Context(cam, max_batch=1, max_local_surfels=16)
    ctx.batch_upload([0], gray[None], depth[None], synth.identity_pose()[None], np.zeros(0, SURFEL_DTYPE), [0, 0])
    # (kernels to run, oracle iterations, last-with-update): seed_init, then (assign, gather, newton) x 3
    for nk, iters, upd in [(2, 1, False), (4, 1, True), (5, 2, False), (7, 2, True), (8, 3, False), (10, 3, True)]:
        ctx.debug_stop_after(nk)
        ctx.batch_run()
        ctx.sync()
        lab_o, seeds_o = ro.debug_iters(gray, depth, iters, upd)
        lab_g, seeds_g = ctx.labels(), ctx.seeds()
        nbad = int((lab_o != lab_g).sum())
        assert nbad == 0, f"after {nk} kernels: {nbad} label mismatches, first {np.argwhere(lab_o != lab_g)[:4].tolist()}"
        for f in ("x", "y", "mean_intensity", "mean_depth"):
            bad = np.nonzero(~bits_equal_nan(seeds_g[f], seeds_o[f]))[0]
            assert len(bad) == 0, f"after {nk} kernels: seed.{f} differs at {bad[:6]}"
        assert (seeds_g["stable"] == seeds_o["stable"]).all(), f"after {nk} kernels: stable differs"
        assert ctx.invariant_violations() == 0
    ctx.debug_stop_after(0)
    ctx.close()
