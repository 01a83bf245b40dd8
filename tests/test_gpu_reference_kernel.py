"""-m gpu: the UNMODIFIED reference CUDA extension (its pcpr kernel, compiled from the reference's own sources by
oracle/build_ref.py) against the oracle and against our kernel (SURVEY.md §8c(3)).  What the reference kernel computed on
a B200 for the two scenes below is stored in tests/golden/reference_pcpr.npz (tests/golden/make_reference_pcpr.py).

The reference kernel is nondeterministic under pixel contention (its lock drops contended writes), so:
  * on a collision-free scene (at most one point per pixel) all three must agree exactly;
  * on a dense scene the reference may only be WORSE than the true z-buffer: ref_depth >= oracle_depth wherever
    both are non-empty, and it never invents coverage.
"""
import numpy as np
import pytest

from conftest import load_golden
from gpu_util import render_gpu, scene_and_cams

pytestmark = pytest.mark.gpu

FREE_W, FREE_H = 64, 48
DENSE_N, DENSE_W, DENSE_H = 300_000, 128, 96


def collision_free_scene():
    ys, xs = np.mgrid[0:FREE_H, 0:FREE_W]
    # one point per pixel centre (identity matrix: u = W(x+1)/2), random depths, shuffled ids
    x = (xs.ravel() + 0.5) / FREE_W * 2 - 1
    y = 1 - (ys.ravel() + 0.5) / FREE_H * 2
    rng = np.random.default_rng(0)
    z = rng.uniform(-0.9, 0.9, x.size)
    xyz = np.stack([x, y, z], 1).astype(np.float32)[rng.permutation(x.size)]
    xyz = np.concatenate([np.full((1, 3), 9, np.float32), xyz])       # id 0 off-screen ("0 denotes empty")
    return xyz, np.eye(4, dtype=np.float32)[None]


def dense_scene():
    return scene_and_cams(DENSE_N, DENSE_W, DENSE_H, [0], depth=60.0)


def checksum(*arrays):
    return [float(np.abs(a.astype(np.float64)).sum()) for a in arrays]


@pytest.fixture(scope="module")
def ref_pcpr():
    return load_golden("reference_pcpr")


def test_collision_free_scene_all_three_agree(oracle_mod, ref_pcpr):
    W, H = FREE_W, FREE_H
    xyz, M = collision_free_scene()
    np.testing.assert_allclose(checksum(xyz, M), ref_pcpr["free_checksum"], rtol=1e-12)
    oi, od = oracle_mod.pcpr_forward(xyz, M, W, H)
    ri, rd = ref_pcpr["free_index"], ref_pcpr["free_depth"]
    gi, gd, _ = render_gpu(xyz, M, W, H, 1)
    assert (oi != 0).all()
    np.testing.assert_array_equal(ri, oi)
    np.testing.assert_array_equal(rd, od)
    np.testing.assert_array_equal(gi[0], oi)
    np.testing.assert_array_equal(gd[0], od)


def test_dense_scene_reference_is_never_better_than_the_zbuffer(oracle_mod, ref_pcpr):
    xyz, M = dense_scene()
    np.testing.assert_allclose(checksum(xyz, M), ref_pcpr["dense_checksum"], rtol=1e-12)
    oi, od = oracle_mod.pcpr_forward(xyz, M, DENSE_W, DENSE_H)
    ri, rd = ref_pcpr["dense_index"], ref_pcpr["dense_depth"]
    assert ((rd == 0) >= (od == 0)).all()                  # reference covers no pixel the z-buffer leaves empty
    both = (rd != 0) & (od != 0)
    assert (rd[both] >= od[both]).all()
    frac_equal = float((ri == oi).mean())
    print(f"reference kernel agrees with the sequential z-buffer on {100 * frac_equal:.2f}% of pixels")
    gi, gd, _ = render_gpu(xyz, M, DENSE_W, DENSE_H, 1)
    np.testing.assert_array_equal(gi[0], oi)               # ours is exact
