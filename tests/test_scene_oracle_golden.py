"""CPU: the ray-generation oracle (oracle/scene_oracle.py) against the reference's own
get_lidar_rays / get_rays outputs (tests/golden/rays_ref.npz, made by oracle/make_golden_rays.py),
plus self-consistency of the occupancy-grid oracle.  Tolerance: the reference evaluates
cos/sin/normalisation in torch fp32 — 2e-6 absolute on unit directions."""
import os

import numpy as np
import pytest

from conftest import GOLDEN

ATOL = 2e-6


@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(GOLDEN, "rays_ref.npz"))


@pytest.fixture(scope="module")
def SO():
    from oracle import scene_oracle
    return scene_oracle


def test_lidar_rays_full_frame(gold, SO):
    o, d = SO.get_lidar_rays(gold["pose_a"], gold["lidar_K"], gold["lidar_K_hoz"], 66, 1030)
    np.testing.assert_allclose(d[gold["lidar_full_a_inds"]], gold["lidar_full_a_d"], rtol=0, atol=ATOL)
    assert np.array_equal(o[0], gold["pose_a"][:3, 3]) and (o == o[0]).all()


@pytest.mark.parametrize("tag", ["a", "b"])
def test_lidar_rays_batch(gold, SO, tag):
    o, d = SO.get_lidar_rays(gold[f"pose_{tag}"], gold["lidar_K"], gold["lidar_K_hoz"], 66, 1030,
                             gold[f"lidar_batch_{tag}_inds"])
    np.testing.assert_allclose(d, gold[f"lidar_batch_{tag}_d"], rtol=0, atol=ATOL)
    if tag == "a":
        np.testing.assert_array_equal(o, gold["lidar_batch_a_o"])


@pytest.mark.parametrize("tag", ["a", "b"])
@pytest.mark.parametrize("kind", ["batch", "patch"])
def test_camera_rays(gold, SO, tag, kind):
    _, d = SO.get_rays(gold[f"pose_{tag}"], gold["cam_K"], 376, 1408, gold[f"cam_{kind}_{tag}_inds"])
    np.testing.assert_allclose(d, gold[f"cam_{kind}_{tag}_d"], rtol=0, atol=ATOL)


def test_camera_rays_small_full(gold, SO):
    _, d = SO.get_rays(gold["pose_a"], gold["cam_K"], 47, 176)
    np.testing.assert_allclose(d, gold["cam_small_full_d"], rtol=0, atol=ATOL)


def test_grid_cell_points_cover_cells(SO):
    """Cell centres land in their own cell of every cascade (round trip through morton3D)."""
    from oracle import raymarching_oracle as RO
    C, H, bound = 2, 16, 2.0
    rng = np.random.default_rng(0)
    x = SO.grid_cell_points(C, H, bound, rng.random((C * H ** 3, 3), dtype=np.float32)).reshape(C, H ** 3, 3)
    for c in range(C):
        bc = min(2 ** c, bound)
        assert np.abs(x[c]).max() <= bc
        # jitter is at most half a cell of the (H-1)-spaced lattice: nearest lattice node = the cell
        node = np.rint((x[c] / (bc - bc / H) + 1) * (H - 1) / 2).astype(np.int32)
        assert np.array_equal(RO.morton3D(node), np.arange(H ** 3, dtype=np.int32))


def test_grid_update_rules(SO):
    g = np.array([0.5, -1.0, 0.2, 0.0, 1.0, 0.3, 0.0, 0.0], np.float32)
    t = np.array([0.1, 0.7, -1.0, 0.4, 0.2, 0.9, 0.0, 0.0], np.float32)
    new, mean, thresh, bits = SO.grid_update(g, t, 0.95, 0.25)
    want = np.array([0.475, -1.0, 0.2, 0.4, 0.95, 0.9, 0.0, 0.0], np.float32)
    np.testing.assert_allclose(new, want, rtol=1e-7)
    assert np.isclose(mean, np.maximum(want, 0).mean())
    assert thresh == np.float32(0.25)
    assert bits.tolist() == [0b00111001]
