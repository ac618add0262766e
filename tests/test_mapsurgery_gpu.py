"""GPU parity of the map-surgery and nearest-neighbour entry points (SURVEY 8(f) #4) through the C ABI: against the
numpy oracle (brute force), against scipy's k-d tree at a size the brute force cannot reach, and against the reference's
own distCUDA2 (simple-knn built unmodified by oracle/build_ref.py; tests/golden/knn_dist_cuda2.npz holds its outputs)."""
import os

import numpy as np
import pytest
import torch

import helpers
from oracle import knn_oracle as ko
from rtg_slam_b200 import mapsurgery, scene

pytestmark = pytest.mark.gpu


def _surface_points(n, seed):
    """Gaussian centres of the surfel room (points on surfaces, as a SLAM map has them) plus exact duplicates."""
    g = scene.surfel_room(n, seed=seed)
    pts = g["xyz"].astype(np.float32).copy()
    pts[n // 2: n // 2 + n // 50] = pts[: n // 50]  # duplicates: distance 0 between different indices
    return pts


def _check_knn(d2, idx, want_d2, query, ref, K):
    d2, idx = d2.cpu().numpy(), idx.cpu().numpy()
    assert d2.shape == want_d2.shape
    assert np.all(np.diff(d2, axis=1) >= 0), "neighbours must be sorted by distance"
    fin = want_d2 < 1e37
    assert np.array_equal(fin, d2 < 1e37)
    assert np.allclose(d2[fin], want_d2[fin], rtol=2e-6, atol=1e-12)   # same fp32 expression, contraction may differ
    # the reported indices realise the reported distances (ties may name another equally near point)
    rr = ref[np.where(fin, idx, 0)]
    dd = ((rr - query[:, None, :]) ** 2).sum(-1)
    assert np.allclose(dd[fin], d2[fin], rtol=2e-6, atol=1e-12)
    assert np.all(idx[~fin] == 2**31 - 1)


@pytest.mark.parametrize("n,K", [(1, 3), (2, 3), (5, 3), (3000, 3), (20_000, 6), (20_000, 8)])
def test_knn_self_matches_brute_force(cuda_device, n, K):
    pts = _surface_points(max(n, 100), seed=3)[:n]
    t = torch.from_numpy(pts).to(cuda_device)
    for skip in (True, False):
        d2, idx = mapsurgery.knn(t, t, K, skip_self=skip)
        want, _ = ko.knn(pts, pts, K, skip_self=skip)
        _check_knn(d2, idx, want, pts, pts, K)
        if skip:
            assert not np.any(idx.cpu().numpy() == np.arange(n)[:, None])


def test_knn_points_api_query_outside_reference_box(cuda_device):
    """Mapping.temp_points_filter: new points against the existing unstable Gaussians (different sets; queries may lie far
    outside the reference points' bounding box)."""
    rng = np.random.default_rng(5)
    ref = _surface_points(8000, seed=7)
    q = np.concatenate([ref[:500] + rng.normal(0, 0.01, (500, 3)), rng.uniform(-20, 20, (300, 3))]).astype(np.float32)
    tq, tr = torch.from_numpy(q).to(cuda_device), torch.from_numpy(ref).to(cuda_device)
    out = mapsurgery.knn_points(tq[None], tr[None], norm=2, K=3, return_nn=True)
    assert out.dists.shape == (1, 800, 3) and out.idx.dtype == torch.int64 and out.knn.shape == (1, 800, 3, 3)
    want, _ = ko.knn(q, ref, 3)
    _check_knn(out.dists[0], out.idx[0].int(), want, q, ref, 3)
    assert torch.equal(out.knn[0], tr[out.idx[0]])
    # gaussians_isolated: K = topk + 1 on the set itself, column 0 is the point itself (mapper.py:903-912)
    iso = mapsurgery.knn_points(tr[None], tr[None], norm=2, K=6, return_nn=True)
    assert float(iso.dists[0, :, 0].max()) == 0.0


def test_dist_cuda2_large_against_kdtree_and_reference(cuda_device):
    from scipy.spatial import cKDTree
    n = 300_000
    pts = _surface_points(n, seed=11)
    t = torch.from_numpy(pts).to(cuda_device)
    mean, idx = mapsurgery.distCUDA2(t)
    assert mean.shape == (n,) and idx.shape == (n, 3) and idx.dtype == torch.int32
    dd, _ = cKDTree(pts.astype(np.float64)).query(pts.astype(np.float64), k=4)
    want = (dd[:, 1:] ** 2).mean(1)
    assert np.allclose(mean.cpu().numpy(), want, rtol=1e-4, atol=1e-10)
    # the reference's own distCUDA2 on the same points, at a seeded sample of them (make_reference_cuda_golden.py)
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "knn_dist_cuda2.npz"))
    rows = helpers.sample_indices(n, helpers.KNN_ROWS, seed=n)
    assert np.allclose(mean.cpu().numpy()[rows], gold["mean"], rtol=2e-6, atol=1e-12)
    a = np.sort(idx.cpu().numpy(), 1)[rows]
    assert (a != gold["idx_sorted"]).any(1).mean() < 0.05  # indices differ only among equidistant neighbours (the planted duplicates)


def test_update_geometry_expression_on_our_knn(cuda_device):
    """GaussianPointCloud.update_geometry (gaussian_pointcloud.py:365-405) evaluated with distCUDA2 from this library and
    from the brute-force oracle: same scales / invalid mask."""
    n = 5000
    pts = _surface_points(n, seed=13)
    radius = np.full(n, 0.004, np.float32)
    t = torch.from_numpy(pts).to(cuda_device)
    _, idx = mapsurgery.distCUDA2(t)
    _, oidx = ko.dist_cuda2(pts)

    def scales(ix):
        ix = ix.astype(np.int64)
        d = [np.linalg.norm(pts - pts[ix[:, k]], axis=1) - 3 * radius[ix[:, k]] for k in range(3)]
        invalid = (d[0] < 0) | (d[1] < 0) | (d[2] < 0)
        return np.sqrt((d[0] ** 2 + d[1] ** 2 + d[2] ** 2) / 3), invalid
    s_a, inv_a = scales(idx.cpu().numpy())
    s_b, inv_b = scales(oidx)
    assert np.array_equal(inv_a, inv_b) and np.allclose(s_a, s_b, rtol=1e-5, atol=1e-9)


@pytest.mark.parametrize("P", [0, 1, 777, 200_000])
def test_soa_delete_remove_cat(cuda_device, P):
    """GaussianPointCloud.delete / remove / cat on the eleven attribute tensors against torch's own boolean indexing."""
    g = torch.Generator(device="cpu").manual_seed(P)
    shapes = dict(xyz=(P, 3), features_dc=(P, 1, 3), features_rest=(P, 15, 3), scaling=(P, 3), rotation=(P, 4), opacity=(P, 1),
                  normal=(P, 3), confidence=(P, 1))
    params = {k: torch.randn(s, generator=g).to(cuda_device) for k, s in shapes.items()}
    for k in ("add_tick", "depth_error_counter", "color_error_counter"):
        params[k] = torch.randint(0, 1000, (P, 1), generator=g, dtype=torch.int32).to(cuda_device)
    assert tuple(params) == mapsurgery.ATTRIBUTES
    mask = (torch.rand(P, generator=g) < 0.3).to(cuda_device)
    new = mapsurgery.delete(params, mask)
    for k, v in params.items():
        assert torch.equal(new[k], v[~mask]), k
        assert new[k].dtype == v.dtype and new[k].shape[1:] == v.shape[1:]
    taken, rest = mapsurgery.remove(params, mask)
    for k, v in params.items():
        assert torch.equal(taken[k], v[mask]) and torch.equal(rest[k], v[~mask]), k
    back = mapsurgery.cat(rest, taken)
    for k, v in params.items():
        assert torch.equal(back[k], torch.cat([v[~mask], v[mask]])), k
    # all / none
    for m in (torch.zeros(P, dtype=torch.bool, device=cuda_device), torch.ones(P, dtype=torch.bool, device=cuda_device)):
        d = mapsurgery.delete(params, m)
        assert all(torch.equal(d[k], params[k][~m]) for k in params)


def test_api_errors(cuda_device):
    t = torch.zeros((10, 3), device=cuda_device)
    with pytest.raises(TypeError):
        mapsurgery.knn(t.double(), t, 3)
    with pytest.raises(Exception):
        mapsurgery.knn(t, t, 9)
    with pytest.raises(TypeError):
        mapsurgery.compact(torch.zeros(10, device=cuda_device), [t])
    with pytest.raises(NotImplementedError):
        mapsurgery.knn_points(t[None], t[None], norm=1, K=1)
