"""GPU parity tests of the rasterizer (through the public operator API -> ctypes -> C ABI -> sm_100a kernels)
against the CPU oracle and the committed golden outputs of the reference's CUDA code (small scenes in full, the timed
configurations and an optimisation loop as seeded samples).

Tolerances (SURVEY.md section 8(c)): float maps L_inf < 1e-4; index maps exact outside pixels whose deciding
alpha / T is within 1e-4 (relative) of a threshold (flagged by the oracle); per-tensor gradient
max|g-g_ref| / max|g_ref| < 1e-3 (and >= 10x the reference's own atomic-order jitter)."""
import os

import numpy as np
import pytest
import torch

import helpers
from golden.make_raster_golden import CASES, build_case
from oracle.splat_oracle import OracleRender
from rtg_slam_b200 import scene

pytestmark = pytest.mark.gpu
NAMES = ("color", "depth", "hit_color", "hit_depth", "hit_color_weight", "hit_depth_weight", "T_map", "radii")
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GRADS = ("means3D", "shs", "opacities", "scales", "rotations")


def oracle_outputs(o):
    return dict(zip(NAMES, o.outputs()))


def check_against_oracle(cam, g, dev, mask=None, label="", **over):
    grads = scene.upstream_grads(cam, seed=5)
    ours = helpers.run_ours(cam, g, dev, tile_mask=mask, grads=grads, **over)
    o = OracleRender(cam, g, tile_mask=mask, precision="f32", tie_eps=1e-4, **over)
    st = helpers.compare_outputs(ours, oracle_outputs(o), tie=o.tie, tol=1e-4, label=label)
    # ceil(3 sigma) may differ by one pixel for a Gaussian whose extent is within rounding of an integer
    assert st["radii_mismatch"] <= max(0, int(1e-5 * g["xyz"].shape[0])), st
    og = o.backward(*grads)
    for k in GRADS:
        e = helpers.rel_err(ours["grads"][k], og[k])
        assert e < 1e-3, f"{label}: d{k} rel err {e:.2e}"
    return ours, o


@pytest.mark.parametrize("name", sorted(CASES))
def test_matches_oracle_on_golden_scenes(cuda_device, name):
    cam, g, mask, _ = build_case(name)
    check_against_oracle(cam, g, cuda_device, mask=mask, label=name)


@pytest.mark.parametrize("name", sorted(CASES))
def test_matches_reference_cuda_golden(cuda_device, name):
    path = os.path.join(GOLD, name + ".npz")
    if not os.path.exists(path):
        pytest.skip("golden fixture missing")
    gold = np.load(path)
    cam, g, mask, grads = build_case(name)
    ours = helpers.run_ours(cam, g, cuda_device, tile_mask=mask, grads=grads)
    o = OracleRender(cam, g, tile_mask=mask, precision="f32", tie_eps=1e-4)  # only for the tie mask
    st = helpers.compare_outputs(ours, {k: gold[k] for k in NAMES}, tie=o.tie, tol=1e-4, label=name)
    assert st["radii_mismatch"] == 0
    for k in GRADS:
        tol = max(1e-3, 10 * float(gold["jitter_" + k]))
        assert helpers.rel_err(ours["grads"][k], gold["grad_" + k]) < tol, k


@pytest.mark.parametrize("camname,P,keep", helpers.LIVE_CASES)
def test_matches_live_reference_cuda(cuda_device, camname, P, keep):
    """The timed configurations against the reference's own CUDA rasterizer, as stored by make_reference_cuda_golden.py:
    pixel maps at a seeded pixel sample, gradients at the sampled rows over the reference's max |g| of the whole tensor,
    radii exactly (digest)."""
    gold = np.load(os.path.join(GOLD, "live_raster_reference.npz"))
    cam, g, mask, grads, c = helpers.live_case(camname, P, keep)
    ours = helpers.run_ours(cam, g, cuda_device, tile_mask=mask, grads=grads)
    rows = gold[f"{c}_rows"]
    a = dict(helpers.pixel_sample(ours, helpers.live_pixels(cam)), radii=ours["radii"][rows])
    b = dict({k: gold[f"{c}_{k}"][:, None] for k in helpers.PIXEL_MAPS}, radii=gold[f"{c}_radii"])
    st = helpers.compare_outputs(a, b, tol=1e-4, max_bad_frac=5e-4, label=f"{camname}/{P}/{keep}")
    assert st["radii_mismatch"] == 0 and helpers.digest(ours["radii"].astype(np.int32)) == str(gold[f"{c}_radii_digest"])
    for k in GRADS:
        jitter = float(gold[f"{c}_jitter_{k}"])
        err = np.abs(ours["grads"][k][rows].astype(np.float64) - gold[f"{c}_grad_{k}"]).max() / (float(gold[f"{c}_gradmax_{k}"]) + 1e-12)
        assert err < max(1e-3, 10 * jitter), (k, err, jitter)


def test_sh_degrees_and_background(cuda_device):
    cam = scene.make_camera("small")
    g = scene.surfel_room(2000, seed=4)
    for deg in (0, 1, 2):
        check_against_oracle(cam, g, cuda_device, label=f"deg{deg}", sh_degree=deg)
    check_against_oracle(cam, g, cuda_device, label="bg", bg=(0.2, 0.5, 0.9))


def test_thresholds_variants(cuda_device):
    cam = scene.make_camera("ragged")
    g = scene.random_blobs(1500, seed=12)
    check_against_oracle(cam, g, cuda_device, label="thr", opaque_threshold=0.3, depth_threshold=0.5,
                         normal_threshold=float(np.cos(np.deg2rad(30.0))), color_sigma=2.0, T_threshold=1e-3)


@pytest.mark.parametrize("P", [30_000, 250_000])
def test_oversized_tile_lists(cuda_device, P):
    """Tile lists longer than the on-chip sort capacity (4096 keys; then 8192; then chunked): the slow paths of the per-tile sort."""
    cam = scene.make_camera("tiny")
    g = scene.dense_blobs(P, seed=21)
    ours, o = check_against_oracle(cam, g, cuda_device, label=f"oversized{P}")
    _, rg = o.binning()
    longest = int((rg[:, 1] - rg[:, 0]).max())
    assert longest > (2 * 4096 if P < 50_000 else 4 * 8192), longest  # ours are shorter (exact culling), still past the limits


def test_equal_depth_ties_follow_gaussian_index(cuda_device):
    """Splats with bit-identical view depth composite in ascending Gaussian index order (the reference's radix sort is
    stable and duplicateWithKeys emits in index order, SURVEY appendix #9)."""
    cam = scene.make_camera("small")
    g0 = scene.random_blobs(1200, seed=31)
    rng = np.random.default_rng(3)
    g = {}
    for k, v in g0.items():  # every Gaussian three times, same centre (=> same depth), different colour / opacity
        g[k] = np.ascontiguousarray(np.concatenate([v, v, v]))
    g["shs"][1200:, 0] = rng.uniform(-1.5, 1.5, (2400, 3)).astype(np.float32)
    g["opacity"][2400:] = rng.uniform(0.05, 0.9, (1200, 1)).astype(np.float32)
    perm = rng.permutation(3600)
    g = {k: np.ascontiguousarray(v[perm]) for k, v in g.items()}
    check_against_oracle(cam, g, cuda_device, label="ties")


def test_backward_with_masked_upstream_gradient(cuda_device):
    """Mapping optimises with a render mask: dL/dcolour is exactly zero outside it (mapper.py:421). Those pixels are
    skipped by the backward; the result must equal the full replay (they only add zeros)."""
    cam = scene.make_camera("small")
    g = scene.surfel_room(3000, seed=14)
    gc, gd = scene.upstream_grads(cam, seed=5)
    rng = np.random.default_rng(2)
    keep = rng.uniform(size=(cam.height, cam.width)) < 0.4
    gc = gc * keep[None]
    ours = helpers.run_ours(cam, g, cuda_device, grads=(gc, gd))
    o = OracleRender(cam, g, precision="f32")
    og = o.backward(gc, gd)
    for k in GRADS:
        assert helpers.rel_err(ours["grads"][k], og[k]) < 1e-3, k


def test_edge_cases(cuda_device):
    from rtg_slam_b200.rasterizer import GaussianRasterizer
    dev = cuda_device
    cam = scene.make_camera("tiny")
    rs = helpers.make_settings(cam, dev)
    # P == 0 (rasterize_points.cu short-circuits; outputs keep their initial values)
    z = lambda *s: torch.zeros(*s, device=dev)
    out = GaussianRasterizer(rs)(means3D=z(0, 3), opacities=z(0, 1), shs=z(0, 16, 3), scales=z(0, 3), rotations=z(0, 4))
    assert out[0].abs().max() == 0 and (out[6] == 1).all() and (out[2] == 0).all() and out[7].numel() == 0
    # everything culled
    g = scene.random_blobs(64, seed=3)
    g["xyz"][:, 2] = -2.0
    r = helpers.run_ours(cam, g, dev, grads=scene.upstream_grads(cam))
    assert (r["radii"] == 0).all() and (r["T_map"] == 1).all() and (r["hit_depth"] == 0).all()
    assert all(np.all(v == 0) for v in r["grads"].values())
    # all tiles masked out
    g = scene.random_blobs(200, seed=5)
    th, tw = cam.tile_grid
    r = helpers.run_ours(cam, g, dev, tile_mask=np.zeros((th, tw), np.int32), grads=scene.upstream_grads(cam))
    assert (r["T_map"] == 1).all() and (r["color"] == 0).all()
    assert all(np.all(v == 0) for v in r["grads"].values())
    assert (r["radii"] > 0).any()  # radii are still reported for visible Gaussians, as in the reference


def test_api_errors(cuda_device):
    from rtg_slam_b200.rasterizer import GaussianRasterizer
    dev = cuda_device
    cam = scene.make_camera("tiny")
    rs = helpers.make_settings(cam, dev)
    t = helpers.to_torch(scene.random_blobs(10, seed=1), dev)
    R = GaussianRasterizer(rs)
    with pytest.raises(Exception, match="excatly one of either SHs or precomputed colors"):
        R(means3D=t["xyz"], opacities=t["opacity"], scales=t["scales"], rotations=t["rotations"])
    with pytest.raises(Exception, match="exactly one of either scale/rotation pair"):
        R(means3D=t["xyz"], opacities=t["opacity"], shs=t["shs"])
    with pytest.raises(ValueError, match="means3D must have dimensions"):
        R(means3D=t["xyz"].reshape(-1), opacities=t["opacity"], shs=t["shs"], scales=t["scales"], rotations=t["rotations"])
    with pytest.raises(TypeError, match="CUDA float32"):
        R(means3D=t["xyz"].cpu(), opacities=t["opacity"], shs=t["shs"], scales=t["scales"], rotations=t["rotations"])


def test_capacity_overflow_is_retried(cuda_device):
    from rtg_slam_b200 import rasterizer
    cam = scene.make_camera("small")
    g = scene.surfel_room(3000, seed=1)
    st = rasterizer._state(cuda_device)
    o = OracleRender(cam, g, precision="f32", tie_eps=1e-4)
    st.reap(block=True)
    try:
        # a forward that waits for its own count ('sync', and the first call of a shape in 'auto') re-runs on overflow
        rasterizer.set_capacity_checks("sync", cuda_device)
        st.r_hint = 16  # far too small: the first attempt must overflow and be re-run
        ours = helpers.run_ours(cam, g, cuda_device)
        helpers.compare_outputs(ours, oracle_outputs(o), tie=o.tie, label="overflow retry")
        assert st.r_hint >= o.num_rendered
        rasterizer.set_capacity_checks("auto", cuda_device)
        st.seen.clear()
        st.r_hint = 16
        ours = helpers.run_ours(cam, g, cuda_device)  # first call of this shape: waits, retries
        helpers.compare_outputs(ours, oracle_outputs(o), tie=o.tie, label="overflow retry (auto, first call)")
        # a forward that does not wait must not fail silently: the overflow surfaces at the frame's own backward ...
        st.r_hint = 16
        with pytest.raises(RuntimeError, match="rendered empty"):
            helpers.run_ours(cam, g, cuda_device, grads=scene.upstream_grads(cam, seed=5))
        assert st.r_hint >= o.num_rendered  # ... and the capacity has been raised: the next frame is complete again
        ours = helpers.run_ours(cam, g, cuda_device, grads=scene.upstream_grads(cam, seed=5))
        helpers.compare_outputs(ours, oracle_outputs(o), tie=o.tie, label="after overflow")
        # ... or, for a forward without a backward, at the next rasterizer call
        st.r_hint = 16
        helpers.run_ours(cam, g, cuda_device)
        torch.cuda.synchronize()
        with pytest.raises(RuntimeError, match="rendered empty"):
            helpers.run_ours(cam, g, cuda_device)
        ours = helpers.run_ours(cam, g, cuda_device)
        helpers.compare_outputs(ours, oracle_outputs(o), tie=o.tie, label="after overflow 2")
    finally:
        rasterizer.set_capacity_checks("auto", cuda_device)
        try:
            st.reap(block=True)
        except RuntimeError:
            pass


def test_two_forwards_then_two_backwards(cuda_device):
    """The saved state of each forward must stay valid if another render happens before its backward (the
    reference allocates fresh buffers per call, rasterize_points.cu:89-96)."""
    from rtg_slam_b200.rasterizer import GaussianRasterizer
    dev = cuda_device
    cams = [scene.make_camera("small"), scene.make_camera("small", c2w=scene.small_pose())]
    g = scene.surfel_room(3000, seed=6)
    t = helpers.to_torch(g, dev)
    leaves = {k: t[k].clone().requires_grad_(True) for k in ("xyz", "shs", "opacity", "scales", "rotations")}
    outs = []
    for cam in cams:
        rs = helpers.make_settings(cam, dev)
        outs.append(GaussianRasterizer(rs)(means3D=leaves["xyz"], opacities=leaves["opacity"], shs=leaves["shs"],
                                           scales=leaves["scales"], rotations=leaves["rotations"]))
    gc, gd = scene.upstream_grads(cams[0], seed=5)
    gct, gdt = torch.from_numpy(gc).to(dev), torch.from_numpy(gd).to(dev)
    total = None
    for i in (1, 0):  # backward in the opposite order
        for v in leaves.values():
            v.grad = None
        ((outs[i][0] * gct).sum() + (outs[i][1] * gdt).sum()).backward()
        o = OracleRender(cams[i], g, precision="f32")
        og = o.backward(gc, gd)
        assert helpers.rel_err(leaves["xyz"].grad.cpu().numpy(), og["means3D"]) < 1e-3
        assert helpers.rel_err(leaves["shs"].grad.cpu().numpy(), og["shs"]) < 1e-3


def test_forward_is_deterministic_and_mark_visible(cuda_device):
    from rtg_slam_b200.rasterizer import GaussianRasterizer
    cam = scene.make_camera("tum")
    g = scene.surfel_room(20000, seed=8)
    a = helpers.run_ours(cam, g, cuda_device)
    b = helpers.run_ours(cam, g, cuda_device)
    for k in NAMES:
        assert np.array_equal(a[k], b[k]), k
    rs = helpers.make_settings(cam, cuda_device)
    vis = GaussianRasterizer(rs).markVisible(torch.from_numpy(g["xyz"]).to(cuda_device)).cpu().numpy()
    assert vis.dtype == np.bool_ and np.all(vis[a["radii"] > 0])


def test_full_size_properties(cuda_device):
    """BASELINE.json's headline configuration (1 M Gaussians, 1200x680): size-independent properties."""
    cam = scene.make_camera("replica")
    g = scene.surfel_room(1_000_000, seed=2024)
    mask = scene.random_tile_mask(cam, 0.5, seed=11)
    grads = scene.upstream_grads(cam, seed=5)
    r = helpers.run_ours(cam, g, cuda_device, tile_mask=mask, grads=grads)
    T = r["T_map"][0]
    assert (T > 0).all() and (T <= 1).all()
    up = np.kron(mask, np.ones((16, 16), np.int32))[: cam.height, : cam.width].astype(bool)
    assert (T[~up] == 1).all() and (r["color"][:, ~up] == 0).all() and (r["hit_depth"][0][~up] == 0).all()
    hit = r["hit_depth"][0]
    assert hit.max() < 1_000_000 and hit[up].min() >= -1
    assert (r["radii"][hit[(hit >= 0) & up]] > 0).all()  # a hit refers to a visible Gaussian
    assert (r["hit_depth_weight"][0][(hit >= 0) & up] >= 0).all()  # alpha*T; T may underflow to 0 behind many translucent splats
    d = r["depth"][0]
    v1, v2 = int(((hit >= 0) & up & ~(d > 0)).sum()), int(((d > 0) & ~((hit >= 0) & up)).sum())
    assert v1 + v2 <= 80, f"depth>0 must coincide with a hit: hit-without-depth {v1}, depth-without-hit {v2}"
    for k, v in r["grads"].items():
        assert np.isfinite(v).all(), k
        assert np.all(v[r["radii"] == 0] == 0), f"culled Gaussians must get exactly zero d{k}"
    # linearity of the backward in the upstream gradient
    r2 = helpers.run_ours(cam, g, cuda_device, tile_mask=mask, grads=(2 * grads[0], 2 * grads[1]))
    for k in GRADS:
        assert helpers.rel_err(r2["grads"][k], 2 * r["grads"][k]) < 1e-4, k


@pytest.mark.gpu
def test_tile_sharded_pieces_reassemble(cuda_device):
    """SURVEY 8(e): the ranks of a tile-sharded frame render disjoint tile subsets of the same map. Emulated on one
    GPU: the union of the pieces is bit-identical to the full render (a tile's result does not depend on which
    other tiles are rendered) and the partial gradients add up to the full gradient."""
    from rtg_slam_b200.parallel import TileShard
    cam = scene.make_camera("replica")
    g = scene.surfel_room(50_000, seed=21)
    grads = scene.upstream_grads(cam, seed=5)
    full = helpers.run_ours(cam, g, cuda_device, grads=grads)
    wts = None
    for world, weighted in ((2, False), (3, True)):
        if weighted:  # per-tile work estimate: Gaussians whose centre falls into the tile
            wts = torch.rand(cam.tile_grid[0] * cam.tile_grid[1], generator=torch.Generator().manual_seed(1))
        pieces = []
        for r in range(world):
            sh = TileShard(cam.height, cam.width, world, r, weights=wts)
            res = helpers.run_ours(cam, g, cuda_device, tile_mask=sh.mask.numpy(), grads=grads)
            pieces.append((sh, res))
        for k in ("color", "depth", "hit_color", "hit_depth", "hit_color_weight", "hit_depth_weight", "T_map"):
            acc = np.zeros_like(full[k])
            for sh, res in pieces:
                pm = sh.pixel_mask.numpy()
                acc = np.where(pm[None], res[k], acc)
                # outside its tiles a rank holds the reference's initial values (rasterize_points.cu:79-87)
                init = 1.0 if k == "T_map" else 0
                assert np.all(res[k][:, ~pm] == init), k
            assert np.array_equal(acc, full[k]), k
        for k in full["grads"]:
            tot = sum(res["grads"][k] for _, res in pieces)
            assert helpers.rel_err(tot, full["grads"][k]) < 1e-4, k


@pytest.mark.gpu
def test_two_phase_backward_with_record_exchange(cuda_device):
    """rtg_splat_backward_render / _finish with an exchange step in between (TileShard.exchange_records). Emulated on
    one GPU: pass 1 captures every shard's gradient records, pass 2 substitutes their sum -- the gradients that come out
    are those of the full frame; without a hook the two-phase path is the one-call path."""
    from rtg_slam_b200 import rasterizer
    from rtg_slam_b200.parallel import TileShard
    cam = scene.make_camera("replica")
    g = scene.surfel_room(40_000, seed=22)
    grads = scene.upstream_grads(cam, seed=5)
    full = helpers.run_ours(cam, g, cuda_device, grads=grads)
    world = 3
    shards = [TileShard(cam.height, cam.width, world, r) for r in range(world)]
    captured = []

    def capture(rec):
        captured.append(rec.clone())
    prev = rasterizer.set_grad_record_hook(capture)
    try:
        for sh in shards:
            helpers.run_ours(cam, g, cuda_device, tile_mask=sh.mask.numpy(), grads=grads)
        assert len(captured) == world and captured[0].shape == (40_000, 16)
        total = sum(captured)
        assert float(total.abs().max()) > 0

        def substitute(rec):
            rec.copy_(total)
        rasterizer.set_grad_record_hook(substitute)
        res = helpers.run_ours(cam, g, cuda_device, tile_mask=shards[1].mask.numpy(), grads=grads)
        for k in full["grads"]:
            assert helpers.rel_err(res["grads"][k], full["grads"][k]) < 1e-4, k
        # identity exchange == single call (records are consumed and cleared either way)
        rasterizer.set_grad_record_hook(lambda rec: None)
        same = helpers.run_ours(cam, g, cuda_device, grads=grads)
    finally:
        rasterizer.set_grad_record_hook(prev)
    again = helpers.run_ours(cam, g, cuda_device, grads=grads)
    for k in full["grads"]:
        assert helpers.rel_err(same["grads"][k], full["grads"][k]) < 1e-5, k
        assert helpers.rel_err(again["grads"][k], full["grads"][k]) < 1e-5, k   # scratch left clean


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 3])
def test_gaussian_sharded_frame_matches_unsharded(cuda_device, world):
    """SURVEY 8(e) / BASELINE configs[4]: Gaussians AND tiles sharded over ranks (parallel.GaussianShard). Emulated on one
    GPU by running the ranks' stages in lock step and doing the two exchanges by hand (all-gather of the per-Gaussian
    records = copying every owner's slice to every rank; reduce-scatter of the gradient records = summing the ranks'
    record buffers and handing each owner its slice). The union of the image pieces is bit-identical to the unsharded
    render, the owners' gradients equal the rows of the unsharded gradient."""
    from rtg_slam_b200.parallel import GaussianShard
    cam = scene.make_camera("replica")
    P = 30_000
    g = scene.surfel_room(P, seed=23)
    grads = scene.upstream_grads(cam, seed=5)
    full = helpers.run_ours(cam, g, cuda_device, grads=grads)
    rs = helpers.make_settings(cam, cuda_device)
    t = helpers.to_torch(g, cuda_device)
    shards = [GaussianShard(P, cam.height, cam.width, cuda_device, world_size=world, r=r) for r in range(world)]
    staged = []
    for sh in shards:
        a, b = sh.p_begin, sh.p_end
        staged.append(sh.forward(rs, t["xyz"][a:b], t["opacity"][a:b], t["shs"][a:b], t["scales"][a:b], t["rotations"][a:b], staged=True))
    for _ in range(2):  # second pass: the first one may have overflowed the initial binning capacity
        for (_, pre, _) in staged:
            pre()
        for sh in shards:  # all-gather by hand
            for dst in shards:
                if dst is sh:
                    continue
                for vs, vd in zip(sh._record_views(), dst._record_views()):
                    vd[sh.p_begin:sh.p_end].copy_(vs[sh.p_begin:sh.p_end])
                dst.radii[sh.p_begin:sh.p_end].copy_(sh.radii[sh.p_begin:sh.p_end])
        ok = [ren() for (_, _, ren) in staged]
        if all(ok):
            break
    assert all(ok)
    assert np.array_equal(shards[0].radii.cpu().numpy(), full["radii"])
    for k in ("color", "depth", "hit_color", "hit_depth", "hit_color_weight", "hit_depth_weight", "T_map"):
        acc = np.zeros_like(full[k])
        for sh, (res, _, _) in zip(shards, staged):
            acc = np.where(sh.tiles.pixel_mask.cpu().numpy()[None], res[k].cpu().numpy(), acc)
        assert np.array_equal(acc, full[k]), k
    gc, gd = torch.from_numpy(grads[0]).to(cuda_device), torch.from_numpy(grads[1]).to(cuda_device)
    stages = [sh.backward(gc, gd, staged=True) for sh in shards]
    for ren, _ in stages:
        ren()
    total = sum(sh.rec_full for sh in shards)  # reduce ...
    for sh in shards:                           # ... scatter
        sh.rec_own.copy_(total[sh.p_begin:sh.p_end])
    for sh, (_, fin) in zip(shards, stages):
        own = fin()
        for k in GRADS:
            want = full["grads"][k][sh.p_begin:sh.p_end]
            assert helpers.rel_err(own[k].cpu().numpy().reshape(want.shape), want) < 1e-4, (k, sh.rank)
        assert float(sh.rec_full.abs().max()) == 0.0  # the record buffer is clean for the next step


@pytest.mark.gpu
def test_optimize_loop_tracks_reference_rasterizer_with_torch_adam(cuda_device):
    """BASELINE configs[3], second half: the optimisation loop of the mapper on top of the hot path -- render -> colour +
    depth L1 -> backward -> Adam, 10 iterations -- run twice from the same state: this library end to end (rasterizer,
    fused loss, FusedAdam) and the reference's own CUDA rasterizer (oracle/_ref) driven by eager torch expressions and
    torch.optim.Adam (eps = 1e-15, lrs of configs/base.yaml:82-86, as Mapping.local_optimize sets it up). The loss must
    follow the same trajectory and the parameters must agree; with eps = 1e-15 Adam's update is sign(g) * lr for a
    gradient of any magnitude, so the handful of elements whose gradient is numerically zero may step the other way
    (atomic-order noise of the reference itself): they are bounded in number and by 2 * lr * iterations. The reference's
    side (losses, the parameters after the loop at a seeded element sample, max |p|, max |p - p0|, its run-to-run spread)
    is stored by make_reference_cuda_golden.py."""
    from rtg_slam_b200.loss import l1_color_depth_loss
    from rtg_slam_b200.optim import FusedAdam
    from rtg_slam_b200.rasterizer import GaussianRasterizer
    gold = np.load(os.path.join(GOLD, "optimize_loop_reference.npz"))
    cam, rs, t, gt_color, gt_depth = helpers.optimize_loop_case(cuda_device)
    lrs, iters = helpers.OPT_LOOP_LRS, helpers.OPT_LOOP_ITERS
    names = tuple(lrs)

    def run():
        p = {k: t[k].clone().requires_grad_(True) for k in names}
        opt = FusedAdam([{"params": [p[k]], "lr": lrs[k]} for k in names], lr=0.0, eps=1e-15)
        losses = []
        for _ in range(iters):
            opt.zero_grad(set_to_none=True)
            out = GaussianRasterizer(rs)(means3D=p["xyz"], opacities=p["opacity"], shs=p["shs"], scales=p["scales"], rotations=p["rotations"])
            loss, _ = l1_color_depth_loss({"render": out[0], "depth": out[1], "depth_index_map": out[3]}, gt_color, gt_depth,
                                          color_weight=0.8, depth_weight=1.0, depth_error_max=0.1)
            loss.backward()
            opt.step()
            losses.append(float(loss.detach()))
        return losses, {k: v.detach().clone() for k, v in p.items()}

    la, pa = run()
    lb = [float(x) for x in gold["losses"]]
    assert lb[-1] < lb[0], ("the loop must make progress", lb)
    for a, b in zip(la, lb):
        assert abs(a - b) < 2e-4 * abs(b), (la, lb)
    report = {}
    for k in names:
        scale = float(gold[f"{k}_scale"])
        moved = float(gold[f"{k}_moved"])
        if lrs[k] == 0.0:
            assert torch.equal(pa[k], t[k]) and moved == 0.0  # opacity_lr is 0 in every shipped config
            continue
        d_ours = np.abs(pa[k].reshape(-1).cpu().numpy()[helpers.optimize_loop_sample(k, t)] - gold[f"{k}_sample"])
        off_ours = float((d_ours > 1e-5 * scale).mean())
        off_self = float(gold[f"{k}_off_self"])
        report[k] = (off_ours, off_self)
        assert moved > 0
        assert float(d_ours.max()) <= 2.0 * lrs[k] * iters + 1e-7, k  # a flipped element is at most 2*lr per step away
    for k, (off_ours, off_self) in report.items():
        # measured: scales 2.1e-3, rotations 1.2e-3, shs 1.3e-4, xyz 0 (reference against itself: 1.5e-4, 5e-5, 1.7e-5, 0): this
        # library's alpha is within 1e-6 of the reference's, an order above fp32 re-association, so more near-cancelling
        # gradient elements change sign -- each such element random-walks by +-lr either way
        assert off_ours <= max(5e-3, 3.0 * off_self), f"{k}: fraction beyond 1e-5 of the range: ours {off_ours:.2e}, reference vs itself {off_self:.2e} ({report})"
