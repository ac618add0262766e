"""Shared test helpers: scene -> torch tensors, calls into the product path, the oracle and (when its
extension has been built into oracle/_ref/) the reference's own CUDA rasterizer."""
from __future__ import annotations

import glob
import hashlib
import importlib.util
import os

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

DEFAULT_SETTINGS = dict(scale_modifier=1.0, color_sigma=3.0, opaque_threshold=0.6, depth_threshold=1.0,
                        normal_threshold=float(np.cos(np.deg2rad(60.0))), T_threshold=1e-4, sh_degree=3)


def to_torch(g, device):
    return {k: torch.from_numpy(v).to(device) for k, v in g.items()}


def make_settings(cam, device, **over):
    from rtg_slam_b200.rasterizer import GaussianRasterizationSettings
    st = dict(DEFAULT_SETTINGS)
    st.update(over)
    return GaussianRasterizationSettings(
        image_height=cam.height, image_width=cam.width, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy,
        bg=torch.tensor(st.get("bg", (0.0, 0.0, 0.0)), dtype=torch.float32, device=device),
        scale_modifier=st["scale_modifier"],
        viewmatrix=torch.from_numpy(cam.viewmatrix).to(device), projmatrix=torch.from_numpy(cam.projmatrix).to(device),
        sh_degree=st["sh_degree"], campos=torch.from_numpy(cam.campos).to(device),
        opaque_threshold=st["opaque_threshold"], normal_threshold=st["normal_threshold"], depth_threshold=st["depth_threshold"],
        prefiltered=False, debug=False, cx=cam.cx, cy=cam.cy, color_sigma=st["color_sigma"], T_threshold=st["T_threshold"])


def run_ours(cam, g, device, tile_mask=None, grads=None, **over):
    """Forward (and backward if `grads`=(dL_dcolor, dL_ddepth) numpy) through the public operator API."""
    from rtg_slam_b200.rasterizer import GaussianRasterizer
    rs = make_settings(cam, device, **over)
    t = to_torch(g, device)
    leaves = {k: t[k].clone().requires_grad_(grads is not None) for k in ("xyz", "shs", "opacity", "scales", "rotations")}
    tm = None if tile_mask is None else torch.from_numpy(np.ascontiguousarray(tile_mask, dtype=np.int32)).to(device)
    out = GaussianRasterizer(rs)(means3D=leaves["xyz"], opacities=leaves["opacity"], shs=leaves["shs"], scales=leaves["scales"],
                                 rotations=leaves["rotations"], tile_mask=tm)
    res = dict(zip(("color", "depth", "hit_color", "hit_depth", "hit_color_weight", "hit_depth_weight", "T_map", "radii"),
                   [o.detach().cpu().numpy() for o in out]))
    if grads is not None:
        gc = torch.from_numpy(grads[0]).to(device)
        gd = torch.from_numpy(grads[1]).to(device)
        loss = (out[0] * gc).sum() + (out[1] * gd).sum()
        loss.backward()
        res["grads"] = dict(means3D=leaves["xyz"].grad.cpu().numpy(), shs=leaves["shs"].grad.cpu().numpy(),
                            opacities=leaves["opacity"].grad.cpu().numpy(), scales=leaves["scales"].grad.cpu().numpy(),
                            rotations=leaves["rotations"].grad.cpu().numpy())
    return res


# ---------------------------------------------------------------- reference CUDA (oracle/_ref)
_REF = None


def ref_cuda_module():
    """The reference's own `_C_depth` extension, built unmodified by oracle/build_ref.py. None if absent."""
    global _REF
    if _REF is None:
        so = glob.glob(os.path.join(ROOT, "oracle", "_ref", "_C_depth*.so"))
        if not so:
            _REF = False
        else:
            spec = importlib.util.spec_from_file_location("_C_depth", so[0])
            mod = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mod)
            _REF = mod
    return _REF or None


def run_ref_cuda(cam, g, device, tile_mask=None, grads=None, **over):
    """Calls rasterize_gaussians / rasterize_gaussians_backward of the reference exactly as its python shim does
    (RAST/diff_gaussian_rasterization_depth/__init__.py:69-97,200-232)."""
    mod = ref_cuda_module()
    assert mod is not None
    st = dict(DEFAULT_SETTINGS)
    st.update(over)
    t = to_torch(g, device)
    H, W = cam.height, cam.width
    th, tw = (H + 15) // 16, (W + 15) // 16
    tm = torch.ones((th, tw), dtype=torch.int32, device=device) if tile_mask is None else \
        torch.from_numpy(np.ascontiguousarray(tile_mask, dtype=np.int32)).to(device)
    bg = torch.tensor(st.get("bg", (0.0, 0.0, 0.0)), dtype=torch.float32, device=device)
    vm = torch.from_numpy(cam.viewmatrix).to(device)
    pm = torch.from_numpy(cam.projmatrix).to(device)
    cp = torch.from_numpy(cam.campos).to(device)
    e = torch.Tensor([])
    args = (bg, t["xyz"], e, t["opacity"], t["scales"], t["rotations"], st["scale_modifier"], e, vm, pm, tm, cam.tanfovx, cam.tanfovy,
            H, W, cam.cx, cam.cy, t["shs"], st["sh_degree"], st["color_sigma"], cp, st["opaque_threshold"], st["depth_threshold"],
            st["normal_threshold"], st["T_threshold"], False, False)
    (num_rendered, num_tile, color, depth, hit_color, hit_depth, hcw, hdw, T_map, radii, geomB, binB, imgB, tile_indices) = \
        mod.rasterize_gaussians(*args)
    res = dict(color=color, depth=depth, hit_color=hit_color, hit_depth=hit_depth, hit_color_weight=hcw, hit_depth_weight=hdw,
               T_map=T_map, radii=radii)
    res = {k: v.cpu().numpy() for k, v in res.items()}
    res["num_rendered"], res["num_tile"] = num_rendered, num_tile
    if grads is not None:
        gc = torch.from_numpy(grads[0]).to(device)
        gd = torch.from_numpy(grads[1]).to(device)
        bargs = (tile_indices, num_tile, bg, t["xyz"], radii, e, t["scales"], t["rotations"], st["scale_modifier"], e, vm, pm,
                 cam.tanfovx, cam.tanfovy, cam.cx, cam.cy, st["depth_threshold"], st["normal_threshold"], gc, gd, t["shs"],
                 st["sh_degree"], cp, geomB, num_rendered, binB, imgB, hit_depth, False)
        (g2d, gcol, gop, gm3, gcov, gsh, gsc, grot) = mod.rasterize_gaussians_backward(*bargs)
        res["grads"] = dict(means3D=gm3.cpu().numpy(), shs=gsh.cpu().numpy(), opacities=gop.cpu().numpy(), scales=gsc.cpu().numpy(),
                            rotations=grot.cpu().numpy(), means2D=g2d.cpu().numpy(), colors=gcol.cpu().numpy(),
                            cov3D=gcov.cpu().numpy())
    return res


# ---------------------------------------------------------------- stored samples of the reference's CUDA extensions
# tests/golden/make_reference_cuda_golden.py runs the reference's own extensions (oracle/_ref) on the inputs below. Their
# full outputs at these sizes are tens of MB, so the fixtures keep a seeded sample of each output plus the whole-array
# figures the assertions need (maxima, run-to-run jitter, a digest where the comparison is exact); the tests draw the
# same samples from the same seeds.
def sample_indices(n, k, seed):
    """`k` distinct indices of range(n), ascending (all of range(n) when k >= n)."""
    if k >= n:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, k, replace=False))


def digest(a):
    """SHA-256 of an array's dtype, shape and values (-0.0 hashed as 0.0): exact equality with an array that is not stored."""
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        a = a + a.dtype.type(0)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()


# (camera, Gaussians, tile-mask keep fraction). The last four are the timed configurations: BASELINE.json configs[1]
# (~300 k @1200x680), the headline scene of bench.py (1 M @1200x680: its longest tile list exceeds the 4096-key
# on-chip sort, i.e. the chunked-merge path), the same with a 50 % tile mask, and configs[2] (1 M @1920x1080).
LIVE_CASES = [("tum", 10_000, None), ("replica", 60_000, None), ("replica", 300_000, None), ("replica", 1_000_000, None),
              ("replica", 1_000_000, 0.5), ("hd", 1_000_000, None)]
LIVE_PIXELS = 2048          # sampled pixels per case: the 5e-4 outlier allowance still admits one
LIVE_ROWS = 128             # sampled visible Gaussians per case, besides the 8 largest gradient rows of each tensor
PIXEL_MAPS = ("color", "depth", "hit_color", "hit_depth", "hit_color_weight", "hit_depth_weight", "T_map")
GRADS = ("means3D", "shs", "opacities", "scales", "rotations")


def live_case(camname, P, keep):
    """Scene, tile mask, upstream gradients and the fixture key of one LIVE_CASES entry."""
    from rtg_slam_b200 import scene
    cam = scene.make_camera(camname)
    g = scene.surfel_room(P, seed=2024)
    mask = None if keep is None else scene.random_tile_mask(cam, keep, seed=11)
    grads = scene.upstream_grads(cam, seed=5)
    return cam, g, mask, grads, f"{camname}_{P}_{keep}"


def live_pixels(cam):
    return sample_indices(cam.height * cam.width, LIVE_PIXELS, seed=cam.height * cam.width)


def pixel_sample(maps, px):
    """The pixel maps of a render at the flat pixel indices `px`, shaped (C, 1, len(px)) for compare_outputs."""
    return {k: maps[k].reshape(maps[k].shape[0], 1, -1)[..., px] for k in PIXEL_MAPS}


# BASELINE configs[3], second half: 10 mapping iterations (render -> colour + depth L1 -> backward -> Adam) on this map.
# Colours / rotations / opacity take the lrs of configs/base.yaml:82-86; position and scale are optimised here in their
# activated form (the mapper steps log-scales), so their lrs are scaled down to keep the 10 steps a descent.
OPT_LOOP_LRS = dict(xyz=1e-4, shs=5e-4, opacity=0.0, scales=1e-4, rotations=1e-3)
OPT_LOOP_ITERS = 10
OPT_LOOP_SAMPLE = 8192      # sampled elements of each optimised parameter tensor


def optimize_loop_case(device):
    """(camera, rasterization settings, initial parameters, target colour (H,W,3), target depth (H,W)): the target frame is
    this library's render of the same map with perturbed colours and positions."""
    from rtg_slam_b200 import scene
    from rtg_slam_b200.rasterizer import GaussianRasterizer
    cam = scene.make_camera("tum")
    g = scene.surfel_room(20_000, seed=31)
    rs = make_settings(cam, device)
    t = to_torch(g, device)
    with torch.no_grad():
        tgt = GaussianRasterizer(rs)(means3D=t["xyz"] + 0.002, opacities=t["opacity"], shs=t["shs"] * 0.9, scales=t["scales"],
                                     rotations=t["rotations"])
    return cam, rs, t, tgt[0].permute(1, 2, 0).contiguous(), tgt[1][0].contiguous()


def optimize_loop_sample(k, t):
    return sample_indices(t[k].numel(), OPT_LOOP_SAMPLE, seed=sum(map(ord, k)))


# GaussianPointCloud.update_geometry's distCUDA2 on a 300 k-point surface map (test_mapsurgery_gpu.py)
KNN_ROWS = 8192


# Mapping's accumulate_gaussian_error (cuda_utils): (H, W, P) cases of test_mapstats_gpu.py
ACCUMULATE_CASES = [(680, 1200, 200_000), (77, 45, 300), (16, 16, 1)]
ACCUMULATE_ROWS = 4096
ACCUMULATE_THRESHOLDS = (0.3, 0.05, 0.5)


def accumulate_inputs(H, W, P, seed):
    """Colour / depth / normal error maps and colour / depth index maps, (H, W, 1) each."""
    rng = np.random.default_rng(seed)
    ce = rng.uniform(0, 1, (H, W, 1)).astype(np.float32) ** 2
    de = rng.uniform(0, 0.2, (H, W, 1)).astype(np.float32)
    ne = rng.uniform(0, 1, (H, W, 1)).astype(np.float32)
    de[rng.uniform(size=(H, W, 1)) < 0.2] = 0
    ci = rng.integers(-1, P, (H, W, 1)).astype(np.int32)     # -1 = no Gaussian
    di = rng.integers(-1, P, (H, W, 1)).astype(np.int32)
    hot = rng.uniform(size=(H, W, 1)) < 0.3                    # many pixels on few Gaussians: contended atomics
    ci[hot] = rng.integers(0, min(P, 17), int(hot.sum()))
    ci[0, 0, 0], di[0, 0, 0] = P, P + 5                        # out of range: skipped
    return ce, de, ne, ci, di


def accumulate_exact(k, check_max):
    """Maxima and integer counts are order-independent (bit-exact); fp32 atomic sums are not."""
    return check_max or k == 3


# ---------------------------------------------------------------- comparison
def rel_err(a, b):
    """max|a-b| / (max|b| + 1e-12): the per-tensor gradient metric of SURVEY.md section 8(c)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-12)) if a.size else 0.0


def compare_outputs(a, b, tie=None, tol=1e-4, max_bad_frac=2e-4, label=""):
    """Float maps: L_inf < tol on all pixels outside `tie` and on all but `max_bad_frac` of the pixels overall.
    Index maps: exact outside `tie`, same outlier allowance. Returns a dict of statistics; raises AssertionError."""
    H, W = a["color"].shape[-2:]
    ok = np.ones((H, W), bool) if tie is None else ~tie.astype(bool)
    idx_equal = (a["hit_color"][0] == b["hit_color"][0]) & (a["hit_depth"][0] == b["hit_depth"][0])
    stats = {}
    bad = ~idx_equal
    for k in ("color", "depth", "hit_color_weight", "hit_depth_weight", "T_map"):
        d = np.abs(a[k].astype(np.float64) - b[k].astype(np.float64)).max(axis=0)
        stats[k] = float(d[ok & idx_equal].max()) if (ok & idx_equal).any() else 0.0
        bad |= d >= tol
    stats["bad_pixels"] = int((bad & ok).sum())
    stats["tie_pixels"] = int((~ok).sum())
    stats["radii_mismatch"] = int((a["radii"] != b["radii"]).sum())
    frac = stats["bad_pixels"] / float(H * W)
    assert frac <= max_bad_frac, f"{label}: {stats['bad_pixels']} pixels differ beyond tol ({frac:.2e} of the image): {stats}"
    return stats


# ---------------------------------------------------------------- map statistics (SURVEY 8(f) #2)
MAPSTATS_SIZES = {"replica": (680, 1200), "ragged": (77, 45)}


def mapstats_inputs(name):
    """Seeded inputs of the tile-mask goldens (tests/golden/make_mapstats_golden.py regenerates them the same way): a
    transmittance-like map (1 where nothing was rendered) and a colour-error image."""
    H, W = MAPSTATS_SIZES[name]
    rng = np.random.default_rng(2024 + H)
    yy, xx = np.mgrid[0:H, 0:W]
    T = np.ones((H, W), np.float32)
    for _ in range(12):
        cy, cx, r = rng.uniform(0, H), rng.uniform(0, W), rng.uniform(5, 0.3 * min(H, W))
        T[(yy - cy) ** 2 + (xx - cx) ** 2 < r * r] = rng.uniform(0, 0.5)
    T[rng.uniform(size=(H, W)) < 0.02] = 0.3
    err = (rng.uniform(size=(H, W)) ** 3).astype(np.float32)
    err[rng.uniform(size=(H, W)) < 0.1] = 0
    return T, err


# ---------------------------------------------------------------- tracker-side frame preprocessing (SURVEY 8(f) #3)
FRAMEPREP_CASES = {
    # thresholds of configs/tum (invalid_confidence_thresh 0.5) and configs/replica (0.2); depth range of base.yaml
    "tum": dict(cam="small", depth_filter=True, min_depth=0.3, max_depth=5.0, thresh=0.5),
    "nofilter_ragged": dict(cam="ragged", depth_filter=False, min_depth=0.5, max_depth=4.0, thresh=0.2),
}


def frameprep_inputs(name):
    """A noisy ray-cast depth image of the box room with holes (zero depth), as a depth sensor delivers it."""
    from rtg_slam_b200 import scene
    cfg = FRAMEPREP_CASES[name]
    cam = scene.make_camera(cfg["cam"])
    rng = np.random.default_rng(77 + cam.width)
    depth = scene.raycast_room_depth(cam).astype(np.float32)
    depth = depth + rng.normal(0, 0.004, depth.shape).astype(np.float32)
    holes = rng.uniform(size=depth.shape) < 0.03
    depth[holes] = 0
    depth[: cam.height // 6, : cam.width // 5] = 0          # a larger missing region
    K = [[cam.fx, 0.0, cam.cx], [0.0, cam.fy, cam.cy], [0.0, 0.0, 1.0]]
    return np.ascontiguousarray(depth, dtype=np.float32), K


# ----------------------------------------------------------------------------- Mapping.history_merge (mapper.py:212-250)
HISTORY_MERGE_SIZES = {"window": 777, "one": 1}


def history_merge_inputs(name):
    """Seeded (history_stat, current state) pair as local_optimize leaves them: the optimisation moved every raw parameter a
    little; a few quaternions moved a lot (the spherical branch of slerp), a few flipped sign (dot < 0), three history
    quaternions are zero (NaN dot -> linear branch). Rows whose |dot| lies within 2e-5 of the 0.9995 branch threshold are
    regenerated away from it (the branch must not depend on the last bit of a norm)."""
    P = HISTORY_MERGE_SIZES[name]
    rng = np.random.default_rng(1000 + P)
    f = np.float32
    hist_conf = rng.integers(0, 40, size=(P, 1)).astype(f)
    conf = hist_conf + rng.integers(0, 51, size=(P, 1)).astype(f)
    if P > 3:
        conf[1], hist_conf[1] = 0, 0                       # a Gaussian that never received a gradient: weight 0 / 1e-6 = 0
    hist = {"confidence": hist_conf, "xyz": rng.normal(size=(P, 3)).astype(f), "features_dc": rng.normal(size=(P, 1, 3)).astype(f),
            "features_rest": (0.1 * rng.normal(size=(P, 15, 3))).astype(f), "scaling": (rng.normal(size=(P, 3)) - 3).astype(f)}
    q = rng.normal(size=(P, 4))
    q /= np.linalg.norm(q, axis=-1, keepdims=True)
    hist["rotation"] = q.astype(f)
    cur = {"confidence": conf}
    for k, sig in (("xyz", 0.01), ("features_dc", 0.05), ("features_rest", 0.02), ("scaling", 0.1)):
        cur[k] = (hist[k] + sig * rng.normal(size=hist[k].shape)).astype(f)
    noise = 0.01 * rng.normal(size=(P, 4))
    big = rng.uniform(size=P) < 0.2
    noise[big] = 0.6 * rng.normal(size=(int(big.sum()), 4))
    raw = (q + noise) * rng.uniform(0.5, 2.0, size=(P, 1))    # the raw rotation is not normalised
    flip = rng.uniform(size=P) < 0.1
    raw[flip] *= -1
    cur["rotation_raw"] = raw.astype(f)
    if P > 10:
        hist["rotation"][5:8] = 0
    rn = cur["rotation_raw"].astype(np.float64)
    rn /= np.linalg.norm(rn, axis=-1, keepdims=True)
    hn = hist["rotation"].astype(np.float64)
    with np.errstate(invalid="ignore"):
        dot = np.abs((hn / np.linalg.norm(hn, axis=-1, keepdims=True) * rn).sum(-1))
    near = np.abs(dot - 0.9995) < 2e-5
    cur["rotation_raw"][near] = (hist["rotation"][near] * 1.5).astype(f)   # collinear: far inside the linear branch
    return hist, cur


def slerp_tolerance(dot, base=4e-7):
    """Per-row bound on |slerp - reference slerp| for fp32 evaluations that differ in libm / summation order: `base` on the
    linear branch, base / sin(theta_0) on the spherical one (s0, s1 = sin(.) / sin(theta_0), SLAM/utils.py:646-648)."""
    with np.errstate(invalid="ignore"):
        d = np.nan_to_num(np.abs(dot.astype(np.float64)), nan=1.0)
        lin = d > 0.9995
        s = np.sqrt(np.maximum(1.0 - np.minimum(d, 1.0) ** 2, 1e-6))
    return np.where(lin, base, base / s + base)


# ----------------------------------------------------------------------------- SSIM term (utils/loss_utils.py:40-100)
SSIM_CASES = {"ragged": (3, 37, 53), "tile": (1, 16, 16), "strip": (2, 5, 40), "smooth": (3, 48, 80)}


def ssim_inputs(name):
    """Seeded (render, frame) pair, float32 (C,H,W) in [0,1]: noise whose upper half is a perturbed copy (high SSIM), or --
    'smooth' -- low-frequency images with a black block each (sigma^2 next to C2, the ill-conditioned regime)."""
    C, H, W = SSIM_CASES[name]
    rng = np.random.default_rng(7000 + H * W)
    if name == "smooth":
        yy, xx = np.meshgrid(np.linspace(0, 1, H), np.linspace(0, 1, W), indexing="ij")
        a = np.stack([0.5 + 0.4 * np.sin(6 * xx + c) * np.cos(4 * yy) for c in range(C)])
        b = np.clip(a + 0.01 * rng.normal(size=a.shape), 0, 1)
        a[:, : H // 4, : W // 3] = 0
        b[:, : H // 5, : W // 4] = 0
    else:
        a = rng.uniform(size=(C, H, W))
        b = rng.uniform(size=(C, H, W))
        b[:, : H // 2] = np.clip(a[:, : H // 2] + 0.02 * rng.normal(size=(C, H // 2, W)), 0, 1)
    return a.astype(np.float32), b.astype(np.float32)
