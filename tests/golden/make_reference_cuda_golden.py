"""Generates the fixtures that hold the GPU tests to the reference's own CUDA extensions, built unmodified into oracle/_ref/
by oracle/build_ref.py (rasterizer `_C_depth`, `cuda_utils`, `simple-knn`). Needs a GPU and those builds:

    python tests/golden/make_reference_cuda_golden.py OUTDIR     # then copy OUTDIR/*.npz into tests/golden/

Full outputs at the tested sizes are tens of MB, so each file keeps a seeded sample of the outputs plus the whole-array
figures the assertions use (tests/helpers.py draws the same samples):

* live_raster_reference.npz -- test_raster_gpu.py::test_matches_live_reference_cuda: per LIVE_CASES entry the pixel maps
  at LIVE_PIXELS pixels, the gradients of the 8 largest rows of each tensor and of LIVE_ROWS visible Gaussians, each
  gradient tensor's max |g| and reference-vs-reference jitter, the digest of the radii.
* optimize_loop_reference.npz -- test_raster_gpu.py::test_optimize_loop_tracks_reference_rasterizer_with_torch_adam: the loss
  trajectory of the reference rasterizer + eager torch loss + torch.optim.Adam, the parameters after the loop at
  OPT_LOOP_SAMPLE elements, their max |p|, max |p - p0| and the fraction the loop moves by more than 1e-5 of max |p| between
  two runs of its own.
* knn_dist_cuda2.npz -- test_mapsurgery_gpu.py::test_dist_cuda2_large_against_kdtree_and_reference: distCUDA2's mean
  squared distance and sorted neighbour indices at KNN_ROWS points.
* mapstats_accumulate.npz -- test_mapstats_gpu.py::test_accumulate_gaussian_error: digests of the order-independent
  outputs, the fp32 atomic sums at ACCUMULATE_ROWS Gaussians.
"""
import glob
import importlib.util
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import helpers  # noqa: E402


def _load(pattern, name):
    so = glob.glob(os.path.join(ROOT, "oracle", "_ref", pattern))
    assert so, f"oracle/_ref/{pattern} is not built (oracle/build_ref.py)"
    spec = importlib.util.spec_from_file_location(name, so[0])
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def raster_live(dev):
    out = {}
    for camname, P, keep in helpers.LIVE_CASES:
        cam, g, mask, grads, c = helpers.live_case(camname, P, keep)
        r = helpers.run_ref_cuda(cam, g, dev, tile_mask=mask, grads=grads)
        r2 = helpers.run_ref_cuda(cam, g, dev, tile_mask=mask, grads=grads)  # atomics jitter of the reference itself
        for k, v in helpers.pixel_sample(r, helpers.live_pixels(cam)).items():
            out[f"{c}_{k}"] = v[:, 0]
        top = [np.argsort(np.abs(r["grads"][k].reshape(P, -1)).max(1))[-8:] for k in helpers.GRADS]
        vis = np.flatnonzero(r["radii"] > 0)
        rows = np.unique(np.concatenate(top + [vis[helpers.sample_indices(len(vis), helpers.LIVE_ROWS, seed=P)]])).astype(np.int64)
        out[f"{c}_rows"] = rows
        out[f"{c}_radii"] = r["radii"][rows]
        out[f"{c}_radii_digest"] = np.array(helpers.digest(r["radii"].astype(np.int32)))
        for k in helpers.GRADS:
            out[f"{c}_grad_{k}"] = r["grads"][k][rows]
            out[f"{c}_gradmax_{k}"] = np.float64(np.abs(r["grads"][k]).max())
            out[f"{c}_jitter_{k}"] = np.float64(helpers.rel_err(r2["grads"][k], r["grads"][k]))
        print(c, "visible", len(vis), "R", r["num_rendered"], "jitter", {k: f"{float(out[f'{c}_jitter_{k}']):.1e}" for k in helpers.GRADS})
    return out


def optimize_loop(dev, mod):
    """The mapper's loop on the reference's own rasterizer, driven by its python shim and eager torch expressions."""
    cam, rs, t, gt_color, gt_depth = helpers.optimize_loop_case(dev)
    H, W = cam.height, cam.width
    st = helpers.DEFAULT_SETTINGS
    names = tuple(helpers.OPT_LOOP_LRS)

    class RefRaster(torch.autograd.Function):  # the reference's python shim, reduced to what the loop needs
        @staticmethod
        def forward(ctx, xyz, shs, opacity, scales, rotations):
            e = torch.Tensor([])
            th, tw = cam.tile_grid
            tm = torch.ones((th, tw), dtype=torch.int32, device=dev)
            out = mod.rasterize_gaussians(rs.bg, xyz, e, opacity, scales, rotations, st["scale_modifier"], e, rs.viewmatrix, rs.projmatrix, tm,
                                          cam.tanfovx, cam.tanfovy, H, W, cam.cx, cam.cy, shs, st["sh_degree"], st["color_sigma"], rs.campos,
                                          st["opaque_threshold"], st["depth_threshold"], st["normal_threshold"], st["T_threshold"], False, False)
            ctx.state = out
            ctx.save_for_backward(xyz, shs, scales, rotations)
            return out[2], out[3], out[5]

        @staticmethod
        def backward(ctx, gc, gd, _):
            (num_rendered, num_tile, color, depth, hit_color, hit_depth, hcw, hdw, T_map, radii, geomB, binB, imgB, tile_indices) = ctx.state
            xyz, shs, scales, rotations = ctx.saved_tensors
            e = torch.Tensor([])
            (g2d, gcol, gop, gm3, gcov, gsh, gsc, grot) = mod.rasterize_gaussians_backward(
                tile_indices, num_tile, rs.bg, xyz, radii, e, scales, rotations, st["scale_modifier"], e, rs.viewmatrix, rs.projmatrix,
                cam.tanfovx, cam.tanfovy, cam.cx, cam.cy, st["depth_threshold"], st["normal_threshold"], gc.contiguous(), gd.contiguous(), shs,
                st["sh_degree"], rs.campos, geomB, num_rendered, binB, imgB, hit_depth, False)
            return gm3, gsh, gop, gsc, grot

    def run():
        p = {k: t[k].clone().requires_grad_(True) for k in names}
        opt = torch.optim.Adam([{"params": [p[k]], "lr": helpers.OPT_LOOP_LRS[k]} for k in names], lr=0.0, eps=1e-15)
        losses = []
        for _ in range(helpers.OPT_LOOP_ITERS):
            opt.zero_grad(set_to_none=True)
            color, depth, hit_depth = RefRaster.apply(p["xyz"], p["shs"], p["opacity"], p["scales"], p["rotations"])
            image, d, di = color.permute(1, 2, 0), depth.permute(1, 2, 0), hit_depth.permute(1, 2, 0)
            color_loss = torch.abs(image - gt_color).mean()
            err = d - gt_depth[..., None]
            valid = (di != -1).squeeze() & (gt_depth > 0) & (err < 0.1).squeeze()
            loss = 1.0 * torch.abs(err[valid]).mean() + 0.8 * color_loss
            loss.backward()
            opt.step()
            losses.append(float(loss.detach()))
        return losses, {k: v.detach().clone() for k, v in p.items()}

    lb, pb = run()
    _, pc = run()  # a second run: the reference's own run-to-run spread (atomic order) is the yardstick
    out = {"losses": np.array(lb, np.float64)}
    for k in names:
        scale = float(pb[k].abs().max())
        out[f"{k}_scale"] = np.float64(scale)
        out[f"{k}_moved"] = np.float64((pb[k] - t[k]).abs().max())
        out[f"{k}_off_self"] = np.float64(((pc[k] - pb[k]).abs() > 1e-5 * scale).float().mean())
        out[f"{k}_sample"] = pb[k].reshape(-1).cpu().numpy()[helpers.optimize_loop_sample(k, t)]
    print("optimize loop losses", lb, {k: float(out[f"{k}_off_self"]) for k in names})
    return out


def dist_cuda2(dev, mod):
    from test_mapsurgery_gpu import _surface_points
    n = 300_000
    pts = _surface_points(n, seed=11)
    rmean, ridx = mod.distCUDA2(torch.from_numpy(pts).to(dev))
    rows = helpers.sample_indices(n, helpers.KNN_ROWS, seed=n)
    return {"mean": rmean.cpu().numpy()[rows], "idx_sorted": np.sort(ridx.cpu().numpy(), 1)[rows]}


def accumulate(dev, mod):
    out = {}
    for H, W, P in helpers.ACCUMULATE_CASES:
        t = [torch.from_numpy(a).to(dev) for a in helpers.accumulate_inputs(H, W, P, seed=H + P)]
        rows = helpers.sample_indices(P, helpers.ACCUMULATE_ROWS, seed=P)
        for check_max in (True, False):
            refs = [r.cpu().numpy() for r in mod.accumulate_gaussian_error(H, W, P, *t, *helpers.ACCUMULATE_THRESHOLDS, check_max)]
            for k, r in enumerate(refs):
                key = f"{H}x{W}x{P}_{int(check_max)}_{k}"
                if helpers.accumulate_exact(k, check_max):
                    out[key + "_digest"] = np.array(helpers.digest(r))
                else:
                    out[key] = r[rows]
    return out


def main():
    dest = sys.argv[1] if len(sys.argv) > 1 else os.path.dirname(os.path.abspath(__file__))
    os.makedirs(dest, exist_ok=True)
    dev = torch.device("cuda", 0)
    rast = helpers.ref_cuda_module()
    assert rast is not None, "oracle/_ref/_C_depth*.so is not built (oracle/build_ref.py)"
    files = {"live_raster_reference": lambda: raster_live(dev),
             "optimize_loop_reference": lambda: optimize_loop(dev, rast),
             "knn_dist_cuda2": lambda: dist_cuda2(dev, _load("simple_knn/_C_simple_knn*.so", "_C_simple_knn")),
             "mapstats_accumulate": lambda: accumulate(dev, _load("cuda_utils/_C*.so", "_C"))}
    for name, make in files.items():
        path = os.path.join(dest, name + ".npz")
        np.savez_compressed(path, **make())
        print(name, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
