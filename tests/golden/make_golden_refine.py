"""tests/golden/make_golden_refine.py -- records render_point.npz by running the REFERENCE's own render_point.

Run in the build container only (needs the reference checkout):  python tests/golden/make_golden_refine.py [--ref DIR]

What is real reference code here (imported unmodified): nerf/refine_utils.py  render_point (projection, NDC flips, alpha from
the squared distance, channel layout, the ignored bg_feat) and fix_poses (the refine stage's camera poses).
What is substituted, because it cannot run here: pytorch3d (third-party CUDA package, not pinned) -> Pointclouds /
rasterize_points / compositing.alpha_composite from oracle/points_ref.py; imageio, tqdm -> MagicMock.  So the fixture pins the
reference's glue around pytorch3d, not pytorch3d itself.

The cloud is thinned of points that sit within a relative 1e-4 of the radius of some pixel centre, or within 1e-5 in depth of
another candidate of the same pixel, at every recorded size: the reference projects with a float32 matmul whose rounding differs
between CPU and GPU, and such points could change their pixel or their place in a pixel's list on a last-bit difference.
"""
import argparse
import math
import os
import random
import sys
import types
from unittest.mock import MagicMock

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

from oracle import points_ref as opr      # noqa: E402
import points_cases as pc                 # noqa: E402

SIZES = (64, 200)
RADIUS = 0.03           # NDC: ~1 px at 64^2, 3 px at 200^2
PPP = 8
N_POINTS = 4000
N_SAMPLE = 4096         # 200^2 outputs are kept at this many seeded pixel positions (fixture size)
SEED = 5


def install_stubs():
    for name in ("imageio", "tqdm"):
        sys.modules[name] = MagicMock()
    p3 = types.ModuleType("pytorch3d")
    structures = types.ModuleType("pytorch3d.structures")
    renderer = types.ModuleType("pytorch3d.renderer")
    compositing = types.ModuleType("pytorch3d.renderer.compositing")
    points = types.ModuleType("pytorch3d.renderer.points")

    class Pointclouds:
        def __init__(self, points, features):
            self._p, self._f = points, features

        def points_packed(self):
            return self._p[0]

        def features_packed(self):
            return self._f[0]

    def rasterize_points(pc3, image_size, radius, points_per_pixel):
        S = image_size[0]
        assert image_size[1] == S
        ndc = pc3.points_packed().detach()
        idx, d = opr.raster_splat(ndc, S, points_per_pixel, radius)
        z = torch.where(idx >= 0, ndc[:, 2][idx.long().clamp(min=0)], torch.full_like(d, -1.0))
        return idx.long()[None], z[None], d[None]

    structures.Pointclouds = Pointclouds
    compositing.alpha_composite = opr.alpha_composite
    renderer.compositing = compositing
    renderer.AlphaCompositor = MagicMock()
    points.rasterize_points = rasterize_points
    renderer.points = points
    p3.structures, p3.renderer = structures, renderer
    sys.modules.update({"pytorch3d": p3, "pytorch3d.structures": structures, "pytorch3d.renderer": renderer,
                        "pytorch3d.renderer.compositing": compositing, "pytorch3d.renderer.points": points})


def robust(xyz, world2cam, Ks):
    """mask of points whose candidacy and depth order do not hinge on the last bit of the projection (float64 analysis)"""
    keep = np.ones(len(xyz), bool)
    for S, K in zip(SIZES, Ks):
        cam = xyz.astype(np.float64) @ world2cam[:3, :3].T.astype(np.float64) + world2cam[:3, 3]
        q = cam @ K.T.astype(np.float64)
        ndc = np.stack([1 - q[:, 0] / q[:, 2] / S * 2, 1 - q[:, 1] / q[:, 2] / S * 2], 1)
        c = opr.pixel_ndc(S).astype(np.float64)
        u = (S - 1) - ((ndc + 1) * S - 1) / 2
        R = math.ceil(RADIUS * S / 2) + 1
        r2 = RADIUS ** 2
        pix, pid, zz = [], [], []
        for oy in range(-R, R + 1):
            for ox in range(-R, R + 1):
                xi, yi = np.round(u[:, 0]).astype(np.int64) + ox, np.round(u[:, 1]).astype(np.int64) + oy
                ok = (xi >= 0) & (xi < S) & (yi >= 0) & (yi < S)
                d2 = (c[np.clip(xi, 0, S - 1)] - ndc[:, 0]) ** 2 + (c[np.clip(yi, 0, S - 1)] - ndc[:, 1]) ** 2
                keep &= ~(ok & (np.abs(d2 - r2) < 1e-4 * r2))
                hit = ok & (d2 <= r2)
                pix.append((yi * S + xi)[hit]), pid.append(np.nonzero(hit)[0]), zz.append(q[hit, 2])
        pix, pid, zz = map(np.concatenate, (pix, pid, zz))
        o = np.lexsort((zz, pix))
        pix, pid, zz = pix[o], pid[o], zz[o]
        close = (pix[1:] == pix[:-1]) & (np.abs(zz[1:] - zz[:-1]) < 1e-5)
        keep[pid[1:][close]] = False
        keep[pid[:-1][close]] = False
    return keep


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref", default=os.environ.get("MI3D_REFERENCE", "/root/reference"))
    args = ap.parse_args()
    install_stubs()
    sys.path.insert(0, args.ref)
    from nerf import refine_utils as ru

    torch.manual_seed(SEED)
    random.seed(SEED)
    c2w, _, _ = ru.fix_poses(1, "cpu", radius_range=[1.0, 1.5], theta_range=[45, 105], phi_range=[-180, 180])
    world2cam = torch.linalg.inv(c2w[0]).float()
    xyz, feats = pc.refine_cloud(N_POINTS, seed=SEED)
    Ks = [pc.intrinsics(S) for S in SIZES]
    keep = robust(xyz, world2cam.numpy(), Ks)
    xyz, feats = xyz[keep], feats[keep]
    out = {"xyz": xyz, "feats": feats, "world2cam": world2cam.numpy(), "radius": np.float64(RADIUS), "ppp": np.int64(PPP),
           "sizes": np.array(SIZES, np.int64)}
    with torch.no_grad():
        for S, K in zip(SIZES, Ks):
            img = ru.render_point(torch.from_numpy(xyz), torch.from_numpy(feats), S, S, torch.from_numpy(K), world2cam, (S, S),
                                  RADIUS, PPP, bg_feat=torch.ones(1, 19, 1, 1))
            out[f"K_{S}"], out[f"out_{S}"] = K, img.numpy()
        S = SIZES[-1]
        ones = torch.ones(len(xyz), 3)
        mask = ru.render_point(torch.from_numpy(xyz), ones, S, S, torch.from_numpy(Ks[-1]), world2cam, (S, S), RADIUS, PPP).numpy()
    pix = np.sort(np.random.default_rng(SEED).choice(S * S, N_SAMPLE, replace=False))
    out["sample_pix"] = pix
    out[f"out_{S}"] = out[f"out_{S}"].reshape(-1, S * S)[:, pix]
    out["mask_out"] = mask.reshape(-1, S * S)[:, pix]
    path = os.path.join(HERE, "render_point.npz")
    np.savez_compressed(path, **out)
    print(f"{path}: {len(xyz)} of {N_POINTS} points kept, {os.path.getsize(path) / 1e3:.0f} kB, "
          f"covered pixels at {S}^2: {(mask[0, 0] > 0).mean():.2f}")


if __name__ == "__main__":
    main()
