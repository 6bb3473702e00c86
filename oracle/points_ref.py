"""Float32 restatement of the refine stage's point renderer (test infrastructure only).

render_point (the reference's nerf/refine_utils.py:306-333) is a few lines of torch glue around pytorch3d's rasterize_points and
compositing.alpha_composite.  pytorch3d is third-party and not available, so its rasteriser is restated here with the two
deviations make-it-3d_b200/csrc/points.cu makes on purpose:
  - a point with a non-finite coordinate is skipped (like z < 0);
  - each pixel keeps its K candidates of smallest (z, point index), a total order (pytorch3d breaks z ties in binning order).
Two rasterisers, written independently, must agree bit for bit:
  raster_brute : per pixel over all points (numpy; small images only)
  raster_splat : per point over its pixel footprint, then one sort by (pixel, z, index) (torch; any device; 800^2 x 1.3 M points)
"""
import math

import numpy as np
import torch


def pixel_ndc(S):
    """NDC centre of pixel rows / columns 0..S-1 (index 0 -> +1): -1 + (2 (S-1-i) + 1) / S, in float64, rounded once to float32."""
    i = np.arange(S, dtype=np.float64)
    return (-1.0 + (2.0 * (S - 1 - i) + 1.0) / S).astype(np.float32)


def _r2(radius):
    r = np.float32(radius)
    return np.float32(r * r)


def raster_brute(pts, S, K, radius):
    """pts [P,3] float32 (NDC x, y, depth z) -> idx [S,S,K] int32 (-1 empty), dists [S,S,K] float32 (-1 empty)."""
    pts = np.asarray(pts, np.float32)
    x, y, z = pts[:, 0], pts[:, 1], pts[:, 2] + np.float32(0)
    ok = np.isfinite(pts).all(axis=1) & (z >= 0)
    ids = np.nonzero(ok)[0]
    x, y, z = x[ids], y[ids], z[ids]
    c = pixel_ndc(S)
    r2 = _r2(radius)
    idx = np.full((S, S, K), -1, np.int32)
    dists = np.full((S, S, K), -1, np.float32)
    for yi in range(S):
        dy = c[yi] - y
        dy2 = dy * dy
        for xi in range(S):
            dx = c[xi] - x
            d2 = dx * dx + dy2
            m = np.nonzero(d2 <= r2)[0]
            if m.size == 0:
                continue
            order = np.lexsort((ids[m], z[m]))[:K]
            idx[yi, xi, :order.size] = ids[m][order]
            dists[yi, xi, :order.size] = d2[m][order]
    return idx, dists


def raster_splat(pts, S, K, radius, chunk=1 << 18):
    """Same contract as raster_brute, for torch tensors on any device.  Returns (idx int32, dists float32) on pts' device."""
    pts = torch.as_tensor(pts, dtype=torch.float32)
    dev = pts.device
    c = torch.from_numpy(pixel_ndc(S)).to(dev)
    r2 = torch.tensor(float(_r2(radius)), dtype=torch.float32, device=dev)
    rpix = float(np.float32(radius)) * S / 2
    R = math.ceil(rpix) + 1                               # footprint half-width around the nearest pixel
    off = torch.arange(-R, R + 1, device=dev)
    pix_l, z_l, id_l, d_l = [], [], [], []
    for b in range(0, pts.shape[0], chunk):
        p = pts[b:b + chunk]
        ok = torch.isfinite(p).all(dim=1) & (p[:, 2] >= 0)
        ids = torch.nonzero(ok).squeeze(1)
        p = p[ids]
        # continuous pixel coordinate of the point: inverse of pixel_ndc
        u = (S - 1) - ((p[:, :2].double() + 1) * S - 1) / 2
        ctr = torch.round(u.clamp(-R - 1, S + R)).long()
        cx = (ctr[:, 0:1] + off[None, :])[:, None, :]      # [n, 1, 2R+1]
        cy = (ctr[:, 1:2] + off[None, :])[:, :, None]      # [n, 2R+1, 1]
        inside = (cx >= 0) & (cx < S) & (cy >= 0) & (cy < S)
        dx = c[cx.clamp(0, S - 1)] - p[:, 0, None, None]
        dy = c[cy.clamp(0, S - 1)] - p[:, 1, None, None]
        d2 = dx * dx + dy * dy
        hit = inside & (d2 <= r2)
        n, i, j = torch.nonzero(hit, as_tuple=True)
        pix_l.append(cy[n, i, 0] * S + cx[n, 0, j])
        z_l.append(p[n, 2] + 0.0)
        id_l.append(ids[n] + b)
        d_l.append(d2[n, i, j])
    pix, z, pid, d2 = (torch.cat(v) for v in (pix_l, z_l, id_l, d_l))
    # (pixel, z, index) order: stable sorts from the least significant key up
    o = torch.sort(pid, stable=True).indices
    o = o[torch.sort(z[o], stable=True).indices]
    o = o[torch.sort(pix[o], stable=True).indices]
    pix, pid, d2 = pix[o], pid[o], d2[o]
    rank = torch.arange(pix.numel(), device=dev) - torch.searchsorted(pix, pix)
    keep = rank < K
    idx = torch.full((S * S, K), -1, dtype=torch.int32, device=dev)
    dists = torch.full((S * S, K), -1.0, dtype=torch.float32, device=dev)
    idx[pix[keep], rank[keep]] = pid[keep].int()
    dists[pix[keep], rank[keep]] = d2[keep]
    return idx.view(S, S, K), dists.view(S, S, K)


def alphas_from_dists(dists, radius):
    """The reference's alpha: 1 - sqrt(clamp(0.1 d / r^2, 1e-3, 1)), in the dtype of dists."""
    r2 = float(_r2(radius))
    return 1 - (0.1 * dists / r2).clamp(min=1e-3, max=1).sqrt()


def alpha_composite(idx, alphas, feats):
    """pytorch3d compositing.alpha_composite: idx / alphas [N,K,H,W], feats [C,P] -> [N,C,H,W]; slots with idx < 0 are skipped.
    out = sum_k T_k a_k feats[:, idx_k], T_0 = 1, T_k+1 = T_k (1 - a_k)."""
    N, K, H, W = idx.shape
    out = feats.new_zeros(N, feats.shape[0], H, W)
    T = torch.ones_like(alphas[:, 0])
    for k in range(K):
        i, a = idx[:, k].long(), alphas[:, k]
        m = (i >= 0).to(feats.dtype)
        f = feats[:, i.clamp(min=0)].permute(1, 0, 2, 3)   # [N,C,H,W]
        out = out + (T * a * m)[:, None] * f
        T = T * (1 - a)
    return out


def composite(idx, dists, feats, radius):
    """idx / dists [S,S,K] (raster output), feats [P,C] -> image [1,C,S,S]; differentiable in feats (use float64 for gradients)."""
    idx = torch.as_tensor(idx).permute(2, 0, 1)[None]
    a = alphas_from_dists(torch.as_tensor(dists).to(feats.dtype).permute(2, 0, 1)[None], radius)
    return alpha_composite(idx.to(feats.device), a.to(feats.device), feats.t())


def project(points_xyz, H, W, K, world2cam):
    """The reference glue: camera = xyz R^T + t, then K, divide x and y by z, to [-1, 1], negate x and y; z stays the depth."""
    cam = torch.matmul(points_xyz, world2cam[:3, :3].T) + world2cam[:3, 3]
    q = torch.matmul(cam, K.T)
    x = q[:, 0] / q[:, 2]
    y = q[:, 1] / q[:, 2]
    x = (x / W * 2 - 1.0) * -1
    y = (y / H * 2 - 1.0) * -1
    return torch.stack([x, y, q[:, 2]], dim=1)


def render_point_ref(points_xyz, points_color, H, W, K, world2cam, image_size, radius, ppp):
    """render_point restated: [1, C, S, S]; background 0."""
    S = image_size if isinstance(image_size, int) else image_size[0]
    ndc = project(points_xyz, H, W, K, world2cam)
    idx, dists = raster_splat(ndc, S, ppp, radius)
    return composite(idx, dists, points_color, radius)
