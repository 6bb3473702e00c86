"""Refine-stage point renderer: drop-in ``render_point`` of the reference's nerf/refine_utils.py (:306-333), on libmi3d.so.

The reference rasterises with pytorch3d's ``rasterize_points`` and composites with ``compositing.alpha_composite``; here both are
the kernels of csrc/points.cu (``mi3d_point_render_forward`` / ``_backward``).  Semantics are pytorch3d's for square images, except
that points with a non-finite coordinate are skipped and each pixel keeps its K nearest-in-depth points ordered by
(z, point index), so that z ties resolve the same way on every run.  Gradients reach the point features only; the point positions
are constant in the refine loop and a position that requires grad is refused rather than given a wrong (zero) gradient.
"""
import ctypes as C

import torch
from torch.autograd import Function

from .. import _lib as L

_WS = {}


def _workspace(device, P, S, K, radius):
    """scratch of the tile binning, cached per (device, P, S, K, radius): the refine loop renders the same three shapes every step"""
    key = (str(device), P, S, K, radius)
    ws = _WS.get(key)
    if ws is None:
        n = L.lib().mi3d_point_render_workspace_bytes(C.c_uint32(P), C.c_uint32(S), C.c_uint32(K), C.c_float(radius))
        if n == 0:
            raise L.Mi3dError("point_render: invalid argument (MI3D_ERR_ARG)")
        if len(_WS) >= 8:
            _WS.clear()
        ws = _WS[key] = torch.empty(n, dtype=torch.uint8, device=device)
    return ws


class _PointRender(Function):
    @staticmethod
    def forward(ctx, points_ndc, features, S, radius, K):
        P, Cf = features.shape
        dev = features.device
        idx = torch.empty(S, S, K, dtype=torch.int32, device=dev)
        dists = torch.empty(S, S, K, dtype=torch.float32, device=dev)
        out = torch.empty(1, Cf, S, S, dtype=torch.float32, device=dev)
        ws = _workspace(dev, P, S, K, radius)
        L.check(L.lib().mi3d_point_render_forward(L.ptr(points_ndc), L.ptr(features), C.c_uint32(P), C.c_uint32(Cf), C.c_uint32(S),
                                                  C.c_uint32(K), C.c_float(radius), L.ptr(idx), L.ptr(dists), L.ptr(out), L.ptr(ws),
                                                  C.c_size_t(ws.numel()), L.stream()), "point_render_forward")
        ctx.save_for_backward(points_ndc, idx, dists)
        ctx.shape = (P, Cf, S, K, radius)
        ctx.mark_non_differentiable(idx, dists)
        return out, idx, dists

    @staticmethod
    def backward(ctx, g_out, _g_idx, _g_dists):
        points_ndc, idx, dists = ctx.saved_tensors
        P, Cf, S, K, radius = ctx.shape
        g_out = L.f32c(g_out)
        g_feats = torch.empty(P, Cf, dtype=torch.float32, device=g_out.device)
        L.check(L.lib().mi3d_point_render_backward(L.ptr(g_out), L.ptr(points_ndc), L.ptr(idx), L.ptr(dists), C.c_uint32(P), C.c_uint32(Cf),
                                                   C.c_uint32(S), C.c_uint32(K), C.c_float(radius), L.ptr(g_feats), L.stream()),
                "point_render_backward")
        return None, g_feats, None, None, None


def point_render(points_ndc, features, image_size, radius, points_per_pixel):
    """Rasterise + alpha-composite P points into a square image.

    points_ndc [P,3]: NDC x, y (+1 = column / row 0) and camera depth z.  features [P,C].  image_size: int S or (S, S).
    radius: NDC radius (float).  points_per_pixel: K in 1..16.
    Returns (image [1,C,S,S], idx [S,S,K] int32 (-1 empty), dists [S,S,K] float32 squared NDC distances (-1 empty)).
    Differentiable in features only."""
    if isinstance(image_size, int):
        S = image_size
    else:
        h, w = image_size
        if h != w:
            raise L.Mi3dError(f"point_render: square images only, got {h}x{w}: invalid argument (MI3D_ERR_ARG)")
        S = h
    L.require_cuda(points_ndc, features)
    if points_ndc.requires_grad:
        raise L.Mi3dError("point_render: point positions carry no gradient (only the features do); detach them")
    if points_ndc.dim() != 2 or points_ndc.shape[1] != 3 or features.dim() != 2 or features.shape[0] != points_ndc.shape[0]:
        raise L.Mi3dError(f"point_render: expected points [P,3] and features [P,C], got {tuple(points_ndc.shape)} and "
                          f"{tuple(features.shape)}")
    return _PointRender.apply(L.f32c(points_ndc), L.f32c(features), int(S), float(radius), int(points_per_pixel))


def render_point(points_xyz_org, points_color, H, W, K, world2cam, image_size, radius, ppp, bg_feat=None, acc='alphacomposite'):
    """Drop-in for the reference's render_point: project the world-space points with world2cam and the intrinsics K, rasterise with
    NDC radius `radius` and `ppp` points per pixel, alpha-composite points_color.  Returns [1, C, h, w].  Like the reference,
    bg_feat and acc are accepted and unused: the background is 0."""
    L.require_cuda(points_xyz_org, points_color)
    if points_xyz_org.requires_grad:
        raise L.Mi3dError("render_point: gradients with respect to point positions are not supported; pass the positions detached")
    cam = torch.matmul(points_xyz_org, world2cam[:3, :3].T) + world2cam[:3, 3]
    q = torch.matmul(cam, K.T)
    z = q[:, 2]
    # pixel -> [-1, 1], then flipped: 1 - u / W * 2 rounds exactly like -(u / W * 2 - 1)
    ndc = torch.stack([1.0 - q[:, 0] / z / W * 2, 1.0 - q[:, 1] / z / H * 2, z], dim=1)
    image, _, _ = point_render(ndc, points_color, image_size, radius, ppp)
    return image
