"""Seeded point clouds for the point-renderer tests (tests/test_points_*.py, tests/measure_point_render.py)."""
import math

import numpy as np

from oracle import points_ref as opr


def edge_cloud(S, n, radius, seed):
    """~n NDC points [P,3] float32 that exercise the rasteriser's corner cases at an S x S image: random points (some off-screen,
    some behind the camera, some non-finite), exact z ties, points on pixel centres, pixel edges and 16-pixel tile boundaries, and
    one pixel with 200 candidates (more than any K)."""
    rng = np.random.default_rng(seed)
    c = opr.pixel_ndc(S)
    m = n // 5
    rand = np.stack([rng.uniform(-1.1, 1.1, m), rng.uniform(-1.1, 1.1, m), rng.uniform(-0.3, 2.0, m)], 1)
    ties = np.stack([rng.uniform(-1, 1, m), rng.uniform(-1, 1, m), rng.choice([0.5, 1.0, 1.5], m)], 1)
    on_ctr = np.stack([c[rng.integers(0, S, m)], c[rng.integers(0, S, m)], rng.uniform(0, 2, m)], 1)
    edge = -1.0 + 2.0 * np.arange(S + 1) / S                            # pixel edges; every 16th is a tile edge
    tile = edge[::16]
    on_edge = np.stack([rng.choice(edge, m), rng.choice(tile, m), rng.choice([0.25, 0.75], m)], 1)
    crowd = np.stack([c[S // 2] + rng.uniform(-0.5, 0.5, 200) * radius, c[S // 3] + rng.uniform(-0.5, 0.5, 200) * radius,
                      rng.choice([1.0, 1.25, 2.0], 200)], 1)
    bad = np.array([[math.nan, 0, 1], [0, math.inf, 1], [0, 0, math.inf], [0, 0, -math.inf], [0, 0, -0.0], [0, 0, -1e-7]])
    pts = np.concatenate([rand, ties, on_ctr, on_edge, crowd, bad]).astype(np.float32)
    return pts[rng.permutation(len(pts))]


def refine_cloud(n=1_300_000, seed=0):
    """A stand-in for the refine stage's point cloud (load_views: ~1.3 M points, <= npoint = 1e6 from the canonical depth plus
    the novel views): a noisy ellipsoidal shell around the origin that fills most of a fov-20 view from distance 1.2, RGB in
    [0,1] and 16 N(0,1) learned features.
    Returns (xyz [n,3], feats [n,19]) float32."""
    rng = np.random.default_rng(seed)
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    r = 0.15 * (1 + 0.15 * rng.normal(size=(n, 1)))
    xyz = (d * r * np.array([1.0, 1.2, 0.8])).astype(np.float32)
    feats = np.concatenate([rng.random((n, 3)), rng.normal(size=(n, 16))], 1).astype(np.float32)
    return xyz, feats


def look_at_world2cam(radius=1.2, theta_deg=60.0, phi_deg=30.0):
    """world -> camera of an orbit camera looking at the origin, in the reference's fix_poses convention (up = -y, camera +z looks
    at the target): the inverse of [right | up | forward | centre]."""
    th, ph = math.radians(theta_deg), math.radians(phi_deg)
    centre = radius * np.array([math.sin(th) * math.sin(ph), math.cos(th), math.sin(th) * math.cos(ph)])
    fwd = -centre / np.linalg.norm(centre)
    right = np.cross(fwd, [0.0, -1.0, 0.0])
    right /= np.linalg.norm(right)
    up = np.cross(right, fwd)
    c2w = np.eye(4)
    c2w[:3, :3] = np.stack([right, up, fwd], 1)
    c2w[:3, 3] = centre
    return np.linalg.inv(c2w).astype(np.float32)


def intrinsics(S, fov_deg=20.0):
    """The refine stage's K at an S x S image: focal = 1 / (2 tan(fov / 2)) of the image side, principal point at the centre."""
    f = 1 / (2 * math.tan(math.radians(fov_deg) / 2))
    return np.array([[f * S, 0, 0.5 * S], [0, f * S, 0.5 * S], [0, 0, 1]], np.float32)


REFINE_RADIUS = 2.0 / 800 * 2.0      # 2 px at 800^2 in NDC, as the refine stage sets it
