"""Shared helpers for the parity tests (test infrastructure; may import oracle/)."""
import math
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import field_ref as fr      # noqa: E402
from oracle import raymarch as orm      # noqa: E402


def sphere_bitfield(radius, H=128, C=1):
    idx = np.arange(H ** 3, dtype=np.int32)
    coords = orm.morton3D_invert(idx)
    xyz = (coords.astype(np.float32) + 0.5) / H * 2 - 1
    grid = (np.linalg.norm(xyz, axis=1) < radius).astype(np.float32)
    return orm.packbits(np.tile(grid, C), 0.5)


def make_table(n_params, seed, scale):
    return ((np.random.default_rng(seed).random(n_params, dtype=np.float32) * 2 - 1) * scale).astype(np.float32)


def camera_rays(HW, radius=1.25, theta=80.0, phi=170.0, fov=20.0):
    pose = fr.orbit_pose(radius, theta, phi)
    focal = HW / (2 * math.tan(math.radians(fov) / 2))
    ro, rd, sc = fr.get_rays_ref(pose, (focal, focal, HW / 2, HW / 2), HW, HW)
    return ro.numpy(), rd.numpy(), sc.numpy()


def march_rows(ro, rd, bits, nears, fars, noises, max_steps=512):
    """The oracle's training march (ray-id order, bit-identical to ours) in N * max_steps caller-allocated rows, the way the
    reference wrapper allocates them: (deltas [N * max_steps, 2], rays [N, 3], number of samples)."""
    _, _, dl, rays, m = orm.march_rays_train(ro, rd, 1.0, bits, 1, 128, nears, fars, noises, 0.0, max_steps, align=-1)
    deltas = np.zeros((ro.shape[0] * max_steps, 2), np.float32)
    deltas[:m] = dl[:m]
    return deltas, rays, m


def field_from_golden(g):
    """oracle FieldRef holding the fixture's parameters."""
    f = fr.FieldRef(bound=1.0, blob_density=5.0, blob_radius=0.1, seed=0)
    table = make_table(f.encoder.params.numel(), int(g["table_seed"]), float(g["table_scale"]))
    with torch.no_grad():
        f.encoder.params.copy_(torch.from_numpy(table))
        for l, (w, b) in enumerate((("w1", "b1"), ("w2", "b2"), ("w3", "b3"))):
            f.sigma_net.net[l].weight.copy_(torch.from_numpy(g[w]))
            f.sigma_net.net[l].bias.copy_(torch.from_numpy(g[b]))
    return f, table


def rel_err(a, b, floor=1e-6):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b) / (np.abs(b) + floor)))


def max_abs(a, b):
    return float(np.max(np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)))) if np.size(a) else 0.0
