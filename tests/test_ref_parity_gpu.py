"""GPU: our CUDA operators and the CPU oracle against the UNMODIFIED reference kernels (the original project's
raymarching/src/raymarching.cu compiled for sm_100a): tests/golden/ref_raymarching.npz holds what those kernels returned for the
inputs built here (recorded by tests/golden/make_golden_ref_raymarching.py; large outputs as a seeded sample).
This is what pins the oracle for rows R1-R4, R6 of SURVEY.md 8a: the reference itself."""
import importlib

import numpy as np
import pytest
import torch

from conftest import load_golden
from helpers import camera_rays, max_abs, orm, sphere_bitfield

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ref():
    return load_golden("ref_raymarching.npz")


@pytest.fixture(scope="module")
def rm():
    return importlib.import_module("make-it-3d_b200.raymarching")


def _cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def test_near_far_morton_packbits_vs_reference_kernels(ref, rm):
    ro, rd, _ = camera_rays(64)
    aabb = np.array([-1, -1, -1, 1, 1, 1], np.float32)
    sel = ref["nf_sel"]
    n, f = rm.near_far_from_aabb(_cu(ro), _cu(rd), _cu(aabb), 0.2)
    torch.cuda.synchronize()
    # the reference binary contracts a*b+c into FMA; ours is built with -fmad=false: allow 2 ulp
    assert max_abs(n.cpu().numpy()[sel], ref["nf_nears"]) < 1e-6 and max_abs(f.cpu().numpy()[sel], ref["nf_fars"]) < 1e-6
    n_o, f_o = orm.near_far_from_aabb(ro, rd, aabb, 0.2)
    assert max_abs(n_o[sel], ref["nf_nears"]) < 1e-6 and max_abs(f_o[sel], ref["nf_fars"]) < 1e-6
    rng = np.random.default_rng(0)
    coords = rng.integers(0, 128, size=(100000, 3), dtype=np.int32)
    idx_o = orm.morton3D(coords)
    np.testing.assert_array_equal(idx_o[ref["morton_sel"]], ref["morton_idx"])
    np.testing.assert_array_equal(rm.morton3D(_cu(coords)).cpu().numpy(), idx_o)
    grid = rng.random((1, 128 ** 3), dtype=np.float32)
    bits_o = orm.packbits(grid.reshape(-1), 0.4)
    np.testing.assert_array_equal(bits_o[ref["pack_sel"]], ref["pack_bits"])
    np.testing.assert_array_equal(rm.packbits(_cu(grid), 0.4).cpu().numpy(), bits_o)


def test_march_train_vs_reference_kernel(ref, rm):
    """Per-ray comparison (the reference's sample ORDER is atomic-arrival, ours is ray-id): counts and positions."""
    ro, rd, _ = camera_rays(96)
    bits = sphere_bitfield(0.25)
    aabb = np.array([-1, -1, -1, 1, 1, 1], np.float32)
    nears, fars = orm.near_far_from_aabb(ro, rd, aabb, 0.2)
    N = ro.shape[0]
    noises = np.random.default_rng(4).random(N, dtype=np.float32)
    x_o, _, dl_o, rays_o_, tot = orm.march_rays_train(ro, rd, 1.0, bits, 1, 128, nears, fars, noises, 0.0, 512, align=-1)
    cnt_r, count_r = ref["mt_counter"], ref["mt_counts"]
    assert cnt_r[1] == N
    same = int((count_r == rays_o_[:, 2]).sum())
    # FMA contraction in the reference binary can move a sample across a voxel face for a handful of rays
    assert same >= 0.999 * N, same
    assert abs(int(cnt_r[0]) - tot) <= 0.001 * tot
    # positions and step sizes of the stored rays (their samples lie back to back in the fixture, in ray order)
    off_r, worst = 0, 0.0
    for n in ref["mt_sel"]:
        c_r, off_o, c_o = int(count_r[n]), int(rays_o_[n, 1]), int(rays_o_[n, 2])
        if c_r == c_o:
            worst = max(worst, float(np.abs(ref["mt_xyzs"][off_r:off_r + c_r] - x_o[off_o:off_o + c_o]).max()))
            assert np.array_equal(ref["mt_dt"][off_r:off_r + c_r], dl_o[off_o:off_o + c_o, 0])
        off_r += c_r
    assert off_r == len(ref["mt_dt"])
    assert worst < 1e-5


def test_composite_vs_reference_kernel(ref, rm):
    ro, rd, _ = camera_rays(64)
    bits = sphere_bitfield(0.3)
    aabb = np.array([-1, -1, -1, 1, 1, 1], np.float32)
    nears, fars = orm.near_far_from_aabb(ro, rd, aabb, 0.2)
    N = ro.shape[0]
    rng = np.random.default_rng(8)
    x, d, dl, rays, tot = orm.march_rays_train(ro, rd, 1.0, bits, 1, 128, nears, fars, rng.random(N, dtype=np.float32), 0.0, 512, align=128)
    m = x.shape[0]
    sig = (rng.random(m, dtype=np.float32) * 20).astype(np.float32); rgb = rng.random((m, 3), dtype=np.float32)
    s_t, c_t = _cu(sig).requires_grad_(), _cu(rgb).requires_grad_()
    ws, dep, img = rm.composite_rays_train(s_t, c_t, _cu(dl), _cu(rays), 1e-4)
    torch.cuda.synchronize()
    sel = ref["cp_sel"]
    assert max_abs(ws.detach().cpu().numpy()[sel], ref["cp_ws"]) < 2e-6 and max_abs(img.detach().cpu().numpy()[sel], ref["cp_img"]) < 2e-6
    assert max_abs(dep.detach().cpu().numpy()[sel], ref["cp_dep"]) < 5e-6
    ws_o, dep_o, img_o = orm.composite_rays_train_forward(sig, rgb, dl, rays, 1e-4)
    assert max_abs(ws_o[sel], ref["cp_ws"]) < 5e-6 and max_abs(img_o[sel], ref["cp_img"]) < 5e-6       # pins the CPU oracle (expf vs __expf)
    gw, gi = rng.standard_normal(N).astype(np.float32), rng.standard_normal((N, 3)).astype(np.float32)
    ((ws * _cu(gw)).sum() + (img * _cu(gi)).sum()).backward()
    torch.cuda.synchronize()
    gsel = ref["cp_gsel"]
    assert max_abs(c_t.grad.cpu().numpy()[gsel], ref["cp_gr"]) < 2e-6
    assert max_abs(s_t.grad.cpu().numpy()[gsel], ref["cp_gs"]) < 1e-5 * max(1.0, float(ref["cp_gs_max"]))
