"""Drop-in boundary B1 at the pybind level: `make-it-3d_b200/backend_mi3d.py::_backend` (the object a maintainer hands to
the REFERENCE's raymarching/raymarching.py:14-25 `get_backend()`) against the reference's own compiled module
(raymarching/src/{raymarching.cu,bindings.cpp} built for sm_100a), called with IDENTICAL positional arguments, caller-allocated
outputs and all -- exactly the calls raymarching/raymarching.py makes.  What the reference module returned for these calls is
stored in tests/golden/ref_raymarching.npz (tests/golden/make_golden_ref_raymarching.py; large outputs as a seeded sample).
The call sites are restated here; tests/test_abi.py::test_backend_mi3d_covers_reference_call_sites checks them against the
calls recorded from the reference's raymarching.py."""
import importlib

import numpy as np
import pytest
import torch

from conftest import load_golden
from helpers import camera_rays, march_rows, max_abs, orm, sphere_bitfield

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def backends():
    ours = importlib.import_module("make-it-3d_b200.backend_mi3d")._backend
    return load_golden("ref_raymarching.npz"), ours


def _cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def test_train_path_calls_match_reference_module(backends):
    """the call sequence of NeRFRenderer.run_cuda's training branch (renderer.py:493-510) through our backend, against what the
    reference module returned for it"""
    ref, ours = backends
    ro, rd, _ = camera_rays(64)
    N = ro.shape[0]
    aabb = _cu(np.array([-1, -1, -1, 1, 1, 1], np.float32))
    rays_o, rays_d = _cu(ro), _cu(rd)
    nears, fars = torch.empty(N, device="cuda"), torch.empty(N, device="cuda")
    ours.near_far_from_aabb(rays_o, rays_d, aabb, N, 0.2, nears, fars)                          # raymarching.py:56
    torch.cuda.synchronize()
    sel = ref["nf_sel"]
    assert max_abs(nears.cpu().numpy()[sel], ref["nf_nears"]) < 1e-6
    assert max_abs(fars.cpu().numpy()[sel], ref["nf_fars"]) < 1e-6
    bits_np, noises_np = sphere_bitfield(0.3), np.random.default_rng(1).random(N, dtype=np.float32)
    bits, noises = _cu(bits_np), _cu(noises_np)
    max_steps, M = 512, N * 512
    n_o, f_o = orm.near_far_from_aabb(ro, rd, aabb.cpu().numpy(), 0.2)        # the march inputs the reference module was given
    xyzs = torch.zeros(M, 3, device="cuda"); dirs = torch.zeros(M, 3, device="cuda"); deltas = torch.zeros(M, 2, device="cuda")
    rays = torch.empty(N, 3, dtype=torch.int32, device="cuda"); counter = torch.zeros(2, dtype=torch.int32, device="cuda")
    ours.march_rays_train(rays_o, rays_d, bits, 1.0, 0.0, max_steps, N, 1, 128, M, _cu(n_o), _cu(f_o), xyzs, dirs, deltas, rays, counter, noises)   # :229
    torch.cuda.synchronize()
    cr, co = ref["dt_counter"], counter.cpu().numpy()
    assert co[1] == cr[1] == N and abs(int(co[0]) - int(cr[0])) <= 0.001 * cr[0]
    # per-ray sample counts (the reference's offsets follow atomic arrival order; ours follow the ray id)
    ru = rays.cpu().numpy()
    assert np.array_equal(ru[:, 0], np.arange(N)) and (ref["dt_counts"] == ru[:, 2]).mean() >= 0.999
    # composite on the oracle's ordered march (the rows ours writes), the same tensors the reference module was given
    deltas_np, rays_np, m = march_rows(ro, rd, bits_np, n_o, f_o, noises_np, max_steps)
    deltas, rays = _cu(deltas_np), _cu(rays_np)
    rng = np.random.default_rng(2)
    sig, rgb = _cu((rng.random(M, dtype=np.float32) * 20)), _cu(rng.random((M, 3), dtype=np.float32))
    ws, dep, img = torch.empty(N, device="cuda"), torch.empty(N, device="cuda"), torch.empty(N, 3, device="cuda")
    ours.composite_rays_train_forward(sig, rgb, deltas, rays, M, N, 1e-4, ws, dep, img)                                     # :271
    torch.cuda.synchronize()
    sel = ref["dt_sel"]
    assert max_abs(ws.cpu().numpy()[sel], ref["dt_ws"]) < 2e-6 and max_abs(img.cpu().numpy()[sel], ref["dt_img"]) < 2e-6
    assert max_abs(dep.cpu().numpy()[sel], ref["dt_dep"]) < 5e-6
    gw, gi = _cu(rng.standard_normal(N).astype(np.float32)), _cu(rng.standard_normal((N, 3)).astype(np.float32))
    gs, gr = torch.zeros(M, device="cuda"), torch.zeros(M, 3, device="cuda")                                               # :295-296
    ours.composite_rays_train_backward(gw, gi, sig, rgb, deltas, rays, ws, img, M, N, 1e-4, gs, gr)                          # :297
    torch.cuda.synchronize()
    gsel = ref["dt_gsel"]
    assert max_abs(gr.cpu().numpy()[gsel], ref["dt_gr"]) < 2e-6
    assert max_abs(gs.cpu().numpy()[gsel], ref["dt_gs"]) < 1e-5 * max(1.0, float(ref["dt_gs_max"]))
    assert m > 0


def test_grid_and_inference_calls_match_reference_module(backends):
    """update_extra_state's morton3D / packbits (renderer.py:607,631) and the eval loop's march_rays / composite_rays (:546,549)"""
    ref, ours = backends
    rng = np.random.default_rng(3)
    coords_np = rng.integers(0, 128, size=(50000, 3), dtype=np.int32)
    grid_np = rng.random((1, 128 ** 3), dtype=np.float32)
    coords, grid = _cu(coords_np), _cu(grid_np)
    idx = torch.empty(50000, dtype=torch.int32, device="cuda")
    ours.morton3D(coords, 50000, idx)                                                         # raymarching.py:110
    back = torch.empty(50000, 3, dtype=torch.int32, device="cuda")
    ours.morton3D_invert(idx, 50000, back)                                                    # :132
    bits_o = torch.empty(128 ** 3 // 8, dtype=torch.uint8, device="cuda")
    ours.packbits(grid, 128 ** 3 // 8, 0.4, bits_o)                                          # raymarching.py:157,162 (N = bytes)
    torch.cuda.synchronize()
    # the reference's outputs at the stored indices, and the oracle (which the stored indices pin) everywhere
    assert np.array_equal(idx.cpu().numpy()[ref["gi_morton_sel"]], ref["gi_morton_idx"]) and torch.equal(back, coords)
    assert np.array_equal(idx.cpu().numpy(), orm.morton3D(coords_np)) and np.array_equal(orm.morton3D(coords_np)[ref["gi_morton_sel"]], ref["gi_morton_idx"])
    assert np.array_equal(bits_o.cpu().numpy()[ref["gi_pack_sel"]], ref["gi_pack_bits"])
    assert np.array_equal(bits_o.cpu().numpy(), orm.packbits(grid_np.reshape(-1), 0.4))
    # inference march + composite, one iteration of the alive-ray loop
    ro, rd, _ = camera_rays(48)
    N = ro.shape[0]
    rays_o, rays_d = _cu(ro), _cu(rd)
    aabb = np.array([-1, -1, -1, 1, 1, 1], np.float32)
    n_o, f_o = orm.near_far_from_aabb(ro, rd, aabb, 0.2)
    nears, fars = _cu(n_o), _cu(f_o)
    bits = _cu(sphere_bitfield(0.3))
    n_alive, n_step = N, 4
    noises = torch.zeros(n_alive, device="cuda")
    rays_alive = torch.arange(n_alive, dtype=torch.int32, device="cuda")
    rays_t = nears.clone()
    xyzs = torch.zeros(n_alive * n_step, 3, device="cuda"); dirs = torch.zeros(n_alive * n_step, 3, device="cuda")
    deltas = torch.zeros(n_alive * n_step, 2, device="cuda")
    ours.march_rays(n_alive, n_step, rays_alive, rays_t, rays_o, rays_d, 1.0, 0.0, 512, 1, 128, bits, nears, fars, xyzs, dirs, deltas, noises)   # :406
    g = torch.Generator(device="cuda").manual_seed(0)
    sig = torch.rand(n_alive * n_step, device="cuda", generator=g) * 30
    rgb = torch.rand(n_alive * n_step, 3, device="cuda", generator=g); nrm = torch.rand(n_alive * n_step, 3, device="cuda", generator=g)
    ws, dep = torch.zeros(N, device="cuda"), torch.zeros(N, device="cuda")
    img, nimg = torch.zeros(N, 3, device="cuda"), torch.zeros(N, 3, device="cuda")
    ours.composite_rays(n_alive, n_step, 1e-2, rays_alive, rays_t, sig, rgb, nrm, deltas, ws, dep, img, nimg)               # :442
    torch.cuda.synchronize()
    res = dict(xyzs=xyzs, ws=ws, dep=dep, img=img, nimg=nimg)
    res = {k: v.cpu().numpy() for k, v in res.items()}
    deltas = deltas.cpu().numpy()
    sel = ref["gi_sel"]                                                # the rays whose positions and composites are stored
    same = (deltas == ref["gi_deltas"]).all(axis=1).mean()
    assert same > 0.999 and max_abs(res["xyzs"].reshape(n_alive, n_step, 3)[sel], ref["gi_xyzs"]) < 1e-2
    agree = (rays_alive.cpu().numpy() == ref["gi_alive"]).mean()
    assert agree > 0.999
    ok = (deltas.reshape(n_alive, n_step, 2) == ref["gi_deltas"].reshape(n_alive, n_step, 2)).all(axis=2).all(axis=1)[sel]
    for k in ("ws", "dep", "img", "nimg"):
        assert max_abs(res[k][sel][ok], ref["gi_" + k][ok]) < 1e-5, k


def test_unbuilt_entry_points_raise(backends):
    _, ours = backends
    L = importlib.import_module("make-it-3d_b200._lib")
    with pytest.raises(L.Mi3dError):
        ours.sph_from_ray(None, None, 1.0, 0, None)
