"""GPU: the refine-stage point renderer (csrc/points.cu, nerf/refine_utils.py) against the float32 oracle (oracle/points_ref.py).
idx / dists are bit-identical (both evaluate the same single-rounding float32 expressions and the same (z, index) order); the image
is within 1e-6; the feature gradient is within 1e-5 of its largest entry of the float64 autograd oracle and bit-identical run to
run (gather, no atomics)."""
import importlib

import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import points_ref as opr
import points_cases as pc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ru(mi3d):
    return importlib.import_module("make-it-3d_b200.nerf.refine_utils")


def bits(t):
    return t.contiguous().view(torch.int32).cpu()


def check_forward(ru, pts, feats, S, K, r):
    out, idx, dists = ru.point_render(pts, feats, S, r, K)
    i_ref, d_ref = opr.raster_splat(pts, S, K, r)
    assert torch.equal(idx.cpu(), i_ref.cpu())
    assert torch.equal(bits(dists), bits(d_ref))
    o_ref = opr.composite(i_ref, d_ref, feats, r)
    assert (out - o_ref).abs().max().item() <= 1e-6
    return out, idx, dists


def test_edge_cases_64_match_brute_force_oracle(ru):
    S, r = 64, 0.05
    pts = pc.edge_cloud(S, 4000, r, seed=1)
    feats = torch.from_numpy(np.random.default_rng(1).normal(size=(len(pts), 19)).astype(np.float32)).cuda()
    for K in (1, 8, 16):
        out, idx, dists = ru.point_render(torch.from_numpy(pts).cuda(), feats, S, r, K)
        i_ref, d_ref = opr.raster_brute(pts, S, K, r)
        assert np.array_equal(idx.cpu().numpy(), i_ref)
        assert np.array_equal(dists.cpu().numpy().view(np.int32), d_ref.view(np.int32))
        assert (out - opr.composite(torch.from_numpy(i_ref), torch.from_numpy(d_ref), feats, r)).abs().max().item() <= 1e-6


@pytest.fixture(scope="module")
def refine_inputs():
    xyz, feats = pc.refine_cloud()
    return torch.from_numpy(xyz).cuda(), torch.from_numpy(feats).cuda()


@pytest.mark.parametrize("S", [800, 400, 200])
def test_refine_sizes_bit_identical(ru, refine_inputs, S):
    xyz, feats = refine_inputs
    pts = opr.project(xyz, S, S, torch.from_numpy(pc.intrinsics(S)).cuda(), torch.from_numpy(pc.look_at_world2cam()).cuda())
    out, idx, _ = check_forward(ru, pts, feats, S, 8, pc.REFINE_RADIUS)
    assert (idx[..., 0] >= 0).float().mean().item() > 0.3


def test_degenerate_cluster_in_one_tile(ru):
    g = torch.Generator().manual_seed(2)
    S, r = 128, 0.04
    pts = torch.stack([0.3 + 0.2 * torch.rand(20000, generator=g) * 2 / 16, -0.1 - 0.2 * torch.rand(20000, generator=g) * 2 / 16,
                       torch.randint(0, 50, (20000,), generator=g).float() / 10], 1)
    feats = torch.randn(20000, 3, generator=g)
    check_forward(ru, pts.cuda(), feats.cuda(), S, 16, r)


def test_all_culled_cloud_renders_zero(ru):
    g = torch.Generator().manual_seed(3)
    pts = torch.rand(5000, 3, generator=g) * 2 - 1
    pts[:, 2] = -pts[:, 2].abs() - 1e-3
    pts[::7, 0] = float("nan")
    pts[::11, 2] = float("inf")
    out, idx, dists = ru.point_render(pts.cuda(), torch.randn(5000, 19).cuda(), 64, 0.1, 8)
    assert torch.count_nonzero(out).item() == 0 and (idx == -1).all() and (dists == -1).all()


def test_feature_gradient_vs_float64_oracle_and_deterministic(ru, refine_inputs):
    xyz, feats = refine_inputs
    S = 400
    pts = opr.project(xyz, S, S, torch.from_numpy(pc.intrinsics(S)).cuda(), torch.from_numpy(pc.look_at_world2cam()).cuda())
    g_out = torch.randn(1, 19, S, S, generator=torch.Generator().manual_seed(4)).cuda()
    f = feats.clone().requires_grad_()
    out, idx, dists = ru.point_render(pts, f, S, pc.REFINE_RADIUS, 8)
    out.backward(g_out)
    g1 = f.grad.clone()
    f.grad = None
    ru.point_render(pts, f, S, pc.REFINE_RADIUS, 8)[0].backward(g_out)
    assert torch.equal(bits(g1), bits(f.grad))
    f64 = feats.double().requires_grad_()
    opr.composite(idx.long(), dists, f64, pc.REFINE_RADIUS).backward(g_out.double())
    ref = f64.grad
    assert ((g1.double() - ref).abs().max() / ref.abs().max()).item() <= 1e-5
    assert torch.count_nonzero(ref).item() > 0.1 * ref.numel()        # ~1/4 of the points are in some pixel's front K


@pytest.fixture(scope="module")
def golden():
    return load_golden("render_point.npz")


def test_render_point_reproduces_reference_fixture(ru, golden):
    """Reference glue + pytorch3d semantics (fixture) vs ours end to end.  The projection is a float32 matmul on the GPU here and on
    the CPU in the fixture; the last-bit differences move alphas by ~1e-7, hence 1e-5 rather than the oracle's 1e-6."""
    g = golden
    xyz, feats, w2c = (torch.from_numpy(g[k]).cuda() for k in ("xyz", "feats", "world2cam"))
    r, ppp, pix = float(g["radius"]), int(g["ppp"]), torch.from_numpy(g["sample_pix"]).cuda()
    for S in g["sizes"]:
        S = int(S)
        K = torch.from_numpy(g[f"K_{S}"]).cuda()
        out = ru.render_point(xyz, feats, S, S, K, w2c, (S, S), r, ppp, bg_feat=torch.ones(1, 19, 1, 1).cuda())
        ref = g[f"out_{S}"]
        assert out.shape == (1, 19, S, S)
        if ref.ndim == 2:
            out = out.reshape(19, -1)[:, pix]
        assert np.abs(out.cpu().numpy() - ref).max() <= 1e-5
    mask = ru.render_point(xyz, torch.ones(len(xyz), 3).cuda(), S, S, K, w2c, (S, S), r, ppp)
    assert np.abs(mask.reshape(3, -1)[:, pix].cpu().numpy() - g["mask_out"]).max() <= 1e-5


def test_rejections(ru, mi3d, golden):
    pts = torch.rand(100, 3).cuda()
    feats = torch.rand(100, 19).cuda()
    with pytest.raises(mi3d.Mi3dError):
        ru.point_render(pts.clone().requires_grad_(), feats, 32, 0.1, 8)
    with pytest.raises(mi3d.Mi3dError):
        ru.point_render(pts.cpu(), feats.cpu(), 32, 0.1, 8)
    with pytest.raises(mi3d.Mi3dError, match="invalid argument"):
        ru.point_render(pts, feats, (32, 48), 0.1, 8)
    with pytest.raises(mi3d.Mi3dError, match="invalid argument"):
        ru.point_render(pts, feats, 32, 0.1, 17)
    K, w2c = torch.from_numpy(pc.intrinsics(32)).cuda(), torch.from_numpy(pc.look_at_world2cam()).cuda()
    with pytest.raises(mi3d.Mi3dError):
        ru.render_point(pts.clone().requires_grad_(), feats, 32, 32, K, w2c, (32, 32), 0.1, 8)
    with pytest.raises(mi3d.Mi3dError):
        ru.render_point(pts.cpu(), feats.cpu(), 32, 32, K.cpu(), w2c.cpu(), (32, 32), 0.1, 8)
    with pytest.raises(mi3d.Mi3dError, match="invalid argument"):
        ru.render_point(pts, feats, 32, 48, K, w2c, (32, 48), 0.1, 8)


def test_gradient_reaches_point_colours_through_render_point(ru, golden):
    g = golden
    S = 64
    xyz, w2c, K = (torch.from_numpy(g[k]).cuda() for k in ("xyz", "world2cam", f"K_{S}"))
    colour = torch.nn.Parameter(torch.from_numpy(g["feats"][:, :3]).cuda())
    learned = torch.nn.Parameter(torch.from_numpy(g["feats"][:, 3:]).cuda())
    wts = torch.rand(1, 19, S, S, generator=torch.Generator().manual_seed(6)).cuda()
    out = ru.render_point(xyz, torch.cat([colour, learned], -1), S, S, K, w2c, (S, S), float(g["radius"]), int(g["ppp"]))
    (out * wts).sum().backward()
    c64 = torch.from_numpy(g["feats"]).double().cuda().requires_grad_()
    ref = opr.render_point_ref(xyz, c64, S, S, K, w2c, (S, S), float(g["radius"]), int(g["ppp"]))
    (ref * wts.double()).sum().backward()
    got = torch.cat([colour.grad, learned.grad], -1).double()
    assert torch.count_nonzero(colour.grad).item() > 0
    assert ((got - c64.grad).abs().max() / c64.grad.abs().max()).item() <= 1e-5
