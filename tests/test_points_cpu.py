"""CPU: the two float32 restatements of the point rasteriser agree bit for bit, and the oracle's render_point reproduces the
reference's (tests/golden/render_point.npz, recorded by tests/golden/make_golden_refine.py)."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import points_ref as opr
import points_cases as pc


@pytest.mark.parametrize("S", [32, 48])
def test_brute_and_splat_rasterisers_agree(S):
    r = 0.05
    pts = pc.edge_cloud(S, 2000, r, seed=S)
    idx_a, d_a = opr.raster_brute(pts, S, 8, r)
    idx_b, d_b = opr.raster_splat(torch.from_numpy(pts), S, 8, r)
    assert np.array_equal(idx_a, idx_b.numpy())
    assert np.array_equal(d_a.view(np.int32), d_b.numpy().view(np.int32))
    # the inputs reach the cases they are there for
    assert (idx_a[..., -1] >= 0).any() and (idx_a[..., 0] < 0).any()           # full and empty pixels
    ok = np.isfinite(pts).all(1) & (pts[:, 2] >= 0)
    assert not np.isin(np.nonzero(~ok)[0], idx_a).any()                        # culled points never selected
    z = pts[:, 2]
    sel = idx_a[idx_a[..., 1] >= 0]
    assert (z[sel[:, 0]] == z[sel[:, 1]]).any()                                # exact z ties resolved by index
    crowd = opr.raster_brute(pts, S, 16, r)[0][S // 3, S // 2]
    assert (crowd >= 0).all()


def test_oracle_render_point_matches_reference_fixture():
    g = load_golden("render_point.npz")
    xyz, feats, w2c = (torch.from_numpy(g[k]) for k in ("xyz", "feats", "world2cam"))
    r, ppp, pix = float(g["radius"]), int(g["ppp"]), g["sample_pix"]
    for S in g["sizes"]:
        S = int(S)
        out = opr.render_point_ref(xyz, feats, S, S, torch.from_numpy(g[f"K_{S}"]), w2c, (S, S), r, ppp).numpy()
        ref = g[f"out_{S}"]
        if ref.ndim == 2:
            out = out.reshape(-1, S * S)[:, pix]
        assert out.shape == ref.shape and np.abs(out - ref).max() <= 1e-6
    S = int(g["sizes"][-1])
    mask = opr.render_point_ref(xyz, torch.ones(len(xyz), 3), S, S, torch.from_numpy(g[f"K_{S}"]), w2c, (S, S), r, ppp).numpy()
    assert np.abs(mask.reshape(3, -1)[:, pix] - g["mask_out"]).max() <= 1e-6
    assert (g["mask_out"] > 0).mean() > 0.2
