"""tests/golden/make_golden_ref_raymarching.py -- fixtures from the REFERENCE's own ray-marching package.

ref_raymarching.npz: what the reference kernels (raymarching/src/{raymarching.cu,bindings.cpp}, compiled unmodified for sm_100a
into oracle/_ref/ by oracle/build_ref.py) return for the inputs that tests/test_ref_parity_gpu.py and
tests/test_backend_dropin_gpu.py build; those tests give our operators the same inputs and compare with these outputs.
Per-ray sample counts, sample totals, and the step sizes and alive list of the inference march are stored whole; other outputs
larger than a few thousand values are stored as a fixed, seeded sample (`<name>_sel` indices + values) to keep the file small.

ref_backend_calls.json: every `get_backend().<name>(...)` call of the reference's raymarching/raymarching.py with its positional
arities (tests/test_abi.py checks backend_mi3d against it).

    python tests/golden/make_golden_ref_raymarching.py [--reference <Make-It-3D checkout>]       (needs a GPU and oracle/_ref/)
"""
import argparse
import ast
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

from helpers import camera_rays, march_rows, orm, sphere_bitfield      # noqa: E402

AABB = np.array([-1, -1, -1, 1, 1, 1], np.float32)
SAMPLE_SEED = 20240
N_IDX = 1024          # sampled morton indices / packed bytes
N_RAYS = 256          # sampled rays of per-ray outputs
N_SAMPLES = 512       # sampled rows of per-sample outputs
N_MARCH_RAYS = 16     # sampled (non-empty) rays whose training-march samples are stored


def _cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _np(t):
    return t.cpu().numpy()


def collect(ref):
    """Every reference-kernel output the two test modules compare with, whole.  The inputs are built exactly as the tests build
    them."""
    z = {}
    # near / far of 64 x 64 rays (parity test and the drop-in train path make the same call)
    ro, rd, _ = camera_rays(64)
    N = ro.shape[0]
    n_r, f_r = torch.empty(N, device="cuda"), torch.empty(N, device="cuda")
    ref.near_far_from_aabb(_cu(ro), _cu(rd), _cu(AABB), N, 0.2, n_r, f_r)
    # morton3D / packbits (parity test)
    rng = np.random.default_rng(0)
    coords = rng.integers(0, 128, size=(100000, 3), dtype=np.int32)
    idx_r = torch.empty(100000, dtype=torch.int32, device="cuda")
    ref.morton3D(_cu(coords), 100000, idx_r)
    grid = rng.random((1, 128 ** 3), dtype=np.float32)
    bits_r = torch.empty(128 ** 3 // 8, dtype=torch.uint8, device="cuda")
    ref.packbits(_cu(grid), 128 ** 3 // 8, 0.4, bits_r)
    torch.cuda.synchronize()
    z.update(nf_nears=_np(n_r), nf_fars=_np(f_r), morton_idx=_np(idx_r), pack_bits=_np(bits_r))

    # training march of 96 x 96 rays (parity test)
    ro, rd, _ = camera_rays(96)
    bits = sphere_bitfield(0.25)
    nears, fars = orm.near_far_from_aabb(ro, rd, AABB, 0.2)
    N = ro.shape[0]
    noises = np.random.default_rng(4).random(N, dtype=np.float32)
    M = N * 512
    xyzs = torch.zeros(M, 3, device="cuda"); dirs = torch.zeros(M, 3, device="cuda"); deltas = torch.zeros(M, 2, device="cuda")
    rays = torch.empty(N, 3, dtype=torch.int32, device="cuda")
    counter = torch.zeros(2, dtype=torch.int32, device="cuda")
    ref.march_rays_train(_cu(ro), _cu(rd), _cu(bits), 1.0, 0.0, 512, N, 1, 128, M, _cu(nears), _cu(fars), xyzs, dirs, deltas, rays,
                         counter, _cu(noises))
    torch.cuda.synchronize()
    cnt = _np(counter)
    z.update(mt_counter=cnt, mt_rays=_np(rays), mt_xyzs=_np(xyzs[:cnt[0]]), mt_deltas=_np(deltas[:cnt[0]]))

    # composite forward / backward on the oracle's march of 64 x 64 rays (parity test)
    ro, rd, _ = camera_rays(64)
    bits = sphere_bitfield(0.3)
    nears, fars = orm.near_far_from_aabb(ro, rd, AABB, 0.2)
    N = ro.shape[0]
    rng = np.random.default_rng(8)
    _, _, dl, rays, _ = orm.march_rays_train(ro, rd, 1.0, bits, 1, 128, nears, fars, rng.random(N, dtype=np.float32), 0.0, 512, align=128)
    m = dl.shape[0]
    sig = (rng.random(m, dtype=np.float32) * 20).astype(np.float32); rgb = rng.random((m, 3), dtype=np.float32)
    ws_r, dep_r, img_r = torch.empty(N, device="cuda"), torch.empty(N, device="cuda"), torch.empty(N, 3, device="cuda")
    ref.composite_rays_train_forward(_cu(sig), _cu(rgb), _cu(dl), _cu(rays), m, N, 1e-4, ws_r, dep_r, img_r)
    gw, gi = rng.standard_normal(N).astype(np.float32), rng.standard_normal((N, 3)).astype(np.float32)
    gs_r, gr_r = torch.zeros(m, device="cuda"), torch.zeros(m, 3, device="cuda")
    ref.composite_rays_train_backward(_cu(gw), _cu(gi), _cu(sig), _cu(rgb), _cu(dl), _cu(rays), ws_r, img_r, m, N, 1e-4, gs_r, gr_r)
    torch.cuda.synchronize()
    z.update(cp_ws=_np(ws_r), cp_dep=_np(dep_r), cp_img=_np(img_r), cp_gs=_np(gs_r), cp_gr=_np(gr_r))

    # drop-in train path: march of 64 x 64 rays, then composite forward / backward on the oracle's (ordered) march
    ro, rd, _ = camera_rays(64)
    N, max_steps = ro.shape[0], 512
    M = N * max_steps
    nears, fars = orm.near_far_from_aabb(ro, rd, AABB, 0.2)
    bits = sphere_bitfield(0.3)
    noises = np.random.default_rng(1).random(N, dtype=np.float32)
    xyzs = torch.zeros(M, 3, device="cuda"); dirs = torch.zeros(M, 3, device="cuda"); deltas = torch.zeros(M, 2, device="cuda")
    rays = torch.empty(N, 3, dtype=torch.int32, device="cuda"); counter = torch.zeros(2, dtype=torch.int32, device="cuda")
    ref.march_rays_train(_cu(ro), _cu(rd), _cu(bits), 1.0, 0.0, max_steps, N, 1, 128, M, _cu(nears), _cu(fars), xyzs, dirs, deltas, rays,
                         counter, _cu(noises))
    dl, rr, m = march_rows(ro, rd, bits, nears, fars, noises, max_steps)
    dl, rr = _cu(dl), _cu(rr)
    rng = np.random.default_rng(2)
    sig, rgb = _cu((rng.random(M, dtype=np.float32) * 20)), _cu(rng.random((M, 3), dtype=np.float32))
    ws, dep, img = torch.empty(N, device="cuda"), torch.empty(N, device="cuda"), torch.empty(N, 3, device="cuda")
    ref.composite_rays_train_forward(sig, rgb, dl, rr, M, N, 1e-4, ws, dep, img)
    gw, gi = _cu(rng.standard_normal(N).astype(np.float32)), _cu(rng.standard_normal((N, 3)).astype(np.float32))
    gs, gr = torch.zeros(M, device="cuda"), torch.zeros(M, 3, device="cuda")
    ref.composite_rays_train_backward(gw, gi, sig, rgb, dl, rr, ws, img, M, N, 1e-4, gs, gr)
    torch.cuda.synchronize()
    z.update(dt_counter=_np(counter), dt_rays=_np(rays), dt_ws=_np(ws), dt_dep=_np(dep), dt_img=_np(img), dt_gs=_np(gs[:m]), dt_gr=_np(gr[:m]))

    # drop-in grid / inference calls
    rng = np.random.default_rng(3)
    coords = rng.integers(0, 128, size=(50000, 3), dtype=np.int32)
    grid = rng.random((1, 128 ** 3), dtype=np.float32)
    idx = torch.empty(50000, dtype=torch.int32, device="cuda")
    ref.morton3D(_cu(coords), 50000, idx)
    back = torch.empty(50000, 3, dtype=torch.int32, device="cuda")
    ref.morton3D_invert(idx, 50000, back)
    bits_r = torch.empty(128 ** 3 // 8, dtype=torch.uint8, device="cuda")
    ref.packbits(_cu(grid), 128 ** 3 // 8, 0.4, bits_r)
    torch.cuda.synchronize()
    assert np.array_equal(_np(back), coords), "reference morton3D_invert does not invert morton3D"
    z.update(gi_morton_idx=_np(idx), gi_pack_bits=_np(bits_r))
    ro, rd, _ = camera_rays(48)
    nears, fars = orm.near_far_from_aabb(ro, rd, AABB, 0.2)
    bits = sphere_bitfield(0.3)
    n_alive, n_step = ro.shape[0], 4
    rays_alive = torch.arange(n_alive, dtype=torch.int32, device="cuda")
    rays_t = _cu(nears).clone()
    xyzs = torch.zeros(n_alive * n_step, 3, device="cuda"); dirs = torch.zeros(n_alive * n_step, 3, device="cuda")
    deltas = torch.zeros(n_alive * n_step, 2, device="cuda")
    ref.march_rays(n_alive, n_step, rays_alive, rays_t, _cu(ro), _cu(rd), 1.0, 0.0, 512, 1, 128, _cu(bits), _cu(nears), _cu(fars), xyzs, dirs,
                   deltas, torch.zeros(n_alive, device="cuda"))
    g = torch.Generator(device="cuda").manual_seed(0)
    sig = torch.rand(n_alive * n_step, device="cuda", generator=g) * 30
    rgb = torch.rand(n_alive * n_step, 3, device="cuda", generator=g); nrm = torch.rand(n_alive * n_step, 3, device="cuda", generator=g)
    ws, dep = torch.zeros(n_alive, device="cuda"), torch.zeros(n_alive, device="cuda")
    img, nimg = torch.zeros(n_alive, 3, device="cuda"), torch.zeros(n_alive, 3, device="cuda")
    ref.composite_rays(n_alive, n_step, 1e-2, rays_alive, rays_t, sig, rgb, nrm, deltas, ws, dep, img, nimg)
    torch.cuda.synchronize()
    z.update(gi_xyzs=_np(xyzs), gi_deltas=_np(deltas), gi_alive=_np(rays_alive), gi_ws=_np(ws), gi_dep=_np(dep), gi_img=_np(img),
             gi_nimg=_np(nimg))
    return z


def _pick(rng, n, k):
    return np.sort(rng.choice(n, size=min(k, n), replace=False)).astype(np.int32)


def _counts(rays, N):
    """per-ray sample counts by ray id (the reference's offsets follow atomic arrival order)"""
    c = np.zeros(N, np.int16)
    c[rays[:, 0]] = rays[:, 2]
    return c


def compact(z):
    """The fixture: whole arrays where they are small or compress well, a seeded sample of the rest."""
    rng = np.random.default_rng(SAMPLE_SEED)
    g = {"nf_sel": _pick(rng, z["nf_nears"].shape[0], N_RAYS)}
    g["nf_nears"], g["nf_fars"] = z["nf_nears"][g["nf_sel"]], z["nf_fars"][g["nf_sel"]]
    for key, sel_key, k in (("morton_idx", "morton_sel", N_IDX), ("pack_bits", "pack_sel", N_IDX),
                            ("gi_morton_idx", "gi_morton_sel", N_IDX), ("gi_pack_bits", "gi_pack_sel", N_IDX)):
        g[sel_key] = _pick(rng, z[key].shape[0], k)
        g[key] = z[key][g[sel_key]]
    # training march: whole per-ray counts and totals, the samples of a few non-empty rays (in ray order)
    rays = z["mt_rays"]
    N = rays.shape[0]
    g["mt_counter"], g["mt_counts"] = z["mt_counter"], _counts(rays, N)
    by_ray = {int(r[0]): (int(r[1]), int(r[2])) for r in rays}
    g["mt_sel"] = np.sort(rng.choice(np.flatnonzero(g["mt_counts"]), size=N_MARCH_RAYS, replace=False)).astype(np.int32)
    rows = np.concatenate([np.arange(by_ray[n][0], by_ray[n][0] + by_ray[n][1]) for n in g["mt_sel"]])
    g["mt_xyzs"], g["mt_dt"] = z["mt_xyzs"][rows], z["mt_deltas"][rows, 0]
    # composites: sampled rays of the forward outputs, sampled rows of the gradients
    for p in ("cp", "dt"):
        g[p + "_sel"] = _pick(rng, z[p + "_ws"].shape[0], N_RAYS)
        for k in ("ws", "dep", "img"):
            g[f"{p}_{k}"] = z[f"{p}_{k}"][g[p + "_sel"]]
        g[p + "_gsel"] = _pick(rng, z[p + "_gs"].shape[0], N_SAMPLES)
        g[p + "_gs"], g[p + "_gr"] = z[p + "_gs"][g[p + "_gsel"]], z[p + "_gr"][g[p + "_gsel"]]
        g[p + "_gs_max"] = np.abs(z[p + "_gs"]).max()          # the scale the sigma-gradient tolerance is relative to
    g["dt_counter"], g["dt_counts"] = z["dt_counter"], _counts(z["dt_rays"], z["dt_rays"].shape[0])
    # inference march + composite: whole step sizes and alive list, sampled rays of the rest
    n_step = z["gi_deltas"].shape[0] // z["gi_alive"].shape[0]
    g["gi_deltas"], g["gi_alive"] = z["gi_deltas"], z["gi_alive"]
    g["gi_sel"] = _pick(rng, z["gi_alive"].shape[0], N_RAYS)
    g["gi_xyzs"] = z["gi_xyzs"].reshape(-1, n_step, 3)[g["gi_sel"]]
    for k in ("ws", "dep", "img", "nimg"):
        g["gi_" + k] = z["gi_" + k][g["gi_sel"]]
    return g


def backend_calls(reference):
    """{name: sorted positional arities} of every `get_backend().<name>(...)` call in the reference's raymarching wrapper."""
    src = open(os.path.join(reference, "raymarching", "raymarching.py")).read()
    calls = {}
    for node in ast.walk(ast.parse(src)):
        if isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute) and isinstance(node.func.value, ast.Call) \
                and getattr(node.func.value.func, "id", "") == "get_backend":
            calls.setdefault(node.func.attr, set()).add(len(node.args))
    return {k: sorted(v) for k, v in sorted(calls.items())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", default=None, help="checkout of the original Make-It-3D project: (re)write ref_backend_calls.json")
    ap.add_argument("--out", default=HERE, help="directory the fixtures are written to")
    ap.add_argument("--full", default=None, help="also write every collected kernel output, unsampled, to this .npz")
    args = ap.parse_args()
    if args.reference:
        with open(os.path.join(args.out, "ref_backend_calls.json"), "w") as f:
            json.dump(backend_calls(args.reference), f, indent=1)
            f.write("\n")
    from oracle import build_ref
    ref = build_ref.load_ref()
    if ref is None or not torch.cuda.is_available():
        raise SystemExit("ref_raymarching.npz needs a GPU and oracle/_ref/_raymarching_ref.so (built by oracle/build_ref.py)")
    z = collect(ref)
    if args.full:
        np.savez_compressed(args.full, **z)
    np.savez_compressed(os.path.join(args.out, "ref_raymarching.npz"), **compact(z))


if __name__ == "__main__":
    main()
