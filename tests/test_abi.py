"""CPU: the C-ABI library builds for sm_100a, loads without a GPU, and exports exactly what include/mi3d.h declares."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    txt = open(os.path.join(ROOT, "include", "mi3d.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(mi3d_[A-Za-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol(mi3d):
    lib = mi3d.lib()
    syms = header_symbols()
    assert len(syms) >= 19
    for s in syms:
        assert hasattr(lib, s), f"libmi3d.so does not export {s}"
    assert sorted(mi3d._lib.SYMBOLS) == syms
    assert b"sm_100a" in lib.mi3d_version()


def test_workspace_queries_are_pure_host(mi3d):
    lib = mi3d.lib()
    assert lib.mi3d_march_rays_train_workspace_bytes(ctypes.c_uint32(16384)) == (1 + 2 * 128) * 4
    assert lib.mi3d_density_grid_workspace_bytes(ctypes.c_uint32(1), ctypes.c_uint32(128)) > 128 ** 3 * 16


def test_hashgrid_geometry_matches_oracle(mi3d):
    """Host helper mi3d_hashgrid_make vs the oracle's level table (tiny-cuda-nn grid.h geometry; SURVEY 8a-E1 sizes)."""
    import importlib
    from oracle import raymarch as orm
    ops = importlib.import_module("make-it-3d_b200.nerf.field_ops")
    hg = ops.make_hashgrid()
    lv = orm.hashgrid_levels()
    assert hg.n_levels == 16 and hg.n_entries == lv["total"] == 6098120
    assert list(hg.sizes) == list(lv["sizes"]) and list(hg.offsets) == list(lv["offsets"]) and list(hg.ress) == list(lv["ress"])
    assert list(hg.sizes)[:5] == [4096, 12168, 29792, 79512, 205384] and all(s == 524288 for s in list(hg.sizes)[5:])
    assert all(abs(a - b) == 0 for a, b in zip(hg.scales, lv["scales"]))


def test_product_path_refuses_cpu_tensors(mi3d):
    """No CPU fallback: the operators raise on CPU tensors instead of silently computing elsewhere."""
    import importlib
    import pytest
    import torch
    ops = importlib.import_module("make-it-3d_b200.nerf.field_ops")
    nt = importlib.import_module("make-it-3d_b200.nerf.network_tcnn")
    enc = nt.HashGridEncoding()
    with pytest.raises(mi3d.Mi3dError):
        enc(torch.rand(4, 3))
    assert ops is not None


def test_state_dict_keys_match_reference(mi3d):
    """nerf/utils.py:1075-1186 checkpoints: same keys / shapes as the reference module tree."""
    import argparse
    import importlib
    nt = importlib.import_module("make-it-3d_b200.nerf.network_tcnn")
    opt = argparse.Namespace(bound=1, min_near=0.1, density_thresh=10, bg_radius=-1, blob_density=5, blob_radius=0.1,
                             lambda_smooth=1, max_depth=10.0)
    sd = nt.NeRFNetwork(opt).state_dict()
    want = {'aabb_train': (6,), 'aabb_infer': (6,), 'density_grid': (1, 128 ** 3), 'density_bitfield': (128 ** 3 // 8,),
            'step_counter': (16, 2), 'encoder.params': (12196240,), 'sigma_net.net.0.weight': (64, 32), 'sigma_net.net.0.bias': (64,),
            'sigma_net.net.1.weight': (64, 64), 'sigma_net.net.1.bias': (64,), 'sigma_net.net.2.weight': (4, 64),
            'sigma_net.net.2.bias': (4,)}
    assert {k: tuple(v.shape) for k, v in sd.items()} == want


def test_committed_bench_line_has_every_contract_key():
    """profiles/r1_final_bench.json is the last line bench.py printed on a B200: the keys the driver parses must all be there"""
    import json
    import os
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "r1_final_bench.json")
    line = json.loads(open(path).read())
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
                "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline"):
        assert key in line, key
    assert line["config"]["workload"] and "model" not in line["config"]
    assert set(("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step")) <= set(line["e2e"])
    assert line["e2e"]["h2d_bytes_per_step"] > 0 and line["e2e"]["d2h_bytes_per_step"] > 0
    assert set(("bound", "achieved", "peak", "unit", "frac", "traffic")) <= set(line["roofline"])
    assert abs(line["roofline"]["frac"] - line["roofline"]["achieved"] / line["roofline"]["peak"]) < 1e-3
    assert set(("value", "unit", "cores", "kind", "sample")) <= set(line["cpu_baseline"])
    assert line["gpu_launches"] > 0 and not set(line["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}


def test_engine_stream_context_is_a_no_op_without_graph_replay():
    """graph_replay=False (engine.stream is None): SDEngine.on_stream() must not touch streams (launches go to the caller's stream)"""
    import importlib
    sd = importlib.import_module("make-it-3d_b200.nerf.sd")

    class _E:
        stream = None
    ran = []
    with sd.SDEngine.on_stream(_E()):
        ran.append(1)
    assert ran == [1]


def test_backend_mi3d_covers_reference_call_sites():
    """Every `get_backend().<name>(...)` call in the REFERENCE's raymarching/raymarching.py must resolve on backend_mi3d._backend
    with the same positional arity (the calls and their arities are recorded in tests/golden/ref_backend_calls.json by
    tests/golden/make_golden_ref_raymarching.py)."""
    import importlib
    import inspect
    import json
    be = importlib.import_module("make-it-3d_b200.backend_mi3d")._backend
    calls = {name: set(arities) for name, arities in json.load(open(os.path.join(ROOT, "tests", "golden", "ref_backend_calls.json"))).items()}
    assert {"near_far_from_aabb", "march_rays_train", "composite_rays_train_forward", "composite_rays_train_backward", "packbits",
            "morton3D", "morton3D_invert", "march_rays", "composite_rays"} <= set(calls)
    for name, arities in calls.items():
        assert hasattr(be, name), name
        fn = getattr(be, name)
        params = list(inspect.signature(fn).parameters.values())
        if any(p.kind == p.VAR_POSITIONAL for p in params):
            continue                                   # the loudly-failing stubs of unreachable entry points
        assert arities == {len(params)}, (name, arities, len(params))
