#!/usr/bin/env python
"""bench.py -- SDS train-steps/sec (NeRF render + SD U-Net) @128x128 on N B200s (BASELINE.json metric).

One step == the SDS branch of Trainer.train_step (nerf/utils.py:461-574) restricted to the hot path (SURVEY.md 8d):
    model.render(128x128 rays, perturb, force_all_rays, max_steps 512, k = 13 field evaluations / sample)
    -> guidance.train_step(text_z, pred_rgb)   [bilinear 512 -> VAE encode -> add_noise -> U-Net x2 (CFG) -> SDS grad
                                                -> latents.backward: VAE input-grad -> composite bwd -> field bwd]
    -> regulariser loss.backward()             [opacity + entropy + orientation + smoothness: second render backward]
    -> (N > 1) all-reduce of hash-grid + MLP gradients
Excluded like SURVEY 8d says: CLIP losses, PNG dumps, the Adan update.  Synthetic data: orbit poses, solid-sphere occupancy
(r = 0.2), seeded random hash table / MLP / SD-2.0-base weights (no weights offline), N(0,1) text embeddings.

  python bench.py --gpus 1 --steps 10 --warmup 3            # one JSON line
  torchrun ... bench.py --gpus N ...                        # one rank per GPU, weak scaling (one view per GPU per step)
  python bench.py --impl reference ...                      # the reference algorithm on the host CPU cores (oracle port)
  python bench.py ... --dump-outputs DIR                    # also write what the last timed step computed to DIR/<name>.npy
"""
import argparse
import importlib
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "SDS train-steps/sec (NeRF render+SD U-Net) @128x128"
UNIT = "view-steps/s"
HW = 128
SPHERE_R = 0.2
WORKLOAD = ("coarse stage 128x128, SD-2.0-base architecture (random-init weights) SDS, hash-grid L=16 F=2 T=2^19 fp32, "
            "solid-sphere occupancy r=0.2, max_steps 512, k=13 field evals/sample (reference defaults lambda_orient/lambda_smooth on)")


def opt_namespace():
    return argparse.Namespace(bound=1, min_near=0.1, density_thresh=10, bg_radius=-1, blob_density=5, blob_radius=0.1,
                              lambda_smooth=1, lambda_orient=1e-2, lambda_opacity=1e-3, lambda_entropy=1, max_depth=10.0,
                              max_steps=512, dt_gamma=0)


def orbit_pose(radius, theta_deg, phi_deg):
    """look-at camera of nerf/provider.py:143-214 (up = -y)"""
    th, ph = math.radians(theta_deg), math.radians(phi_deg)
    c = np.array([radius * math.sin(th) * math.sin(ph), radius * math.cos(th), radius * math.sin(th) * math.cos(ph)], np.float32)
    fwd = -c / np.linalg.norm(c)
    right = np.cross(fwd, np.array([0, -1, 0], np.float32)); right /= np.linalg.norm(right)
    up = np.cross(right, fwd); up /= np.linalg.norm(up)
    pose = np.eye(4, dtype=np.float32)
    pose[:3, 0], pose[:3, 1], pose[:3, 2], pose[:3, 3] = right, up, fwd, c
    return pose


def synth_pose(index, rng):
    """radius U[1,1.5], theta U[70,110], phi U[0,360), fovy U[15,25] (main.py:72-76); index % 4 == 0 is the front view."""
    if index % 4 == 0:
        return orbit_pose(1.0, 90.0, 180.0), 20.0
    return orbit_pose(rng.uniform(1.0, 1.5), rng.uniform(70, 110), rng.uniform(0, 360)), rng.uniform(15, 25)


def sphere_bitfield_numpy(radius, H=128):
    def spread(v):
        v = (v * 0x00010001) & 0xFF0000FF; v = (v * 0x00000101) & 0x0F00F00F
        v = (v * 0x00000011) & 0xC30C30C3; v = (v * 0x00000005) & 0x49249249
        return v
    idx = np.arange(H, dtype=np.uint32)
    s = spread(idx.astype(np.uint64)).astype(np.uint32)
    xs, ys, zs = np.meshgrid(idx, idx, idx, indexing="ij")
    morton = (s[xs] | (s[ys] << 1) | (s[zs] << 2)).reshape(-1)
    c = (np.stack([xs, ys, zs], -1).reshape(-1, 3).astype(np.float32) + 0.5) / H * 2 - 1
    occ = np.zeros(H ** 3, np.uint8)
    occ[morton] = (np.linalg.norm(c, axis=1) < radius)
    return np.packbits(occ, bitorder="little")


class ClockSampler:
    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", "--query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap",
                 "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def build_models(device, seed, defer_backward=False):
    nt = importlib.import_module("make-it-3d_b200.nerf.network_tcnn")
    sdm = importlib.import_module("make-it-3d_b200.nerf.sd")
    torch.manual_seed(seed)
    model = nt.NeRFNetwork(opt_namespace())
    with torch.no_grad():
        g = torch.Generator().manual_seed(3)
        # "trained-like" table amplitude so densities / colours vary (init U(-1e-4,1e-4) would make the field a pure blob)
        model.encoder.params.copy_((torch.rand(model.encoder.params.numel(), generator=g) * 2 - 1) * 0.5)
    model = model.to(device).train()
    model.density_bitfield = torch.from_numpy(sphere_bitfield_numpy(SPHERE_R)).to(device)
    guidance = sdm.StableDiffusion(device, seed=0, defer_backward=defer_backward)
    return model, guidance


def regulariser_loss(out, opt):
    """nerf/utils.py:519-548 for global_step >= diff_iters (opacity, entropy x10, orientation x(1+10), smoothness)."""
    ws = out["weights_sum"]
    loss = opt.lambda_opacity * (ws ** 2).mean()
    a = ws.clamp(1e-5, 1 - 1e-5)
    loss = loss + opt.lambda_entropy * 10 * (-a * torch.log2(a) - (1 - a) * torch.log2(1 - a)).mean()
    loss = loss + opt.lambda_orient * out["loss_orient"] * 11
    loss = loss + opt.lambda_smooth * out["loss_smooth"]
    return loss


def dump_outputs(path, out, loss, model):
    """What the last timed step handed its caller: the render outputs, the total loss, and the gradients it left on the NeRF
    parameters (SDS + regularisers, summed over ranks), one float32 .npy per array (about 47 MiB in all)."""
    os.makedirs(path, exist_ok=True)
    arrays = dict(out, loss=loss, grad_encoder=model.encoder.params.grad)
    arrays.update({"grad_sigma_net." + n: p.grad for n, p in model.sigma_net.named_parameters()})
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t.detach().float().cpu().numpy())


def run_ours(args):
    par = importlib.import_module("make-it-3d_b200.parallel")
    field_ops = importlib.import_module("make-it-3d_b200.nerf.field_ops")
    utils = importlib.import_module("make-it-3d_b200.nerf.utils")
    rank, local, world = par.init_distributed()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU: the hot path has no CPU fallback (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    model, guidance = build_models(device, seed=0, defer_backward=args.defer_backward)
    opt = model.opt
    reducer = par.GradientAllReduce(model.encoder.params, list(model.sigma_net.parameters()), op="sum")
    ray_par = par.RayParallel() if (world > 1 and args.render_split == "rays") else None
    torch.manual_seed(par.rank_seed(0, rank))
    text_z = torch.randn(2, 77, 1024, generator=torch.Generator().manual_seed(0)).to(device)
    n_steps = args.warmup + args.steps + 8
    N = HW * HW
    # ---- the G = world views of every step (pose sequence shared by all ranks: view v of step s is pose index s*G + v, rank v owns it)
    rng = np.random.default_rng(0)
    cams_host, cams_dev = [], []
    for s in range(n_steps):
        rows = []
        for v in range(world):
            pose, fov = synth_pose(par.pose_index(s, v, world), rng)
            focal = HW / (2 * math.tan(math.radians(fov) / 2))
            rows.append(np.concatenate([pose[:3].reshape(-1), np.array([focal, focal, HW / 2, HW / 2], np.float32)]))
        tab = torch.from_numpy(np.stack(rows).astype(np.float32))
        if ray_par is None:
            tab = tab[rank:rank + 1]                       # view-parallel render: this rank sees its own view only
        cams_host.append(tab.contiguous().pin_memory())
        cams_dev.append(tab.to(device))
    text_host = text_z.cpu().pin_memory()
    h2d_bytes = cams_host[0].numel() * 4 + text_host.numel() * 4
    t_cycle = (250, 450, 600)          # islarge=True keeps every step on the SDS branch (nerf/sd.py:153)
    G = cams_dev[0].shape[0]
    gen_shared = torch.Generator(device=device).manual_seed(4242)      # same draws on every rank (per-view background colours)
    result_dev = torch.zeros(4, device=device)
    result_host = torch.zeros(4).pin_memory()
    m_log = torch.zeros(n_steps + 16, dtype=torch.int32, device=device)     # this rank's marched samples per executed step
    state = {"i": 0}

    def step(s, e2e, explicit_rays=False, marks=None):
        if e2e:
            cams = cams_host[s % n_steps].to(device, non_blocking=True)
            tz = text_host.to(device, non_blocking=True)
        else:
            cams, tz = cams_dev[s % n_steps], text_z
        model.zero_grad(set_to_none=True)
        bg = torch.rand(world, 3, device=device, generator=gen_shared)
        bg = bg if ray_par is not None else bg[rank]
        kw = dict(bg_color=bg, staged=False, perturb=True, ambient_ratio=1.0, shading='albedo', force_all_rays=True, **vars(opt))
        if marks is not None:
            marks.append(_ev())
        if explicit_rays:            # per-kernel timing leg: the same kernels through the unfused entry points (events around the field calls)
            rays = utils.get_rays(torch.cat([cams[:, :12].view(1, 3, 4), torch.tensor([[[0., 0., 0., 1.]]], device=device)], 1),
                                  tuple(float(x) for x in cams[0, 12:].tolist()), HW, HW, -1)
            out = model.render(rays['rays_o'], rays['rays_d'], depth_scale=rays['depth_scale'], **kw)
        else:
            out = model.render(None, None, cam_table=cams, cam_hw=(HW, HW), ray_parallel=ray_par,
                               step_seed=par.shared_seed(0, s) if ray_par is not None else None, **kw)
        ws = list(model._workspaces.values())[0]
        m_log[state["i"] % m_log.numel()].copy_(ws.counter[0]); state["i"] += 1
        if marks is not None:
            marks.append(_ev())
        pred_rgb = out['image'].reshape(1, HW, HW, 3).permute(0, 3, 1, 2).contiguous()
        loss, _ = guidance.train_step(tz, pred_rgb, islarge=True, guidance_scale=10, t=t_cycle[s % 3])
        if marks is not None:
            marks.append(_ev())
        loss = loss + regulariser_loss(out, opt)
        loss.backward()
        state["out"] = {k: v.detach() for k, v in out.items()}
        state["loss"] = loss.detach()
        if marks is not None:
            marks.append(_ev())
        reducer()
        if marks is not None:
            marks.append(_ev())
        if e2e:
            result_dev[0] = loss.detach(); result_dev[1] = out['loss_orient'].detach(); result_dev[2] = out['loss_smooth'].detach()
            result_dev[3] = out['weights_sum'].mean().detach()
            result_host.copy_(result_dev, non_blocking=True)
        return loss

    def _ev():
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def timed(n, e2e, first):
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for s in range(n):
            step(first + s, e2e)
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()
        return par.max_over_ranks(e0.elapsed_time(e1), device)

    for s in range(max(args.warmup, 3)):
        step(s, False)
    torch.cuda.synchronize()
    if args.launch_list:
        torch.cuda.nvtx.range_push("timed_steps")
        for s in range(args.steps):
            step(args.warmup + s, False)
        torch.cuda.synchronize()
        torch.cuda.nvtx.range_pop()
        if world > 1:
            torch.distributed.destroy_process_group()
        return
    def timeline(n_steps):
        # per-rank CUDA-event table of the step phases (profiles/: where a multi-GPU step spends its time on every rank)
        rows = []
        for s in range(n_steps):
            if world > 1:
                torch.distributed.barrier()
            marks = []
            step(args.warmup + s, False, marks=marks)
            torch.cuda.synchronize()
            rows.append([marks[i].elapsed_time(marks[i + 1]) for i in range(4)] + [int(m_log[(state["i"] - 1) % m_log.numel()])])
        t = torch.tensor(rows, dtype=torch.float64, device=device)
        allt = [torch.zeros_like(t) for _ in range(world)]
        if world > 1:
            torch.distributed.all_gather(allt, t)
        else:
            allt = [t]
        if rank != 0:
            return None
        out = {"n_gpus": world, "render_split": args.render_split if world > 1 else "single", "steps": n_steps,
               "columns": ["render_fwd_ms (incl. its collectives)", "sd_guidance_ms (VAE enc, U-Net, SDS backward to the field)",
                           "regulariser_backward_ms", "grad_allreduce_ms", "samples_marched_by_rank"],
               "per_rank": [[[round(float(x), 3) for x in r] for r in a.tolist()] for a in allt]}
        arr = np.array(out["per_rank"])
        out["mean_per_rank"] = [[round(float(x), 3) for x in arr[r].mean(0)] for r in range(world)]
        out["step_ms_max_over_ranks_mean"] = round(float(arr[:, :, :4].sum(2).max(0).mean()), 3)
        return out

    if args.timeline:
        out = timeline(args.steps)
        if rank == 0:
            print(json.dumps(out))
        if world > 1:
            torch.distributed.destroy_process_group()
        return
    # ---- launch count (one profiled step, outside the timed region) ----
    launches_per_step = None
    cupti = {}
    try:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            step(0, False)
            torch.cuda.synchronize()
        mine = ("k_field", "k_bwd", "k_march", "k_composite", "k_tc_gemm", "sdk::", "sd::k_", "k_loss_finalize", "k_near_far", "k_packbits", "k_grid",
                "k_view_", "k_get_rays", "k_flash_attn", "k_splitk")
        launches_per_step = sum(1 for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA and any(m in ev.name for m in mine))
        # CUPTI kernel durations of that step IN PIPELINE CONTEXT (graph replay on, no per-launch events): reported beside the
        # event-timed roofline numbers, which run the lists as plain launches with an event pair around every tile launch
        for ev in prof.events():
            if ev.device_type != torch.autograd.DeviceType.CUDA:
                continue
            for key in ("k_tc_gemm", "k_flash_attn", "k_field_fwd_tc", "k_field_bwd_tc", "k_bwd_enc_scatter", "k_gn_", "k_march_train", "k_composite_train"):
                if key in ev.name:
                    cupti[key] = cupti.get(key, 0.0) + (ev.device_time if hasattr(ev, "device_time") else ev.cuda_time) * 1e-3
    except Exception:
        launches_per_step = None
    clocks = ClockSampler(local)
    clocks.start()
    time.sleep(0.3)
    i_first = state["i"]
    ms = timed(args.steps, False, args.warmup)
    m_timed = m_log[[(i_first + k) % m_log.numel() for k in range(args.steps)]].cpu().numpy().astype(np.int64)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, state["out"], state["loss"], model)
    # ---- per-kernel live timing of the dominant kernels (CUDA events on the launching stream) ----
    import ctypes as C
    L = importlib.import_module("make-it-3d_b200._lib")
    n_prof = 3
    L.check(L.lib().mi3d_sd_profile(guidance.engine.h, C.c_int(1), None, None), "sd_profile")
    prof_steps = []
    if world == 1:
        for s in range(n_prof):
            field_ops.PROFILE = []
            step(args.warmup + s, False, explicit_rays=True)
            torch.cuda.synchronize()
            rows = {}
            for name, s0, e0, info in field_ops.PROFILE:
                key = name + ("_full" if info.get("full") else ("_image" if name == "k_field_bwd" else ""))
                rows[key] = rows.get(key, 0.0) + s0.elapsed_time(e0)
            rows["M"] = int(m_log[(state["i"] - 1) % m_log.numel()])
            prof_steps.append(rows)
        field_ops.PROFILE = None
    else:
        for s in range(n_prof):
            step(args.warmup + s, False)
        torch.cuda.synchronize()
    gemm_ms, gemm_n = C.c_float(0), C.c_int(0)
    # one line per timed launch: M N K block_n splits conv batch epi ms (in a scratch directory: the tree may be read-only)
    with tempfile.TemporaryDirectory() as tmp:
        dump_path = os.path.join(tmp, "sd_launches.txt")
        L.check(L.lib().mi3d_sd_profile_dump(guidance.engine.h, C.c_int(0), C.byref(gemm_ms), C.byref(gemm_n), dump_path.encode()), "sd_profile_dump")
        launches = open(dump_path).read().splitlines()
    tile_flops = attn_flops = attn_ms = 0.0
    attn_n = 0
    for ln in launches:
        f = ln.split()
        Mm, Nn, Kk, conv, batch, ms_l = int(f[0]), int(f[1]), int(f[2]), int(f[5]), int(f[6]), float(f[8])
        if conv == 2:
            attn_flops += 4.0 * Mm * Nn * Kk * batch; attn_ms += ms_l; attn_n += 1
        else:
            tile_flops += 2.0 * Mm * Nn * Kk * batch
    for s in range(2):                      # untimed: first-use allocations of the host-input staging path
        step(s, True)
    ms_e2e = timed(args.steps, True, args.warmup)
    clock_info = clocks.stop()

    value = world * args.steps / (ms * 1e-3)
    e2e_value = world * args.steps / (ms_e2e * 1e-3)
    split = ("ray-parallel render (every rank marches every %d-th pixel of all %d views) + view-parallel SD" % (world, world)) if ray_par is not None \
        else ("view-parallel render + SD" if world > 1 else "single GPU")
    line = {
        "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32 render / fp16 SD (fp32 accumulate)",
        "data": "synthetic (orbit poses, sphere occupancy, random-init hash table / MLP / SD-2.0-base weights, N(0,1) text embeddings)",
        "config": {"workload": WORKLOAD, "rays": N, "samples_per_step_M_mean": int(m_timed.mean()), "samples_per_step_M_min_max": [int(m_timed.min()), int(m_timed.max())],
                   "samples_note": "samples marched by rank 0 in the timed steps (depends on the pose: index % 4 == 0 is the close front view)",
                   "field_evals_per_sample": 13, "views_per_step": world,
                   "parallelism": f"dp{world}: {split}", "l2": "inputs larger than L2: 1.8 GB of SD weights + activations stream through L2 every step "
                   "(the 48.8 MB hash table is re-fetched after each SD pass)", "excluded": "CLIP losses, PNG I/O, Adan update (SURVEY 8d)",
                   "sd_launch_lists": "CUDA-graph replay" if guidance.engine.graph_replays() else "plain launches",
                   "render_backward_passes": 1 if args.defer_backward else 2,
                   "sds_backward": "deferred into the one loss.backward() (--defer-backward: same gradients, one render backward)" if args.defer_backward
                   else "immediate, inside guidance.train_step like nerf/sd.py:171 (two render backward passes per step)"},
        "e2e": {"value": round(e2e_value, 3), "unit": UNIT, "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": int(result_host.numel() * 4),
                "inputs": "pinned host camera table [views,16] + text embeddings [2,77,1024] copied in every step (rays are generated in the march kernel); 4 loss scalars copied out"},
        "gpu_launches": (launches_per_step * args.steps) if launches_per_step is not None else None,
        "clocks": clock_info,
    }
    # roofline of the dominant kernel = the tcgen05 tile kernel k_tc_gemm (every conv / linear product of the U-Net and the VAE: the
    # largest share of the step).  achieved = 2*M*N*K over the engine's own launch list of the profiled steps / summed duration of
    # those launches, timed live with CUDA events around each launch (plain launches: graph replay is suspended while profiling).
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    tf_peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    summary = {}
    try:
        summary = json.load(open(os.path.join(ROOT, "profiles", "r2_summary.json")))
    except Exception:
        pass
    gemm_ms_step = gemm_ms.value / n_prof
    flops = tile_flops / n_prof
    line["roofline"] = {
        "kernel": "tc::k_tc_gemm<64|128|160|256> (tcgen05.mma/TMEM/TMA tile kernel; all launches of one step: every conv / linear of the U-Net and the VAE)", "bound": "tensor",
        "achieved": round(flops / (gemm_ms_step * 1e-3) / 1e12, 1), "peak": tf_peak, "unit": "TFLOP/s",
        "frac": round(flops / (gemm_ms_step * 1e-3) / 1e12 / tf_peak, 4),
        "traffic": summary.get("k_tc_gemm", {}).get("dram_bytes_per_launch"),
        "traffic_source": "ncu --set full capture committed under profiles/ (per-launch mean; not measured by this run)",
        "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (of measured; kernel timed inside a long step)" if peaks else "fallback 1400 TFLOP/s (of fallback)",
        "ms_per_step": round(gemm_ms_step, 3), "launches_per_step": gemm_n.value // n_prof, "algorithmic_flops_per_step": flops,
    }
    if cupti.get("k_tc_gemm"):
        line["roofline"]["in_pipeline"] = {"source": "CUPTI kernel durations (torch.profiler) of one step with the launch lists replayed as CUDA graphs",
                                           "ms_per_step": round(cupti["k_tc_gemm"], 3), "achieved": round(flops / (cupti["k_tc_gemm"] * 1e-3) / 1e12, 1),
                                           "frac": round(flops / (cupti["k_tc_gemm"] * 1e-3) / 1e12 / tf_peak, 4)}
        line["kernel_ms_in_pipeline"] = {k: round(v, 3) for k, v in cupti.items()}
    if attn_n:
        line["roofline"]["attention"] = {"kernel": "attn::k_flash_attn (tcgen05, scores in TMEM)", "ms_per_step": round(attn_ms / n_prof, 3),
                                         "launches_per_step": attn_n // n_prof, "achieved": round(attn_flops / (attn_ms * 1e-3) / 1e12, 1), "unit": "TFLOP/s",
                                         "frac": round(attn_flops / (attn_ms * 1e-3) / 1e12 / tf_peak, 4)}
    # second roofline: the render kernels against the HBM roofline the north_star names.  Bytes and times come from the SAME profiled
    # steps: step i marched M_i samples -> E_i = 13 * pad128(M_i) evaluations -> algorithmic bytes E_i*1024 (+ per-ray terms) forward,
    # E_i*2048 backward (SURVEY 8d); frac = sum(bytes_i) / sum(ms_i) / peak.
    if prof_steps:
        fb = ft = bb = bt = 0.0
        for r in prof_steps:
            m_pad = r["M"] + 128 - r["M"] % 128
            if "k_field_fwd" in r:
                fb += 13 * m_pad * 1024 + N * 44 + 262144; ft += r["k_field_fwd"]
            if "k_field_bwd_full" in r:
                bb += 13 * m_pad * 2048 + N * 16; bt += r["k_field_bwd_full"]
        line["roofline_render"] = {"bound": "hbm", "peak": hbm, "unit": "GB/s", "profiled_steps": prof_steps,
                                   "traffic": {k: summary.get(k, {}).get("dram_bytes_per_launch") for k in ("k_field_fwd_tc", "k_bwd_enc_scatter", "k_field_bwd_tc")},
                                   "traffic_source": "ncu --set full capture committed under profiles/ (not measured by this run)"}
        if ft:
            line["roofline_render"]["fwd"] = {"algorithmic_bytes": int(fb), "ms": round(ft, 3), "achieved": round(fb / (ft * 1e-3) / 1e9, 1), "frac": round(fb / (ft * 1e-3) / 1e9 / hbm, 4)}
        if bt:
            line["roofline_render"]["bwd"] = {"algorithmic_bytes": int(bb), "ms": round(bt, 3), "achieved": round(bb / (bt * 1e-3) / 1e9, 1), "frac": round(bb / (bt * 1e-3) / 1e9 / hbm, 4)}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(args)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if args.timeline_out:
        tl = timeline(8)
        if rank == 0:
            with open(args.timeline_out, "w") as f:
                f.write(json.dumps(tl) + "\n")
    if world > 1:
        torch.distributed.destroy_process_group()


def cpu_baseline(args, steps=1):
    """The oracle port of the reference algorithm (oracle/: C ray-march + PyTorch fp32 field / U-Net / VAE) on the host cores.
    Bounded sample of the SAME workload: the FULL-size SD guidance step once + the render forward/backward (k = 13, reference
    regularisers on) on every 4th pixel of the 128x128 view -- 4096 rays in two 2048-ray chunks, large enough that torch's CPU
    kernels run at their full-size efficiency -- scaled by the measured ratio of marched samples (whole view / sample).
    A reported baseline, not the target."""
    from oracle import field_ref as fr
    from oracle import raymarch as orm
    from oracle import sd_ref
    # more threads than ~32 make torch's CPU kernels slower on these many-core hosts (measured: 128 threads -> 30x slower)
    torch.set_num_threads(min(32, os.cpu_count()))
    cores = torch.get_num_threads()
    pose = orbit_pose(1.25, 80.0, 170.0)
    focal = HW / (2 * math.tan(math.radians(20.0) / 2))
    ro, rd, sc = fr.get_rays_ref(pose, (focal, focal, HW / 2, HW / 2), HW, HW)
    ro, rd, sc = ro.numpy(), rd.numpy(), sc.numpy()
    field = fr.FieldRef(seed=0, table_scale=0.5)
    bits = sphere_bitfield_numpy(SPHERE_R)
    rng = np.random.default_rng(0)
    noises = rng.random(HW * HW, dtype=np.float32)
    aabb = np.array([-1, -1, -1, 1, 1, 1], np.float32)
    nears, fars = orm.near_far_from_aabb(ro, rd, aabb, 0.2)
    m_full = int(orm.march_rays_train(ro, rd, 1.0, bits, 1, 128, nears, fars, noises, 0.0, 512, align=-1)[4])      # whole view, march only
    sel = np.arange(0, HW * HW, 4)
    m_sample, t_render = 0, 0.0
    for chunk in np.array_split(sel, 2):
        t0 = time.time()
        out = fr.render_train_ref(field, ro[chunk], rd[chunk], bits, noises=noises[chunk], light_d=np.array([0, 0.6, 0.8], np.float32),
                                  bg_color=rng.random(3, dtype=np.float32), depth_scale=sc[chunk], max_steps=512, shading="albedo", lambda_smooth=1.0)
        (out["image"].sum() + out["loss_orient"] + out["loss_smooth"]).backward()
        t_render += time.time() - t0
        m_sample += int(out["total"])
    t_render_full = t_render * m_full / max(1, m_sample)
    unet = sd_ref.UNet2DConditionModel(sd_ref.sd20_unet_config()).eval()
    vae = sd_ref.AutoencoderKLEncoder(sd_ref.sd_vae_config()).eval()
    for p in list(unet.parameters()) + list(vae.parameters()):
        p.requires_grad_(False)
    g = torch.Generator().manual_seed(0)
    rgb = torch.rand(1, 3, HW, HW, generator=g).requires_grad_()
    t0 = time.time()
    sd_ref.sds_train_step_ref(unet, vae, torch.randn(2, 77, 1024, generator=g), rgb, 500, torch.randn(1, 4, 64, 64, generator=g),
                              torch.randn(1, 4, 64, 64, generator=g), guidance_scale=10.0)
    t_sd = time.time() - t0
    return {"value": round(1.0 / (t_render_full + t_sd), 5), "unit": UNIT, "cores": cores, "kind": "port", "extrapolated": True,
            "sample": f"full-size SD guidance step measured once ({t_sd:.1f} s) + render fwd/bwd (k=13) measured on every 4th pixel "
                      f"({len(sel)} of {HW * HW} rays, {m_sample} of {m_full} samples: {t_render:.1f} s) and scaled by the sample ratio to the whole "
                      f"view ({t_render_full:.1f} s); oracle PORT of the reference algorithm, not the reference's own code (tcnn / diffusers absent)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb = cpu_baseline(args)
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": 1, "warmup": 0,
            "ms_per_step": round(1000.0 / cb["value"], 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32",
            "data": "synthetic", "config": {"workload": WORKLOAD, "note": "reference algorithm (oracle port: C ray-march + PyTorch fp32 field/U-Net/VAE) on host CPU cores; "
                                            "the reference's own CUDA/tcnn/diffusers path cannot run without its third-party packages and SD weights"},
            "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--render-split", default="rays", choices=["rays", "views"],
                    help="N > 1: 'rays' = ray-parallel render (balanced, default), 'views' = round-1 view-parallel render (A/B)")
    ap.add_argument("--defer-backward", action="store_true",
                    help="StableDiffusion(defer_backward=True): the SDS gradient joins the regularisers in ONE render backward (A/B; off = reference order)")
    ap.add_argument("--timeline-out", default=None, help="after the timed regions, also write the per-rank phase timeline of a few extra steps to this file")
    ap.add_argument("--timeline", action="store_true",
                    help="print a per-rank CUDA-event table of the step phases instead of the bench line (for profiles/)")
    ap.add_argument("--launch-list", action="store_true",
                    help="profiling aid: warm up, run --steps steps of the same step function and exit (use under "
                         "`ncu --metrics gpu__time_duration.sum`; numbers printed under a profiler are never bench values)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last one computed (render outputs, loss, parameter gradients) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.timeline or args.launch_list):
        ap.error("--dump-outputs writes the outputs of the timed steps: not with --impl reference, --timeline or --launch-list")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
