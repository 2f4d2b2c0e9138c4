#!/usr/bin/env python
"""bench.py -- SDS iterations/sec at 512x512 with an 8-view batch (BASELINE.json metric).

One "step" = one full score-distillation iteration over a batch of synthetic views:
PBR Monte-Carlo render (200+128 rays/pixel, BVH occlusion) -> VAE encode (with grad) -> ControlNet + UNet
for the 3 CFG branches -> CSD gradient -> backward through the VAE and the shader into the hash grid /
MLP -> (all-reduce when sharded) -> Adam.  SD-2.1-base / ControlNet / VAE topology with seeded random
weights (no checkpoints offline), fp16 storage + fp32 accumulation like the reference default.

    python bench.py --gpus N --steps K --warmup W            our arm (torchrun for N > 1)
    python bench.py --impl reference ...                     the reference algorithm (CPU oracle port) on host cores
    python bench.py --impl torch-cuda ...                    the same algorithm through stock PyTorch CUDA ops on this GPU
    python bench.py --views 4 | --res 1024 --dtype bf16 | --views 64 (8 GPUs) | --shading splitsum    BASELINE configs 2 / 3 / 4 / a5
    python bench.py --gpus 2 --check                         + gradient identity of the sharded step vs one process
    python bench.py --dump-outputs DIR                       + what the last timed step computed, as DIR/<name>.npy
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DENSE_TFLOP_PER_VIEW = 5.50    # SURVEY.md section 8(d): UNet 2.41 + ControlNet 0.86 + VAE fwd 1.12 + VAE dgrad 1.12
UNET_CN_TFLOP_PER_VIEW = 3.27


def burst_tflops():
    """burst bf16/fp16 tensor peak for a kernel timed alone (MEASURED_PEAKS.json `bf16_tflops`), else the recipe's fallback"""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)["bf16_tflops"], "measured"
    except Exception:
        return 1650.0, "fallback"


def kernel_roofline(dtype):
    """Roofline of the dominant tensor kernel, timed ALONE with CUDA events on the launching stream: the CTA-pair
    implicit-GEMM convolution on the UNet's 16x16-latent layer of the 8-view batch (conv3x3 24x16x16, 1280 -> 1280).
    Algorithmic flops per launch = 2 * 6144 * 1280 * 11520; `traffic` is the DRAM read+write of the same launch from the
    committed ncu --set full capture (profiles/r01c_launches_summary.md: 45.3 + 1.3 MB; algorithmic 29.5 MB weights +
    15.7 MB input + 15.7 MB output, the nine taps re-read L2 only)."""
    import torch
    from dreammat_b200 import dense_ops as D
    x = torch.randn(24, 16, 16, 1280, device="cuda").to(dtype)
    w = (torch.randn(1280, 9 * 1280, device="cuda") * 0.01).to(dtype)
    for _ in range(5):
        D.conv2d(x, w, 3)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 50
    e0.record()
    for _ in range(n):
        D.conv2d(x, w, 3)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    flops = 2.0 * 24 * 256 * 1280 * 1280 * 9
    peak, src = burst_tflops()
    ach = flops / (ms * 1e-3) / 1e12
    return {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": 46.6e6,
            "kernel": "tc_gemm_pair_kernel<256> conv3x3 24x16x16 1280->1280 (timed alone, %d launches, %.1f us each)" % (n, ms * 1e3),
            "peak_source": src + " burst bf16", "traffic_source": "ncu --set full, profiles/r01c_launches_summary.md"}


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return p["hbm_gbs"], p.get("bf16_tflops_sustained", p["bf16_tflops"]), "measured"
    except Exception:
        return 6650.0, 1400.0, "fallback"


class ClockSampler:
    def __init__(self, dev):
        self.p = None
        try:
            self.p = subprocess.Popen(
                ["nvidia-smi", "-i", str(dev), "--query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                 "clocks_event_reasons.sw_power_cap", "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill()
            out = ""
        sm, mx, reasons = [], 0, set()
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx = max(mx, float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ our arm


def build_system(device, res, n_faces, env_hw, seed, dtype, shading="mc"):
    import torch
    from dreammat_b200 import weights as Wt
    from dreammat_b200.guidance import PromptProcessorOutput, StableDiffusionLightGuidance
    from dreammat_b200.scene import DataConfig, FixCameraSet, procedural_mesh, synthetic_envmap
    from dreammat_b200.system import DreamMat, DreamMatMaterial, DreamMatMesh, RaytraceRender
    mesh = procedural_mesh(n_faces, 0.8, seed)
    geo = DreamMatMesh({"shape_init": "procedural", "shape_init_params": 0.8}, device, mesh=mesh, seed=seed)
    envs = [synthetic_envmap(env_hw[0], env_hw[1], seed + i) for i in range(5)]
    fg = None
    if shading == "splitsum":
        # the reference's load/lights/bsdf_256_256.bin is not on the box: an analytic stand-in with the same layout / ranges
        u = (torch.arange(256, dtype=torch.float32) + 0.5) / 256
        ndv, rough = torch.meshgrid(u, u, indexing="xy")
        fg = torch.stack([(1 - rough) * (0.3 + 0.7 * ndv), 0.04 + 0.5 * (1 - ndv) ** 5 * (1 - rough)], -1).reshape(1, 256, 256, 2)
    mat = DreamMatMaterial({"environment_texture": "synthetic", "environment_scale": 2.0, "use_bump": False,
                            "use_raytracing": shading == "mc", "diffuse_sample_num": 200, "specular_sample_num": 128}, device, envs,
                           fg_lut=fg)
    ren = RaytraceRender({"context_type": "cuda"}, geo, mat, None, device)
    ucfg, vcfg = Wt.UNetConfig(), Wt.VAEConfig()
    gcfg = dict(use_controlnet=True, control_types=["light"], cond_scale=1.05, uncond_scale=[0, -1.0, -0.5, 2000],
                null_scale=[0, 0.0, -0.5, 2000], noise_scale=0.0, min_step_percent=[500, 0.2, 0.02, 501],
                max_step_percent=[500, 0.8, 0.5, 501], control_anneal_start_step=700, condition_scales=[1.0],
                condition_scales_anneal=[0.8])     # configs/dreammat.yaml:54-71
    wu, wc, wv = Wt.random_unet(ucfg, device, 10), Wt.random_controlnet(ucfg, device, 11), Wt.random_vae(vcfg, device, 12)
    guid = StableDiffusionLightGuidance(gcfg, ucfg, vcfg, wu, wc, wv, device, dtype)
    del wu, wc, wv
    torch.cuda.empty_cache()
    g = torch.Generator().manual_seed(seed + 100)
    D = ucfg.cross_attention_dim
    vd, uvd, null = torch.randn(4, 77, D, generator=g), torch.randn(4, 77, D, generator=g), torch.randn(1, 77, D, generator=g)
    pu = PromptProcessorOutput(vd[:1].to(device), uvd[:1].to(device), null.to(device), vd.to(device), uvd.to(device))
    sysm = DreamMat(None, geo, mat, ren, guid, pu, device)
    cams = FixCameraSet(DataConfig(batch_size=1, width=res, height=res), torch.Generator().manual_seed(seed))
    return sysm, cams


FP32_LANES_PER_SM = 128


def run_ours(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = f"cuda:{local}"
    # the step's device-side draws (jitter, MC samples, timesteps, noise, VAE posterior) come from the default CUDA
    # generator, which PyTorch otherwise seeds at random per process: fixed here so a run's inputs repeat; one stream per rank
    torch.cuda.manual_seed(rank)
    if world > 1:
        # NCCL_DEBUG is left exactly as the launcher set it (its banner goes to stderr with everything else, see main())
        dist.init_process_group("nccl", device_id=torch.device(device))
    from dreammat_b200 import _cabi
    _cabi.check(_cabi.lib().dm_device_check(local), "dm_device_check")   # fails loudly without the sm_100a library
    if args.no_pdl:
        _cabi.lib().dm_tune(b"pdl", 0)
    dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float16
    V = args.views
    assert V % world == 0, "global view batch must divide over the ranks"
    Vl = V // world
    sysm, cams = build_system(device, args.res, args.faces, (args.env_h, args.env_w), 0, dtype, args.shading)
    sysm.world_size, sysm.rank = world, rank
    sysm.balance_pixels = not args.no_balance
    res = args.res
    gres = 512 if sysm.resize_to_vae else res                    # renders that are not 512^2 are resized before the VAE
    # N1: the pre-rendered condition maps (depth fp32, normal / 6 light maps uint8; data/uncond.py:532-582) live on the device
    # -- 3.3 GB for 128 views x 5 envs at 512^2 -- and are gathered + de-quantised inside the ControlNet graph by (view, env) id
    from dreammat_b200.parallel import global_pixel_count, quiesce_host_gc, shard_slice
    from dreammat_b200.scene import FixViewMaps
    n_fix, n_env = cams.cfg.fix_view_num, 5
    maps = FixViewMaps.synthetic(n_fix, n_env, gres, gres, device=device, seed=7)
    sysm.guidance.maps = maps
    if not args.no_graphs:
        sysm.guidance.enable_graphs(Vl, gres, gres, maps=maps)    # dense section as three captured CUDA graphs
    # a1: per-view camera tensors (fixed set) on the host (pinned: what the data module hands over each step) and on the
    # device; G-buffers produced once per fixed view (a2: costs 0 ms inside the timed step by construction -- fixed mesh, fixed cameras)
    all_ids = torch.arange(n_fix)
    cam_keys = ("mvp_mtx", "w2c", "elevation", "azimuth", "camera_distances")
    cam_host = {k: [] for k in cam_keys}
    for v0 in range(0, n_fix, 16):
        c = cams.cameras(all_ids[v0:v0 + 16])
        for j in range(c["mvp_mtx"].shape[0]):
            one = {k: (val[j:j + 1].to(device) if torch.is_tensor(val) else val) for k, val in c.items()}
            sysm.renderer.gbuffer(one["rays_o"], one["rays_d"], one["mvp_mtx"], one["w2c"], v0 + j)
        for k in cam_keys:
            cam_host[k].append(c[k].float())
    cam_host = {k: torch.cat(v, 0).pin_memory() for k, v in cam_host.items()}
    cam_dev = {k: v.to(device) for k, v in cam_host.items()}
    # per-view device rows: building a batch is a torch.cat of resident tensors (indexing a CUDA tensor with a CPU index tensor
    # would issue a synchronous H2D copy of the indices per key -- measured: 5 ms / step of CPU stall at 8 GPUs)
    cam_rows = [{k: cam_dev[k][v:v + 1] for k in cam_keys} for v in range(n_fix)]
    pn = [sysm.renderer._cache[i]["pn"] for i in range(n_fix)]
    sysm.prepare_balanced(range(n_fix))          # one MIN all-reduce: all ranks agree on balanced shading
    gsel = torch.Generator().manual_seed(1234)   # shared by all ranks -> the global batch is a function of the step
    stage = {k: torch.empty(Vl, *v.shape[1:], device=device) for k, v in cam_host.items()}
    def make_batch(mode):
        """mode: 'device' (ids + cameras already resident) | 'e2e' (this step's ids + camera tensors come from pinned host memory)"""
        view_id, env_id = cams.collate(gsel, V)
        tot_pn = global_pixel_count(pn, view_id)
        mine = shard_slice(V, rank, world)
        vid, eid = view_id[mine], env_id[mine]
        b = {"view_id": vid, "env_id": eid, "height": res, "width": res, "global_view_id": view_id, "global_env_id": env_id}
        h2d = 0
        if mode == "device":
            for k in cam_keys:
                b[k] = torch.cat([cam_rows[int(v)][k] for v in vid], 0)
        else:
            for k in cam_keys:
                for i, v in enumerate(vid):
                    stage[k][i].copy_(cam_host[k][int(v)], non_blocking=True)
                b[k] = stage[k]
                h2d += stage[k].numel() * 4
            h2d += 2 * Vl * 4                                    # the (view, env) ids the graph reads (graph_step copies them)
        return b, tot_pn, h2d

    class _Rays:   # the G-buffer cache is keyed by view id; rays are not needed again
        def __getitem__(self, i):
            return None

    h2d_seen = {}

    def step(mode="device"):
        b, tot_pn, h2d = make_batch(mode)
        h2d_seen[mode] = h2d
        b["rays_o"] = b["rays_d"] = _Rays()
        out = sysm.training_step_fused(b, global_views=V, total_pn_global=tot_pn)
        if mode != "device":
            return float(out["loss"])      # D2H read of the step's result
        return out

    def timed(n_warm, n_steps, mode):
        for _ in range(n_warm):
            step(mode)
        if not args.no_gc_freeze:
            quiesce_host_gc()      # what the plugin does in on_fit_start: no 30-40 ms full-GC pause on any rank inside a step
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        gr = sysm.guidance.graphs
        l0 = _cabi.lib().dm_launch_count() + (gr.replayed_launches if gr else 0)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(n_steps + 1)]
        ev[0].record()
        host, seg0 = [time.perf_counter()], torch.cuda.memory_stats().get("num_device_alloc", 0)
        for i in range(n_steps):
            if i + 1 < n_steps:
                step(mode)
            else:
                last = step(mode)      # only the final result is held: earlier steps free theirs as soon as they return
            ev[i + 1].record()
            host.append(time.perf_counter())
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = torch.tensor([ev[0].elapsed_time(ev[-1])], device=device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        l1 = _cabi.lib().dm_launch_count() + (gr.replayed_launches if gr else 0)
        raw = [ev[i].elapsed_time(ev[i + 1]) for i in range(n_steps)]
        worst = max(range(n_steps), key=lambda i: raw[i])
        per = sorted(raw)
        spread = {"median_ms": per[len(per) // 2], "min_ms": per[0], "max_ms": per[-1],
                  "steps_over_1p5x_median": sum(1 for x in per if x > 1.5 * per[len(per) // 2]),
                  "slowest_step": {"index": worst, "host_ms": (host[worst + 1] - host[worst]) * 1e3,
                                   "cudaMalloc_calls_in_region": torch.cuda.memory_stats().get("num_device_alloc", 0) - seg0}}
        return float(ms) / n_steps, (l1 - l0) // n_steps, spread, last

    sampler = ClockSampler(local) if rank == 0 else None
    ms_step, launches, spread, last = timed(args.warmup, args.steps, "device")
    if args.dump_outputs and rank == 0:
        # before the profiled and e2e steps below: they overwrite the captured graphs' canvas that comp_rgb views
        dump_outputs(args.dump_outputs, last)
    del last
    # section split (one extra profiled step, outside the timed region)
    sec = sysm.profile_step(lambda: make_batch("device")[:2], V) if hasattr(sysm, "profile_step") else {}
    ms_e2e, _, spread_e2e, _ = timed(max(1, args.warmup // 2), args.steps, "e2e")
    parity = gradient_identity_check(sysm, make_batch, cam_dev, V, world, rank, device) if args.check else None
    clocks = sampler.stop() if sampler else None
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    hbm, tf, src = peaks()
    value = 1000.0 / ms_step
    weak = args.views != 8 and args.views == 8 * world           # BASELINE config 4: 8 views per GPU
    cfg_name = ("north-star" if (V == 8 and res == 512 and args.shading == "mc") else
                "config 2 (run_examples.sh: 4 views / iteration)" if (V == 4 and res == 512) else
                "config 3 (1024^2 render)" if res == 1024 else
                "config 4 (8 views per GPU, weak scaling)" if weak else "custom")
    out = {"metric": "SDS iters/sec at 512x512, 8-view batch", "value": value, "unit": "it/s", "n_gpus": world,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
           "scaling": "weak" if weak else "strong", "vs_baseline": None, "dtype": "f16" if dtype == torch.float16 else "bf16",
           "data": "synthetic (procedural %d-face mesh, synthetic HDR env maps and uint8 condition maps, seeded random SD-2.1-base/ControlNet/VAE weights)" % args.faces,
           "config": {"workload": "%s: %dx%d render, %d-view batch (%d/GPU), %s, 5 env maps, 128 fixed views" % (
                          cfg_name, res, res, V, Vl, "200+128 MC rays/px" if args.shading == "mc" else "split-sum shading"),
                      "views": V, "resolution": res, "shading": args.shading,
                      "parallelism": "dp%d (views sharded; shading pixels balanced over ranks by 2 small all-to-alls; 1 all-reduce of 50.4 MB grads)" % world,
                      "l2": "working set (2.5 GB weights + activations) exceeds the 126 MB L2 every step",
                      "g_buffer": "rasterisation (row a2) is hoisted out of the step: fixed mesh + 128 fixed cameras -> per-view G-buffer cache built before timing",
                      "condition_maps": "resident on the device as uint8 (%.2f GB), gathered by (view, env) id inside the ControlNet graph" % (maps.nbytes / 1e9)},
           "step_time_spread": spread, "clocks": clocks, "gpu_launches": int(launches),
           "e2e": {"value": 1000.0 / ms_e2e, "unit": "it/s", "h2d_bytes_per_step": int(h2d_seen.get("e2e", 0)),
                   "d2h_bytes_per_step": 4, "step_time_spread": spread_e2e,
                   "note": "per step: this batch's camera tensors + (view, env) ids from pinned host memory, loss read back; the "
                           "condition maps are a device-resident dataset (N1), like the weights"}}
    if parity is not None:
        out["parity_check"] = parity
    t_dense = sec.get("dense_ms")
    if t_dense:
        ach = DENSE_TFLOP_PER_VIEW * Vl / (t_dense / 1000.0)
        out["roofline"] = {"bound": "tensor", "achieved": ach, "peak": tf, "unit": "TFLOP/s", "frac": ach / tf,
                           "traffic": None, "kernel": "tc_gemm_pair_kernel + tc_gemm_kernel + attention_kernel over the dense section",
                           "peak_source": src + " sustained bf16",
                           "note": "section-level: algorithmic flops of ALL dense kernels / CUDA-event time of the section inside the timed "
                                   "step (GroupNorm, softmax etc. included); the dominant tensor kernel alone is in roofline_kernel, the "
                                   "shader in roofline_shading"}
        out["sections_ms"] = sec
        try:
            out["roofline_kernel"] = kernel_roofline(dtype)
        except Exception as ex:  # noqa: BLE001 -- the section-level roofline above stands on its own
            out["roofline_kernel"] = {"error": str(ex)[:200]}
        t_r = sec.get("render_fwd_ms")
        if t_r:
            pn_step = float(sec.get("pn_local", 0))
            sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
            fp32_peak = 148 * FP32_LANES_PER_SM * 2 * sm_mhz * 1e6
            if args.shading == "mc":
                # NOT HBM-bound (BVH traversal + FP32 ALU).  SURVEY 8d: rays/s, the FP32-lane fraction and the HBM fraction
                # from the byte formula (200 B per covered pixel + one 16 B texel per unoccluded sample; upper bound: every sample)
                byts = pn_step * (200.0 + 16.0 * 328)
                instr = MC_THREAD_INSTR_PER_RAY * pn_step * 328
                out["roofline_shading"] = {"bound": "hbm", "achieved": byts / (t_r * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                                           "frac": byts / (t_r * 1e-3) / 1e9 / hbm, "traffic": None,
                                           "rays_per_s": pn_step * 328 / (t_r * 1e-3), "covered_pixels": pn_step,
                                           "fp32_frac": 2.0 * instr / (t_r * 1e-3) / fp32_peak,
                                           "fp32_note": "lane-level instructions of the shader (ncu smsp__thread_inst_executed, %d per ray, "
                                                        "profiles/r02_shade_frontier.md) x 2 flop / (148 SM x 128 lanes x 2 x %.0f MHz)" % (MC_THREAD_INSTR_PER_RAY, sm_mhz),
                                           "note": "latency/issue-bound BVH any-hit traversal (shared-origin frontier); bytes are an upper bound (every sample unoccluded)"}
            else:
                byts = pn_step * 124.0          # forward only inside render_fwd (76 B more in the backward section)
                out["roofline_shading"] = {"bound": "hbm", "achieved": None, "peak": hbm, "unit": "GB/s", "frac": None, "traffic": None,
                                           "covered_pixels": pn_step,
                                           "note": "render_fwd also holds 2 hash-grid evaluations, jitter, scatter, antialias; the split-sum kernel alone is timed below"}
                out["roofline_shading"].update(splitsum_kernel_roofline(sysm, hbm))
        out["unet_controlnet_ms_per_step"] = sec.get("unet_cn_ms")
    if world == 1 and not args.no_gpu_baseline:
        try:
            out["gpu_baseline"] = torch_cuda_baseline(args, sysm, pn, dtype, sec)
        except Exception as ex:  # noqa: BLE001
            out["gpu_baseline"] = {"error": str(ex)[:300]}
    if world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(args, sum(pn) / len(pn))
    emit(out)
    if world > 1:
        dist.destroy_process_group()


MC_THREAD_INSTR_PER_RAY = 2290     # measured: ncu thread-level instructions of shade_mc_kernel / rays (profiles/r02_shade_frontier.md)


def splitsum_kernel_roofline(sysm, hbm):
    """dm_shade_splitsum_fwd + dm_shade_bwd timed alone on one cached view (CUDA events on the launching stream):
    algorithmic bytes = 124 B (fwd) + 76 B (bwd) per covered pixel (SURVEY.md section 8d)."""
    import ctypes as C
    import torch
    from dreammat_b200._cabi import check, lib, ptr, stream_ptr
    mat, ren = sysm.material, sysm.renderer
    ge = max(ren._cache.values(), key=lambda g: g["pn"])
    n = ge["pn"]
    dev = ge["pts"].device
    f, fj = torch.randn(n, 5, device=dev), torch.randn(n, 5, device=dev)
    color, jac, reg = torch.empty(n, 3, device=dev), torch.empty(n, 9, device=dev), torch.zeros(2, device=dev)
    dcol, df, dfj = torch.randn(n, 3, device=dev), torch.empty(n, 5, device=dev), torch.empty(n, 5, device=dev)
    dcube, mips = mat.envlight[0]
    st = stream_ptr()

    def fwd():
        check(lib().dm_shade_splitsum_fwd(C.byref(mat.ss_cfg), ptr(mat.FG_LUT), mat.FG_LUT.shape[0], ptr(dcube), dcube.shape[1], mat._mip_ptrs[0],
                                          len(mips), mips[0].shape[1], ptr(ge["nrm"]), ptr(ge["vd"]), ptr(f), ptr(fj), n, ptr(color), ptr(jac),
                                          ptr(reg), *([None] * 7), st), "dm_shade_splitsum_fwd")

    def bwd():
        check(lib().dm_shade_bwd(C.byref(mat.ss_cfg), ptr(f), ptr(fj), ptr(dcol), ptr(jac), 1e-6, 1e-6, n, ptr(df), ptr(dfj), st), "dm_shade_bwd")
    res = {}
    for name, fn, byts in (("fwd", fwd, 124.0), ("bwd", bwd, 76.0)):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            fn()
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) / 20 * 1e3
        res[name] = {"us": us, "GBps": byts * n / (us * 1e-6) / 1e9}
    ach = 200.0 * n / ((res["fwd"]["us"] + res["bwd"]["us"]) * 1e-6) / 1e9
    return {"achieved": ach, "frac": ach / hbm, "kernel": "shade_splitsum_kernel + shade_bwd_kernel timed alone on one view (%d covered px; "
            "fwd %.1f us = %.0f GB/s, bwd %.1f us = %.0f GB/s)" % (n, res["fwd"]["us"], res["fwd"]["GBps"], res["bwd"]["us"], res["bwd"]["GBps"]),
            "algorithmic_bytes_per_pixel": 200}


def gradient_identity_check(sysm, make_batch, cam_dev, V, world, rank, device):
    """--check: one step with explicit randomness (identical on every rank) computed (a) sharded over the ranks as in the
    timed loop -- views split, pixel-balanced shading if enabled, gradient all-reduce -- and (b) by rank 0 alone over the whole
    global batch; the flat parameter gradients must agree (the sum over views is the only cross-view coupling).  Done twice:
    in the timed precision (fp16: two evaluations batch the networks differently, so they agree to the fp16 run-to-run
    noise, which is measured alongside) and with the dense half in the fp32 high-precision mode (a crisp identity)."""
    import torch
    import torch.distributed as dist
    from dreammat_b200 import weights as Wt
    from dreammat_b200.guidance import StableDiffusionLightGuidance
    geo, ren = sysm.geometry, sysm.renderer
    b, tot_pn, _ = make_batch("device")
    gvid = [int(v) for v in b["global_view_id"]]
    g = torch.Generator().manual_seed(99)
    rng = {k: [] for k in ("rand_ang", "normal_eps", "rand_d", "rand_s")}
    for v in gvid:
        n = ren._cache[v]["pn"]
        rng["rand_ang"].append(torch.rand(n, generator=g)); rng["normal_eps"].append(torch.randn(n, generator=g) * 0.05)
        rng["rand_d"].append(torch.rand(n, generator=g)); rng["rand_s"].append(torch.rand(n, generator=g))
    h = (512 if sysm.resize_to_vae else b["height"]) // 8
    rng.update(t=torch.randint(20, 981, (V,), generator=g), noise=torch.randn(V, 4, h, h, generator=g), vae_eps=torch.randn(V, 4, h, h, generator=g),
               indexed_by="global_view")

    class _Rays:
        def __getitem__(self, i):
            return None
    state = (geo.params.clone(), sysm.m.clone(), sysm.v.clone(), sysm.global_step)
    maps = sysm.guidance.maps

    def restore():
        geo.params.copy_(state[0]); sysm.m.copy_(state[1]); sysm.v.copy_(state[2]); sysm.global_step = state[3]

    def one_precision():
        # (a) sharded
        b["rays_o"] = b["rays_d"] = _Rays()
        b["condition_map"] = maps.condition_map(b["view_id"], b["env_id"])
        sysm.training_step_fused(b, global_views=V, total_pn_global=tot_pn, rng=rng, apply_optimizer=False)
        g_sharded = geo.grads.clone()
        restore()
        # (b) rank 0 alone, whole global batch (no collective inside: world_size is 1 for it)
        err = floor = None
        if rank == 0:
            ws, bal = sysm.world_size, sysm.balance_pixels
            sysm.world_size, sysm.balance_pixels = 1, False
            try:
                vid, eid = b["global_view_id"], b["global_env_id"]
                full = {"view_id": vid, "env_id": eid, "height": b["height"], "width": b["width"], "rays_o": _Rays(), "rays_d": _Rays()}
                for k in ("mvp_mtx", "w2c", "elevation", "azimuth", "camera_distances"):
                    full[k] = cam_dev[k][vid.to(device)]
                full["condition_map"] = maps.condition_map(vid, eid)
                sysm.training_step_fused(full, global_views=V, total_pn_global=tot_pn, rng=rng, apply_optimizer=False)
                g_single = geo.grads.clone()
                err = float((g_sharded.double() - g_single.double()).norm() / (g_single.double().norm() + 1e-30))
                # the same single-process evaluation once more: its own run-to-run noise (fp32 atomics in split-K / GroupNorm
                # statistics / hash-grid scatter) is the floor the sharded result has to be read against
                restore()
                sysm.training_step_fused(full, global_views=V, total_pn_global=tot_pn, rng=rng, apply_optimizer=False)
                floor = float((geo.grads.double() - g_single.double()).norm() / (g_single.double().norm() + 1e-30))
            finally:
                sysm.world_size, sysm.balance_pixels = ws, bal
            restore()
        if world > 1:
            dist.barrier()
        return err, floor
    err16, floor16 = one_precision()
    # fp32 high-precision dense half (same seeded weights, half_precision_weights=false)
    guid16 = sysm.guidance
    ucfg, vcfg = Wt.UNetConfig(), Wt.VAEConfig()
    gcfg = dict(guid16.cfg.__dict__, half_precision_weights=False)
    guid32 = StableDiffusionLightGuidance(gcfg, ucfg, vcfg, Wt.random_unet(ucfg, device, 10), Wt.random_controlnet(ucfg, device, 11),
                                          Wt.random_vae(vcfg, device, 12), device)
    guid32.maps = maps
    sysm.guidance = guid32
    try:
        err32, floor32 = one_precision()
    finally:
        sysm.guidance = guid16
        del guid32
        torch.cuda.empty_cache()
    return {"grad_rel_err": err16, "single_process_run_to_run": floor16, "grad_rel_err_fp32_mode": err32, "single_process_run_to_run_fp32_mode": floor32,
            "what": "flat [grid | W1 | W2] gradient of one step: %d ranks (views sharded, balanced shading %s, all-reduce) vs rank 0 alone on the "
                    "same global batch and randomness; fp16 (the timed precision) and fp32 high-precision dense half" % (world, "on" if sysm.balance_pixels else "off")}


# ------------------------------------------------------------------------------------------------ stock PyTorch CUDA arm


def torch_cuda_baseline(args, sysm, pn, dtype, sec):
    """The "same box" bar (SURVEY.md section 8d, BASELINE.md section 4): the reference's algorithm through STOCK PyTorch CUDA
    ops on this GPU -- cuDNN / cuBLAS / SDPA for the dense half at the reference's precision (fp16 weights and activations),
    unfused [pn,328,.] tensor ops with autograd for the Monte-Carlo shading (oracle/render.py + oracle/sd.py are plain torch
    and run on any device; here they are the thing being TIMED, never the product path).  The ray tracer and the hash grid
    are native extensions in the reference too (_raytracing, tiny-cuda-nn): this leg uses our dm_bvh_trace / hash-grid kernels
    for them, so the comparison isolates shading + dense kernels.  Times are CUDA events after warm-up."""
    import torch
    from dreammat_b200 import render_ops as R
    from dreammat_b200 import weights as Wt
    from oracle import render as OR
    from oracle import sd as OS
    dev = sysm.device
    V = args.views
    ucfg, vcfg = OS.UNetConfig(), OS.VAEConfig()
    tdt = dtype

    def evt(fn, reps=2, warm=1):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps
    out = {"what": "oracle/{sd,render}.py (plain torch) on cuda:0, %s dense half, fp32 shading with autograd" % ("fp16" if tdt == torch.float16 else "bf16"),
           "views": V}
    g = torch.Generator(device=dev).manual_seed(0)
    # ---- dense half
    wv = {k: v.to(tdt) for k, v in Wt.random_vae(Wt.VAEConfig(), dev, 12).items()}
    x = (torch.rand(V, 3, 512, 512, device=dev, generator=g) * 2 - 1).to(tdt).requires_grad_(True)
    eps = torch.randn(V, 4, 64, 64, device=dev, generator=g).to(tdt)
    dz = torch.randn(V, 4, 64, 64, device=dev, generator=g).to(tdt)

    def vae():
        x.grad = None
        z = OS.vae_sample(OS.vae_encode_moments(wv, vcfg, x), eps, vcfg.scaling_factor)
        z.backward(dz)
    out["vae_fwd_bwd_ms"] = evt(vae)
    del wv
    wu = {k: v.to(tdt) for k, v in Wt.random_unet(Wt.UNetConfig(), dev, 10).items()}
    wc = {k: v.to(tdt) for k, v in Wt.random_controlnet(Wt.UNetConfig(), dev, 11).items()}
    z3 = torch.randn(3 * V, 4, 64, 64, device=dev, generator=g).to(tdt)
    t3 = torch.full((3 * V,), 500, device=dev, dtype=torch.long)
    ctx = torch.randn(3 * V, 77, 1024, device=dev, generator=g).to(tdt)
    cond = torch.rand(V, 22, 512, 512, device=dev, generator=g).to(tdt)

    def unet_cn():
        with torch.no_grad():
            d, m = OS.controlnet_forward(wc, ucfg, z3, t3, ctx, cond, 1.0)
            OS.unet_forward(wu, ucfg, z3, t3, ctx, d, m)
    import oracle.sd as _osd
    _te = _osd.timestep_embedding
    _osd.timestep_embedding = lambda t, dim: _te(t.cpu(), dim).to(device=t.device, dtype=tdt)   # the oracle builds this table on the CPU
    try:
        out["unet_controlnet_ms"] = evt(unet_cn)
    finally:
        _osd.timestep_embedding = _te
    del wu, wc
    torch.cuda.empty_cache()
    out["dense_ms"] = out["vae_fwd_bwd_ms"] + out["unet_controlnet_ms"]
    # ---- Monte-Carlo shading of the batch's views (forward + backward through autograd), one view at a time
    mat, ren = sysm.material, sysm.renderer
    if mat.cfg.use_raytracing:
        views = sorted(ren._cache)[:2]        # two views (the [pn,328,.] autograd graph of one view is tens of GB); reported per pixel
        env = mat.light[0][..., :3].contiguous()

        def trace_fn(o, d):
            t, tri, _ = ren.ray_tracer.trace(o, d)
            return tri >= 0

        def shade():
            for v in views:
                ge = ren._cache[v]
                n = ge["pn"]
                f = torch.randn(n, 5, device=dev, generator=g, requires_grad=True)
                fj = torch.randn(n, 5, device=dev, generator=g, requires_grad=True)
                al, me, ro, reg = OR.material_params(f, fj)
                o = OR.shade_raytracing(ge["pts"], ge["nrm"], ge["vd"], env, me, ro, al, torch.rand(n, 1, 1, device=dev, generator=g),
                                        torch.rand(n, 1, 1, device=dev, generator=g), trace_fn)
                (o["color"].sum() + reg).backward()
        out["shading_fwd_bwd_ms"] = evt(shade, reps=1, warm=1)
        out["shading_pixels"] = int(sum(ren._cache[v]["pn"] for v in views))
        ours_shade = (sec.get("render_fwd_ms") or 0) + (sec.get("render_bwd_adam_ms") or 0)
        if ours_shade:
            px_ours = float(sec.get("pn_local", 0)) or 1.0
            out["ours_over_stock"] = {"dense": out["dense_ms"] / sec["dense_ms"] if sec.get("dense_ms") else None,
                                      "shading_per_pixel": (out["shading_fwd_bwd_ms"] / out["shading_pixels"]) / (ours_shade / px_ours),
                                      "note": "> 1 means our kernels are faster; our shading figure also contains hash grid, canvas, antialias, all-reduce, Adam"}
    elif sec.get("dense_ms"):
        out["ours_over_stock"] = {"dense": out["dense_ms"] / sec["dense_ms"]}
    return out


def run_torch_cuda(args):
    """--impl torch-cuda: the stock-PyTorch-CUDA leg on its own (one JSON line)."""
    import torch
    torch.cuda.set_device(0)
    dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float16
    sysm, cams = build_system("cuda:0", args.res, args.faces, (args.env_h, args.env_w), 0, dtype, args.shading)
    for v0 in range(0, args.views):
        c = cams.cameras(torch.tensor([v0]))
        sysm.renderer.gbuffer(c["rays_o"].cuda(), c["rays_d"].cuda(), c["mvp_mtx"].cuda(), c["w2c"].cuda(), v0)
    pn = [sysm.renderer._cache[i]["pn"] for i in range(args.views)]
    b = torch_cuda_baseline(args, sysm, pn, dtype, {})
    ms = b["dense_ms"] + b.get("shading_fwd_bwd_ms", 0.0)
    emit({"impl": "torch-cuda", "metric": "SDS iters/sec at 512x512, 8-view batch", "value": 1000.0 / ms, "unit": "it/s", "n_gpus": 1,
          "ms_per_step": ms, "higher_is_better": True, "dtype": args.dtype, "data": "synthetic",
          "config": {"workload": "stock PyTorch CUDA ops (cuDNN/cuBLAS/SDPA + unfused torch shading), %d views, %dx%d" % (args.views, args.res, args.res)},
          "sections_ms": b})


# ------------------------------------------------------------------------------------------------ CPU arm


def _cpu_sample(state):
    """One bounded sample of the reference algorithm on host cores (oracle port), at the REAL per-unit sizes:
    (a) ControlNet+UNet forward for ONE VIEW's three CFG branches (batch 3, the shape of the reference's call per view) at 64x64
        latents (22-channel condition at 512x512),
    (b) VAE encode forward + input-gradient backward of ONE 512x512 image,
    (c) MC shading (200+128 rays/px) + hash-grid forward/backward of ONE 128x128 render.  Returns seconds (a, b, c)."""
    import torch
    from oracle import render as OR
    from oracle import sd as OS
    ucfg, vcfg, wu, wc, wv, sc, grid, W1, W2, meta = state
    g = torch.Generator().manual_seed(0)
    t0 = time.perf_counter()
    with torch.no_grad():
        z = torch.randn(3, 4, 64, 64, generator=g); t = torch.tensor([500] * 3); ctx = torch.randn(3, 77, 1024, generator=g)
        cond = torch.rand(1, 22, 512, 512, generator=g)
        d, m = OS.controlnet_forward(wc, ucfg, z, t, ctx, cond)
        OS.unet_forward(wu, ucfg, z, t, ctx, d, m)
    t1 = time.perf_counter()
    x = torch.rand(1, 3, 512, 512, generator=g, requires_grad=True)
    mom = OS.vae_encode_moments(wv, vcfg, x)
    mom.square().sum().backward()
    t2 = time.perf_counter()
    gp = grid.clone().requires_grad_(True)
    f = OR.geometry_forward(sc["pts"], gp, W1, W2, meta)
    fj = OR.geometry_forward(OR.jitter_positions(sc["pts"], sc["nrm"], sc["rand_ang"], sc["normal_eps"]), gp, W1, W2, meta)
    al, me, ro, reg = OR.material_params(f, fj)
    out = OR.shade_raytracing(sc["pts"], sc["nrm"], sc["vd"], sc["env"], me, ro, al, sc["rand_d"], sc["rand_s"],
                              lambda o, dd: sc["tracer"].trace(o, dd)[1])
    (out["color"].sum() + reg).backward()
    t3 = time.perf_counter()
    return t1 - t0, t2 - t1, t3 - t2


def _cpu_state():
    import torch
    from oracle import render as OR
    from oracle import sd as OS
    from tests._fixtures import make_scene
    ucfg, vcfg = OS.UNetConfig(), OS.VAEConfig()
    wu, wc, wv = OS.random_unet_weights(ucfg, 10), OS.random_controlnet_weights(ucfg, 11), OS.random_vae_weights(vcfg, 12)
    sc = make_scene(res=128, subdiv=5, bump=0.12, seed=0)
    meta, total = OR.hashgrid_meta()
    g = torch.Generator().manual_seed(0)
    grid = (torch.rand(total * 2, generator=g) * 2 - 1) * 1e-4
    W1 = (torch.rand(64, 32, generator=g) * 2 - 1) / 32 ** 0.5
    W2 = (torch.rand(5, 64, generator=g) * 2 - 1) / 8
    return (ucfg, vcfg, wu, wc, wv, sc, grid, W1, W2, meta)


def _cpu_its(ta, tb, tc, views, px_sample, px_per_view):
    """One full iteration from the measured units: per view the 3-branch ControlNet+UNet batch (measured at the real size),
    one VAE forward+backward (measured at the real size), and the shading of the view's covered pixels (measured per pixel
    on a 128^2 render; shading is per-pixel independent, so the cost is linear in covered pixels)."""
    per_view = ta + tb + tc * (px_per_view / px_sample)
    return 1.0 / (views * per_view)


SAMPLE_DESC = ("full-size SD-2.1-base topology, fp32, oracle port on the host cores: the 3-branch CFG batch of ControlNet+UNet for one view at "
               "64x64 latents (real size), 1 VAE encode fwd+bwd at 512x512 (real size), MC shading + hash grid fwd/bwd of a 128x128 render; "
               "one iteration = views x (UNet/CN batch + VAE + shading x covered-pixel ratio); every unit = its BEST time over the runs, "
               "which alternate between all host threads and 16 (small-tensor stages slow down when oversubscribed)")


def _cpu_measure(reps):
    import torch
    cores = min(os.cpu_count() or 1, 64)   # torch-CPU conv throughput degrades beyond ~64 threads on this path
    st = _cpu_state()
    runs = []
    for i in range(reps):                  # the CPU gets its best case: per unit the fastest run, over two thread counts
        torch.set_num_threads(cores if i % 2 == 0 else min(cores, 16))
        runs.append(_cpu_sample(st))
    torch.set_num_threads(cores)
    best = [min(r[i] for r in runs) for i in range(3)]
    spread = [[min(r[i] for r in runs), max(r[i] for r in runs)] for i in range(3)]
    return cores, best, spread, st[5]["pn"]


def cpu_baseline(args, px_per_view):
    reps = 2
    cores, (ta, tb, tc), spread, px_sample = _cpu_measure(reps)
    return {"value": _cpu_its(ta, tb, tc, args.views, px_sample, px_per_view), "unit": "it/s", "cores": cores, "kind": "port",
            "sample": SAMPLE_DESC, "reps": reps,
            "sample_seconds": {"unet_controlnet_3branch_batch_64x64_latents": ta, "vae_512_fwd_bwd": tb, "shade_128x128_render": tc,
                               "min_max": spread, "covered_pixels_of_the_sample_render": px_sample, "covered_pixels_per_view_of_the_workload": px_per_view}}


def run_reference(args):
    """The reference's algorithm on the host CPUs (the reference itself is CUDA-only and cannot be installed
    offline: pytorch_lightning / diffusers / nvdiffrast / tinycudann / _raytracing are absent), i.e. the oracle port."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    reps = max(2, min(args.steps, 4))      # each unit is tens of seconds of CPU work: keep the arm to a few minutes; >= 2 so both thread counts run
    cores, (ta, tb, tc), spread, px_sample = _cpu_measure(reps)
    px_per_view = 0.40 * args.res * args.res   # typical coverage of the 128 fixed views of the bench mesh (measured 0.22 .. 0.75)
    its = _cpu_its(ta, tb, tc, args.views, px_sample, px_per_view)
    cb = {"value": its, "unit": "it/s", "cores": cores, "kind": "port", "sample": SAMPLE_DESC, "reps": reps,
          "sample_seconds": {"unet_controlnet_3branch_batch_64x64_latents": ta, "vae_512_fwd_bwd": tb, "shade_128x128_render": tc, "min_max": spread,
                             "covered_pixels_of_the_sample_render": px_sample, "covered_pixels_per_view_assumed": px_per_view}}
    out = {"impl": "reference", "metric": "SDS iters/sec at 512x512, 8-view batch", "value": its, "unit": "it/s",
           "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": reps, "warmup": 0,
           "ms_per_step": 1000.0 / its, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
           "data": "synthetic", "config": {"workload": "north-star: %dx%d, %d-view batch, 200+128 MC rays/px (oracle port on the host cores: every unit of the step measured at its real size, composed to the full step)" % (args.res, args.res, args.views),
                                           "views": args.views, "resolution": args.res},
           "cpu_baseline": cb,
           "e2e": {"value": its, "unit": "it/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(out)


DUMP_MAX_ELEMS = 1 << 23        # 32 MB of float32: comp_rgb of the default workload (8 x 512 x 512 x 3) fits whole


def dump_outputs(out_dir, out):
    """--dump-outputs: what one training step hands its caller -- every entry of training_step_fused's result (the losses,
    the logged norms, comp_rgb) -- as float32 DIR/<name>.npy.  A larger comp_rgb (more views, higher resolution) is written
    as a fixed sample of its flattened values (seeded, sorted indices), so two builds of the project compare element for
    element.  The parameters after Adam are left out: with eps = 1e-15 a near-zero gradient entry moves by +-lr whatever
    its sign, so they differ between two runs of the same build far more than any output does."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in out.items():
        t = t.detach().float()
        if t.numel() > DUMP_MAX_ELEMS:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_MAX_ELEMS].sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


_RESULT_FD = None


def emit(obj):
    line = json.dumps(obj) + "\n"
    sys.stdout.flush()
    if _RESULT_FD is None:
        sys.stdout.write(line); sys.stdout.flush()
    else:
        os.write(_RESULT_FD, line.encode())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "torch-cuda"])
    ap.add_argument("--shading", default="mc", choices=["mc", "splitsum"], help="use_raytracing true | false (dreammat_material.py:747-762)")
    ap.add_argument("--check", action="store_true", help="add parity_check: gradient identity of the sharded step vs one process")
    ap.add_argument("--no-gpu-baseline", action="store_true", help="skip the stock-PyTorch-CUDA leg (gpu_baseline)")
    ap.add_argument("--views", type=int, default=8)
    ap.add_argument("--res", type=int, default=512)
    ap.add_argument("--faces", type=int, default=100000)
    ap.add_argument("--env-h", type=int, default=2048)
    ap.add_argument("--env-w", type=int, default=4096)
    ap.add_argument("--dtype", default="f16", choices=["f16", "bf16"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graphs", action="store_true")
    ap.add_argument("--no-pdl", action="store_true", help="disable programmatic dependent launch of the dense kernels")
    ap.add_argument("--no-gc-freeze", action="store_true", help="A/B: leave Python's full collections inside the timed region")
    ap.add_argument("--no-balance", action="store_true", help="multi-GPU: every rank shades only its own views")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    # stdout carries exactly one JSON line: libraries that write to fd 1 (NCCL's version banner, nvcc/ninja chatter)
    # are sent to stderr for the whole run and the result line is written to the saved descriptor.
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "torch-cuda":
        run_torch_cuda(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
