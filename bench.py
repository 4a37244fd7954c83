#!/usr/bin/env python
"""bench.py — denoise-steps/sec of the Cosmos-7B GEN3C DiT (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --steps K --warmup W    # the reference algorithm on the host CPU (oracle port)
  python bench.py --steps K --warmup W --dump-outputs DIR  # + the last timed step's outputs as DIR/<name>.npy

One step = one loop body of generate_samples_from_batch (reference model_v2w.py:130-149): sampler glue +
cond forward + uncond forward of the 28-block 7B DiT over the 121-frame / 704x1280 latent [16,16,88,160]
(56 320 tokens), bf16 weights/activations, fp32 accumulation, random-init weights in the real checkpoint
layout, synthetic latents / poses / text context (no network for checkpoints or data).
N > 1 (torchrun): total work is fixed -> "scaling": "strong".  Default layout ("cfgxcp"): the conditional and the
unconditional forward of a step run on two halves of the ranks (CFG-parallel, one 14 MB peer-memory exchange of the
network outputs per step) and each half shards the 16 latent frames context-parallel (cp = N/2, one K and one V^T
exchange per self-attention layer); "--parallelism cp" is the reference's layout (cp = N, general_dit.py:524-543).
Before the timed region every multi-GPU run checks the sharded denoise step against the unsharded one on a tiny net
and aborts on mismatch.  The same JSON line carries a "path_r" object: the 3D-cache render (121 target frames of
704x1280 from one cached frame) with its own roofline / e2e / cpu_baseline.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from (which may be read-only)

FLOP_PER_FORWARD = 2.2096e15  # SURVEY.md §8d / BASELINE.md §2
FLOP_PER_STEP = 2 * FLOP_PER_FORWARD
SELF_ATTN_FLOP_PER_LAUNCH_FULL = 4.0 * 56320 * 56320 * 4096  # 5.197e13 at cp = 1
LAT = (16, 16, 88, 160)
CTX = (512, 1024)
DUMP_SAMPLE = 1 << 20  # elements kept of each Path R output (1.7 GB per render) by --dump-outputs


def seeded_sample(torch, t):
    """The same DUMP_SAMPLE elements of any tensor of t's size, so that two builds can be compared output for output."""
    idx = torch.randint(t.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0))
    return t.reshape(-1)[idx.to(t.device)]


def dump_outputs(dump_dir, outputs):
    """Writes each tensor as dump_dir/<name>.npy in float32."""
    import numpy as np

    os.makedirs(dump_dir, exist_ok=True)
    for name, t in outputs.items():
        np.save(os.path.join(dump_dir, name + ".npy"), t.float().cpu().numpy())


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"tflops_burst": d["bf16_tflops"], "tflops_sustained": d["bf16_tflops_sustained"], "hbm_gbs": d["hbm_gbs"],
                "source": "measured"}
    return {"tflops_burst": 1590.0, "tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback"}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self._halt = index, [], threading.Event()

    def run(self):
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([s.strip() for s in out.split(",")])
            except Exception:  # noqa: BLE001
                pass
            self._halt.wait(0.2)

    def finish(self):
        self._halt.set()
        self.join(timeout=3)
        sm = sorted(int(float(s[0])) for s in self.samples if s and s[0].replace(".", "").isdigit())
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        mx = max((int(float(s[1])) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()), default=None)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port of the reference algorithm on the host cores
# ------------------------------------------------------------------------------------------------------
def cpu_sample_seconds(threads: int, repeats: int = 1):
    """One FA-CA-MLP block at full width (D=4096, 32 heads, ctx 512x1024) on ONE latent frame (3 520 tokens),
    fp32, torch CPU ops = the reference's graph with the TE ops restated (oracle/dit_oracle.py).
    Returns (seconds per sample, FLOPs of the sample)."""
    import torch

    from oracle import dit_oracle

    torch.set_num_threads(threads)
    cfg = dit_oracle.DitCfg(num_blocks=1)
    g = torch.Generator().manual_seed(0)
    sd = {k: (0.02 * torch.randn(s, generator=g)) for k, s in dit_oracle.state_dict_shapes(cfg).items()}
    T, H, W = 1, 88, 160
    x = torch.randn(16, T, H, W, generator=g)
    mask = torch.zeros(1, T, H, W)
    pose = torch.randn(64, T, H, W, generator=g)
    ctx = torch.randn(*CTX, generator=g)
    L, D = T * 44 * 80, 4096
    flops = 28.0 * L * D * D + 4.0 * L * L * D + 4.0 * 512 * 1024 * D + 4.0 * L * 512 * D + 2.0 * L * 328 * D + 2.0 * L * D * 64
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        with torch.no_grad():
            dit_oracle.forward(sd, cfg, x, mask, pose, None, 0.5, ctx)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return best, flops


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = min(os.cpu_count() or 1, 64)  # torch's CPU GEMM/SDPA stop scaling (and regress) beyond this
    cpu_sample_seconds(threads)  # page-in / warm
    for _ in range(max(0, args.warmup - 1)):
        cpu_sample_seconds(threads)
    ts = []
    flops = 0.0
    for _ in range(args.steps):
        dt, flops = cpu_sample_seconds(threads)
        ts.append(dt)
    t = sum(ts) / len(ts)
    sps = 1.0 / (t * FLOP_PER_STEP / flops)
    sample = ("1 FA-CA-MLP block of the 7B DiT (D=4096, 32 heads, ctx 512x1024) on 1 latent frame (3 520 tokens), fp32 "
              "torch-CPU oracle port; steps/s extrapolated by FLOPs (x%.0f) to the full 2-forward step" % (FLOP_PER_STEP / flops))
    line = {"impl": "reference", "metric": "denoise-steps/sec, 7B DiT, 121-frame 720p latent", "value": sps,
            "unit": "steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 / sps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "Cosmos-7B GEN3C DiT denoise step (2 forwards), latent [16,16,88,160], ctx 512x1024",
                       "note": "CPU-extrapolated; the reference has no CPU path of its own (model_t2w.py:56)"},
            "cpu_baseline": {"value": sps, "unit": "steps/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": sps, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    fps, dt, thr = path_r_cpu_frames_per_s(8)
    line["path_r"] = {"metric": "cache-render frames/sec, 704x1280, 1 cached frame -> 121 target poses", "value": fps,
                      "unit": "frames/s", "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": thr, "kind": "port",
                                                           "sample": "oracle port of forward_warp (numpy f32) on 8 of the 121 target frames, %.1f s" % dt}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------
# this repo's arm
# ------------------------------------------------------------------------------------------------------
def build_net(torch, device):
    from gen3c_b200.dit import VideoExtendGeneralDIT

    net = VideoExtendGeneralDIT(device=device)  # GEN3C_Cosmos_7B defaults
    g = torch.Generator(device=device).manual_seed(1234)
    with torch.no_grad():
        for k, p in net.state_dict(keep_vars=True).items():
            if k == "pos_embedder.seq":
                continue
            if p.dim() == 1:
                p.copy_((1.0 + 0.05 * torch.randn(p.shape, device=device, generator=g)).to(p.dtype))
            else:
                p.copy_((0.02 * torch.randn(p.shape, device=device, generator=g)).to(p.dtype))
    return net


# ------------------------------------------------------------------------------------------------------
# Path R leg: Cache3D render of 121 target frames (SURVEY.md §8d)
# ------------------------------------------------------------------------------------------------------
R_FRAMES, R_H, R_W = 121, 704, 1280
R_BYTES_PER_PX = 44  # read points 12 + image 12 + mask 4, write image 12 + mask 4 (SURVEY.md §8d, DESIGN.md §3.4)


def path_r_cpu_frames_per_s(n_frames: int = 4):
    """The oracle port of forward_warp (numpy, float32) on n_frames 704x1280 target frames, chunks of 2 like
    cache_3d.py:175-223.  Returns (frames/s, seconds, threads)."""
    import numpy as np

    from oracle import cases, warp_oracle

    depth = cases.smooth_depth(R_H, R_W)[None, None]
    K = cases.intrinsics(R_H, R_W)[None]
    img = np.random.RandomState(0).uniform(-1, 1, (1, 3, R_H, R_W)).astype(np.float32)
    pts = warp_oracle.unproject_points(depth, np.eye(4, dtype=np.float32)[None], K)
    w2cs = cases.pan_trajectory(R_FRAMES, 0.3)[:n_frames]
    t0 = time.perf_counter()
    for i in range(0, n_frames, 2):
        c = w2cs[i:i + 2]
        b = c.shape[0]
        warp_oracle.forward_warp(np.repeat(img, b, 0), None, np.repeat(pts, b, 0), c, np.repeat(K, b, 0))
    dt = time.perf_counter() - t0
    return n_frames / dt, dt, 1


def bench_path_r(torch, dev, peaks, steps: int, warmup: int, cpu_baseline: bool, outputs=None):
    """outputs: dict that receives a seeded sample of the pixels and masks of the last timed render, or None."""
    import numpy as np

    from gen3c_b200 import warp
    from gen3c_b200.cache_3d import Cache3D_Buffer
    from oracle import cases  # synthetic inputs only (seeded depth / trajectory); nothing is computed by the oracle here

    depth_h = torch.from_numpy(cases.smooth_depth(R_H, R_W)[None, None]).pin_memory()
    img_h = (torch.rand(1, 3, R_H, R_W, generator=torch.Generator().manual_seed(0)) * 2 - 1).pin_memory()
    K_h = torch.from_numpy(cases.intrinsics(R_H, R_W)[None]).pin_memory()
    eye_h = torch.eye(4)[None].pin_memory()
    w2cs_h = torch.from_numpy(cases.pan_trajectory(R_FRAMES, 0.3))[None].pin_memory()
    Ks_h = K_h[None].expand(1, R_FRAMES, 3, 3).contiguous().pin_memory()
    cov_h = torch.empty(R_FRAMES).pin_memory()

    def make_cache(non_blocking=True):
        return Cache3D_Buffer(frame_buffer_max=2, noise_aug_strength=0, generator=None,
                              input_image=img_h.to(dev, non_blocking=non_blocking),
                              input_depth=depth_h.to(dev, non_blocking=non_blocking),
                              input_w2c=eye_h.to(dev, non_blocking=non_blocking),
                              input_intrinsics=K_h.to(dev, non_blocking=non_blocking), device=dev)

    cache = make_cache()
    w2cs, Ks = w2cs_h.to(dev), Ks_h.to(dev)
    pts, img = cache.input_points[:, :, :, 0], cache.input_image[:, :, :, 0]

    def resident(_):
        return warp.render_cache(pts, img, None, w2cs, Ks)

    def e2e(_):
        c = make_cache()
        pix, msk = warp.render_cache(c.input_points[:, :, :, 0], c.input_image[:, :, :, 0], None,
                                     w2cs_h.to(dev, non_blocking=True), Ks_h.to(dev, non_blocking=True))
        cov_h.copy_(msk.mean(dim=(0, 2, 3, 4, 5)), non_blocking=True)
        return pix

    def timed(fn, n):
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for i in range(n):
            out = fn(i)
        e.record()
        torch.cuda.synchronize()
        return s.elapsed_time(e) / n, out

    for i in range(max(3, warmup)):
        resident(i)
    n = steps
    ms, (pix, msk) = timed(resident, n)
    if outputs is not None:
        outputs["path_r_pixels_sample"] = seeded_sample(torch, pix)
        outputs["path_r_masks_sample"] = seeded_sample(torch, msk)
    del pix, msk
    e2e(0)
    ms_e2e, _ = timed(e2e, n)
    px = R_FRAMES * R_H * R_W
    gbs = px * R_BYTES_PER_PX / (ms * 1e-3) / 1e9
    h2d = sum(t.numel() * t.element_size() for t in (depth_h, img_h, K_h, eye_h, w2cs_h, Ks_h))
    out = {"metric": "cache-render frames/sec, 704x1280, 1 cached frame -> 121 target poses", "value": R_FRAMES / (ms * 1e-3),
           "unit": "frames/s", "ms_per_render": ms, "dtype": "f32", "steps": n,
           "config": {"workload": "Cache3D_Buffer.render_cache: unprojected 704x1280 frame -> 121-pose left pan "
                                  "(project + soft-z bilinear splat + normalise), outputs 1.7 GB per render > L2"},
           "gpu_launches": (1 + 2 * ((R_FRAMES + 3) // 4)) * n,  # k_project_max + (k_splat_points, k_normalise) per pass of 4
           "e2e": {"value": R_FRAMES / (ms_e2e * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": h2d,
                   "d2h_bytes_per_step": R_FRAMES * 4,
                   "note": "host image/depth/cameras -> Cache3D_Buffer (H2D + unproject) -> render; the rendered frames "
                           "stay on the GPU as in the reference (cache_3d.py:236), per-frame coverage is read back"},
           "roofline": {"bound": "hbm", "kernel": "k_splat_points (+ k_project_max, k_normalise)", "achieved": gbs,
                        "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
                        "traffic": ncu_traffic_bytes("r02_splat_ncu_summary.txt"),
                        "algorithmic_bytes_per_render": px * R_BYTES_PER_PX, "peak_source": peaks["source"]}}
    if cpu_baseline:
        fps, dt, thr = path_r_cpu_frames_per_s(4)
        out["cpu_baseline"] = {"value": fps, "unit": "frames/s", "cores": thr, "kind": "port",
                               "sample": "oracle port of forward_warp (numpy f32) on 4 of the 121 target frames, %.1f s" % dt}
    return out


# ------------------------------------------------------------------------------------------------------
# multi-GPU correctness gate: sharded denoise step == unsharded denoise step (tiny net), before anything is timed
# ------------------------------------------------------------------------------------------------------
def sharded_step_parity(torch, dist, dev, setup_parallel, cp_size, cp_rank):
    from gen3c_b200 import sampler
    from gen3c_b200.dit import VideoExtendGeneralDIT

    T_local, H, W, M = 2, 16, 16, 128          # 2 * 8 * 8 = 128 tokens per rank
    T = T_local * cp_size
    bf = torch.bfloat16
    kw = dict(max_img_h=64, max_img_w=64, max_frames=16, model_channels=256, num_blocks=2, num_heads=2,
              crossattn_emb_channels=64, adaln_lora_dim=32, device=dev)
    g = torch.Generator().manual_seed(77)      # identical on every rank

    def rnd(*shape, s=1.0):
        return (s * torch.randn(*shape, generator=g)).to(bf).to(dev)

    ref = VideoExtendGeneralDIT(**kw)
    sd = {}
    for k, p in ref.state_dict().items():
        if k == "pos_embedder.seq":
            sd[k] = p
        elif p.dim() == 1:
            sd[k] = (1.0 + 0.1 * torch.randn(p.shape, generator=g)).to(bf).to(dev)
        else:
            sd[k] = (0.04 * torch.randn(p.shape, generator=g)).to(bf).to(dev)
    ref.load_state_dict(sd)
    par = VideoExtendGeneralDIT(**kw)
    par.load_state_dict(sd)
    setup_parallel(par)
    sigma, sigma_next, guidance = 0.67, 0.47, 1.5
    x, gt = rnd(16, T, H, W, s=0.8), rnd(16, T, H, W, s=0.5)
    noise = torch.randn(16, T, H, W, generator=g).to(dev)
    ind = torch.zeros(T, device=dev)
    ind[0] = 1.0
    mask = torch.zeros(1, T, H, W, device=dev, dtype=bf)
    mask[:, 0] = 1
    pose, pad = rnd(64, T, H, W, s=0.5), torch.zeros(H, W, device=dev, dtype=bf)
    ctx_c, ctx_u = rnd(M, 64), rnd(M, 64)
    o_ref = torch.empty_like(x)
    x_ref = sampler.denoise_step(ref, x, gt, noise, ind, mask, pose, pad, ctx_c, ctx_u, sigma, sigma_next, guidance,
                                 net_output=o_ref)
    sl = slice(cp_rank * T_local, (cp_rank + 1) * T_local)
    loc = lambda t: t[:, sl].contiguous()  # noqa: E731
    o_par = torch.empty_like(loc(x))
    x_par = sampler.denoise_step(par, loc(x), loc(gt), loc(noise), ind[sl].contiguous(), loc(mask), loc(pose), pad, ctx_c,
                                 ctx_u, sigma, sigma_next, guidance, net_output=o_par)
    torch.cuda.synchronize()

    def rel(a, b):
        return (a.float() - b.float()).norm() / b.float().norm()

    err = torch.stack([rel(o_par, loc(o_ref)), rel(x_par, loc(x_ref))])
    dist.all_reduce(err, op=dist.ReduceOp.MAX)
    e_out, e_x = float(err[0]), float(err[1])
    par._teardown_barrier()
    del par, ref
    # both sides are bf16 computations that differ in accumulation order (K/V chunk order, tile partition); on this small
    # net the CFG-combined output (guidance 1.5: forward differences x 2.9) sits at 3.8e-3 and x_(t-1) at 9e-4 for cp = 2..4
    # (0 for pure CFG parallelism); a dropped K/V chunk, a stale flag or swapped branches gives >= 1e-1
    return {"net_output_rel_l2_max_over_ranks": e_out, "x_next_rel_l2_max_over_ranks": e_x, "tol": 1e-2, "tol_x": 2.5e-3,
            "case": f"2-block D=256 net, T={T} latent frames (2 per cp rank), sharded vs unsharded g3c_denoise_step"}


def attention_ab(torch, dev):
    """The dominant kernel against torch's fused SDPA on the same tensors (one full-size self-attention: 56 320 x 56 320,
    32 heads): device time of 3 launches each, after one warm-up."""
    from gen3c_b200 import ops

    L, Hh = LAT[1] * 44 * 80, 32
    g = torch.Generator(device=dev).manual_seed(5)
    q, k, v = ((torch.randn(L, Hh * 128, device=dev, generator=g)).to(torch.bfloat16) for _ in range(3))
    vt = v.T.contiguous()

    def ours():
        return ops.attention(q, k, vt, Hh)

    qh, kh, vh = (t.view(L, Hh, 128).permute(1, 0, 2)[None] for t in (q, k, v))

    def sdpa():
        return torch.nn.functional.scaled_dot_product_attention(qh, kh, vh)

    res = {}
    for name, fn in (("ours", ours), ("torch_sdpa", sdpa)):
        fn()
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(3):
            fn()
        e.record()
        torch.cuda.synchronize()
        ms = s.elapsed_time(e) / 3
        res[name] = {"ms": ms, "tflops": SELF_ATTN_FLOP_PER_LAUNCH_FULL / (ms * 1e-3) / 1e12}
    return res


def gpu_reference_graph_steps_per_s(torch, net, devt, sig):
    """SURVEY.md §8d "unmodified graph" arm: the reference's op graph (oracle/dit_oracle.py restates it op for op) in
    bf16 on this GPU with torch's own kernels — cuBLAS Linears, fused SDPA, unfused element-wise ops — for the same
    2-forward step.  A baseline beside the product number; nothing of this repo's CUDA runs in it."""
    from oracle import dit_oracle

    cfg = dit_oracle.DitCfg()
    sd = dict(net.state_dict())

    def fwd(x_in, t, cond):
        return dit_oracle.forward(sd, cfg, x_in, devt["mask"], devt["pose"] if cond else None, devt["pad"], t,
                                  devt["ctx_c"] if cond else devt["ctx_u"], compute_dtype=torch.bfloat16)

    ind = devt["ind"]

    def step(i):
        return dit_oracle.denoise_step(fwd, devt["xt"].float(), devt["gt"].float(), devt["noise"], ind, sig[i], sig[i + 1], 1.0)

    with torch.no_grad():
        step(0)
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        step(1)
        e.record()
        torch.cuda.synchronize()
    return 1e3 / s.elapsed_time(e)


def run_ours(args):
    import torch
    import torch.distributed as dist

    from gen3c_b200 import _lib, sampler

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    peaks = measured_peaks()
    # ---- layout: cfg (1 or 2) x cp
    layout = args.parallelism
    if layout == "auto":
        layout = "cfgxcp" if world >= 2 else "cp"
    cfg_size = 2 if (layout == "cfgxcp" and world >= 2) else 1
    cp_size = world // cfg_size
    assert cfg_size * cp_size == world and LAT[1] % cp_size == 0, "16 latent frames must divide over the cp ranks"
    cfg_role, cp_rank = rank // cp_size, rank % cp_size
    cp_group = pair_group = None
    if world > 1:
        # every rank creates every group, in the same order
        cp_groups = [dist.new_group(list(range(c * cp_size, (c + 1) * cp_size))) for c in range(cfg_size)]
        pair_groups = [dist.new_group([i, i + cp_size]) for i in range(cp_size)] if cfg_size == 2 else []
        cp_group = cp_groups[cfg_role] if cp_size > 1 else None
        pair_group = pair_groups[cp_rank] if cfg_size == 2 else None

    def setup_parallel(n):
        if cp_group is not None:
            n.enable_context_parallel(cp_group, mode=args.cp_mode)
        if pair_group is not None:
            n.enable_cfg_parallel(pair_group)

    parity = None
    if world > 1:
        parity = sharded_step_parity(torch, dist, dev, setup_parallel, cp_size, cp_rank)
        if not (parity["net_output_rel_l2_max_over_ranks"] < parity["tol"] and parity["x_next_rel_l2_max_over_ranks"] < parity["tol_x"]):
            raise SystemExit(f"multi-GPU parity check FAILED, nothing timed: {parity}")
    net = build_net(torch, dev)
    setup_parallel(net)
    Tl = LAT[1] // cp_size
    t0 = cp_rank * Tl
    bf = torch.bfloat16
    g = torch.Generator().manual_seed(1)  # host-side synthetic inputs (pinned), same on every rank
    sch = sampler.EDMEulerScheduler().set_timesteps(35)

    def pin(t):
        return t.contiguous().pin_memory()

    full = {
        "xt": (torch.randn(LAT, generator=g) * sch.init_noise_sigma).to(bf),
        "gt": (0.5 * torch.randn(LAT, generator=g)).to(bf),
        "noise": sampler.arch_invariant_rand(LAT, 1),
        "pose": (0.5 * torch.randn(64, *LAT[1:], generator=g)).to(bf),
        "mask": torch.zeros(1, *LAT[1:]).to(bf),
        "ctx_c": torch.randn(CTX, generator=g).to(bf),
        "ctx_u": torch.randn(CTX, generator=g).to(bf),
        "pad": torch.zeros(LAT[2], LAT[3]).to(bf),
    }
    full["mask"][:, 0] = 1
    ind_full = torch.zeros(LAT[1])
    ind_full[0] = 1.0
    host = {k: pin(v[:, t0:t0 + Tl] if v.dim() == 4 else v) for k, v in full.items()}
    host["ind"] = pin(ind_full[t0:t0 + Tl])
    devt = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
    out_host = torch.empty((16, Tl, LAT[2], LAT[3]), dtype=bf).pin_memory()
    sig = [float(s) for s in sch.sigmas]
    lib = _lib.load()

    def step_resident(i):
        return sampler.denoise_step(net, devt["xt"], devt["gt"], devt["noise"], devt["ind"], devt["mask"], devt["pose"],
                                    devt["pad"], devt["ctx_c"], devt["ctx_u"], sig[i % 34], sig[i % 34 + 1], 1.0)

    h2d_bytes = sum(host[k].numel() * host[k].element_size() for k in ("xt", "gt", "noise", "pose", "mask", "ctx_c", "ctx_u", "pad", "ind"))
    d2h_bytes = out_host.numel() * out_host.element_size()

    def step_e2e(i):
        d = {k: host[k].to(dev, non_blocking=True) for k in host}
        o = sampler.denoise_step(net, d["xt"], d["gt"], d["noise"], d["ind"], d["mask"], d["pose"], d["pad"], d["ctx_c"],
                                 d["ctx_u"], sig[i % 34], sig[i % 34 + 1], 1.0)
        out_host.copy_(o, non_blocking=True)
        return o

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for i in range(steps):
            out = fn(i)
        e.record()
        barrier()
        ms = torch.tensor([s.elapsed_time(e)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms) / steps, out

    for i in range(max(3, args.warmup)):
        step_resident(i)
    barrier()
    launches_per_step = net.last_launch_count()
    clocks = ClockSampler(local)
    clocks.start()
    # -- timed region 1: inputs resident in HBM, profiling events on (per-category device time)
    _lib.check(lib.g3c_dit_profile(net._engine(), 1), "g3c_dit_profile")
    ms_resident, x_next = timed(step_resident, args.steps)
    outputs = {"x_next": x_next.float().cpu()} if args.dump_outputs else None
    del x_next
    cat_ms = (C.c_float * 6)()
    cat_n = (C.c_int * 6)()
    _lib.check(lib.g3c_dit_profile_read(net._engine(), cat_ms, cat_n, 6), "g3c_dit_profile_read")
    wait_ms = C.c_float(0.0)
    _lib.check(lib.g3c_dit_profile_wait_ms(net._engine(), C.byref(wait_ms)), "g3c_dit_profile_wait_ms")
    _lib.check(lib.g3c_dit_profile(net._engine(), 0), "g3c_dit_profile")
    # -- timed region 2: same step through the public API with pinned host buffers (H2D + D2H inside)
    step_e2e(0)
    ms_e2e, _ = timed(step_e2e, args.steps)
    clk = clocks.finish()
    if rank != 0:
        if world > 1:
            net._teardown_barrier()
            dist.destroy_process_group()
        return
    names = ["gemm", "attn_self", "attn_cross", "eltwise", "comm", "vector"]
    breakdown = {n: {"ms_per_step": cat_ms[i] / args.steps, "launches_per_step": cat_n[i] // max(1, args.steps)}
                 for i, n in enumerate(names)}
    breakdown["kv_wait_exposed_upper_bound"] = {
        "ms_per_step": wait_ms.value / args.steps,
        "note": "mean over CTAs of the time the attention kernel's loader warps spent polling peer K/V flags (inside attn_self)"}
    # dominant kernel: self-attention (65.9 % of the FLOPs); algorithmic FLOPs per launch on this rank
    attn_launches = max(1, cat_n[1])
    attn_ms = cat_ms[1] / attn_launches
    attn_flop = SELF_ATTN_FLOP_PER_LAUNCH_FULL / cp_size
    achieved = attn_flop / (attn_ms * 1e-3) / 1e12 if attn_ms > 0 else 0.0
    peak = peaks["tflops_sustained"]
    sps = 1e3 / ms_resident
    par_name = (f"cfg{cfg_size}xcp{cp_size}" if cfg_size > 1 else f"cp{cp_size}")
    if cp_size > 1:
        par_name += f" ({args.cp_mode or os.environ.get('G3C_CP_MODE', 'p2p')} K/V exchange)"
    line = {
        "metric": "denoise-steps/sec, 7B DiT, 121-frame 720p latent", "value": sps, "unit": "steps/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_resident,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "Cosmos-7B GEN3C DiT denoise step (cond + uncond forward + EDM Euler glue), latent "
                               "[16,16,88,160] = 56 320 tokens, ctx 512x1024, guidance 1, random-init weights",
                   "parallelism": par_name, "l2": "inputs larger than L2 (14.5 GB weights, 0.9 GB residual stream)"},
        "e2e": {"value": 1e3 / ms_e2e, "unit": "steps/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes},
        "gpu_launches": launches_per_step * args.steps,
        "roofline": {"bound": "tensor", "kernel": "k_attn_fwd1t (self-attention)", "achieved": achieved, "peak": peak,
                     "unit": "TFLOP/s", "frac": achieved / peak,
                     # DRAM bytes of one launch from the committed ncu --set full capture of this kernel at the cp = 1
                     # shape; not meaningful for the sharded shapes, hence null there
                     "traffic": ncu_traffic_bytes("r02_attn_ncu_summary.txt", "r01_attn_ncu_summary.txt") if cp_size == 1 else None,
                     "peak_source": peaks["source"] + " (sustained)",
                     "step_tflops": FLOP_PER_STEP * sps / 1e12 / world, "step_frac": FLOP_PER_STEP * sps / 1e12 / world / peak},
        "kernel_breakdown": breakdown,
        "clocks": clk,
        "workspace_gb": net.workspace_bytes() / 1e9,
    }
    if parity is not None:
        line["sharded_parity"] = parity
    if world == 1 and not args.no_cpu_baseline:
        threads = min(os.cpu_count() or 1, 64)
        try:
            cpu_sample_seconds(threads)
            dt, flops = cpu_sample_seconds(threads)
            line["cpu_baseline"] = {
                "value": 1.0 / (dt * FLOP_PER_STEP / flops), "unit": "steps/s", "cores": threads, "kind": "port",
                "sample": "1 FA-CA-MLP block (D=4096) on 1 latent frame (3 520 tokens), fp32 torch-CPU oracle port, %.1f s; "
                          "extrapolated by FLOPs (x%.0f)" % (dt, FLOP_PER_STEP / flops)}
        except Exception as ex:  # noqa: BLE001 - a reported baseline, never worth the headline line
            line["cpu_baseline"] = {"error": repr(ex)[:300]}
    if world == 1 and not args.no_extras:
        try:
            line["attention_ab"] = attention_ab(torch, dev)
            line["gpu_reference_graph"] = {
                "value": gpu_reference_graph_steps_per_s(torch, net, devt, sig), "unit": "steps/s",
                "what": "the reference's op graph (oracle restatement) in bf16 with torch kernels on this GPU: cuBLAS Linears, "
                        "fused SDPA, unfused element-wise ops; same 2-forward step, 1 timed step after 1 warm-up"}
        except Exception as ex:  # noqa: BLE001 - extras must never cost the headline line
            line["extras_error"] = repr(ex)[:300]
    if world == 1 and not args.no_path_r:
        del devt
        torch.cuda.empty_cache()
        try:
            line["path_r"] = bench_path_r(torch, dev, peaks, args.steps, args.warmup, not args.no_cpu_baseline, outputs)
        except Exception as ex:  # noqa: BLE001 - the second leg must never cost the headline line
            line["path_r"] = {"error": repr(ex)[:300]}
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(line), flush=True)
    if world > 1:
        net._teardown_barrier()
        dist.destroy_process_group()


def ncu_traffic_bytes(*names):
    """DRAM bytes (read + write) of one launch of the named kernel, from the first committed `ncu --set full` summary found
    under profiles/ (written by tools/ncu_summary.py from the capture of the same shape); None when absent.  Static
    evidence: bench.py cannot read DRAM counters itself (a number printed under a profiler is never a bench value)."""
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    for name in names:
        path = os.path.join(ROOT, "profiles", name)
        tot, seen = 0.0, 0
        try:
            for ln in open(path):
                if ln.startswith("--") and seen >= 2:
                    break
                for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    if ln.startswith(key):
                        unit = ln[ln.index("[") + 1:ln.index("]")]
                        tot += float(ln.split("=")[1]) * scale[unit]
                        seen += 1
        except (OSError, ValueError, KeyError):
            continue
        if seen >= 2:
            return tot
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the attention A/B and the torch-kernel reference-graph arm")
    ap.add_argument("--no-path-r", action="store_true", help="skip the 3D-cache render leg")
    ap.add_argument("--parallelism", default="auto", choices=["auto", "cp", "cfgxcp"],
                    help="N > 1: cfgxcp (default) = cond / uncond forward on two halves of the ranks x context parallel "
                         "inside each half; cp = context parallel over all ranks (the reference's layout)")
    ap.add_argument("--cp-mode", default=None, choices=[None, "p2p", "nccl"],
                    help="context-parallel K/V exchange: p2p = fused projection -> peer-memory all-gather (default), nccl = ncclAllGather")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32): the "
                         "denoise step's x_(t-1) and a seeded sample of the Path R render")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.gpus != 1):
        ap.error("--dump-outputs needs --impl ours and --gpus 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
