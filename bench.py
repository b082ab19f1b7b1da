#!/usr/bin/env python
"""bench.py — BASELINE.json metric on B200: 512x512 50-step SAM+ControlNet-inpaint images/sec and
the fused ControlNet x2 + UNet + CFG + DDIM step time.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): SD1.5 topology, 512x512 image -> 64x64 latents, 1 image per
GPU + classifier-free guidance (B = 2), SAM-ControlNet + inpaint-ControlNet, 77-token context,
DDIM eta = 0; synthetic inputs and seeded random weights (no checkpoints / network here).
A "step" is one denoising step.  `value` (images/s) = n_gpus / (50 * step + SAM encode), both
components device-timed in this run and reported in `config`.
One process per GPU; images shard one per GPU (weak scaling) with a single NCCL all-gather of the
final latents/images at the end — no data-path collective inside the step.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

STEP_TFLOP = 2.740        # algorithmic 2*MAC per fused step at configs[1] (BASELINE.md §2)
SAM_TFLOP = 5.96          # SAM ViT-H image encoder, one 1024x1024 image (BASELINE.md §2)
DDIM_STEPS = 50
DUMP_MAX_BYTES = 64 << 20


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1442.5), d.get("bf16_tflops", 1682.0), d.get("hbm_gbs", 6585.4), "measured"
    return 1400.0, 1590.0, 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self._stop_evt = index, [], threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([s.strip() for s in out.split(",")])
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=3)
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        mx = max([int(s[1]) for s in self.samples if s[1].isdigit()] or [0])
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for s in self.samples for i in range(4) if len(s) > 2 + i and s[2 + i] == "Active"})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": reasons,
                "samples": len(self.samples)}


def make_inputs(cfg, B, lat, L, seed):
    """B = 2 * images (CFG halves: [uncond x n; cond x n])."""
    """Same synthetic inputs as oracle/inputs.py (SURVEY.md §8d); duplicated here so the product arm
    imports nothing from oracle/."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, cfg.in_channels, lat, lat, generator=g)
    ctx = torch.randn(B, L, cfg.context_dim, generator=g)
    h0 = torch.randint(0, 256, (1, 3, 8 * lat, 8 * lat), generator=g).float()
    h0[:, 2] = 0
    h1 = torch.rand(1, 3, 8 * lat, 8 * lat, generator=g)
    q = 2 * lat
    h1[:, :, q:8 * lat - q, q:8 * lat - q] = -1.0
    return x, ctx, [h0.repeat(B, 1, 1, 1), h1.repeat(B, 1, 1, 1)]


def _gemm_traffic():
    """DRAM bytes per ea_gemm launch (read + write, averaged over one step's launches) from the committed
    ncu launch list of this same command (profiles/gemm_traffic.json, written by
    tools/summarize_launches.py --traffic-json); None when no capture is committed."""
    path = os.path.join(ROOT, "profiles", "gemm_traffic.json")
    try:
        doc = json.load(open(path))
        n = rd = 0
        for k, v in doc["kernels"].items():
            if "ea_gemm" in k:
                n += v["launches"]
                rd += v["dram_bytes_per_launch"] * v["launches"]
        if n:
            return round(rd / n), "ncu dram__bytes_read.sum + dram__bytes_write.sum per launch, profiles/gemm_traffic.json (" + doc.get("source", "") + ")"
    except (OSError, KeyError, ValueError):
        pass
    return None, "no ncu capture committed"


class GemmProbe:
    """Wraps editanything_b200.ops and records every ea_gemm call of one step (arguments + algorithmic
    FLOPs).  The recorded launches are then re-issued back to back inside ONE CUDA graph and the graph
    replay is timed with CUDA events: that is the dominant kernel's average launch duration inside
    the timed region without the ~25 us of Python/ctypes/tensor-map-encode cost per launch."""

    def __init__(self, ops):
        self._ops, self.records = ops, []

    def __getattr__(self, n):
        return getattr(self._ops, n)

    @staticmethod
    def _flops(a, w, kw):
        conv = kw.get("conv")
        M = conv[0] * conv[1] * conv[2] if conv else (kw.get("M") or a.shape[0])
        return 2.0 * M * w.shape[0] * w.shape[1]

    def gemm(self, a, w, out=None, **kw):
        r = self._ops.gemm(a, w, out, **kw)
        kw2 = dict(kw)
        if out is None and kw.get("out_f32") is None:
            out = r
        self.records.append((a, w, out, kw2, self._flops(a, w, kw)))
        return r

    def gemm_grouped(self, calls):
        """One launch for several networks (ea_gemm_grouped): recorded as ONE launch carrying every group's FLOPs."""
        outs = self._ops.gemm_grouped(calls)
        calls2 = [(a, w, o if o is not None else r, dict(kw)) for (a, w, o, kw), r in zip(calls, outs)]
        self.records.append(("grouped", calls2, None, None, sum(self._flops(a, w, kw) for a, w, _, kw in calls2)))
        return outs

    def _issue(self, rec):
        if rec[0] == "grouped":
            self._ops.gemm_grouped(rec[1])
        else:
            a, w, out, kw, _ = rec
            self._ops.gemm(a, w, out, **kw)

    def replay_time_ms(self, reps=3):
        ops = self._ops
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for rec in self.records:
                self._issue(rec)
        torch.cuda.current_stream().wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for rec in self.records:
                self._issue(rec)
        g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps


def dump_outputs(out_dir, **arrays):
    """Writes each array as out_dir/<name>.npy in float32 so that two builds can be compared output for output; an
    array over DUMP_MAX_BYTES keeps its leading rows (whole images) up to that size."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().float()
        rows = max(1, DUMP_MAX_BYTES // max(1, t[:1].numel() * 4))
        np.save(os.path.join(out_dir, name + ".npy"), t[:rows].cpu().numpy())


def _all_gather_list(t, world):
    import torch.distributed as dist
    bufs = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(bufs, t.contiguous())
    return bufs


def measure_batch_block(eng, cfg, n_img, rank, sust, args, ts, a, ap):
    """Device-timed fused steps at n_img images per GPU (BASELINE.json configs[3] = 4 per GPU => B = 8), same
    engine and weights: returns the `config.batchN` block."""
    x, ctx, hints = make_inputs(cfg, 2 * n_img, 64, 77, 31 + rank)
    eng.prepare(ctx, hints, [0.5, 1.0], cfg_duplicated=True)
    eng.set_schedule(ts, a, ap)
    eng.begin(x[:n_img], guidance=9.0, use_graph=not args.no_graph)
    for _ in range(3):
        eng.step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k = 10
    e0.record()
    for _ in range(k):
        eng.step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / k
    tf = STEP_TFLOP * n_img
    return {"images_per_gpu": n_img, "network_batch": 2 * n_img, "ms_per_step": round(ms, 4), "steps_timed": k,
            "step_tflop": round(tf, 3), "achieved_tflops": round(tf / (ms * 1e-3), 1),
            "frac_of_sustained_peak": round(tf / (ms * 1e-3) / sust, 4),
            "images_per_s_denoise_only": round(n_img * 1000.0 / (DDIM_STEPS * ms), 4),
            "launches_per_step": int(getattr(eng, "launches_per_step", 0) or 0),
            "outputs_finite": bool(torch.isfinite(eng.latents()).all().item())}


def run_ours(args, rank, world, local_rank):
    import torch.distributed as dist
    from editanything_b200 import ops
    from editanything_b200.denoise import DenoiseEngine, ddim_schedule
    from editanything_b200.unet_spec import SD15, make_state_dict
    dev = torch.device(f"cuda:{local_rank}")
    torch.cuda.set_device(dev)
    cfg = SD15
    sust, burst, hbm, peak_src = _peaks()

    usd = make_state_dict(cfg, "unet", 101, device=dev)
    csds = [make_state_dict(cfg, "controlnet", 102, device=dev), make_state_dict(cfg, "controlnet", 103, device=dev)]
    eng = DenoiseEngine(cfg, usd, csds, dev)
    del usd, csds
    torch.cuda.empty_cache()
    n_img = max(1, args.images_per_gpu)          # images per GPU; the network batch is 2 * n_img (CFG)
    x, ctx, hints = make_inputs(cfg, 2 * n_img, 64, 77, 11 + rank)
    ts, a, ap = ddim_schedule(DDIM_STEPS)

    def run_steps(k):
        """k fused steps: ONE graph launch each; the per-step scalars (DDIM coefficients, time-embedding rows) are
        rows of device tables indexed by a device counter (DenoiseEngine.set_schedule).  Past the 50th step the
        counter stays on the last row - the same kernels on the same shapes."""
        for _ in range(k):
            eng.step()

    # ---- device-resident timed region: exactly K denoising steps --------------------------------
    eng.prepare(ctx, hints, [0.5, 1.0], cfg_duplicated=True)
    eng.set_schedule(ts, a, ap)
    eng.begin(x[:n_img], guidance=9.0, use_graph=not args.no_graph)
    run_steps(args.warmup)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ops.reset_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    if args.profiler_range:
        torch.cuda.profiler.start()          # ncu --profile-from-start off: capture the timed region only
    e0.record()
    run_steps(args.steps)
    e1.record()
    torch.cuda.synchronize()
    if args.profiler_range:
        torch.cuda.profiler.stop()
    if world > 1:
        dist.barrier()
    clocks = sampler.stop()
    ms_total = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms_total], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = t.item()
    ms_step = ms_total / args.steps
    launches_per_step = getattr(eng, "launches_per_step", None)
    if launches_per_step is None:
        launches_per_step = ops.launch_count() // max(1, args.steps)
    finite = bool(torch.isfinite(eng.latents()).all().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, latents=eng.latents())

    # ---- SAM ViT-H encoder (once per image) -----------------------------------------------------
    sam_ms, sam_note, sam = None, "skipped (--no-sam): images/s below is denoise-only", None
    try:
        if args.no_sam:
            raise ImportError("skipped")
        from editanything_b200.sam import SamEncoderEngine, make_sam_state_dict, SAM_VIT_H
        ssd = make_sam_state_dict(SAM_VIT_H, 201, device=dev)
        sam = SamEncoderEngine(SAM_VIT_H, ssd, dev)
        del ssd
        img = torch.randn(1, 3, 1024, 1024, device=dev)
        for _ in range(2):
            sam.encode(img)
        torch.cuda.synchronize()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(3):
            sam.encode(img)
        s1.record()
        torch.cuda.synchronize()
        sam_ms = s0.elapsed_time(s1) / 3
        sam_note = "SAM ViT-H 1024x1024 encode, device-timed, 3 iterations"
    except ImportError:
        pass

    # ---- first-stage decoder (once per image; SURVEY.md 8f N1) -----------------------------------
    vae_ms, vae_enc_ms, vae = None, None, None
    if not args.no_vae:
        from editanything_b200.vae import SD_VAE, VaeEngine, make_vae_state_dict
        vsd = dict(make_vae_state_dict(SD_VAE, 412, device=dev, part="encoder"))
        vsd.update(make_vae_state_dict(SD_VAE, 402, device=dev))
        vae = VaeEngine(SD_VAE, vsd, dev)
        del vsd
        lat = eng.latents().float()[:1]
        src = torch.rand(1, 3, 512, 512, device=dev) * 2 - 1          # the masked source image (prepare_masked_image_latents)

        def _time(fn):
            for _ in range(2):
                fn()
            torch.cuda.synchronize()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record()
            for _ in range(3):
                fn()
            s1.record()
            torch.cuda.synchronize()
            return s0.elapsed_time(s1) / 3
        vae_ms = _time(lambda: vae.decode_latents(lat))
        vae_enc_ms = _time(lambda: vae.encode(src))

    # n_img images per GPU share the 50 steps; SAM encode, VAE encode and decode run once per image
    # per-request preparation (prompt K/V of every attention layer + the ControlNet hint stacks), device-timed
    torch.cuda.synchronize()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    for _ in range(3):
        eng.prepare(ctx, hints, [0.5, 1.0], cfg_duplicated=True)
    p1.record()
    torch.cuda.synchronize()
    prepare_ms = p0.elapsed_time(p1) / 3
    img_ms = DDIM_STEPS * ms_step + n_img * ((sam_ms or 0.0) + (vae_ms or 0.0) + (vae_enc_ms or 0.0))
    value = world * n_img * 1000.0 / img_ms
    step_tflop = STEP_TFLOP * n_img

    # ---- roofline of the dominant kernel (ea_gemm_kernel), live CUDA events ----------------------
    probe = GemmProbe(ops)
    eng_ops_saved = (eng.ops, eng.runner.ops, eng.unet.ops, [c.ops for c in eng.cns])
    eng.ops = eng.runner.ops = eng.unet.ops = probe
    for c in eng.cns:
        c.ops = probe
    eng._use_graph = False
    j = (args.warmup + args.steps) % DDIM_STEPS
    eng.step(int(ts[j]), float(a[j]), float(ap[j]))
    probe.records.clear()
    eng.step(int(ts[j]), float(a[j]), float(ap[j]))
    torch.cuda.synchronize()
    g_fl = sum(r[4] for r in probe.records)
    n_gemm = len(probe.records)
    g_ms = probe.replay_time_ms()
    eng.ops, eng.runner.ops, eng.unet.ops = eng_ops_saved[0], eng_ops_saved[1], eng_ops_saved[2]
    for c, o in zip(eng.cns, eng_ops_saved[3]):
        c.ops = o
    achieved = g_fl / (g_ms * 1e-3) / 1e12 if g_ms > 0 else 0.0
    # operand bytes the algorithm needs per launch (A + W + out (+ residual)), averaged over the step's launches
    alg_bytes = 0
    flat = []
    for rec in probe.records:
        flat += [(a_, w_, o_, k_, 0) for a_, w_, o_, k_ in rec[1]] if rec[0] == "grouped" else [rec]
    for a_, w_, out_, kw_, _ in flat:
        conv = kw_.get("conv")
        Mrows = conv[0] * conv[1] * conv[2] if conv else (kw_.get("M") or a_.shape[0])
        Kin = conv[3] if conv else w_.shape[1]
        n_out = w_.shape[0] // 2 if kw_.get("act") == 3 else w_.shape[0]
        alg_bytes += 2 * (Mrows * Kin + w_.numel() + Mrows * n_out * (2 if kw_.get("residual") is not None else 1))
    traffic, traffic_src = _gemm_traffic()
    roofline = {"bound": "tensor", "kernel": "ea_gemm_kernel", "achieved": round(achieved, 1), "peak": sust,
                "unit": "TFLOP/s", "frac": round(achieved / sust, 4), "traffic": traffic,
                "traffic_note": traffic_src, "algorithmic_bytes_per_launch": round(alg_bytes / max(n_gemm, 1)),
                "peak_source": f"{peak_src} bf16_tflops_sustained (kernel timed inside a long step)",
                "launches": n_gemm, "gemm_ms_per_step": round(g_ms, 3),
                "timing": "all ea_gemm launches of one step re-issued back to back in one CUDA graph, CUDA events",
                "gemm_tflop_per_step": round(g_fl / 1e12, 3),
                "whole_step": {"tflop": step_tflop, "achieved": round(step_tflop / (ms_step * 1e-3), 1),
                               "frac": round(step_tflop / (ms_step * 1e-3) / sust, 4)}}

    # ---- e2e: host buffers in, host result out, through the public engine API ---------------------
    e2e = None
    if (rank == 0 or world > 1) and not args.no_e2e:
        # n_img images per GPU end to end through the public engine API, inputs in PINNED HOST memory:
        #   H2D preprocessed image -> SAM ViT-H encode -> D2H embedding (what the mask decoder / AMG consume)
        #   H2D prompt embeddings, ControlNet conditioning images, initial noise -> prepare (ctx K/V, hint
        #   stacks) -> 50 fused steps (one graph launch each) -> VAE decode -> uint8 image tiles [n, H, W, 3]
        #   -> (world > 1) ONE NCCL all-gather of every rank's tiles (SURVEY.md 8e) -> D2H.
        # One untimed warm-up pass (CUDA-graph capture, allocator), then n_rep timed passes.
        hx, hctx = x[:n_img].pin_memory(), ctx.pin_memory()
        hh = [h.pin_memory() for h in hints]
        himg = torch.randn(1, 3, 1024, 1024).pin_memory() if sam is not None else None
        hsrc = (torch.rand(1, 3, 512, 512) * 2 - 1).pin_memory() if vae is not None else None
        n_rep = 5
        from editanything_b200.sharding import gather_sharded

        def one_pass():
            emb = None
            for _ in range(n_img):
                if sam is not None:
                    emb = sam.encode(himg.to(dev, non_blocking=True)).cpu()
                if vae is not None:  # masked-image latents (utils/...inpaint.py:1056-1105); consumed by the blend
                    vae.encode(hsrc.to(dev, non_blocking=True)).latent_dist.sample()
            eng.prepare(hctx.to(dev, non_blocking=True), [h.to(dev, non_blocking=True) for h in hh], [0.5, 1.0], cfg_duplicated=True)
            eng.set_schedule(ts, a, ap)
            eng.begin(hx.to(dev, non_blocking=True), guidance=9.0, use_graph=not args.no_graph)
            for _ in range(DDIM_STEPS):
                eng.step()
            if vae is not None:   # decoded images as uint8 tiles (what numpy_to_pil makes of them, :333-335)
                img = torch.cat([vae.decode_latents(eng.latents()[i:i + 1].float()) for i in range(n_img)])
                res = (img.permute(0, 2, 3, 1) * 255).round().to(torch.uint8).contiguous()
            else:
                res = eng.latents()
            if world > 1:
                res = gather_sharded(res, world * n_img, rank, world) if n_img == 1 else \
                    torch.cat(_all_gather_list(res, world))          # the single end-of-job collective
            return res.cpu(), emb

        import gc
        one_pass()
        one_pass()
        torch.cuda.synchronize()
        # the timed passes run with the cyclic garbage collector parked, as a serving process would (gc.freeze() after
        # start-up): a generation-2 collection over the imported module graph is a 50-200 ms host stall that landed in
        # some runs' timed region and not in others (e2e 362 vs 417-437 ms / image at the same device time)
        gc.collect()
        gc.freeze()
        gc.disable()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        pass_ms = []
        for _ in range(n_rep):
            tp = time.perf_counter()
            res, emb = one_pass()          # ends with a D2H copy of the result: the pass is complete when it returns
            pass_ms.append(round((time.perf_counter() - tp) * 1e3, 1))
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        gc.enable()
        if world > 1:
            t = torch.tensor([dt], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = t.item()
            assert res.shape[0] == world * n_img
        h2d = (hx.numel() + hctx.numel() + sum(h.numel() for h in hh)) * 4 + n_img * (
            (himg.numel() if himg is not None else 0) + (hsrc.numel() if hsrc is not None else 0)) * 4
        d2h = res.numel() * res.element_size() + n_img * (emb.numel() * 4 if emb is not None else 0)
        e2e = {"value": round(world * n_img * n_rep / dt, 4), "unit": "images/s",
               "h2d_bytes_per_step": h2d // DDIM_STEPS, "d2h_bytes_per_step": d2h // DDIM_STEPS,
               "ms_per_image": round(dt / (n_rep * n_img) * 1e3, 2), "images_timed": n_rep * n_img,
               "pass_ms": pass_ms,
               "note": "per image: pinned host image -> H2D -> SAM ViT-H encode -> D2H embedding; pinned host source "
                       "image -> H2D -> VAE encode; pinned host ctx / hints / noise -> H2D -> prepare (ctx K/V, hint "
                       "stacks) -> 50 fused steps (one graph launch per step) -> VAE decode -> uint8 tiles -> "
                       "(N > 1: one NCCL all-gather of all ranks' tiles, inside the timed region) -> D2H; 2 untimed "
                       "warm-up passes, garbage collector parked; text encoder / SAM mask decoder not included (SURVEY.md 8f)"}

    line = {
        "metric": "512x512 50-step SAM+ControlNet-inpaint images/sec; fused ControlNetx2+UNet+CFG+DDIM step ms",
        "value": round(value, 4), "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms_step, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp16 storage / fp32 accumulate" if ops.half_dtype() == torch.float16 else "bf16 storage / fp32 accumulate",
        "data": "synthetic inputs, seeded random weights (SD1.5 topology, 859.5M + 2x361.3M params)",
        "config": {"workload": ("BASELINE.json configs[1]: SD1.5 ControlNet-inpaint 512x512, 50 DDIM steps, batch=1/GPU "
                                "(+CFG => B=2), SAM+inpaint ControlNets, L=77") if n_img == 1 else
                               (f"BASELINE.json configs[3] shard: SD1.5 ControlNet-inpaint 512x512, 50 DDIM steps, "
                                f"batch={n_img}/GPU (+CFG => B={2 * n_img}), SAM+inpaint ControlNets, L=77"),
                   "global_batch": world * n_img,
                   "parallelism": f"dp{world} ({n_img} image(s) per GPU, final all-gather of uint8 tiles)",
                   "l2": "weights touched per step (3.16 GB) exceed the 126 MB L2; no explicit flush",
                   "cuda_graph": not args.no_graph, "sam_ms_per_image": sam_ms, "sam": sam_note,
                   "vae_decode_ms_per_image": vae_ms, "vae_encode_ms_per_image": vae_enc_ms,
                   "image": "image_ms = 50 x ms_per_step + images_per_gpu x (SAM encode + VAE encode of the masked source "
                            "image (512x512 -> 64x64 latents) + VAE decode (64x64 -> 512x512), kl-f8); "
                            "value = n_gpus x images_per_gpu x 1000 / image_ms",
                   "images_per_gpu": n_img, "prepare_ms_per_request": round(prepare_ms, 3),
                   "image_ms": round(img_ms, 3), "outputs_finite": finite},
        "gpu_launches": int(launches_per_step) * args.steps, "launches_per_step": int(launches_per_step),
        "clocks": clocks, "roofline": roofline, "e2e": e2e,
    }
    if n_img == 1 and not args.no_batch4:
        # BASELINE.json configs[3] (4 images per GPU): where the weight-bound 8x8 / 16x16 levels amortise
        line["config"]["batch4"] = measure_batch_block(eng, cfg, 4, rank, sust, args, ts, a, ap)
        if world > 1:
            t = torch.tensor([line["config"]["batch4"]["ms_per_step"]], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            b4 = line["config"]["batch4"]
            b4["ms_per_step"] = round(t.item(), 4)
            b4["images_per_s_denoise_only"] = round(world * 4 * 1000.0 / (DDIM_STEPS * t.item()), 4)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(sample_steps=1)
    if rank == 0:
        print(json.dumps(line), file=_JSON_OUT, flush=True)


def _oracle_step_fn(cfg):
    """Builds the CPU step (ControlNet x2 -> UNet -> CFG -> DDIM) at configs[1] size: the REFERENCE's own
    cldm.ControlNet / ControlledUnetModel modules when they are available (oracle/_ref, made by oracle/build_ref.py
    in the build container and shipped with the snapshot; kind "reference"), else the oracle port (kind "port").
    Returns (step, kind)."""
    from editanything_b200.unet_spec import build_topology, make_state_dict
    from oracle import ref_shim
    from oracle import unet_oracle as O
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    usd = {k: v.cpu() for k, v in make_state_dict(cfg, "unet", 101, device=dev).items()}
    csds = [{k: v.cpu() for k, v in make_state_dict(cfg, "controlnet", s, device=dev).items()} for s in (102, 103)]
    ut, ct = build_topology(cfg), build_topology(cfg, with_decoder=False)
    x, ctx, hints = make_inputs(cfg, 2, 64, 77, 11)
    ts, a, ap = O.make_ddim_schedule(DDIM_STEPS)
    state = {"lat": x[:1].clone(), "i": len(ts) - 1}
    kind, ref_nets = "port", None
    if ref_shim.available():
        try:
            ref_nets = ref_shim.build_reference_nets(cfg, usd, csds)
            kind = "reference"
            usd = csds = None
        except Exception as e:          # e.g. a missing third-party import on this box: fall back to the port
            sys.stderr.write(f"reference modules unusable ({type(e).__name__}: {e}); timing the oracle port\n")

    def step():
        i = state["i"]
        xx = torch.cat([state["lat"], state["lat"]])
        tt = torch.full((2,), int(ts[i]))
        with torch.no_grad():
            if ref_nets is not None:
                e, _ = ref_shim.reference_apply_model(ref_nets[0], ref_nets[1], xx, tt, ctx, hints, [0.5, 1.0])
            else:
                e = O.apply_model(usd, ut, [(sd, ct) for sd in csds], xx, tt, ctx, hints, [0.5, 1.0])
        state["lat"], _ = O.ddim_step(state["lat"], e[:1], e[1:], 9.0, float(a[i]), float(ap[i]))
        state["i"] = i - 1 if i > 0 else len(ts) - 1
    return step, kind


def usable_cores():
    """Host threads this process may actually run on: the scheduler affinity mask capped by the
    cgroup CPU quota (a 128-thread box that grants the container fewer CPUs thrashes when torch
    spawns one thread per logical CPU: 151 s/step measured vs 12.8 s on 8 dedicated cores), and by
    64, beyond which the oracle's small-batch convolutions stop scaling."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(per))))
    except Exception:
        pass
    return max(1, min(n, 64))


def _oracle_sam_seconds():
    """One SAM ViT-H image-encoder pass (1024x1024) of the CPU oracle, fp32, no warm-up (~30-60 s)."""
    from editanything_b200.sam_spec import SAM_VIT_H, make_sam_state_dict
    from oracle import sam_oracle as S
    sd = make_sam_state_dict(SAM_VIT_H, 201)
    img = torch.randn(1, 3, 1024, 1024, generator=torch.Generator().manual_seed(3))
    t0 = time.perf_counter()
    with torch.no_grad():
        S.image_encoder(sd, SAM_VIT_H, img)
    return time.perf_counter() - t0


def _oracle_vae_seconds():
    """One first-stage encode (512x512 -> 64x64) + decode (64x64 -> 512x512) of the CPU oracle, fp32 (~15-30 s)."""
    from editanything_b200.vae_spec import SD_VAE, make_vae_state_dict
    from oracle import vae_oracle as V
    sd = make_vae_state_dict(SD_VAE, 402)
    esd = make_vae_state_dict(SD_VAE, 412, part="encoder")
    lat = torch.randn(1, 4, 64, 64, generator=torch.Generator().manual_seed(4)) * SD_VAE.scaling_factor
    src = torch.rand(1, 3, 512, 512, generator=torch.Generator().manual_seed(5)) * 2 - 1
    t0 = time.perf_counter()
    with torch.no_grad():
        V.encode_moments(src, esd, SD_VAE)
        V.decode_latents(lat, sd, SD_VAE)
    return time.perf_counter() - t0


def cpu_baseline(sample_steps=1):
    from editanything_b200.unet_spec import SD15
    cores = usable_cores()
    torch.set_num_threads(cores)
    step, kind = _oracle_step_fn(SD15)
    step()  # warm-up (allocator, thread pool)
    t0 = time.perf_counter()
    for _ in range(sample_steps):
        step()
    dt = (time.perf_counter() - t0) / sample_steps
    sam_s = _oracle_sam_seconds()
    vae_s = _oracle_vae_seconds()
    return {"value": round(1.0 / (DDIM_STEPS * dt + sam_s + vae_s), 6), "unit": "images/s", "cores": cores, "kind": kind,
            "step_impl": "the reference's own cldm.ControlNet x2 + ControlledUnetModel (oracle/_ref)" if kind == "reference"
                         else "oracle port of the reference's ldm/cldm modules",
            "ms_per_step": round(dt * 1e3, 1), "sam_ms_per_image": round(sam_s * 1e3, 1),
            "vae_encode_decode_ms_per_image": round(vae_s * 1e3, 1),
            "sample": f"{sample_steps} full-size fused step(s) (2 ControlNets + UNet + CFG + DDIM, B=2, 64x64, fp32) of the "
                      f"CPU arm on {cores} host threads after 1 warm-up + 1 SAM ViT-H encode + 1 VAE encode + decode of the oracle "
                      f"port (segment_anything / diffusers are absent); images/s = 1/(50*step + SAM + VAE)"}


def run_reference(args, rank, world):
    """Reference arm: the reference's own algorithm (oracle port of its ldm/cldm modules; the
    reference is pure Python and cannot travel to the box) on the host cores, rank 0 only."""
    if rank != 0:
        return
    from editanything_b200.unet_spec import SD15
    cores = usable_cores()
    torch.set_num_threads(cores)
    step, kind = _oracle_step_fn(SD15)
    budget_s = 240.0
    t0 = time.perf_counter()
    step()
    first = time.perf_counter() - t0
    n_w = max(0, min(args.warmup - 1, int(budget_s * 0.2 / max(first, 1e-3))))
    for _ in range(n_w):
        step()
    k = max(1, min(args.steps, int(budget_s * 0.8 / max(first, 1e-3))))
    t0 = time.perf_counter()
    for _ in range(k):
        step()
    dt = (time.perf_counter() - t0) / k
    sam_s = _oracle_sam_seconds()
    vae_s = _oracle_vae_seconds()
    v = round(1.0 / (DDIM_STEPS * dt + sam_s + vae_s), 6)
    sample = (f"{k} of the requested {args.steps} steps timed (each a full-size configs[1] fused step on CPU, fp32, "
              f"{cores} threads; bounded to ~{int(budget_s)} s) + 1 SAM ViT-H encode ({sam_s:.1f} s) + 1 VAE encode + decode "
              f"({vae_s:.1f} s); images/s = 1/(50*step + SAM + VAE)")
    line = {"impl": "reference",
            "metric": "512x512 50-step SAM+ControlNet-inpaint images/sec; fused ControlNetx2+UNet+CFG+DDIM step ms",
            "value": v, "unit": "images/s", "n_gpus": world, "steps": k, "warmup": 1 + n_w,
            "ms_per_step": round(dt * 1e3, 2), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "fp32", "data": "synthetic inputs, seeded random weights",
            "config": {"workload": "BASELINE.json configs[1]: SD1.5 ControlNet-inpaint 512x512, 50 DDIM steps, batch=1 "
                                   "(+CFG => B=2), SAM+inpaint ControlNets, L=77 - on the host CPU: " +
                                   ("the reference's own cldm modules (oracle/_ref)" if kind == "reference" else "oracle port")},
            "cpu_baseline": {"value": v, "unit": "images/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), file=_JSON_OUT, flush=True)


_JSON_OUT = sys.stdout


def main():
    # stdout carries exactly ONE line (the JSON): anything a library prints on the way (the reference's modules announce
    # a missing xformers at import) goes to stderr
    # ... including what C libraries write to file descriptor 1 (NCCL announces its version there): fd 1 is pointed at
    # stderr and the JSON line goes to a duplicate of the original stdout
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = sys.stderr
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-vae", action="store_true", help="skip the first-stage decode (kernel profiling runs)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profiler-range", action="store_true",
                    help="bracket the timed region with cudaProfilerStart/Stop (for ncu --profile-from-start off)")
    ap.add_argument("--no-sam", action="store_true", help="profiling runs only: skip the SAM encoder leg")
    ap.add_argument("--no-e2e", action="store_true", help="profiling runs only (ncu): skip the e2e leg")
    ap.add_argument("--images-per-gpu", type=int, default=1,
                    help="images per GPU (network batch = 2x with CFG); 4 = BASELINE.json configs[3]")
    ap.add_argument("--no-batch4", action="store_true", help="skip the extra configs[3] (4 images per GPU) block")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what their last step produced (the latents, [images, 4, 64, 64]) "
                         "as DIR/latents.npy, float32; rank 0 only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(3, args.warmup)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
