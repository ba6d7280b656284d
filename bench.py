#!/usr/bin/env python
"""Headline benchmark: denoise-step latents/sec, Wan2.1-T2V-14B 720p x 81f (BASELINE.json configs[1]).

One "step" = scheduler.step_pre + model.infer (cond + uncond forwards, CFG combine; 2 x 40 DiT blocks over 75 600 tokens,
pre/post-infer included) + scheduler.step_post — the body of DefaultRunner.run's loop (lightx2v/models/runners/default_runner.py:97-114).
Synthetic latents / prompt embeddings / random-init weights of the named shapes (no datasets or checkpoints offline).

    python bench.py [--gpus N --steps K --warmup W]            our sm_100a path  (N > 1: torchrun, Ulysses over the token axis)
    python bench.py --impl reference [...]                     the reference's CPU torch path (oracle port) on the host cores,
                                                               bounded sample extrapolated by the FLOP model of SURVEY.md §8d
    python bench.py --workload <name> ...                      the other BASELINE configs (fp8 distill, i2v, HunyuanVideo + VAE, ...)
    python bench.py ... --dump-outputs DIR                     also write what the last timed step computed as DIR/<name>.npy

Prints ONE JSON line on stdout (rank 0, flushed); progress lines with wall-clock stamps go to stderr.  The whole run is sized
against --budget-s (default 480 s of wall clock per process): the W warm-up and K timed steps are always run as asked; the
end-to-end (host-buffer) loop runs as many of K steps as still fit (>= 1, reported as e2e.steps); the side legs (VAE decode, the
reference's GPU path, cpu_baseline) run only at N = 1 outside torchrun and only while budget remains.
Weights and inputs are drawn from fixed seeds, so the same arguments give the same inputs on every run and two builds can be
compared output for output with --dump-outputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

T0 = time.time()
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def log(msg):
    if int(os.environ.get("RANK", "0")) == 0:
        print(f"[bench +{time.time() - T0:7.1f}s] {msg}", file=sys.stderr, flush=True)


log("importing torch")
import torch  # noqa: E402

log("torch imported")

METRIC = "denoise-step latents/sec (Wan2.1-14B 720p x 81f)"
WORKLOADS = {
    # name: dims of the DiT + latent shape
    "wan2.1-t2v-14b-720p-81f": dict(dim=5120, num_heads=40, ffn_dim=13824, num_layers=40, target_shape=(16, 21, 90, 160), infer_steps=50,
                                    enable_cfg=True, sample_guide_scale=5.0, sample_shift=5.0),
    # BASELINE config 3: w8a8-fp8 linears (weights quantised per out-channel at load), 4-step distilled sampler, no CFG
    "wan2.1-t2v-14b-fp8-distill-720p-81f": dict(dim=5120, num_heads=40, ffn_dim=13824, num_layers=40, target_shape=(16, 21, 90, 160), infer_steps=4,
                                                enable_cfg=False, sample_guide_scale=1.0, sample_shift=5.0, fp8=True, distill=True),
    # north_star's w4a4-nvfp4 weight path on the same distilled sampler (the reference ships the kernels but no model wiring for it)
    "wan2.1-t2v-14b-nvfp4-distill-720p-81f": dict(dim=5120, num_heads=40, ffn_dim=13824, num_layers=40, target_shape=(16, 21, 90, 160), infer_steps=4,
                                                  enable_cfg=False, sample_guide_scale=1.0, sample_shift=5.0, nvfp4=True, distill=True),
    # BASELINE config 4: image-to-video (36 input channels = 16 noise + 4 mask + 16 VAE-encoded image, 257 CLIP tokens in a second cross-attention)
    "wan2.1-i2v-14b-720p-81f": dict(dim=5120, num_heads=40, ffn_dim=13824, num_layers=40, target_shape=(16, 21, 90, 160), infer_steps=50,
                                    enable_cfg=True, sample_guide_scale=5.0, sample_shift=5.0, task="i2v"),
    "wan2.1-t2v-1.3b-480p-17f": dict(dim=1536, num_heads=12, ffn_dim=8960, num_layers=30, target_shape=(16, 5, 60, 104), infer_steps=50,
                                     enable_cfg=True, sample_guide_scale=5.0, sample_shift=5.0),   # quick self-test of this script
}
HUNYUAN = "hunyuan-13b-720p-129f"          # BASELINE config 5: DiT block stack + 3D VAE decode


class Budget:
    """Wall-clock budget of this process (seconds since interpreter start)."""

    def __init__(self, total_s):
        self.total = float(total_s)

    def left(self):
        return self.total - (time.time() - T0)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d["bf16_tflops_sustained"], d["hbm_gbs"], "MEASURED_PEAKS.json (sustained: the kernel is timed inside a long step)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel, shape):
    """DRAM read+write bytes per launch of `kernel` at `shape` from the committed `ncu --set full` summaries (profiles/roofline_traffic.json,
    each entry naming the summary file it was read from); None when no capture of that shape is committed."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    try:
        for e in json.load(open(p))["entries"]:
            if e["kernel"] == kernel and list(e["shape"]) == list(shape):
                return e["dram_bytes_per_launch"], e["source"]
    except Exception:
        pass
    return None, None


def step_flops(cfg):
    from oracle.wan_oracle import block_flops  # FLOP model only (SURVEY.md §8d); not on the measured path
    C, Fr, H, W = cfg["target_shape"]
    S = Fr * (H // 2) * (W // 2)
    per_fwd = cfg["num_layers"] * block_flops(S, cfg["dim"], cfg["ffn_dim"], 512, i2v=cfg.get("task") == "i2v")
    return S, per_fwd * (2 if cfg["enable_cfg"] else 1)


def synth_weights(cfg, device, seed=42):
    """Random-init weights with the checkpoint's key names and shapes (SURVEY.md §8d recipe), generated on the device."""
    g = torch.Generator(device=device).manual_seed(seed)
    D, F_, L = cfg["dim"], cfg["ffn_dim"], cfg["num_layers"]
    W = {}

    def rnd(*shape, scale=0.02):
        return (torch.randn(*shape, generator=g, device=device, dtype=torch.float32) * scale).to(torch.bfloat16)

    def lin(name, n, k):
        W[name + ".weight"] = rnd(n, k)
        W[name + ".bias"] = rnd(n)

    i2v = cfg.get("task") == "i2v"
    W["patch_embedding.weight"] = rnd(D, 36 if i2v else 16, 1, 2, 2, scale=0.05)
    W["patch_embedding.bias"] = rnd(D)
    lin("text_embedding.0", D, 4096)
    lin("text_embedding.2", D, D)
    lin("time_embedding.0", D, 256)
    lin("time_embedding.2", D, D)
    lin("time_projection.1", 6 * D, D)
    lin("head.head", 64, D)
    W["head.modulation"] = rnd(1, 2, D, scale=0.1)
    for i in range(L):
        p = f"blocks.{i}."
        W[p + "modulation"] = rnd(1, 6, D, scale=0.1)
        for nm in ("q", "k", "v", "o"):
            lin(p + "self_attn." + nm, D, D)
            lin(p + "cross_attn." + nm, D, D)
        for nm in ("self_attn.norm_q", "self_attn.norm_k", "cross_attn.norm_q", "cross_attn.norm_k", "norm3"):
            W[p + nm + ".weight"] = (1.0 + rnd(D, scale=0.05).float()).to(torch.bfloat16)
        W[p + "norm3.bias"] = rnd(D)
        lin(p + "ffn.0", F_, D)
        lin(p + "ffn.2", D, F_)
        if i2v:
            lin(p + "cross_attn.k_img", D, D)
            lin(p + "cross_attn.v_img", D, D)
            W[p + "cross_attn.norm_k_img.weight"] = (1.0 + rnd(D, scale=0.05).float()).to(torch.bfloat16)
    if i2v:                                                       # img_emb.proj: LN(1280) -> Linear(1280, 1280) -> GELU -> Linear(1280, D) -> LN(D)
        W["img_emb.proj.0.weight"], W["img_emb.proj.0.bias"] = (1.0 + rnd(1280, scale=0.05).float()).to(torch.bfloat16), rnd(1280)
        lin("img_emb.proj.1", 1280, 1280)
        lin("img_emb.proj.3", D, 1280)
        W["img_emb.proj.4.weight"], W["img_emb.proj.4.bias"] = (1.0 + rnd(D, scale=0.05).float()).to(torch.bfloat16), rnd(D)
    return W


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = sorted(float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 7 and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


def dist_env():
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    return world, rank, local_rank


def init_dist(dev, world):
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
        log(f"NCCL process group up ({world} ranks)")


def barrier(world):
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()


def timed_loop(step_fn, n_steps, world):
    """EXACTLY n_steps of step_fn bracketed by barrier + synchronize on both sides; CUDA events on the current stream. -> ms per step (this rank)."""
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(world)
    t0.record()
    for _ in range(n_steps):
        step_fn()
    t1.record()
    barrier(world)
    return t0.elapsed_time(t1) / n_steps


DUMP_LIMIT_BYTES = 64 * 2**20


def dump_outputs(out_dir, arrays):
    """Write each tensor of `arrays` as <out_dir>/<name>.npy in float32."""
    import numpy as np
    total = sum(t.numel() * 4 for t in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())
    log(f"outputs of the last timed step written to {out_dir}: {', '.join(f'{k}{list(v.shape)}' for k, v in arrays.items())}")


def max_over_ranks(vals, dev, world):
    if world > 1:
        t = torch.tensor(vals, device=dev, dtype=torch.float64)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return t.tolist()
    return list(vals)


def roofline_from_profile(prof, want, peak_tf, peak_src, kernel_name):
    """prof: lib.prof_fmha_end() records (ms, sq, sk, heads, d); `want` selects the dominant launches."""
    fm = [r for r in prof if want(r) and r[0] > 0]
    if not fm:
        return None
    avg_ms = sum(r[0] for r in fm) / len(fm)
    _, sq, sk, h, d = fm[0]
    fl = 4.0 * sq * sk * h * d
    ach = fl / (avg_ms * 1e-3) / 1e12
    traffic, tsrc = ncu_traffic(kernel_name, (sq, sk, h, d))
    return {"kernel": kernel_name + " (self-attention)", "bound": "tensor", "achieved": round(ach, 1), "peak": peak_tf, "unit": "TFLOP/s",
            "frac": round(ach / peak_tf, 4), "traffic": traffic, "traffic_unit": "bytes/launch (ncu dram__bytes_read.sum + dram__bytes_write.sum)",
            "traffic_source": tsrc, "launch_ms": round(avg_ms, 3), "launches_timed": len(fm), "algorithmic_flop_per_launch": fl,
            "timing": "CUDA event pair recorded by the library around every attention launch on the launching stream (b200_prof_fmha_begin/_end)",
            "peak_source": peak_src}


# ===================================================================================================================== Wan workloads
def run_ours(args):
    from lightx2v_b200 import lib
    from lightx2v_b200.host import ulysses
    from lightx2v_b200.host.wan_model import WanModel
    from lightx2v_b200.host.wan_scheduler import WanScheduler

    budget = Budget(args.budget_s)
    world, rank, local_rank = dist_env()
    under_torchrun = "WORLD_SIZE" in os.environ
    side_legs = world == 1 and not under_torchrun

    cfg = dict(WORKLOADS[args.workload])
    cfg.update(task=cfg.get("task", "t2v"), freq_dim=256, text_len=512, in_dim=36 if cfg.get("task") == "i2v" else 16, out_dim=16, seed=42, mm_config={},
               patch_size=(1, 2, 2))
    S, flops_step = step_flops(cfg)

    # ---- the reference's CPU path first (no GPU involved, hard time cap), so a later stall can never take it along
    cpu_base = None
    if args.cpu_baseline and side_legs and rank == 0:
        log("cpu_baseline: oracle port on the host cores (bounded sample)")
        cpu_base = cpu_reference_sample(cfg, flops_step, budget_s=min(args.cpu_budget, max(3.0, budget.left() * 0.05)))
        log(f"cpu_baseline done: {cpu_base['value']:.3e} latents/s on {cpu_base['cores']} threads")

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    init_dist(dev, world)
    lib.load()
    log(f"libb200dit.so loaded, {lib.load().b200_num_sms()} SMs")

    if cfg.get("fp8"):
        from lightx2v_b200.host.ops import FP8_MM_KEY
        cfg["mm_config"] = {"mm_type": FP8_MM_KEY, "weight_auto_quant": True}
    if cfg.get("nvfp4"):
        from lightx2v_b200.host.ops import NVFP4_MM_KEY
        cfg["mm_config"] = {"mm_type": NVFP4_MM_KEY}
    if cfg.get("distill"):
        cfg["denoising_step_list"] = [1000, 750, 500, 250]
    # The library's default schedule is measured: one native b200_wan_block_fwd call per block when eligible (bf16 linears, single GPU),
    # the per-op entry points otherwise (fp8 / nvfp4 / sequence parallel).  Launches and attention timings are counted below the C ABI.
    cfg["b200_native_block"] = not args.per_op
    W = synth_weights(cfg, dev)
    model = WanModel.from_weight_dict(cfg, W)
    graphed = bool(args.graph) and world == 1 and not cfg.get("distill")
    if cfg.get("distill"):
        from lightx2v_b200.host.wan_scheduler import WanStepDistillScheduler
        sched = WanStepDistillScheduler(cfg, device=dev)
    elif graphed:
        from lightx2v_b200.host.wan_graph import WanSchedulerDevice
        sched = WanSchedulerDevice(cfg, device=dev)
    else:
        sched = WanScheduler(cfg, device=dev)
    sched.prepare()
    model.set_scheduler(sched)
    log(f"model built: {args.workload}, {S} tokens, {torch.cuda.memory_allocated() / 2**30:.1f} GiB allocated")
    g = torch.Generator(device=dev).manual_seed(7)
    ctx = {"context": torch.randn(512, 4096, generator=g, device=dev).to(torch.bfloat16),
           "context_null": torch.randn(512, 4096, generator=g, device=dev).to(torch.bfloat16)}
    inputs = {"text_encoder_output": ctx, "image_encoder_output": None}
    if cfg["task"] == "i2v":      # synthetic encoder outputs of the published shapes (SURVEY.md 8d): CLIP ViT-H tokens, VAE-encoded image + mask
        ts = cfg["target_shape"]
        inputs["image_encoder_output"] = {"clip_encoder_out": torch.randn(257, 1280, generator=g, device=dev).to(torch.bfloat16),
                                          "vae_encode_out": torch.randn(20, ts[1], ts[2], ts[3], generator=g, device=dev).to(torch.bfloat16)}

    if world > 1:
        sp_mode = args.sp
        if args.parallel == "cfg" and cfg["enable_cfg"] and world % 2 == 0:
            sp_mode = ulysses.parallelize_wan_cfg(model, S, lib.fmha, sp=args.sp)
        elif sp_mode == "fused":
            ulysses.parallelize_wan_fused(model, S)         # raises if symmetric memory is unavailable: no silent change of the measured path
        else:
            ulysses.parallelize_wan(model, S, lib.fmha)
        log(f"sequence parallel installed: {sp_mode}")
    else:
        sp_mode = "none"

    den = None
    if graphed:
        from lightx2v_b200.host.wan_graph import GraphedDenoiser
        den = GraphedDenoiser(model, sched, inputs)

    def one_step(i):
        i = i % max(1, sched.infer_steps - 1)
        if den is not None:                      # one CUDA graph per step kind (host/wan_graph.py); the history of step 0 is reset by its kind
            den.step(i)
            return
        if i == 0 and not cfg.get("distill"):
            sched.set_timesteps(sched.infer_steps, shift=sched.sample_shift)   # fresh multistep history when the 50-step grid wraps
        sched.step_pre(i)
        model.infer(inputs)
        sched.step_post()

    state = {"i": 0}

    def step():
        one_step(state["i"])
        state["i"] += 1

    log(f"warm-up: {args.warmup} steps")
    tw = time.time()
    for _ in range(args.warmup):
        step()
    barrier(world)
    est_step_s = (time.time() - tw) / max(1, args.warmup)
    log(f"warm-up done: ~{est_step_s:.2f} s/step; budget left {budget.left():.0f} s")

    # ---------------- timed region 1: inputs resident in HBM
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    if den is None:
        lib.prof_fmha_begin(8192)          # (events recorded inside a captured graph would be overwritten by every replay)
    l0 = lib.launch_count()
    g0 = den.replayed_launches if den is not None else 0
    torch.cuda.nvtx.range_push("timed")          # ncu --nvtx --nvtx-include "timed/" captures exactly this region
    ms_resident = timed_loop(step, args.steps, world)
    torch.cuda.nvtx.range_pop()
    launches = lib.launch_count() - l0
    if den is not None:
        launches = den.replayed_launches - g0
    prof = lib.prof_fmha_end(8192)
    clk = clocks.stop() if rank == 0 else None
    log(f"timed region: {args.steps} steps, {ms_resident:.1f} ms/step (this rank), {launches} launches; budget left {budget.left():.0f} s")
    if args.dump_outputs and rank == 0:
        # what one denoise step hands its caller: the updated latents, and the CFG-combined model prediction (a graph replay keeps
        # that prediction in a buffer of whichever graph was captured last, so it is only written from the eager loop)
        dump_outputs(args.dump_outputs, {"latents": sched.latents} if den is not None else {"latents": sched.latents, "noise_pred": sched.noise_pred})

    # ---------------- timed region 2: end to end through the public API with HOST buffers (H2D inputs, D2H result per step)
    reserve = 75.0 if side_legs else 20.0
    n_e2e = int(max(1, min(args.steps, (budget.left() - reserve) / max(ms_resident * 1e-3, 1e-3))))
    if world > 1:                                  # every rank must run the same number of steps
        n_e2e = int(min(max_over_ranks([-n_e2e], dev, world)[0] * -1, n_e2e))
    h_lat = torch.empty(cfg["target_shape"], dtype=torch.float32).pin_memory()
    h_lat.copy_(sched.latents.float().cpu())
    h_ctx = {k: v.cpu().pin_memory() for k, v in ctx.items()}
    h_out = torch.empty(cfg["target_shape"], dtype=torch.float32).pin_memory()
    h2d = h_lat.numel() * 4 + sum(v.numel() * 2 for v in h_ctx.values())
    d2h = h_out.numel() * 4

    def e2e_step():
        if den is not None:                  # graph replay reads static buffers: the H2D copies land in them
            sched.s_lat.copy_(h_lat, non_blocking=True)
            for k, v in h_ctx.items():
                ctx[k].copy_(v, non_blocking=True)
        else:
            sched.latents = h_lat.to(dev, non_blocking=True)
            inputs["text_encoder_output"] = {k: v.to(dev, non_blocking=True) for k, v in h_ctx.items()}
        step()
        h_out.copy_(sched.latents.float(), non_blocking=True)

    log(f"e2e region: {n_e2e} steps with host buffers")
    ms_e2e = timed_loop(e2e_step, n_e2e, world)
    log(f"e2e region done: {ms_e2e:.1f} ms/step; budget left {budget.left():.0f} s")

    ms_resident, ms_e2e = max_over_ranks([ms_resident, ms_e2e], dev, world)

    if rank == 0:
        peak_tf, peak_gbs, peak_src = peaks()
        roof = roofline_from_profile(prof, lambda r: r[1] == r[2] and r[1] >= S, peak_tf, peak_src, "fmha_fwd_kernel<128>")
        native = cfg["b200_native_block"] and world == 1 and not (cfg.get("fp8") or cfg.get("nvfp4"))
        out = {
            "metric": METRIC, "value": round(1000.0 / ms_resident, 5), "unit": "latents/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms_resident, 2), "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "fp8-e4m3 linears, bf16 attention" if cfg.get("fp8") else ("nvfp4 (e2m1 + ue4m3/16) linears, bf16 attention" if cfg.get("nvfp4") else "bf16"),
            "data": "synthetic latents/prompt embeddings, random-init weights of the named shapes",
            "config": {"workload": args.workload, "tokens": S, "forwards_per_step": 2 if cfg["enable_cfg"] else 1, "blocks": cfg["num_layers"],
                       "parallelism": (sp_mode if sp_mode.startswith("cfg2") else f"ulysses{world}") if world > 1 else "single", "sp_exchange": sp_mode,
                       "block_schedule": ("one CUDA graph per denoise step (host/wan_graph.py), " if den is not None else "") + ("library default: one native b200_wan_block_fwd call per block" if native else "per-op C-ABI entry points"),
                       "l2": "activations (774 MB/tensor) and weights (28 GB) exceed the 126 MB L2",
                       "scheduler": "step-distill 4-step (x0 re-noising)" if cfg.get("distill") else "UniPC order 2 (flow), 50-step sigma grid"},
            "achieved_tflops": round(flops_step / (ms_resident * 1e-3) / 1e12, 1),
            "model_tflop_per_step": round(flops_step / 1e12, 1),
            "e2e": {"value": round(1000.0 / ms_e2e, 5), "unit": "latents/s", "ms_per_step": round(ms_e2e, 2), "steps": n_e2e, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches),
            "gpu_launches_source": "b200_launch_count(): counted inside libb200dit.so at every kernel launch (this rank)",
            # where the step goes: the self-attention launches (CUDA events inside the library) vs everything else (GEMMs, row-wise kernels,
            # pre/post-infer, scheduler, and - at N > 1 - the exchange kernels and the two symmetric-memory barriers per block)
            "step_breakdown_ms": (lambda fm: {"self_attention": round(fm, 1), "everything_else": round(ms_resident - fm, 1)})(
                sum(r[0] for r in prof if r[1] == r[2] and r[1] >= S and r[0] > 0) / max(1, args.steps)),
            "clocks": clk,
            "roofline": roof,
        }
        if cpu_base is not None:
            out["cpu_baseline"] = cpu_base
        if side_legs and args.vae and budget.left() > 45:
            log("side leg: Wan VAE decode")
            del model, W
            sched.latents = None
            torch.cuda.empty_cache()
            out["vae_decode"] = vae_decode_bench(cfg, dev, with_reference=args.gpu_reference and budget.left() > 60)
            log(f"VAE leg done; budget left {budget.left():.0f} s")
        if side_legs and args.gpu_reference and budget.left() > 30:
            log("side leg: the reference's GPU path (flash-attn 2 + torch) on one block")
            out["gpu_reference"] = gpu_reference_sample(cfg, S, dev)
        out["wall_s"] = round(time.time() - T0, 1)
        print(json.dumps(out), flush=True)
        log("JSON line printed")
    if world > 1:
        torch.distributed.destroy_process_group()


# ===================================================================================================================== HunyuanVideo (config 5)
def run_hunyuan(args):
    """BASELINE config 5: HunyuanVideo 13B bf16, 720p x 129f = 118 800 image tokens + 256 text tokens (77 valid), 20 double-stream + 40
    single-stream blocks, one forward per step (embedded guidance, no CFG), then the 3-D VAE decode of the [1,16,33,90,160] latent.
    N > 1: image tokens Ulysses-sharded over the ranks (text replicated; lightx2v/attentions/distributed/ulysses/wrap.py:5-50,
    utils/hunyuan/processor.py:5-72), VAE tiles dealt round-robin to the ranks (HunyuanVAEB200.decode_dist)."""
    from lightx2v_b200 import lib
    from lightx2v_b200.host import ulysses
    from lightx2v_b200.host.hunyuan_infer import HunyuanTransformerInfer, HunyuanTransformerWeights

    budget = Budget(args.budget_s)
    world, rank, local_rank = dist_env()
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    init_dist(dev, world)
    lib.load()
    D, M, H, ND, NS = 3072, 12288, 24, 20, 40
    Li, Lt, valid = 33 * 45 * 80, 256, 77
    g = torch.Generator(device=dev).manual_seed(42)

    def rnd(*shape, scale=0.02):
        return (torch.randn(*shape, generator=g, device=dev, dtype=torch.float32) * scale).to(torch.bfloat16)

    W = {}

    def lin(name, n, k, scale=0.02):
        W[name + ".weight"] = rnd(n, k, scale=scale)
        W[name + ".bias"] = rnd(n)

    for i in range(ND):
        p = f"double_blocks.{i}."
        for s in ("img", "txt"):
            lin(p + s + "_mod.linear", 6 * D, D, 0.01); lin(p + s + "_attn_qkv", 3 * D, D); lin(p + s + "_attn_proj", D, D)
            lin(p + s + "_mlp.fc1", M, D); lin(p + s + "_mlp.fc2", D, M)
            W[p + s + "_attn_q_norm.weight"] = (1 + rnd(128, scale=0.05).float()).to(torch.bfloat16)
            W[p + s + "_attn_k_norm.weight"] = (1 + rnd(128, scale=0.05).float()).to(torch.bfloat16)
    for i in range(NS):
        p = f"single_blocks.{i}."
        lin(p + "linear1", 3 * D + M, D); lin(p + "linear2", D, D + M); lin(p + "modulation.linear", 3 * D, D, 0.01)
        W[p + "q_norm.weight"] = (1 + rnd(128, scale=0.05).float()).to(torch.bfloat16)
        W[p + "k_norm.weight"] = (1 + rnd(128, scale=0.05).float()).to(torch.bfloat16)
    cfg = dict(task="t2v", mm_config={}, double_blocks_num=ND, single_blocks_num=NS)
    weights = HunyuanTransformerWeights(cfg)
    weights.load(W)
    infer = HunyuanTransformerInfer(cfg)
    if Li % world != 0:
        raise SystemExit(f"{Li} image tokens do not split over {world} ranks")
    s_rows = Li // world
    sl = slice(rank * s_rows, (rank + 1) * s_rows)
    img0, txt0, vec = rnd(Li, D, scale=1.0), rnd(Lt, D, scale=1.0), rnd(1, D, scale=1.0)     # same on every rank (same seed)
    ang = torch.rand(Li, 64, generator=g, device=dev) * 6.28
    freqs = (ang.cos().repeat_interleave(2, 1).to(torch.bfloat16)[sl].contiguous(), ang.sin().repeat_interleave(2, 1).to(torch.bfloat16)[sl].contiguous())
    cu = [0, Li + valid, Li + Lt]
    if world > 1:
        ulysses.parallelize_hunyuan(infer, lib.fmha)
    full = torch.empty(Li, D, dtype=torch.bfloat16, device=dev)
    log(f"HunyuanVideo blocks built: {Li}+{Lt} tokens, {world} rank(s), {torch.cuda.memory_allocated() / 2**30:.1f} GiB")

    def step(img_src=None, txt_src=None):
        img = (img0 if img_src is None else img_src)[sl].clone()
        out, _ = infer.infer(weights, img, (txt0 if txt_src is None else txt_src).clone(), vec, cu, Li + Lt, freqs)
        if world > 1:
            torch.distributed.all_gather_into_tensor(full, out.contiguous())      # post-process of processor.py:52-72
            return full
        return out

    tw = time.time()
    for _ in range(args.warmup):
        step()
    barrier(world)
    log(f"warm-up done: ~{(time.time() - tw) / max(1, args.warmup):.2f} s/step")
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    lib.prof_fmha_begin(8192)
    l0 = lib.launch_count()
    last = {}
    ms = timed_loop(lambda: last.update(out=step()), args.steps, world)
    launches = lib.launch_count() - l0
    prof = lib.prof_fmha_end(8192)
    clk = clocks.stop() if rank == 0 else None
    log(f"timed region: {ms:.1f} ms/step; budget left {budget.left():.0f} s")
    if args.dump_outputs and rank == 0:
        # the image-token stream after the block stack is far above the size limit: a fixed seeded sample of its rows, sorted, so
        # that every run and every build writes the same rows
        out = last["out"]
        rows = torch.randperm(out.shape[0], generator=torch.Generator().manual_seed(0))[:4096].sort().values
        dump_outputs(args.dump_outputs, {"img_out_rows": out[rows.to(out.device)]})
    # e2e: image / text token streams from pinned host memory every step, result back to the host
    h_img, h_txt = img0.cpu().pin_memory(), txt0.cpu().pin_memory()
    h_out = torch.empty(Li, D, dtype=torch.bfloat16).pin_memory()
    n_e2e = int(max(1, min(args.steps, (budget.left() - 60.0) / max(ms * 1e-3, 1e-3))))
    if world > 1:
        n_e2e = int(-max_over_ranks([-n_e2e], dev, world)[0])

    def e2e_step():
        r = step(h_img.to(dev, non_blocking=True), h_txt.to(dev, non_blocking=True))
        h_out.copy_(r, non_blocking=True)

    ms_e2e = timed_loop(e2e_step, n_e2e, world)
    ms, ms_e2e = max_over_ranks([ms, ms_e2e], dev, world)
    vae = None
    if args.vae and budget.left() > 30:
        del weights, W, infer
        torch.cuda.empty_cache()
        log("Hunyuan VAE decode leg")
        vae = hunyuan_vae_decode_bench(dev, world, rank, with_reference=world == 1 and args.gpu_reference)
    if rank == 0:
        L = Li + Lt
        flops = 60 * (4.0 * L * L * D + 24.0 * L * D * D)          # SURVEY.md 8d
        peak_tf, _, peak_src = peaks()
        roof = roofline_from_profile(prof, lambda r: r[1] >= Li, peak_tf, peak_src, "fmha_fwd_kernel<128>")
        print(json.dumps({"metric": "denoise-step latents/sec (HunyuanVideo 13B 720p x 129f, DiT block stack); VAE decode MPix/s", "value": round(1000.0 / ms, 5),
                          "unit": "latents/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 1), "higher_is_better": True,
                          "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                          "config": {"workload": args.workload, "img_tokens": Li, "txt_tokens": Lt, "txt_valid": valid, "blocks": "20 double + 40 single",
                                     "parallelism": f"ulysses{world} (NCCL all-to-all: image tokens sharded, text replicated)" if world > 1 else "single",
                                     "l2": "activations (730 MB/tensor) exceed the 126 MB L2"},
                          "achieved_tflops": round(flops / (ms * 1e-3) / 1e12, 1), "model_tflop_per_step": round(flops / 1e12, 1),
                          "e2e": {"value": round(1000.0 / ms_e2e, 5), "unit": "latents/s", "ms_per_step": round(ms_e2e, 1), "steps": n_e2e,
                                  "h2d_bytes_per_step": (Li + Lt) * D * 2, "d2h_bytes_per_step": Li * D * 2},
                          "gpu_launches": int(launches), "clocks": clk, "roofline": roof, "vae_decode": vae, "wall_s": round(time.time() - T0, 1)}), flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()


def hunyuan_vae_decode_bench(dev, world=1, rank=0, with_reference=True):
    """HunyuanVideo VAE decode of the 720p x 129f latent [1,16,33,90,160] with the reference's tiling (3 temporal x 28 spatial tiles),
    through HunyuanVAEB200.decode (N > 1: decode_dist, tiles dealt to the ranks), next to the torch restatement of the reference's fp16
    cuDNN path on ONE full tile [16,17,32,32] of the same GPU (bounded sample; diffusers is absent on the box, so the reference
    classes themselves cannot be imported there)."""
    from oracle import hunyuan_vae_oracle as HV
    from lightx2v_b200.host.hunyuan_vae import HunyuanVAEB200

    cfg = dict(HV.HUNYUAN_VAE_CFG)
    W = {k: v.to(dev) for k, v in HV.synth_vae_weights(cfg, seed=5).items()}
    vae = HunyuanVAEB200(W, device=dev)
    g = torch.Generator(device=dev).manual_seed(1)
    lat = torch.randn(1, 16, 33, 90, 160, generator=g, device=dev)
    vae.decode_device(lat[:, :, :5, :32, :32])                                   # warm-up (kernel attribute setup, allocator)
    barrier(world)
    torch.cuda.reset_peak_memory_stats()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    s.record()
    if world > 1:
        out = vae.decode_dist(lat, to_cpu=False)
        e.record()
        barrier(world)
        out = out.cpu().float() if rank == 0 else out
    else:
        img = vae.decode_device(lat)
        e.record()
        out = img.cpu().float()
    wall = time.time() - t0
    ms = max_over_ranks([s.elapsed_time(e)], dev, world)[0]
    mpix = out.shape[2] * out.shape[3] * out.shape[4] / 1e6
    res = {"unit": "MPix/s", "output": list(out.shape[1:]), "mpix": round(mpix, 2), "value": round(mpix / (ms * 1e-3), 1), "ms": round(ms, 1), "n_gpus": world,
           "wall_s_with_d2h": round(wall, 2), "tiles": "3 temporal x 4 x 7 spatial (25 % overlap, linear blends)" + (f", dealt round-robin to {world} ranks" if world > 1 else ""),
           "dtype": "bf16 activations, fp32 accumulate, fp32/fp64 GroupNorm statistics", "peak_mem_gb": round(torch.cuda.max_memory_allocated() / 2 ** 30, 1)}
    if with_reference:
        tile = lat[:, :, :17, :32, :32]
        s.record()
        vae.decoder.decode_tile(tile[0])
        e.record()
        torch.cuda.synchronize()
        ms_tile = s.elapsed_time(e)
        Wh = {k: v.half() for k, v in W.items()}
        with torch.no_grad():
            zt = (tile / cfg["scaling_factor"]).half()
            HV.tile_decode(Wh, zt[:, :, :3, :8, :8], cfg)                            # cuDNN warm-up
            torch.cuda.synchronize()
            s.record()
            HV.tile_decode(Wh, zt, cfg)
            e.record()
            torch.cuda.synchronize()
        ms_ref = s.elapsed_time(e)
        res["gpu_reference"] = {"sample": "one full tile [16,17,32,32] -> [3,65,256,256], torch fp16 (cuDNN) restatement of the reference decoder",
                                "ms_tile_reference": round(ms_ref, 1), "ms_tile_ours": round(ms_tile, 1), "speedup": round(ms_ref / ms_tile, 2),
                                "value": round(mpix / (ms * 1e-3) * ms_tile / ms_ref, 1), "unit": "MPix/s (extrapolated by the tile ratio)"}
    return res


# ===================================================================================================================== side legs
def host_threads():
    """Cores this process may actually run on (cgroup / affinity aware), not the machine's core count."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def cpu_reference_sample(cfg, flops_step, budget_s=12.0):
    """The reference's CPU torch path (oracle port, pinned to the real reference by tests/golden) on the host cores:
    ONE block of the workload's width on a bounded token count, extrapolated to the full step by the FLOP model.  Attention is
    under-represented in the sample (9 % of the FLOPs at 1024 tokens vs 72 % at 75 600), so this is an optimistic CPU number."""
    from oracle import wan_oracle as O
    D, F_, H = cfg["dim"], cfg["ffn_dim"], cfg["num_heads"]
    grid = (4, 16, 16)                                      # 1024 tokens
    S = grid[0] * grid[1] * grid[2]
    W = O.synth_block_weights(1, D, F_, seed=1)
    x, embed0, context = O.synth_block_inputs(S, D, seed=2)
    freqs = O.wan_freqs_table(128)
    t_start = time.time()
    threads = min(host_threads(), 32)                       # torch CPU GEMMs stop scaling (and oversubscribe shared hosts) beyond that
    torch.set_num_threads(threads)
    O.infer_blocks(W, 1, x.clone(), embed0, grid, freqs, context, H)          # warm-up
    n, t0 = 0, time.time()
    while True:
        O.infer_blocks(W, 1, x.clone(), embed0, grid, freqs, context, H)
        n += 1
        if time.time() - t_start > budget_s or n >= 5:
            break
    sec = (time.time() - t0) / n
    fl = O.block_flops(S, D, F_, 512)
    tflops = fl / sec / 1e12
    est_step_s = flops_step / (tflops * 1e12)
    return {"value": 1.0 / est_step_s, "unit": "latents/s", "cores": threads, "kind": "port",
            "sample": f"1 DiT block (D={D}, F={F_}) at {S} tokens, {n} runs, {sec:.2f} s/block = {tflops:.3f} TFLOP/s on {threads} threads; "
                      f"extrapolated to the {flops_step / 1e12:.0f} TFLOP step by the FLOP model (SURVEY.md 8d); attention is 9 % of the sample's FLOPs "
                      f"vs 72 % of the real step, so the CPU figure is optimistic"}


def vae_decode_bench(cfg, dev, with_reference=True):
    """Second half of BASELINE.json's metric: Wan VAE decode MPix/s on the workload's latent ([16, 21, 90, 160] -> 81 x 720 x 1280)."""
    from lightx2v_b200.host.wan_vae import WanVAEDecoderB200
    from oracle import vae_oracle as V           # synthetic weights + (optional) the reference decode loop as GPU baseline
    C, Fr, Hh, Ww = cfg["target_shape"]
    Wd = V.synth_vae_weights(0)
    resident = torch.cuda.memory_allocated()     # what the denoiser legs still hold in this process (weights, workspaces): not the decoder's
    dec = WanVAEDecoderB200(Wd, device=dev)
    g = torch.Generator(device=dev).manual_seed(3)
    zs = torch.randn(C, Fr, Hh, Ww, generator=g, device=dev)
    mpix = (1 + 4 * (Fr - 1)) * Hh * 8 * Ww * 8 / 1e6
    res = {"unit": "MPix/s", "output": [3, 1 + 4 * (Fr - 1), Hh * 8, Ww * 8], "mpix": round(mpix, 2), "dtype": "bf16 activations, fp32 accumulate"}
    try:
        img = dec.decode(zs)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        n = 2
        for _ in range(n):
            img = dec.decode(zs)
        e.record()
        torch.cuda.synchronize()
        ms = s.elapsed_time(e) / n
        res.update(value=round(mpix / (ms * 1e-3), 1), ms=round(ms, 1), effective_tflops=round(639.3 / (ms * 1e-3), 1),   # the reference algorithm's 639.3 TFLOP (SURVEY 8d) / time
                   peak_mem_gb=round((torch.cuda.max_memory_allocated() - resident) / 2**30, 1),   # decoder weights + latent + activations + output
                   resident_other_gb=round(resident / 2**30, 1))
        del img
    except Exception as ex:  # noqa
        res["error"] = str(ex)[:300]
    if with_reference:
        try:
            del dec
            torch.cuda.empty_cache()
            Wg = {k: v.to(dev) for k, v in Wd.items()}
            zs_small = zs[:, :6]                                   # the reference loop is per latent frame: 6 frames -> 21 video frames
            V.vae_decode(Wg, zs_small[:, :2])
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            V.vae_decode(Wg, zs_small)
            e.record()
            torch.cuda.synchronize()
            frames = 1 + 4 * (zs_small.shape[1] - 1)
            mp = frames * Hh * 8 * Ww * 8 / 1e6
            res["gpu_reference"] = {"value": round(mp / (s.elapsed_time(e) * 1e-3), 1), "unit": "MPix/s",
                                    "sample": f"reference per-frame decode loop (fp32, cuDNN TF32), {zs_small.shape[1]} latent frames -> {frames} frames"}
        except Exception as ex:  # noqa
            res["gpu_reference"] = {"unavailable": str(ex)[:200]}
    return res


def gpu_reference_sample(cfg, S, dev):
    """The reference's own GPU path: ONE block at the full token count through the REAL LightX2V classes (WanTransformerWeights +
    WanTransformerInfer with their stock ops: torch.addmm, F.layer_norm, the bf16 RMSNorm fallback, fp64 RoPE, flash_attn_varlen_func),
    byte-compiled unmodified into oracle/_ref (oracle/build_ref.py), x blocks x forwards.  When that build is absent the pinned
    restatement (oracle/wan_oracle.py, bit-identical to those classes: tests/test_gpu_reference_dropin.py) runs instead and the line says
    so.  Extra information beside the contract's CPU reference arm."""
    from oracle import ref_loader as R
    from oracle import wan_oracle as O
    D, F_, H, L = cfg["dim"], cfg["ffn_dim"], cfg["num_heads"], cfg["num_layers"]
    C, Fr, Hh, Ww = cfg["target_shape"]
    grid = (Fr, Hh // 2, Ww // 2)
    try:
        W = O.synth_block_weights(1, D, F_, seed=1, device=dev)
        x, embed0, context = O.synth_block_inputs(S, D, seed=2, device=dev)
        freqs = O.wan_freqs_table(128).to(dev)
        impl = "oracle restatement (reference copy not present)"
        run = lambda: O.infer_blocks(W, 1, x.clone(), embed0, grid, freqs, context, H, attn="flash_attn2")   # noqa: E731
        if R.import_reference():
            from lightx2v.models.networks.wan.infer.transformer_infer import WanTransformerInfer as RefInfer
            from lightx2v.models.networks.wan.weights.transformer_weights import WanTransformerWeights as RefWeights
            rcfg = R.ref_config(D, H, F_, 1, "t2v", mm_type=None, attn_type="flash_attn2")
            rw = RefWeights(rcfg)
            rw.load(W)
            rinfer = RefInfer(rcfg)
            gs, sl = torch.tensor([list(grid)]), torch.tensor([S], device=dev)
            run = lambda: rinfer.infer(rw, gs, None, x.clone(), embed0, sl, freqs, context)   # noqa: E731
            impl = "real LightX2V classes (oracle/_ref, unmodified): mm Default (torch.addmm), flash_attn2, torch norms"
        run()
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        n = 2
        for _ in range(n):
            run()
        e.record()
        torch.cuda.synchronize()
        ms_block = s.elapsed_time(e) / n
        fw = 2 if cfg["enable_cfg"] else 1
        return {"value": 1000.0 / (ms_block * L * fw), "unit": "latents/s", "ms_per_block": round(ms_block, 2), "impl": impl,
                "sample": f"1 block at {S} tokens, x{L} blocks x{fw} forwards"}
    except Exception as ex:  # noqa
        return {"unavailable": str(ex)[:200]}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on the host cores (rank 0 only)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cfg = dict(WORKLOADS[args.workload])
    S, flops_step = step_flops(cfg)
    vals = []
    per = max(2.0, min(args.cpu_budget / 2, 0.6 * args.budget_s / max(1, args.warmup + args.steps)))
    for i in range(args.warmup + args.steps):
        vals.append(cpu_reference_sample(cfg, flops_step, budget_s=per))
        log(f"reference sample {i + 1}/{args.warmup + args.steps}: {vals[-1]['value']:.3e} latents/s")
    timed = vals[args.warmup:] or vals
    v = sum(x["value"] for x in timed) / len(timed)
    base = dict(timed[-1])
    base["value"] = v
    out = {"impl": "reference", "metric": METRIC, "value": v, "unit": "latents/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": 1000.0 / v, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16",
           "data": "synthetic", "config": {"workload": args.workload, "tokens": S},
           "cpu_baseline": base, "e2e": {"value": v, "unit": "latents/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError(f"must be >= 1, got {v}")
    return v


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=2, help="timed steps")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="wan2.1-t2v-14b-720p-81f", choices=list(WORKLOADS) + [HUNYUAN, "hunyuan-13b-720p-129f-blocks"])
    ap.add_argument("--no-cpu-baseline", dest="cpu_baseline", action="store_false")
    ap.add_argument("--no-gpu-reference", dest="gpu_reference", action="store_false")
    ap.add_argument("--no-vae", dest="vae", action="store_false")
    ap.add_argument("--graph", action="store_true", help="N = 1: replay each denoise step as a CUDA graph with the device-resident scheduler (host/wan_graph.py)")
    ap.add_argument("--per-op", action="store_true", help="drive the per-op C-ABI entry points from Python instead of the native per-block call")
    ap.add_argument("--sp", default="fused", choices=["fused", "nccl"], help="Ulysses exchange: peer-memory kernels (default) or NCCL all-to-all")
    ap.add_argument("--parallel", default="ulysses", choices=["ulysses", "cfg"],
                    help="N > 1: Ulysses over all ranks, or CFG-parallel (cond / uncond on rank halves) x Ulysses inside each half")
    ap.add_argument("--cpu-budget", type=float, default=12.0)
    ap.add_argument("--budget-s", type=float, default=480.0, help="wall-clock budget of the whole run; the e2e loop and the side legs shrink to fit")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last of them computed as DIR/<name>.npy (float32, "
                                                           "at most 64 MB; a fixed seeded sample where the output is larger)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA path; --impl reference only times a sample")
    if args.workload.startswith("hunyuan"):
        if args.impl == "reference":
            print(json.dumps({"impl": "reference", "unavailable": "no CPU port of the HunyuanVideo step is timed; the Wan workload carries the reference arm"}), flush=True)
            return
        args.workload = HUNYUAN
        run_hunyuan(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
