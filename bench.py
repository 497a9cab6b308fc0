#!/usr/bin/env python
"""bench.py — BAGEL-7B-MoT text->image denoising throughput on B200 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

Workload (BASELINE.json configs[1], SURVEY.md §8d cfg 2): BAGEL-7B-MoT random-init, 1024x1024 (4096 latent tokens
+ soi/eoi per sample), 50 timesteps = 49 velocity evaluations, text CFG (cfg_text_scale 2.0 -> 2 branches, both run
as one packed LM call), batch 8 per GPU, 66-token text context per sample, cfg_renorm "global".

A "step" is ONE denoising step of the whole batch: latent-in -> 28 MoT layers over both CFG branches -> latent-out
-> CFG + renorm + Euler update (every step costs the same, 49 of them make one image batch). Reported:
  value   images/s (whole job, all GPUs) = global_batch / (49 * s_per_step); x_t and all inputs resident in HBM,
          W warm-up steps, exactly K timed steps, CUDA events, max over ranks. The activations + weights touched
          per step (> 30 GB) far exceed the 126 MB L2, so no explicit L2 flush is needed (config.l2: "working set").
  e2e     the same metric through the public API: Bagel.generate_image(**prepare_vae_latent(...)) from host
          (pinned) init noise to host latents, including planning, H2D/D2H, and for N > 1 the NCCL all-gather of
          the final latents.
  roofline   the dominant kernel (SwiGLU gate/up GEMM, tcgen05): algorithmic FLOPs / CUDA-event time per launch.
  cpu_baseline  the oracle (CPU port of the reference path) on this box's host cores, bounded sample.
--impl reference times the reference's CPU path (the oracle port: the Python reference cannot travel to the
box) with all host threads on a bounded sample of the same workload and prints the same JSON shape.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

EVALS_PER_IMAGE = 49            # num_timesteps 50 -> timesteps[:-1] (bagel.py:693-696)
METRIC = "denoised images/sec @1024^2, 50 steps, BAGEL-7B-MoT"
UNIT = "images/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=12)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=8, help="images per GPU")
    ap.add_argument("--image-size", type=int, default=1024)
    ap.add_argument("--layers", type=int, default=None, help="debug only: fewer layers (marks the run invalid)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-no-graph", action="store_true", help="A/B: run the e2e generate_image without CUDA-graph capture")
    ap.add_argument("--no-taylorseer", action="store_true", help="skip the informational enable_taylorseer=True run")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true",
                    help="skip the blocks for the other BASELINE configs (attn, und_prefill, decode, edit, "
                         "gpu_library_baseline, parity, strong_scaling)")
    ap.add_argument("--blocks", default="attn,und,edit,library,strong",
                    help="comma list of extra blocks to run (default: all)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the latents they produced as DIR/<name>.npy (float32), so that "
                         "two builds can be compared output for output on identical seeded inputs")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the oracle port of the reference path on the host cores, bounded sample
# ------------------------------------------------------------------------------------------------------
def cpu_reference_sample(image_size: int, threads: int):
    """One MoT decoder layer (mode "gen": 4096 latent rows through the gen expert, soi/eoi through the und
    expert, 66 cached context tokens, non-causal packed attention) for ONE 1024^2 sample at BAGEL-7B dims,
    executed by the oracle. One image = 28 layers x 98 LM forwards of this, so
    images/s = 1 / (t_layer * 28 * 98)  (latent in/out and CFG are < 0.1 % and omitted)."""
    import torch
    from oracle import fixtures, qwen2_mot as om

    torch.set_num_threads(threads)
    cfg7 = fixtures.BAGEL_7B_LM
    cfg = om.LMConfig(hidden_size=cfg7.hidden_size, intermediate_size=cfg7.intermediate_size, num_hidden_layers=1,
                      num_attention_heads=cfg7.num_attention_heads, num_key_value_heads=cfg7.num_key_value_heads,
                      vocab_size=8)
    sd = fixtures.lm_state_dict(cfg, seed=0, dtype=torch.bfloat16, w_std=0.02, lm_head=False)
    ntok = (image_size // 16) ** 2
    n, ctx = ntok + 2, 66
    g = torch.Generator().manual_seed(3)
    x = torch.randn(n, cfg.hidden_size, generator=g).to(torch.bfloat16)
    cache = om.KVCache(1)
    cache.key_cache[0] = torch.randn(ctx, cfg.num_key_value_heads, cfg.head_dim, generator=g).to(torch.bfloat16)
    cache.value_cache[0] = torch.randn(ctx, cfg.num_key_value_heads, cfg.head_dim, generator=g).to(torch.bfloat16)
    kw = dict(query_lens=torch.tensor([n], dtype=torch.int32), packed_query_position_ids=torch.full((n,), ctx),
              packed_query_indexes=torch.arange(ctx, ctx + n), past_key_values=cache,
              key_values_lens=torch.tensor([ctx], dtype=torch.int32), packed_key_value_indexes=torch.arange(ctx),
              update_past_key_values=False, is_causal=False, mode="gen",
              packed_vae_token_indexes=torch.arange(1, n - 1), packed_text_indexes=torch.tensor([0, n - 1]))
    times = []
    with torch.no_grad():
        om.lm_forward_inference(sd, cfg, x, **kw)  # warm-up
        # give the CPU arm its best thread count: bf16 matmuls on a 128-thread host are often faster with fewer threads
        best_thr, best_t = threads, None
        for thr in sorted({threads, max(1, threads // 2), max(1, threads // 4), max(1, threads // 8)}, reverse=True):
            torch.set_num_threads(thr)
            t0 = time.time()
            om.lm_forward_inference(sd, cfg, x, **kw)
            dt = time.time() - t0
            if best_t is None or dt < best_t:
                best_thr, best_t = thr, dt
        torch.set_num_threads(best_thr)
        threads = best_thr
        t_end = time.time() + 12.0
        while len(times) < 3 or (time.time() < t_end and len(times) < 10):
            t0 = time.time()
            om.lm_forward_inference(sd, cfg, x, **kw)
            times.append(time.time() - t0)
    t_layer = statistics.median(times)
    img_s = 1.0 / (t_layer * cfg7.num_hidden_layers * 2 * EVALS_PER_IMAGE)
    sample = (f"oracle (CPU port of the reference path), 1 of 28 MoT layers x 1 sample x 1 CFG branch at "
              f"{image_size}^2 ({n} query tokens + {ctx} ctx), median of {len(times)} runs = {t_layer:.3f} s on "
              f"{threads} threads (fastest of a thread-count sweep); images/s = 1/(t*28*98)")
    return img_s, sample, t_layer, threads


def cpu_reference_full_forward_flow(image_size: int, threads: int):
    """ONE full velocity evaluation (`_forward_flow`, bagel.py:757-907) of ONE 1024^2 sample at BAGEL-7B dims on the
    host cores with the oracle: latent-in, all 28 MoT layers (main branch, 66 cached context tokens), latent-out.
    images/s = 1 / (t * 2 branches * 49 evaluations). The 28 layers share one set of random weights (the timing is
    the same: 0.93 GB per layer does not stay in any CPU cache; drawing 14 G random parameters on the host would take
    longer than the measurement)."""
    import torch
    from oracle import bagel_flow as obf, fixtures, qwen2_mot as om

    torch.set_num_threads(threads)
    c7 = fixtures.BAGEL_7B_LM
    cfg1 = om.LMConfig(hidden_size=c7.hidden_size, intermediate_size=c7.intermediate_size, num_hidden_layers=1,
                       num_attention_heads=c7.num_attention_heads, num_key_value_heads=c7.num_key_value_heads, vocab_size=8)
    one = fixtures.lm_state_dict(cfg1, seed=0, dtype=torch.bfloat16, w_std=0.02, lm_head=False)
    L = c7.num_hidden_layers
    cfg = om.LMConfig(hidden_size=c7.hidden_size, intermediate_size=c7.intermediate_size, num_hidden_layers=L,
                      num_attention_heads=c7.num_attention_heads, num_key_value_heads=c7.num_key_value_heads, vocab_size=8)
    sd = {}
    for k, v in one.items():
        if k.startswith("model.layers.0."):
            for li in range(L):
                sd["language_model." + k.replace("model.layers.0.", f"model.layers.{li}.")] = v
        else:
            sd["language_model." + k] = v
    sd.update(fixtures.bagel_extra_state_dict(cfg.hidden_size, seed=1, w_std=0.02))
    sd["latent_pos_embed.pos_embed"] = obf.sincos_2d_table(cfg.hidden_size, 64).to(torch.bfloat16)
    fc = obf.FlowConfig(lm=cfg, max_latent_size=64)
    ctx = 66
    g = torch.Generator().manual_seed(3)
    cache = om.KVCache(L)
    for li in range(L):
        cache.key_cache[li] = torch.randn(ctx, cfg.num_key_value_heads, cfg.head_dim, generator=g).to(torch.bfloat16)
        cache.value_cache[li] = torch.randn(ctx, cfg.num_key_value_heads, cfg.head_dim, generator=g).to(torch.bfloat16)
    torch.manual_seed(2)
    gi = obf.prepare_vae_latent(fc, [ctx], [ctx], [(image_size, image_size)], 1, 2)
    x = gi["packed_init_noises"]
    t = torch.full((x.shape[0],), 0.9)
    with torch.no_grad():
        t0 = time.time()
        obf.forward_flow(sd, fc, x, t, gi["packed_vae_token_indexes"], gi["packed_vae_position_ids"], gi["packed_text_ids"],
                         gi["packed_text_indexes"], gi["packed_indexes"], gi["packed_position_ids"], gi["packed_seqlens"],
                         gi["key_values_lens"], cache, gi["packed_key_value_indexes"])
        dt = time.time() - t0
    img_s = 1.0 / (dt * 2 * EVALS_PER_IMAGE)
    sample = (f"oracle (CPU port of the reference path): ONE full _forward_flow (28 MoT layers, 1 sample, main CFG branch, "
              f"{x.shape[0]} latent tokens + soi/eoi + {ctx} ctx) at {image_size}^2 = {dt:.1f} s on {threads} threads; "
              f"images/s = 1/(t*2*49)")
    return img_s, sample, dt


def run_reference_arm(args):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    # thread count from the single-layer sweep (bf16 CPU matmuls are often fastest well below the core count), then one
    # FULL velocity evaluation at that thread count as the measured sample
    v1, sample1, t_layer, used = cpu_reference_sample(args.image_size, threads)
    v, sample, t_full = cpu_reference_full_forward_flow(args.image_size, used)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 / (v * EVALS_PER_IMAGE) * args.batch if v > 0 else None,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "BAGEL-7B-MoT random-init T2I 1024^2, 49 evals, text CFG (2 branches), CPU oracle port",
                   "global_batch": args.batch, "parallelism": "cpu"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": used, "kind": "port", "sample": sample,
                         "extrapolated": True, "factor": 2 * EVALS_PER_IMAGE,
                         "single_layer_cross_check": {"value": v1, "t_layer_s": t_layer, "factor": 28 * 2 * EVALS_PER_IMAGE}},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _emit(line)


# ------------------------------------------------------------------------------------------------------
DUMP_BYTES_MAX = 60 << 20       # all ranks together: stays under 64 MB with the .npy headers


def dump_latents(out_dir: str, latents, rank: int, world: int):
    """--dump-outputs: the per-sample latents x_t after the last timed step (what FlowRunner.latents() hands a
    caller) as one float32 array [samples, tokens, 64]. Above this rank's share of DUMP_BYTES_MAX, a fixed seeded
    subset of token rows [k, 64] in their original order, so every build stores the same elements."""
    import numpy as np
    import torch

    x = torch.stack(latents, 0).float().cpu()
    cap = DUMP_BYTES_MAX // world
    if x.numel() * 4 > cap:
        rows = x.reshape(-1, x.shape[-1])
        k = cap // (rows.shape[1] * 4)
        idx = torch.randperm(rows.shape[0], generator=torch.Generator().manual_seed(0))[:k].sort().values
        x = rows[idx]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "latents.npy" if world == 1 else f"latents_rank{rank}.npy"), x.numpy())


_JSON_FD = None


def _claim_stdout():
    """The driver parses ONE JSON line from stdout. Libraries print there too (NCCL's version banner under torchrun), so
    keep a private duplicate of the real stdout for the result line and point fd 1 at stderr for everything else."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def _emit(line: dict):
    _claim_stdout()
    os.write(_JSON_FD, (json.dumps(line) + "\n").encode())


def main():
    args = parse_args()
    _claim_stdout()
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (bagel_b200 has no CPU path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    from bagel_b200 import _cabi, ops, synthetic
    from bagel_b200.dist import gather_latents

    B = args.batch
    model = synthetic.build_random_bagel(device=dev, seed=rank, num_layers=args.layers)
    cfg = model.config.llm_config
    gen_input, cfg_text, ctxs = synthetic.t2i_inputs(model, B, (args.image_size, args.image_size), seed=1 + rank,
                                                     noise_seed=2 + rank)
    gen_kwargs = dict(
        num_timesteps=EVALS_PER_IMAGE + 1, timestep_shift=3.0, cfg_renorm_min=0.0, cfg_renorm_type="global",
        cfg_interval=[0.0, 1.0], cfg_text_scale=2.0, cfg_img_scale=1.0,
        cfg_text_packed_position_ids=cfg_text["cfg_packed_position_ids"],
        cfg_text_packed_query_indexes=cfg_text["cfg_packed_query_indexes"],
        cfg_text_key_values_lens=cfg_text["cfg_key_values_lens"],
        cfg_text_packed_key_value_indexes=cfg_text["cfg_packed_key_value_indexes"],
        cfg_text_past_key_values=ctxs["cfg_text"])

    # ---------------- device-resident timing: W warm-up + K timed denoising steps ----------------
    # per-kernel CUDA-event timing (roofline) needs individually launched kernels: the device-resident region runs the
    # launch sequence eagerly; the end-to-end region below replays it as a CUDA graph (the product default)
    model.use_cuda_graph = False
    runner = model.make_flow_runner(past_key_values=ctxs["main"], **gen_input, **gen_kwargs)
    for i in range(args.warmup):
        runner.step(i % EVALS_PER_IMAGE)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ops.kernel_timer_start("swiglu")
    l0 = _cabi.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        runner.step((args.warmup + i) % EVALS_PER_IMAGE)
    e1.record()
    torch.cuda.synchronize()
    launches = _cabi.launch_count() - l0
    swiglu_ms = ops.kernel_timer_stop()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = float(t.item()) / args.steps
    value = (B * world) / (EVALS_PER_IMAGE * ms_per_step / 1000.0)
    if args.dump_outputs:
        dump_latents(args.dump_outputs, runner.latents(), rank, world)
    del runner

    # ---------------- roofline of the dominant kernel ----------------
    peaks, peak_src = measured_peaks()
    rows = 2 * B * ((args.image_size // 16) ** 2 + 2)  # both CFG branches in one packed call
    flops_launch = 2.0 * rows * (2 * cfg.intermediate_size) * cfg.hidden_size
    roof = None
    traffic, traffic_src = None, None
    prof = os.path.join(ROOT, "profiles", "r02_gemm2_swiglu_ncu_full.csv")
    if os.path.exists(prof) and rows == 65568:   # the capture was taken on exactly this launch shape
        try:
            vals = {}
            for ln in open(prof):
                if ln.startswith('"dram__bytes_read.sum",') or ln.startswith('"dram__bytes_write.sum",'):
                    name, unit, v = [x.strip().strip('"') for x in ln.split(",")]
                    vals[name] = float(v) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}[unit]
            traffic = vals["dram__bytes_read.sum"] + vals["dram__bytes_write.sum"]
            traffic_src = "profiles/r02_gemm2_swiglu_ncu_full.csv (ncu --set full, one launch of this kernel/shape, this build)"
        except Exception:
            traffic = None
    if swiglu_ms:
        avg_ms = statistics.mean(swiglu_ms)
        ach = flops_launch / (avg_ms * 1e-3) / 1e12
        peak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops")))
        roof = {"kernel": "gemm2_bf16_kernel<SWIGLU> (CTA-pair tcgen05 cta_group::2; gate|up projection + SiLU*up epilogue)",
                "bound": "tensor",
                "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": traffic,
                "traffic_unit": "bytes/launch (dram read+write)", "traffic_source": traffic_src,
                "algorithmic_bytes_per_launch": 2.0 * (rows * cfg.hidden_size + 2 * cfg.intermediate_size * cfg.hidden_size
                                                       + rows * cfg.intermediate_size),
                "peak_source": f"{peak_src} bf16_tflops_sustained (kernel timed inside a long step)",
                "launches_timed": len(swiglu_ms), "avg_launch_ms": avg_ms,
                "flops_per_launch": flops_launch}
    model_flops_img = 98 * (4098 * 13.05e9 + 4 * 4098 * (4098 + 66) * 3584 * 28)  # SURVEY.md §6
    mfu = value / world * model_flops_img / (float(peaks.get("bf16_tflops_sustained", 1400.0)) * 1e12)

    # ---------------- end to end through the public API ----------------
    e2e = None
    model.use_cuda_graph = not args.e2e_no_graph
    if not args.no_e2e:
        noise_host = gen_input["packed_init_noises"].pin_memory()
        gi = dict(gen_input)
        gi["packed_init_noises"] = noise_host
        h2d = noise_host.numel() * 4 + sum(v.numel() * v.element_size() for k, v in gi.items()
                                           if k != "packed_init_noises" and torch.is_tensor(v))
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        lat = model.generate_image(past_key_values=ctxs["main"], **gi, **gen_kwargs)
        local = torch.stack(lat, 0)                       # [B, 4096, 64] fp32 on device
        full = gather_latents(local) if world > 1 else local
        host = full.to("cpu")                             # D2H of the result
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
        assert torch.isfinite(host).all()
        e2e = {"value": (B * world) / dt, "unit": UNIT, "h2d_bytes_per_step": int(h2d // EVALS_PER_IMAGE),
               "d2h_bytes_per_step": int(host.numel() * 4 // EVALS_PER_IMAGE), "seconds_per_batch": dt,
               "h2d_bytes_per_generate": int(h2d), "d2h_bytes_per_generate": int(host.numel() * 4),
               "note": "one full generate_image (49 evals) per GPU incl. planning, H2D noise, D2H latents"
                       + (", NCCL all-gather" if world > 1 else "")}

    # ---------------- same call with the reference's step cache (informational; NOT the headline) ----------------
    e2e_ts = None
    if not args.no_e2e and not args.no_taylorseer:
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        lat = model.generate_image(past_key_values=ctxs["main"], **gi, **gen_kwargs, enable_taylorseer=True)
        local = torch.stack(lat, 0)
        full = gather_latents(local) if world > 1 else local
        host = full.to("cpu")
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
        assert torch.isfinite(host).all()
        e2e_ts = {"value": (B * world) / dt, "unit": UNIT, "seconds_per_batch": dt,
                  "note": "generate_image(enable_taylorseer=True): the reference's TaylorSeer schedule computes 19 of "
                          "the 49 evaluations and extrapolates 30 (different numerics from the headline run)"}

    # ---------------- the other BASELINE configs + library baseline + parity (tools/bench_blocks.py) ----------------
    extra = {}
    blocks = set() if args.no_extra or args.layers is not None else set(args.blocks.split(","))
    if blocks:
        from tools import bench_blocks as bb
        torch.cuda.empty_cache()

        def guarded(name, fn):
            """A failing block must not take the headline line down with it: record the error instead."""
            try:
                return fn()
            except Exception as e:  # noqa: BLE001
                import traceback
                traceback.print_exc()
                torch.cuda.synchronize()
                return {"error": f"{type(e).__name__}: {e}"[:300]}

        if world == 1 and "library" in blocks:
            tok = synthetic.RandomIdTokenizer(1 + rank)
            prompt_ids = [tok.encode("64") for _ in range(B)]
            r = guarded("library", lambda: bb.library_baseline_and_parity(model, gen_input, cfg_text, ctxs["main"], gen_kwargs,
                                                                          prompt_ids, dev, ms_per_step, B))
            extra.update(r if "error" not in r else {"gpu_library_baseline": r, "parity": r})
            torch.cuda.empty_cache()
        if world == 1 and "attn" in blocks:
            extra["attn"] = guarded("attn", lambda: bb.attn_block(peaks, dev))
        if world > 1 and "strong" in blocks and 8 % world == 0:
            # configs[1] with the GLOBAL batch fixed at 8 images (SURVEY.md §8e: "cfg 2: B=8 -> 1/GPU")
            def strong():
                bs = 8 // world
                gi_s, ct_s, cx_s = synthetic.t2i_inputs(model, bs, (args.image_size, args.image_size), seed=11 + rank,
                                                        noise_seed=12 + rank)
                kw_s = dict(gen_kwargs)
                kw_s.update(cfg_text_packed_position_ids=ct_s["cfg_packed_position_ids"],
                            cfg_text_packed_query_indexes=ct_s["cfg_packed_query_indexes"],
                            cfg_text_key_values_lens=ct_s["cfg_key_values_lens"],
                            cfg_text_packed_key_value_indexes=ct_s["cfg_packed_key_value_indexes"],
                            cfg_text_past_key_values=cx_s["cfg_text"])
                model.use_cuda_graph = False
                rn = model.make_flow_runner(past_key_values=cx_s["main"], **gi_s, **kw_s)
                for i in range(3):
                    rn.step(i)
                torch.cuda.synchronize()
                dist.barrier()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                ks = 8
                for i in range(ks):
                    rn.step(3 + i)
                b.record()
                torch.cuda.synchronize()
                tt_ = torch.tensor([a.elapsed_time(b)], device=dev)
                dist.all_reduce(tt_, op=dist.ReduceOp.MAX)
                msps = float(tt_.item()) / ks
                return {"workload": "BASELINE configs[1] strong-scaled: GLOBAL batch 8 images (SURVEY.md 8e), "
                                    f"{bs} per GPU on {world} GPUs, 2 CFG branches", "global_batch": 8, "per_gpu_batch": bs,
                        "steps": ks, "warmup": 3, "ms_per_step": msps, "value": 8 / (EVALS_PER_IMAGE * msps / 1e3),
                        "unit": UNIT, "scaling": "strong"}
            extra["strong_scaling"] = guarded("strong", strong)
        need_vit = ("und" in blocks and world == 1) or "edit" in blocks
        if need_vit:
            r = guarded("vit", lambda: synthetic.attach_random_vit(model, seed=5))
            if isinstance(r, dict):
                extra["und_prefill"] = extra["edit"] = r
                need_vit = False
        if need_vit and world == 1 and "und" in blocks:
            extra.update(guarded("und", lambda: bb.und_prefill_and_decode_block(model, dev)))
            torch.cuda.empty_cache()
        if need_vit and "edit" in blocks:
            def edit():
                vae = synthetic.build_random_vae(dev)
                model.use_cuda_graph = True
                if world > 1:
                    dist.barrier()
                r = bb.edit_block(model, vae, dev, samples=2)
                tt_ = torch.tensor([r["seconds"]], device=dev)
                if world > 1:
                    dist.all_reduce(tt_, op=dist.ReduceOp.MAX)
                sec = float(tt_.item())
                return {"workload": "BASELINE configs[3]: image edit (VAE encode 1024^2 + SigLIP 980^2 + 64-token prompt, 49 "
                                    "evals x 3 CFG branches, VAE decode) through InterleaveInferencer, 2 samples per GPU"
                                    + (f" = batch {2 * world} over {world} GPUs, no collective" if world > 1 else ""),
                        "global_batch": 2 * world, "seconds": sec, "s_per_image_per_gpu": sec / 2,
                        "images_per_s": 2 * world / sec}
            extra["edit"] = guarded("edit", edit)

    # ---------------- CPU baseline (rank 0, N=1 only) ----------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        v, sample, _, used = cpu_reference_sample(args.image_size, threads)
        cpu = {"value": v, "unit": UNIT, "cores": used, "kind": "port", "sample": sample, "extrapolated": True,
               "factor": 28 * 2 * EVALS_PER_IMAGE,
               "note": "bounded sample (1 of 28 layers x 1 of 2 branches x 1 of 49 evaluations); `--impl reference` times one "
                       "full _forward_flow (factor 98)"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "BAGEL-7B-MoT random-init text->image 1024^2, 50 timesteps (49 evals), text CFG "
                                   "scale 2 (2 branches packed in one LM call), batch 8 per GPU; step = one "
                                   "denoising step of the batch; images/s = global_batch/(49*s_per_step)",
                       "model": "BAGEL-7B-MoT (random init)", "global_batch": B * world, "per_gpu_batch": B,
                       "image_size": args.image_size, "layers": cfg.num_hidden_layers,
                       "parallelism": f"replica-dp{world}", "l2": "working set per step >> 126 MB L2 (no flush needed)"},
            "per_gpu_images_per_s": value / world, "mfu_vs_sustained_peak": mfu,
            "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
            "e2e_taylorseer": e2e_ts,
        }
        line.update(extra)
        if args.layers is not None:
            line["invalid"] = "debug run with a reduced layer count"
        _emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
