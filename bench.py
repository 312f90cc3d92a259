#!/usr/bin/env python
"""bench.py — YUME denoise-step benchmark on B200 (driver contract: one JSON line on stdout from rank 0).

Workload at N=1 = BASELINE.json configs[1]: one Yume-5B-720P denoise step (WanModel.forward, wan23 tree) on an
81-frame 704x1280 latent [48,21,44,80] -> L = 18 480 tokens, random-init bf16-valued weights, synthetic Gaussian
latent and text context, t = 500. metric = latent frames produced per second by the denoise forward (`ms_per_step`
is the denoise-step latency BASELINE.json names).

  value      device-resident inputs (latent, t, context already in HBM), CUDA-event timed
  e2e        the same step through the reference-facing `WanModel.forward(x, t, context, seq_len, flag=False)`
             with pinned HOST inputs: H2D copies and the D2H read of the result are inside the timed region
  roofline   the dominant kernel (self-attention, attention_kernel<true>) timed live with CUDA events on the
             launching stream inside the timed steps: achieved = 4*L^2*C FLOP / mean launch time
  cpu_baseline / --impl reference: the oracle port of the reference forward (oracle/wan_dit.py) on the host cores,
             on a bounded sample (one WanAttentionBlock of the same workload, extrapolated by FLOPs).
N > 1: Ulysses sequence parallelism over NCCL (one process per GPU, torchrun) — strong scaling of the same step.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

CFG_5B = dict(variant="5b", dim=3072, ffn_dim=14336, num_heads=24, num_layers=30, in_dim=48, out_dim=48,
              text_len=512, text_dim=4096, freq_dim=256)
CFG_14B = dict(variant="14b", dim=5120, ffn_dim=13824, num_heads=40, num_layers=40, in_dim=36, out_dim=16,
               text_len=512, text_dim=4096, freq_dim=256, clip_dim=1280)
LATENT = (48, 21, 44, 80)          # 81 frames @ 704x1280 through the Wan2.2 VAE (stride 4,16,16)
SEQ_LEN = 21 * 22 * 40             # 18 480 tokens
CTX_LEN = 512


def block_flops(L: int, C: int, F: int, S: int) -> float:
    """SURVEY.md §8(d): 8LC^2 + 4L^2C + 4LC^2 + 4SC^2 + 4LSC + 4LCF."""
    return 8 * L * C * C + 4 * L * L * C + 4 * L * C * C + 4 * S * C * C + 4 * L * S * C + 4 * L * C * F


def synthetic_state_dict(cfg: dict, device, seed: int = 0):
    """Random-init weights with the reference's state-dict keys, generated on the device, bf16-representable
    (the reference zero-inits head.head — model.py:914 — which would make the output 0; we use N(0, 0.02))."""
    g = torch.Generator(device=device).manual_seed(seed)
    C, Fd, cin, cout = cfg["dim"], cfg["ffn_dim"], cfg["in_dim"], cfg["out_dim"]

    def rn(*shape, std=1.0):
        return (torch.randn(*shape, generator=g, device=device) * std).to(torch.bfloat16).to(torch.float32)

    sd = {}
    for name, k in (("patch_embedding", 2), ("patch_embedding_2x", 4), ("patch_embedding_4x", 8),
                    ("patch_embedding_8x", 16), ("patch_embedding_16x", 32)):
        sd[name + ".weight"] = rn(C, cin, 1, k, k, std=1 / math.sqrt(cin * k * k))
        sd[name + ".bias"] = rn(C, std=0.02)
    sd["patch_embedding_2x_f.weight"] = rn(cin, cin, 1, 4, 4, std=1 / math.sqrt(cin * 16))
    sd["patch_embedding_2x_f.bias"] = rn(cin, std=0.02)
    sd["text_embedding.0.weight"], sd["text_embedding.0.bias"] = rn(C, cfg["text_dim"], std=1 / 64), rn(C, std=0.02)
    sd["text_embedding.2.weight"], sd["text_embedding.2.bias"] = rn(C, C, std=C ** -0.5), rn(C, std=0.02)
    sd["time_embedding.0.weight"], sd["time_embedding.0.bias"] = rn(C, cfg["freq_dim"], std=1 / 16), rn(C, std=0.02)
    sd["time_embedding.2.weight"], sd["time_embedding.2.bias"] = rn(C, C, std=C ** -0.5), rn(C, std=0.02)
    sd["time_projection.1.weight"], sd["time_projection.1.bias"] = rn(6 * C, C, std=C ** -0.5), rn(6 * C, std=0.02)
    img = cfg["variant"] == "14b"
    if img:
        cd = cfg["clip_dim"]
        sd["img_emb.proj.0.weight"], sd["img_emb.proj.0.bias"] = 1 + rn(cd, std=0.1), rn(cd, std=0.02)
        sd["img_emb.proj.1.weight"], sd["img_emb.proj.1.bias"] = rn(cd, cd, std=cd ** -0.5), rn(cd, std=0.02)
        sd["img_emb.proj.3.weight"], sd["img_emb.proj.3.bias"] = rn(C, cd, std=cd ** -0.5), rn(C, std=0.02)
        sd["img_emb.proj.4.weight"], sd["img_emb.proj.4.bias"] = 1 + rn(C, std=0.1), rn(C, std=0.02)
    for i in range(cfg["num_layers"]):
        p = f"blocks.{i}"
        for att in ("self_attn", "cross_attn"):
            for pr in ("q", "k", "v", "o") + (("k_img", "v_img") if (img and att == "cross_attn") else ()):
                sd[f"{p}.{att}.{pr}.weight"], sd[f"{p}.{att}.{pr}.bias"] = rn(C, C, std=C ** -0.5), rn(C, std=0.02)
            sd[f"{p}.{att}.norm_q.weight"] = 1 + rn(C, std=0.1)
            sd[f"{p}.{att}.norm_k.weight"] = 1 + rn(C, std=0.1)
            if img and att == "cross_attn":
                sd[f"{p}.{att}.norm_k_img.weight"] = 1 + rn(C, std=0.1)
        sd[f"{p}.norm3.weight"], sd[f"{p}.norm3.bias"] = 1 + rn(C, std=0.1), rn(C, std=0.02)
        sd[f"{p}.ffn.0.weight"], sd[f"{p}.ffn.0.bias"] = rn(Fd, C, std=C ** -0.5), rn(Fd, std=0.02)
        sd[f"{p}.ffn.2.weight"], sd[f"{p}.ffn.2.bias"] = rn(C, Fd, std=Fd ** -0.5), rn(C, std=0.02)
        sd[f"{p}.modulation"] = rn(1, 6, C, std=C ** -0.5)
    sd["head.head.weight"], sd["head.head.bias"] = rn(4 * cout, C, std=0.02), rn(4 * cout, std=0.02)
    sd["head.modulation"] = rn(1, 2, C, std=C ** -0.5)
    return sd


DUMP_LIMIT_BYTES = 64 << 20
DUMP_SAMPLE = 1 << 19              # elements kept of a supplementary output (2 MB): the headline output is written whole
DUMP_SAMPLE_ONE = 1 << 22          # elements kept of the one output of a --workload vae* run (16 MB of a 0.9 - 1 GB video)


def dump_sample(t: torch.Tensor, n: int = DUMP_SAMPLE) -> torch.Tensor:
    """`t` flattened, or a fixed sample of n of its elements when it has more: the positions are drawn from a seeded generator
    and depend only on t.numel(), so two runs of the same workload sample the same elements."""
    flat = t.detach().reshape(-1)
    if flat.numel() <= n:
        return flat.float().cpu()
    idx = torch.randint(flat.numel(), (n,), generator=torch.Generator().manual_seed(0)).sort().values
    return flat[idx.to(flat.device)].float().cpu()


def dump_outputs(out_dir, arrays: dict) -> None:
    """Write every output as <out_dir>/<name>.npy in float32 (at most DUMP_LIMIT_BYTES in all)."""
    import numpy as np
    arrays = {name: t.detach().float().cpu().numpy() for name, t in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT_BYTES, f"outputs to dump are {total} bytes, more than {DUMP_LIMIT_BYTES}"
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out_dir / f"{name}.npy", a)


def measured_peaks():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        d = json.loads(f.read_text())
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"], bf16_sustained=d.get("bf16_tflops_sustained"),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_sustained=1400.0, source="fallback (B200_PROFILING.md)")


# ------------------------------------------------------------------------------------------------------------
# CPU reference arm (the one place bench.py executes oracle/ on the CPU): bounded, FIXED sample of the same workload
# ------------------------------------------------------------------------------------------------------------
CPU_SAMPLE_L, CPU_SAMPLE_GRID, CPU_SAMPLE_REPS = 2310, (21, 11, 10), 5


def cpu_reference_sample():
    """Times the oracle port of WanAttentionBlock.forward (oracle/wan_dit.py <- wan23/modules/model.py:272-316) at the
    real 5B width on the host cores. The sample is FIXED — one block at L' = 2310 tokens (1/8 of the sequence), 1 warm-up +
    5 timed repetitions (best taken), independent of --steps / --warmup — so every invocation (product line, BENCH reference arm, SCALE
    reference arm) measures the same thing; it is extrapolated to the 30-block step by algorithmic FLOPs."""
    from oracle import synth
    from oracle.wan_dit import WanOracle, grid_freqs

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = dict(synth.CFG_5B, num_layers=1)
    sd = synth.make_state_dict(cfg, 1, num_layers=1)
    m = WanOracle(sd, **synth.oracle_kwargs(cfg))
    C, F, S = cfg["dim"], cfg["ffn_dim"], cfg["text_len"]
    L, grid = CPU_SAMPLE_L, CPU_SAMPLE_GRID
    g = torch.Generator().manual_seed(0)
    x = torch.randn(1, L, C, generator=g)
    e = 0.5 * torch.randn(1, L, 6, C, generator=g)
    ctx = torch.randn(1, S, C, generator=g)
    fr = grid_freqs(m.tables, *grid)

    def run():
        t0 = time.perf_counter()
        with torch.no_grad():
            m.block(0, x, e, fr, ctx)
        return time.perf_counter() - t0

    run()                                                      # first touch of weights / thread pool: discarded
    times = [run() for _ in range(CPU_SAMPLE_REPS)]
    # best of the repetitions: the host is shared and noisy (2.0 - 5.5 s for the same sample on the same box); the minimum is the
    # reproducible figure and the one most favourable to the reference arm
    t_sample = min(times)
    step_flops = CFG_5B["num_layers"] * block_flops(SEQ_LEN, C, F, S)
    factor = step_flops / block_flops(L, C, F, S)
    return dict(t_sample_s=t_sample, t_step_s=t_sample * factor, cores=cores, L=L, times_s=times, factor=factor,
                sample=f"1 of 30 WanAttentionBlocks (oracle port, fp32 weights, bf16 SDPA) at L={L} of 18480 tokens: "
                       f"best of {CPU_SAMPLE_REPS} reps after 1 warm-up: {t_sample:.2f} s (mean {sum(times) / len(times):.2f}, max {max(times):.2f}), "
                       f"extrapolated to the 30-block step by algorithmic FLOPs (x{factor:.1f})")


def cpu_baseline_isolated() -> dict:
    """The `cpu_baseline` object of the product line: the SAME fixed sample as `--impl reference`, run the same way — a fresh process
    without a CUDA context — so that both arms measure one thing. (The shared 128-core host is noisy: 1.9 - 5.5 s for the identical
    sample across runs on the same box; best-of-5 and process isolation remove what can be removed.) Falls back to the in-process sample."""
    import subprocess
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT")}
    env["CUDA_VISIBLE_DEVICES"] = ""
    try:
        r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                           capture_output=True, text=True, timeout=600, env=env)
        rec = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
        cb = rec["cpu_baseline"]
        cb["ms_per_step"] = rec["ms_per_step"]
        cb["measured_in"] = "a separate process (`bench.py --impl reference`), no CUDA context"
        return cb
    except Exception as e:
        r = cpu_reference_sample()
        return {"value": LATENT[1] / r["t_step_s"], "unit": "latent-frames/s", "cores": r["cores"], "kind": "port",
                "sample": r["sample"], "ms_per_step": r["t_step_s"] * 1e3, "sample_seconds": r["times_s"],
                "extrapolation_factor": r["factor"], "measured_in": f"this process (isolated run failed: {type(e).__name__})"}


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_sample()
    value = LATENT[1] / r["t_step_s"]
    line = {
        "impl": "reference", "metric": "latent_frames_per_sec", "value": value, "unit": "latent-frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["t_step_s"] * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32 (bf16 attention inputs)",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "timing": "time.perf_counter on host; fixed sample (see cpu_baseline.sample), "
                                                   "not a function of --steps/--warmup"},
        "cpu_baseline": {"value": value, "unit": "latent-frames/s", "cores": r["cores"], "kind": "port",
                         "sample": r["sample"], "sample_seconds": r["times_s"], "extrapolation_factor": r["factor"]},
        "e2e": {"value": value, "unit": "latent-frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------
# GPU comparator: the reference's own eager regime (PyTorch ops + SDPA under autocast bf16) on the same B200
# ------------------------------------------------------------------------------------------------------------
def gpu_comparator(dev):
    """The oracle port of WanAttentionBlock.forward run ON THE GPU the way the reference runs its model: stock PyTorch
    eager kernels under torch.autocast(bf16), attention through F.scaled_dot_product_attention (the library FMHA; the
    reference calls flash_attn, absent here — SDPA is the faster of the two on sm_100, profiles/README.md), RoPE in
    complex128 as the reference does. One block at the full L = 18 480, x 30 blocks. BASELINE.md §4."""
    from oracle import synth
    from oracle.wan_dit import WanOracle, grid_freqs
    cfg = dict(synth.CFG_5B, num_layers=1)
    sd = {k: v.to(dev) for k, v in synth.make_state_dict(cfg, 1, num_layers=1).items()}
    m = WanOracle(sd, **synth.oracle_kwargs(cfg))
    m.tables = tuple(t.to(dev) for t in m.tables)
    C, S, L = cfg["dim"], cfg["text_len"], SEQ_LEN
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.randn(1, L, C, generator=g, device=dev)
    e = 0.5 * torch.randn(1, L, 6, C, generator=g, device=dev)
    ctx = torch.randn(1, S, C, generator=g, device=dev)
    fr = grid_freqs(m.tables, 21, 22, 40)
    times = []
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        for i in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            m.block(0, x, e, fr, ctx)
            e1.record()
            torch.cuda.synchronize()
            if i:
                times.append(e0.elapsed_time(e1))
    ms_block = sum(times) / len(times)
    del sd, m, x, e, ctx, fr
    torch.cuda.empty_cache()
    return {"what": "oracle port of the reference block on the same GPU: PyTorch eager + SDPA under autocast(bf16), one "
                    "WanAttentionBlock at L=18480, 3 timed reps after 1 warm-up, x30 blocks (embeddings/head excluded)",
            "ms_per_block": ms_block, "ms_per_step": 30 * ms_block, "value": LATENT[1] / (30 * ms_block * 1e-3),
            "unit": "latent-frames/s"}


# ------------------------------------------------------------------------------------------------------------
# product arm
# ------------------------------------------------------------------------------------------------------------
WORKLOAD = ("Yume-5B-720P single denoise step (WanModel.forward, flag=False), 81-frame 704x1280 latent [48,21,44,80], "
            "L=18480 tokens, 512-token text context, t=500")


def _rand_sd(shapes: dict, dev, gamma_like=lambda n: n.endswith(".gamma"), wscale=0.8):
    g = torch.Generator(device=dev).manual_seed(0)
    sd = {}
    for name, shape in shapes.items():
        t = torch.randn(shape, generator=g, device=dev)
        if name.endswith(".bias"):
            t = 0.05 * t
        elif gamma_like(name) or (len(shape) == 1):
            t = 1 + 0.1 * t
        else:
            t = t * (wscale / math.sqrt(math.prod(shape[1:])))
        sd[name] = t
    return sd


def _timed_simple(fn, steps, warmup, dev_index=0):
    """(ms per call, clocks summary, launches per call, algorithmic TFLOP per call) of fn on one GPU."""
    from yume_b200 import ops
    from yume_b200.utils import ClockSampler
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    with ClockSampler(dev_index) as clocks:
        ops.reset_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return ms, clocks.summary(), ops.launch_count() // steps, ops.flop_count() / steps / 1e12, out


def supplementary(args, dev, eng5, world, rank, peaks, dumps=None):
    """The other BASELINE.json configs, run AFTER the headline so the bench line holds them too (each with its own
    clocks and roofline): configs[3] 5B 4-step distilled loop (+SDE), a 14B FramePack-chunk forward and a 5-step slice of
    configs[2] (50-step ODE with CFG), and at N = 1 the three VAE decodes (configs[4] hyvideo; Wan2.2 / Wan2.1).
    With `dumps`, rank 0 stores there a sample (dump_sample) of each entry's result from its last timed repetition."""
    import torch.distributed as dist

    from yume_b200 import ops, sampler
    from yume_b200.model import WanModel14B
    from yume_b200.utils import ClockSampler
    peak = peaks["bf16_sustained"] or peaks["bf16_tflops"]
    out = {}
    li = dev.index or 0

    def loop_entry(name, fn, new_frames, fwd_per_loop, flops_per_fwd, reps=2, parity_engine=None):
        fn()                                                   # warm-up (fills the context cache / captures graphs)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        with ClockSampler(li) as clocks:
            ops.reset_launch_count()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                res = fn()
            e1.record()
            torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1) / reps], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        ms = float(ms)
        if dumps is not None and rank == 0:
            dumps[name] = dump_sample(res)
        tf = flops_per_fwd * fwd_per_loop / (ms * 1e-3) / 1e12
        out[name] = {"ms_per_loop": ms, "forwards_per_loop": fwd_per_loop, "ms_per_forward": ms / fwd_per_loop,
                     "value": new_frames / (ms * 1e-3), "unit": "new latent-frames/s (new_frames / loop time)",
                     "new_frames": new_frames, "finite": bool(torch.isfinite(res).all()),
                     "gpu_launches_per_loop": ops.launch_count() // reps, "clocks": clocks.summary(),
                     "roofline": {"bound": "tensor", "achieved": tf, "peak": peak, "unit": "TFLOP/s", "frac": tf / peak,
                                  "note": "whole loop: algorithmic FLOPs of all forwards (all ranks) / loop time / GPUs"
                                          if world > 1 else "whole loop: algorithmic FLOPs of all forwards / loop time"}}
        if world > 1:
            out[name]["roofline"]["achieved"] = tf / world
            out[name]["roofline"]["frac"] = tf / world / peak
            if parity_engine is not None:                      # correctness on the record: same engine, rank 0 alone, same inputs
                dist.barrier()
                if rank == 0:
                    with parity_engine.sequence_parallel_disabled():
                        r1 = fn()
                    torch.cuda.synchronize()
                    out[name]["parity_vs_n1"] = float((res.float() - r1.float()).norm() / r1.float().norm())
                    del r1
                dist.barrier()

    # ---- configs[3]: Yume-5B 4-step distilled sampling of one FramePack chunk (5 history + 8 new latent frames) ----
    g = torch.Generator(device=dev).manual_seed(2)
    ctx5 = torch.randn(CTX_LEN, CFG_5B["text_dim"], generator=g, device=dev).to(torch.bfloat16)
    hist = torch.randn(48, 5, 44, 80, generator=g, device=dev)
    noise = torch.randn(48, 8, 44, 80, generator=g, device=dev)
    model5 = eng5["model"]
    e5 = eng5["engine"]
    e5.context_cache = True
    arg_c = dict(context=[ctx5], seq_len=9460)
    fl5 = CFG_5B["num_layers"] * block_flops(9460, CFG_5B["dim"], CFG_5B["ffn_dim"], CTX_LEN)

    def loop5(sde):
        return lambda: sampler.denoise_chunk_5b(model5, torch.cat([hist, noise], 1), hist, 8, 4, arg_c, shift=7.0, sde=sde)
    loop_entry("5b-chunk-4step", loop5(False), 8, 4, fl5, parity_engine=e5)
    loop_entry("5b-chunk-4step-sde", loop5(True), 8, 4, fl5)
    if world == 1:
        e5.use_cuda_graph = True
        loop_entry("5b-chunk-4step-cudagraph", loop5(False), 8, 4, fl5)
        e5.use_cuda_graph = False
    out["5b-chunk-4step"]["config"] = ("BASELINE configs[3]: sample_5b.py:941-1034 loop, 4 Euler steps shift 7.0, L=9460 (5 history "
                                       "+ 8 new latent frames @44x80), per-token t; context K/V cached across the steps")
    # free the 5B engine before the 14B one is built
    eng5.clear()
    del model5, e5
    torch.cuda.empty_cache()

    # ---- configs[2]: Yume-I2V-540P (14B): one FramePack-chunk forward, and a 5-step slice of the 50-step CFG ODE ----
    if not args.no_14b:
        cfg = CFG_14B
        sd = synthetic_state_dict(cfg, dev, seed=0)
        with torch.device("meta"):
            m14 = WanModel14B(model_type="i2v", text_len=cfg["text_len"], in_dim=cfg["in_dim"], dim=cfg["dim"],
                              ffn_dim=cfg["ffn_dim"], freq_dim=cfg["freq_dim"], text_dim=cfg["text_dim"],
                              out_dim=cfg["out_dim"], num_heads=cfg["num_heads"], num_layers=cfg["num_layers"])
        m14.install(dev, state_dict=sd)
        del sd
        torch.cuda.empty_cache()
        e14 = m14._yb_engine
        if world > 1:
            e14.enable_sequence_parallel(dist.group.WORLD, transport=args.sp_transport)
        ctx_c = torch.randn(CTX_LEN, cfg["text_dim"], generator=g, device=dev).to(torch.bfloat16)
        ctx_n = torch.randn(CTX_LEN, cfg["text_dim"], generator=g, device=dev).to(torch.bfloat16)
        x14 = torch.randn(16, 13, 68, 120, generator=g, device=dev)
        mi14 = torch.randn(16, 13, 68, 120, generator=g, device=dev)
        y14 = torch.randn(20, 13, 68, 120, generator=g, device=dev)
        clip = torch.randn(1, 257, 1280, generator=g, device=dev)
        L14, S14 = 21930, CTX_LEN + 257
        fl14 = cfg["num_layers"] * block_flops(L14, cfg["dim"], cfg["ffn_dim"], S14)
        a_c = dict(context=[ctx_c], clip_fea=clip, y=[y14], seq_len=L14)
        a_n = dict(context=[ctx_n], clip_fea=clip, y=[y14], seq_len=L14)
        t14 = torch.tensor([500.0], device=dev)
        e14.context_cache = False
        loop_entry("14b-chunk", lambda: m14([x14], t=t14, rand_num_img=0.6, latent_frame_zero=8, **a_c)[0], 8, 1, fl14, reps=3,
                   parity_engine=e14)
        out["14b-chunk"]["config"] = ("Yume-I2V-540P (14B: dim 5120, 40 heads, 40 layers) single FramePack-chunk forward, 13 latent "
                                      "frames @68x120 (5 history + 8 new), L=21930, 257 CLIP + 512 text context rows; no caching")
        e14.context_cache = True
        loop_entry("14b-cfg-ode-5of50", lambda: sampler.denoise_chunk_14b(m14, x14, mi14, 8, 50, a_c, a_n, rand_num_img=0.6,
                                                                         shift=3.0, guidance=5.0, first_steps=5), 8, 10, fl14, reps=1)
        out["14b-cfg-ode-5of50"]["config"] = ("BASELINE configs[2] slice: first 5 of the 50 Euler steps of sample.py:755-790 (CFG 5.0 -> "
                                              "2 forwards per step, shift 3.0); value extrapolates nothing: 8 new frames / (10 forwards)")
        out["14b-cfg-ode-5of50"]["ms_per_50_steps_extrapolated"] = out["14b-cfg-ode-5of50"]["ms_per_loop"] * 10
        try:
            # the full 81-frame regular grid (no FramePack packing): L = 21 x 34 x 60 = 42 840 tokens, the largest 14B forward
            xg = torch.randn(16, 21, 68, 120, generator=g, device=dev)
            yg = torch.randn(20, 21, 68, 120, generator=g, device=dev)
            Lg = 42840
            flg = cfg["num_layers"] * block_flops(Lg, cfg["dim"], cfg["ffn_dim"], S14)
            e14.context_cache = False
            a_g = dict(context=[ctx_c], clip_fea=clip, y=[yg], seq_len=Lg)
            loop_entry("14b-grid-81f", lambda: m14([xg], t=t14, rand_num_img=0.3, **a_g)[0], 21, 1, flg, reps=2, parity_engine=e14)
            out["14b-grid-81f"]["config"] = ("Yume-I2V-540P (14B) single forward on the full 81-frame 544x960 grid, latent [16,21,68,120], "
                                             "L=42840 (regular-grid RoPE path, rand_num_img < 0.4), 257 CLIP + 512 text context rows; no caching")
            del xg, yg
        except Exception as e:   # never lose the other entries to the largest one
            out["14b-grid-81f"] = {"error": f"{type(e).__name__}: {e}"[:500]}
        del m14, e14
        torch.cuda.empty_cache()

    # ---- VAE decodes (one GPU) ----
    if world == 1 and not args.no_vae:
        from yume_b200.vae import CONFIG_884_16C, HyVaeDecoder
        from yume_b200.vae import decoder_param_shapes as hy_shapes
        from yume_b200.vae21 import Wan21VaeDecoder
        from yume_b200.vae21 import decoder_param_shapes as v21_shapes
        from yume_b200.vae22 import Wan22VaeDecoder
        from yume_b200.vae22 import decoder_param_shapes as v22_shapes

        def vae_entry(name, eng, z, frames_of, config, encode=False):
            ms, clocks, launches, tflop, res = _timed_simple((lambda: eng.encode(z)) if encode else (lambda: eng.decode(z)), 2, 1, li)
            if dumps is not None:
                dumps[name] = dump_sample(res)
            frames = frames_of(res)
            out[name] = {"ms_per_decode": ms, "value": frames / (ms * 1e-3), "unit": ("encoded" if encode else "decoded") + " frames/s",
                         "frames": frames,
                         "gpu_launches": launches, "finite": bool(torch.isfinite(res).all()), "clocks": clocks, "config": config,
                         "roofline": {"bound": "tensor", "achieved": tflop / (ms * 1e-3), "peak": peak, "unit": "TFLOP/s",
                                      "frac": tflop / (ms * 1e-3) / peak, "tflop_per_decode": tflop,
                                      "note": "algorithmic FLOPs of every conv / GEMM launch of the decode (counted per "
                                              "launch by ops.flop_count) / whole-decode time, glue kernels included in the time"}}
            del res
            torch.cuda.empty_cache()

        hy = HyVaeDecoder(_rand_sd(hy_shapes(), dev, wscale=1.5), device=dev, **CONFIG_884_16C)
        hy.enable_tiling()
        vae_entry("hyvae", hy, torch.randn(1, 16, 21, 90, 160, generator=g, device=dev), lambda r: r.shape[2],
                  "BASELINE configs[4]: hyvideo AutoencoderKLCausal3D tiled decode z[1,16,21,90,160] -> [1,3,81,720,1280], 56 tiles")
        del hy
        v22 = Wan22VaeDecoder(_rand_sd(v22_shapes(), dev), device=dev)
        vae_entry("vae22", v22, torch.randn(48, 21, 44, 80, generator=g, device=dev), lambda r: r.shape[1],
                  "Wan2.2 VAE one-pass decode z[48,21,44,80] -> [3,81,704,1280] (what sample_5b.py decodes with)")
        del v22
        v21 = Wan21VaeDecoder(_rand_sd(v21_shapes(), dev), device=dev)
        vae_entry("vae21", v21, torch.randn(16, 21, 68, 120, generator=g, device=dev), lambda r: r.shape[1],
                  "Wan2.1 VAE one-pass decode z[16,21,68,120] -> [3,81,544,960] (what sample.py decodes with)")
        del v21
        torch.cuda.empty_cache()
        # ---- VAE encodes (SURVEY.md §8(f) rank 3): the history / first-frame conditioning encodes of the two samplers ----
        from yume_b200.vae_enc import Wan21VaeEncoder, Wan22VaeEncoder, encoder_param_shapes_21, encoder_param_shapes_22
        e22 = Wan22VaeEncoder(_rand_sd(encoder_param_shapes_22(), dev), device=dev)
        vae_entry("vae22-encode", e22, torch.randn(3, 81, 704, 1280, generator=g, device=dev).clamp_(-1, 1), lambda r: 81,
                  "Wan2.2 VAE one-pass encode video[3,81,704,1280] -> mu[48,21,44,80] (sample_5b.py:892-893 history encode)", encode=True)
        del e22
        e21 = Wan21VaeEncoder(_rand_sd(encoder_param_shapes_21(), dev), device=dev)
        vae_entry("vae21-encode", e21, torch.randn(3, 81, 544, 960, generator=g, device=dev).clamp_(-1, 1), lambda r: 81,
                  "Wan2.1 VAE one-pass encode video[3,81,544,960] -> mu[16,21,68,120] (wan/image2video.py:348-367 conditioning encode)",
                  encode=True)
        del e21
        torch.cuda.empty_cache()
    return out


def product_arm(args):
    import torch.distributed as dist

    from yume_b200 import ops
    from yume_b200.model import WanModel5B
    from yume_b200.utils import ClockSampler

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if world != args.gpus and rank == 0:
        print(f"warning: --gpus {args.gpus} but WORLD_SIZE={world}", file=sys.stderr)

    cfg = CFG_5B
    sd = synthetic_state_dict(cfg, dev, seed=0)
    with torch.device("meta"):
        model = WanModel5B(model_type="ti2v", text_len=cfg["text_len"], in_dim=cfg["in_dim"], dim=cfg["dim"],
                           ffn_dim=cfg["ffn_dim"], freq_dim=cfg["freq_dim"], text_dim=cfg["text_dim"],
                           out_dim=cfg["out_dim"], num_heads=cfg["num_heads"], num_layers=cfg["num_layers"])
    model.install(dev, state_dict=sd)
    del sd
    eng = model._yb_engine
    # the headline is ONE denoise step: everything a step computes is computed inside the timed region — the
    # cross-step context cache (a sampling-loop optimisation, timed in `supplementary`) is switched off
    eng.context_cache = False
    if world > 1:
        eng.enable_sequence_parallel(dist.group.WORLD, transport=args.sp_transport)

    g = torch.Generator().manual_seed(1)
    x_host = torch.randn(*LATENT, generator=g).pin_memory()
    ctx_host = torch.randn(CTX_LEN, cfg["text_dim"], generator=g).to(torch.bfloat16).pin_memory()
    t_host = torch.tensor([500.0]).pin_memory()
    out_host = torch.empty(LATENT, dtype=torch.float32).pin_memory()
    x_dev, ctx_dev, t_dev = x_host.to(dev), ctx_host.to(dev), t_host.to(dev)

    def step_device():
        return eng.forward(x_dev, t_dev, ctx_dev, SEQ_LEN, packed=False)

    def step_e2e():
        xd = x_host.to(dev, non_blocking=True)
        cd = ctx_host.to(dev, non_blocking=True)
        td = t_host.to(dev, non_blocking=True)
        out = model([xd], td, [cd], seq_len=SEQ_LEN, flag=False)[0]
        out_host.copy_(out, non_blocking=True)
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """(total ms of `steps` calls of fn, what the last call returned)"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out

    n_warm = args.warmup if args.quick else max(3, args.warmup)
    for _ in range(n_warm):
        step_device()
    torch.cuda.synchronize()

    # ---- value: K steps, device-resident inputs, NO per-kernel instrumentation inside the timed region ----
    with ClockSampler(local_rank) as clocks:
        ops.reset_launch_count()
        total_ms, last = timed(step_device, args.steps)
        launches = ops.launch_count()
    dumps = None
    if args.dump_outputs and rank == 0:
        dumps = {"latent_out": last.float().cpu()}                 # the denoised latent [48, 21, 44, 80] of the last timed step
    del last
    # ---- e2e: the same step through the reference-facing WanModel.forward with pinned HOST tensors ----
    if args.quick:
        e2e_ms = float("nan")
    else:
        for _ in range(2):
            step_e2e()
        e2e_ms, _ = timed(step_e2e, args.steps)
    # ---- per-kernel table: a SEPARATE instrumented pass (CUDA events around tagged launches on the launching stream) ----
    k_steps = min(args.steps, 5)
    eng.timer.reset()
    eng.timer.active = True
    instr_ms, _ = timed(step_device, k_steps)
    eng.timer.active = False
    kern = eng.timer.summary()

    # ---- multi-GPU correctness on the record: the SP output against the SAME engine run on rank 0 alone ----
    parity = None
    if world > 1:
        out_sp = step_device()
        barrier()
        if rank == 0:
            with eng.sequence_parallel_disabled():
                out_1 = eng.forward(x_dev, t_dev, ctx_dev, SEQ_LEN, packed=False)
            torch.cuda.synchronize()
            parity = {"parity_vs_n1": float((out_sp - out_1).norm() / out_1.norm()),
                      "finite": bool(torch.isfinite(out_sp).all()), "max_abs_diff": float((out_sp - out_1).abs().max()),
                      "what": "rel-Frobenius of the N-GPU Ulysses output vs the same engine run without sequence "
                              "parallelism on rank 0, same inputs, full 5B size (bar: < 5e-3)"}
            del out_1
        barrier()
        del out_sp

    ms_per_step = total_ms / args.steps
    e2e_ms_per_step = e2e_ms / args.steps
    frames = LATENT[1]
    peaks = measured_peaks()
    C, F, L = cfg["dim"], cfg["ffn_dim"], SEQ_LEN
    step_flops = cfg["num_layers"] * block_flops(L, C, F, CTX_LEN)
    # dominant kernel: self-attention (4*L^2*C algorithmic FLOP per launch; with P GPUs each rank does 1/P of the heads)
    att = kern.get("self_attention")
    att_flops = 4.0 * L * L * C / world
    roof = None
    if att:
        ach = att_flops / (att["mean_ms"] * 1e-3) / 1e12
        peak = peaks["bf16_sustained"] or peaks["bf16_tflops"]
        traffic, traffic_src = None, None
        tf = ROOT / "profiles" / "r02_attention_traffic.json"
        if world == 1 and tf.exists():
            tj = json.loads(tf.read_text())
            traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
        roof = {"bound": "tensor", "kernel": "yb::attention kernel (self-attention launch)", "achieved": ach, "peak": peak,
                "unit": "TFLOP/s", "frac": ach / peak,
                "traffic": traffic, "traffic_unit": "bytes/launch",
                "traffic_source": traffic_src or "none this run (offline `ncu --set full` capture; see profiles/)",
                "peak_source": peaks["source"] + ", sustained cuBLAS bf16 (kernel timed inside a long step)",
                "mean_launch_ms": att["mean_ms"], "launches_timed": att["count"],
                "share_of_step": att["total_ms"] / instr_ms,
                "timing": f"CUDA events around each launch in a separate {k_steps}-step instrumented pass "
                          f"({instr_ms / k_steps:.2f} ms/step vs {ms_per_step:.2f} uninstrumented)"}
    gemm_flops = {"gemm_qkv": 6.0 * L * C * C, "gemm_o": 2.0 * L * C * C, "gemm_ffn1": 2.0 * L * C * F,
                  "gemm_ffn2": 2.0 * L * C * F}
    kernels = {}
    for tag, s_ in kern.items():
        k = {"mean_ms": s_["mean_ms"], "count": s_["count"], "share_of_step": s_["total_ms"] / instr_ms}
        if tag in gemm_flops:
            k["tflops"] = gemm_flops[tag] / world / (s_["mean_ms"] * 1e-3) / 1e12
        if tag == "ln_modulate":
            k["gbps"] = (L / world) * C * 6 / (s_["mean_ms"] * 1e-3) / 1e9
        if tag == "qk_norm_rope":
            k["gbps"] = (L / world) * C * 8 / (s_["mean_ms"] * 1e-3) / 1e9
        kernels[tag] = k

    line = None
    if rank == 0:
        line = {
            "metric": "latent_frames_per_sec", "value": frames / (ms_per_step * 1e-3), "unit": "latent-frames/s",
            "n_gpus": world, "steps": args.steps, "warmup": n_warm, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "model": "Yume-5B-720P (Wan2.2-TI2V-5B geometry: dim 3072, ffn 14336, 24 heads, 30 layers), random init",
                       "parallelism": "single GPU" if world == 1 else
                       f"ulysses sp{world} (transport {eng.sp_transport}: "
                       f"{'NVLink peer-memory exchange fused into kernels' if eng._sp_p2p else 'NCCL all-to-all'})",
                       "l2": "per-step working set (10 GB of bf16 weights + 1.5 GB activations) >> 126 MB L2; no flush needed",
                       "caching": "none: text embedding and all 30 cross-attention K/V projections are recomputed inside every timed step",
                       "step_tflop": step_flops / 1e12},
            "step_tflops_achieved": step_flops / (ms_per_step * 1e-3) / 1e12,
            "e2e": {"value": frames / (e2e_ms_per_step * 1e-3), "unit": "latent-frames/s", "ms_per_step": e2e_ms_per_step,
                    "h2d_bytes_per_step": x_host.numel() * 4 + ctx_host.numel() * 2 + 4,
                    "d2h_bytes_per_step": out_host.numel() * 4,
                    "api": "yume_b200.model.WanModel5B.forward(x, t, context, seq_len, flag=False) with pinned host tensors"},
            "gpu_launches": launches,
            "roofline": roof,
            "kernels": kernels,
            "clocks": clocks.summary(),
        }
        if parity is not None:
            line.update(parity)
    if world == 1 and not args.no_cpu_baseline and not args.quick and rank == 0:
        line["cpu_baseline"] = cpu_baseline_isolated()
        try:
            line["gpu_comparator"] = gpu_comparator(dev)
        except Exception as e:  # the comparator is context, never a reason to lose the bench line
            line["gpu_comparator"] = {"error": f"{type(e).__name__}: {e}"}
    if not args.quick and not args.no_supplementary:
        holder = {"model": model, "engine": eng}
        del model, eng
        try:
            sup = supplementary(args, dev, holder, world, rank, peaks, dumps)
        except Exception as e:
            import traceback
            sup = {"error": f"{type(e).__name__}: {e}", "traceback": traceback.format_exc()[-1500:]}
        if rank == 0:
            line["supplementary"] = sup
    if dumps is not None:
        dump_outputs(args.dump_outputs, dumps)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def chunk_arm(args):
    """Supplementary workloads (BASELINE.json configs[2]/[3]): one FramePack-chunk denoise forward.
      5b-chunk : Yume-5B, 13 latent frames @44x80 (5 history + 8 new), L = 9460, per-token t (0 / 900)
      14b-chunk: Yume-I2V-540P (14B), 13 latent frames @68x120, latent_frame_zero 8, L = 21930, CLIP + text context"""
    from yume_b200 import ops
    from yume_b200.dit import WanDiT

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    five = args.config == "5b-chunk"
    cfg = CFG_5B if five else CFG_14B
    sd = synthetic_state_dict(cfg, dev, seed=0)
    kw = {k: cfg[k] for k in ("dim", "ffn_dim", "num_heads", "num_layers", "in_dim", "out_dim", "text_len", "freq_dim")}
    eng = WanDiT(sd, cfg["variant"], device=dev, **kw)
    del sd
    torch.cuda.empty_cache()
    g = torch.Generator(device=dev).manual_seed(1)
    ctx = torch.randn(CTX_LEN, cfg["text_dim"], generator=g, device=dev).to(torch.bfloat16)
    if five:
        x = torch.randn(48, 13, 44, 80, generator=g, device=dev)
        fwd = lambda: eng.forward(x, torch.tensor([[0.0, 900.0]], device=dev), ctx, 0, latent_frame_zero=8, packed=True)  # noqa: E731
        L, S = 9460, CTX_LEN
    else:
        x = torch.randn(16, 13, 68, 120, generator=g, device=dev)
        y = torch.randn(20, 13, 68, 120, generator=g, device=dev)
        clip = torch.randn(1, 257, 1280, generator=g, device=dev)
        fwd = lambda: eng.forward(x, torch.tensor([500.0], device=dev), ctx, 0, y=y, clip_fea=clip, latent_frame_zero=8,  # noqa: E731
                                  packed=True)
        L, S = 21930, CTX_LEN + 257
    for _ in range(max(3, args.warmup)):
        out = fwd()
    torch.cuda.synchronize()
    ops.reset_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out = fwd()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"latent_out": out})
    flops = cfg["num_layers"] * block_flops(L, cfg["dim"], cfg["ffn_dim"], S)
    print(json.dumps({"metric": "latent_frames_per_sec", "value": 8 / (ms * 1e-3), "unit": "latent-frames/s", "n_gpus": 1,
                      "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms, "higher_is_better": True,
                      "dtype": "bf16", "data": "synthetic",
                      "config": {"workload": f"{args.config}: FramePack chunk forward, L={L}, out {tuple(out.shape)}",
                                 "step_tflop": flops / 1e12},
                      "step_tflops_achieved": flops / (ms * 1e-3) / 1e12, "gpu_launches": ops.launch_count(),
                      "finite": bool(torch.isfinite(out).all())}), flush=True)


def vae_arm(args):
    """Supplementary workload (BASELINE.json configs[4]): hyvideo causal 3D VAE tiled decode of z [1,16,21,90,160]
    (81 frames 720x1280) with the upstream 884-16c config, random-init weights. Prints the same JSON schema."""
    import math as _m

    from yume_b200 import ops
    from yume_b200.vae import CONFIG_884_16C, HyVaeDecoder, decoder_param_shapes

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    g = torch.Generator(device=dev).manual_seed(0)
    sd = {}
    for name, shape in decoder_param_shapes().items():
        t = torch.randn(shape, generator=g, device=dev)
        if name.endswith(".bias"):
            t = 0.05 * t
        elif len(shape) == 1:
            t = 1 + 0.1 * t
        else:
            t = t * (1.5 / _m.sqrt(_m.prod(shape[1:])))
        sd[name] = t
    eng = HyVaeDecoder(sd, device=dev, **CONFIG_884_16C)
    eng.enable_tiling()
    T, H, W = (21, 90, 160) if not args.quick else (5, 40, 40)
    z = torch.randn(1, 16, T, H, W, generator=g, device=dev)
    for _ in range(args.warmup):
        eng.decode(z)
    torch.cuda.synchronize()
    ops.reset_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out = eng.decode(z)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"video": dump_sample(out, DUMP_SAMPLE_ONE)})
    frames = out.shape[2]
    print(json.dumps({"metric": "decoded_frames_per_sec", "value": frames / (ms * 1e-3), "unit": "frames/s", "n_gpus": 1,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                      "dtype": "bf16", "data": "synthetic",
                      "config": {"workload": f"hyvideo AutoencoderKLCausal3D tiled decode z[1,16,{T},{H},{W}] -> {tuple(out.shape)}",
                                 "tiles": "spatial 32x32 stride 24, temporal 17 stride 12 (upstream 884-16c)"},
                      "gpu_launches": ops.launch_count(), "finite": bool(torch.isfinite(out).all())}), flush=True)


def vae22_arm(args):
    """Supplementary workloads (SURVEY.md §8(f) rank 1), random-init weights at the real widths:
    vae22 — Wan2.2 VAE decode of the 5B sampler's latent z [48,21,44,80] -> video [3,81,704,1280] (`Wan2_2_VAE.decode`);
    vae21 — Wan2.1 VAE decode of the 14B sampler's 540p latent z [16,21,68,120] -> [3,81,544,960] (`WanVAE.decode`)."""
    from yume_b200 import ops
    if args.workload == "vae22":
        from yume_b200.vae22 import Wan22VaeDecoder as Decoder, decoder_param_shapes
        zc, full, label = 48, (21, 44, 80), "Wan2.2 VAE"
    else:
        from yume_b200.vae21 import Wan21VaeDecoder as Decoder, decoder_param_shapes
        zc, full, label = 16, (21, 68, 120), "Wan2.1 VAE"

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    g = torch.Generator(device=dev).manual_seed(0)
    sd = {}
    for name, shape in decoder_param_shapes().items():
        t = torch.randn(shape, generator=g, device=dev)
        if name.endswith(".bias"):
            t = 0.05 * t
        elif name.endswith(".gamma"):
            t = 1 + 0.1 * t
        else:
            t = t * (0.8 / math.sqrt(math.prod(shape[1:])))
        sd[name] = t
    eng = Decoder(sd, device=dev)
    T, H, W = full if not args.quick else (5, 16, 16)
    z = torch.randn(zc, T, H, W, generator=g, device=dev)
    for _ in range(args.warmup):
        eng.decode(z)
    torch.cuda.synchronize()
    ops.reset_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out = eng.decode(z)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"video": dump_sample(out, DUMP_SAMPLE_ONE)})
    print(json.dumps({"metric": "decoded_frames_per_sec", "value": out.shape[1] / (ms * 1e-3), "unit": "frames/s", "n_gpus": 1,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                      "dtype": "bf16", "data": "synthetic",
                      "config": {"workload": f"{label} whole-sequence decode z[{zc},{T},{H},{W}] -> {tuple(out.shape)}"},
                      "gpu_launches": ops.launch_count(), "peak_mem_gb": torch.cuda.max_memory_allocated() / 2**30,
                      "finite": bool(torch.isfinite(out).all())}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="dit", choices=["dit", "vae", "vae22", "vae21"])
    ap.add_argument("--config", default="5b-720p", choices=["5b-720p", "5b-chunk", "14b-chunk"],
                    help="5b-720p is the headline workload (BASELINE.json configs[1]); the others are supplementary")
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps (at least 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="yume_b200", choices=["yume_b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-supplementary", action="store_true", help="headline only (no configs[2]/[3]/[4] side runs)")
    ap.add_argument("--no-14b", action="store_true", help="supplementary: skip the 14B runs")
    ap.add_argument("--no-vae", action="store_true", help="supplementary: skip the VAE decodes")
    ap.add_argument("--sp-transport", default="auto", choices=["auto", "p2p", "p2p_gemm", "nccl"])
    ap.add_argument("--gemm-split-k", type=int, default=0, choices=[0, 1], help="tail split-K of the gate+residual GEMMs: 0 automatic, 1 never (A/B)")
    ap.add_argument("--quick", action="store_true", help="profiling runs: exact --warmup, no e2e leg, no CPU baseline")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float32; the headline "
                         "latent whole, each supplementary result and a VAE video as a fixed seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    torch.manual_seed(0)     # draws without an explicit generator (the SDE loop's noise) repeat from run to run
    if args.gemm_split_k:
        from yume_b200 import ops as _ops
        _ops.GEMM_SPLIT_K = args.gemm_split_k
    if args.workload == "vae":
        vae_arm(args)
    elif args.workload in ("vae22", "vae21"):
        vae22_arm(args)
    elif args.config != "5b-720p":
        chunk_arm(args)
    elif args.impl == "reference":
        reference_arm(args)
    else:
        product_arm(args)


if __name__ == "__main__":
    main()
