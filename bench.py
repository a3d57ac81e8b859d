#!/usr/bin/env python
"""bench.py — frames/sec of the Self-Forcing hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One STEP = one generation block of the server loop (release_server.py:636-736) at
BASELINE configs[1]: Krea-14B dims (40 layers, d=5120, ffn 13824, 40 heads), 832x480,
kv_cache_num_frames=3, 4 denoise steps: 1 KV-recompute DiT pass + 4 denoise DiT passes + VAE
decode of 3 latent frames -> 12 pixel frames.  Synthetic seeded weights / prompt embedding /
noise (no checkpoints, no network).  Warm-up covers block 0 (no recompute, 6 frames), so every
timed step is a steady-state block.

value : frames/s with inputs resident in HBM, timed with CUDA events, max over ranks.
e2e   : same loop through the same public API (realtime_video_b200/dropin wrappers) with the
        block's noise copied from pinned host memory every step and the decoded fp32 frames
        copied back to pinned host memory inside the timed region.
N > 1 : ONE video stream on all N GPUs (strong scaling; realtime_video_b200/parallel.py: token rows sharded for
        everything token-wise, heads sharded for self-attention, the rows<->heads exchange written straight into the
        peers' buffers over NVLink by the kernels).  value = frames of that one stream / max-over-ranks time.
        The throughput-oriented alternative (N independent replicas, no data-path collective) is measured in
        the same run and reported as the secondary key "replicas".  --parallel replicas makes it the headline.
--workload vae_decode : VAE-decode-only throughput (BASELINE configs[4]): a stream of 3-latent-frame blocks through
        the decoder with a warm feature cache; frames/s, conv TF/s and algorithmic HBM GB/s vs the measured peak.
--impl reference : the reference algorithm on the host CPU cores (oracle port, torch fp32, all
        threads) on a bounded sample of the same workload, scaled to frames/s.
--dump-outputs DIR : after the timed steps, write what the last timed step returned as DIR/<name>.npy (float32):
        ``frames`` [1, 12, 3, 480, 832] and, for the block workload, that block's denoised ``latents``
        [1, 3, 16, 60, 104].  Weights, prompt and noise are seeded, so two builds run with the same arguments can
        be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

WORKLOAD = "krea14b_832x480_4step_kv3_block12f"
FRAMES_PER_STEP = 12
D, FFN, HEADS, LAYERS, TEXT = 5120, 13824, 40, 40, 512
LQ, LKV = 4680, 9360


def layer_flops(lq, lkv):
    """SURVEY.md §8d: Lq*(12 d^2 + 4 d ffn + 4 d (Lkv + 512))."""
    return lq * (12 * D * D + 4 * D * FFN + 4 * D * (lkv + TEXT))


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        j = json.loads(p.read_text())
        return {"tensor": j.get("bf16_tflops_sustained", 1425.5), "hbm": j.get("hbm_gbs", 6480.8),
                "source": "MEASURED_PEAKS.json (sustained cuBLAS bf16; kernel timed inside a long step)"}
    return {"tensor": 1400.0, "hbm": 6650.0, "source": "fallback of B200_PROFILING.md"}


# ---------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ---------------------------------------------------------------------------------------------
class Clocks:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=f, stderr=subprocess.DEVNULL)
        except Exception:  # noqa: BLE001
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                c = [x.strip() for x in line.split(",")]
                if len(c) < 7:
                    continue
                try:
                    sm.append(float(c[0])); mx.append(float(c[1]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:  # noqa: BLE001
            pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


# ---------------------------------------------------------------------------------------------
# CPU baseline: the oracle port on the host cores, bounded sample
# ---------------------------------------------------------------------------------------------
def _best_thread_count() -> int:
    """fp32 GEMM throughput of this host at a few thread counts (oversubscribed SMT / NUMA hosts
    are often fastest below os.cpu_count()); returns the fastest."""
    cores = os.cpu_count() or 1
    a, b = torch.randn(2048, 2048), torch.randn(2048, 2048)
    best, best_t = cores, None
    for n in sorted({cores, max(1, cores // 2), max(1, cores // 4), min(cores, 32)}, reverse=True):
        torch.set_num_threads(n)
        a @ b
        t0 = time.time()
        for _ in range(3):
            a @ b
        dt = time.time() - t0
        if best_t is None or dt < best_t:
            best, best_t = n, dt
    torch.set_num_threads(best)
    return best


class CpuReference:
    """The oracle port (torch fp32) on DiT layer-forwards at the full C2 size: Lq=4680 new tokens
    against Lkv=9360 cached keys, d=5120, ffn 13824.  One 12-frame block = 4 denoise passes x 40
    layers at Lkv=9360 + 1 recompute pass x 40 layers at Lkv=4680 (+ VAE, not sampled); a measured
    per-layer time is scaled by FLOPs to that block."""

    def __init__(self):
        from oracle import dit_oracle as O
        self.O = O
        self.threads = _best_thread_count()
        cfg = O.DiTConfig(dim=D, ffn_dim=FFN, num_heads=HEADS, num_layers=1)
        g = torch.Generator().manual_seed(0)

        def rnd(*shape, s=0.02):
            return torch.randn(*shape, generator=g) * s

        p = {"blocks.0.modulation": rnd(1, 6, D, s=D ** -0.5)}
        for pre in ("blocks.0.self_attn.", "blocks.0.cross_attn."):
            for n in "qkvo":
                p[pre + n + ".weight"], p[pre + n + ".bias"] = rnd(D, D), rnd(D)
            p[pre + "norm_q.weight"], p[pre + "norm_k.weight"] = torch.ones(D), torch.ones(D)
        p["blocks.0.norm3.weight"], p["blocks.0.norm3.bias"] = torch.ones(D), torch.zeros(D)
        p["blocks.0.ffn.0.weight"], p["blocks.0.ffn.0.bias"] = rnd(FFN, D), rnd(FFN)
        p["blocks.0.ffn.2.weight"], p["blocks.0.ffn.2.bias"] = rnd(D, FFN), rnd(D)
        self.orc = O.DiTOracle(cfg, p)
        self.x, self.e0, self.ctx = rnd(LQ, D, s=1.0), rnd(3, 6, D, s=0.1), rnd(TEXT, D, s=1.0)
        self.kv = O.new_kv_cache(cfg, LKV, torch.float32)[0]
        self.kv["k"].normal_(generator=g)
        self.kv["v"].normal_(generator=g)
        self.ca = O.new_crossattn_cache(cfg, torch.float32)[0]
        self.times = []

    def layer_forward(self) -> float:
        self.kv["global_end_index"], self.kv["local_end_index"] = LQ, LQ   # 3 context frames cached
        t0 = time.time()
        with torch.no_grad():
            self.orc.block(0, self.x, self.e0, (3, 30, 52), self.ctx, self.kv, self.ca, LQ, None)
        dt = time.time() - t0
        self.times.append(dt)
        return dt

    @staticmethod
    def fps_from_layer_time(t_layer: float) -> float:
        block_flops = 4 * LAYERS * layer_flops(LQ, LKV) + LAYERS * layer_flops(LQ, LQ)
        return FRAMES_PER_STEP / (t_layer * block_flops / layer_flops(LQ, LKV))

    def describe(self, t_layer: float, n: int) -> dict:
        return {"value": self.fps_from_layer_time(t_layer), "unit": "frames/s", "cores": self.threads,
                "kind": "port",
                "sample": f"{n} DiT layer-forward(s) (Lq=4680, Lkv=9360, d=5120, ffn 13824, fp32 torch oracle, "
                          f"{self.threads} of {os.cpu_count()} host threads = fastest measured), "
                          f"{t_layer:.2f} s/layer; scaled by FLOPs to the 200 layer-passes of a 12-frame "
                          f"block; VAE decode not included (would lower it further)"}


def cpu_reference_sample(budget_s: float = 25.0, max_layers: int = 8) -> dict:
    ref = CpuReference()
    t_all = time.time()
    for i in range(max_layers):
        ref.layer_forward()
        if time.time() - t_all > budget_s and i >= 1:
            break
    t_layer = min(ref.times[1:]) if len(ref.times) > 1 else ref.times[0]    # first call warms up
    return ref.describe(t_layer, len(ref.times))


def run_reference_arm(args, rank, world):
    """--impl reference: every STEP is one DiT layer-forward of the oracle port (a bounded sample of
    the 200 layer-passes + VAE that make one 12-frame block), scaled to frames/s."""
    if rank != 0:
        return
    steps = max(1, args.steps)
    ref = CpuReference()
    for _ in range(max(1, args.warmup)):
        ref.layer_forward()
    t0 = time.time()
    ts = [ref.layer_forward() for _ in range(steps)]
    t_layer = (time.time() - t0) / steps
    v = ref.fps_from_layer_time(t_layer)
    line = {"impl": "reference", "metric": "frames_per_second_832x480_4step_t2v", "value": v, "unit": "frames/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * t_layer, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "note": "reference algorithm (oracle port pinned to the reference) on "
                       "host CPU cores; one step = one DiT layer-forward at full size, value scaled by FLOPs to "
                       "frames/s of a whole 12-frame block"},
            "cpu_baseline": ref.describe(t_layer, len(ts)),
            "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
_JSON_FD = None


def _claim_stdout():
    """stdout must carry exactly ONE JSON line: park the real stdout and point fd 1 at stderr, so
    anything a library prints (e.g. NCCL's version banner) cannot land in front of it."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


DUMP_LIMIT_BYTES = 64 * 10 ** 6


def dump_outputs(path: str, arrays: dict):
    """Write each host tensor of ``arrays`` as ``path/<name>.npy`` in float32."""
    import numpy as np
    total = sum(a.numel() * 4 for a in arrays.values())
    assert total <= DUMP_LIMIT_BYTES, f"outputs to dump take {total} bytes, over {DUMP_LIMIT_BYTES}"
    out = Path(path)
    out.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out / f"{name}.npy", a.to(torch.float32).numpy())


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def _flat_roofline(prof: dict, ms_step: float, peaks: dict, traffic_db: dict) -> dict:
    """roofline object for the dominant kernel family (the tcgen05 GEMMs) + flat per-kernel scalars.
    ``prof`` comes from ONE separately profiled step (CUDA events around every launch of a family), never from the
    timed region; ``share`` = family time / that step's time."""
    def fam(name):
        g = prof.get(name)
        if not g or g["ms"] <= 0:
            return None, None, 0
        return g["flops"] / (g["ms"] * 1e-3) / 1e12, g["ms"] / ms_step, g["n"]
    gem, gem_share, gem_n = fam("gemm")
    out = {"bound": "tensor",
           "kernel": "kr_gemm (tcgen05: gemm2_tn_kernel CTA-pair + gemm_tn_kernel single-CTA, all DiT linears)",
           "achieved": gem, "peak": peaks["tensor"], "unit": "TFLOP/s", "frac": (gem / peaks["tensor"]) if gem else None,
           "peak_source": peaks["source"], "launches_timed": gem_n, "share_of_step": gem_share,
           "how": "algorithmic FLOPs of the launches / their CUDA-event time, from one extra profiled step after the "
                  "timed region (the timed region itself carries no per-launch events)"}
    by_kernel = {}
    for label, key in (("gemm2", "gemm/gemm2_tn_kernel"), ("gemm1", "gemm/gemm_tn_kernel"),
                       ("gemm_streamk", "gemm/gemm_sk_kernel"), ("gemm_flex", "gemm/gemm_flex_kernel"),
                       ("attn", "attention"), ("vae_conv", "vae_conv")):
        a, share, n = fam(key)
        out[label + "_tflops"] = a
        out[label + "_frac"] = (a / peaks["tensor"]) if a else None
        out[label + "_share"] = share
        if a is not None:
            by_kernel[label] = {"achieved": a, "frac": a / peaks["tensor"], "launches_timed": n, "share_of_step": share}
    dominant = max(("gemm2_tn_kernel", "gemm_tn_kernel"),
                   key=lambda k: (prof.get("gemm/" + k) or {"ms": 0})["ms"])
    out["traffic"] = traffic_db.get(dominant, {}).get("dram_bytes_per_launch")
    out["traffic_kernel"] = dominant
    out["by_kernel"] = by_kernel
    return out


def _traffic_db() -> dict:
    for name in ("r02_gemm_traffic.json", "r01_gemm_traffic.json"):
        tp = ROOT / "profiles" / name
        if tp.exists():
            try:
                return json.loads(tp.read_text())
            except Exception:  # noqa: BLE001
                pass
    return {}


def _reference_host_egress_ms(px: torch.Tensor, reps: int = 2):
    """The reference's own frame egress on this box's host cores, timed on the block just decoded: fp32 download to
    pinned memory, ``add_(1).mul_(0.5).clamp_(0, 1)`` (release_server.py:979-983), then per frame
    ``to_pil_image(...).save(JPEG, quality=90)`` in a 24-thread pool (release_server.py:945-946, :973)."""
    try:
        import io
        from concurrent.futures import ThreadPoolExecutor

        import torchvision.transforms.functional as TF
        host = torch.empty(px.shape, dtype=torch.float32)
        if px.is_cuda:
            host = host.pin_memory()

        def enc(frame):
            buf = io.BytesIO()
            TF.to_pil_image(frame, "RGB").save(buf, format="JPEG", quality=90)
            return buf.getvalue()
        with ThreadPoolExecutor(max_workers=24) as pool:
            ts = []
            for _ in range(reps + 1):
                t0 = time.time()
                host.copy_(px)
                norm = host.add_(1.0).mul_(0.5).clamp_(0.0, 1.0)
                list(pool.map(enc, [norm[0, i] for i in range(norm.shape[1])]))
                ts.append(time.time() - t0)
        return 1e3 * min(ts[1:])
    except Exception:  # noqa: BLE001 - Pillow / torchvision missing: no host comparison
        return None


def assemble_line(args, world, sp_mode, pp_mode, use_graphs, main_run, e2e_run, egress, egress_jpeg, fp8_line, secondary,
                  cpu) -> dict:
    """The ONE JSON line of the block workload from the measured pieces (pure: no GPU, unit-tested on the CPU in
    tests/test_bench_line_cpu.py so that a key error cannot cost a finished multi-minute run its result)."""
    K, W = args.steps, args.warmup
    streams = 1 if sp_mode else world
    ms = main_run["ms"]
    value = streams * K * FRAMES_PER_STEP / (ms / 1e3)
    e2e = streams * K * FRAMES_PER_STEP / (e2e_run["ms"] / 1e3)
    peaks = measured_peaks()
    roofline = _flat_roofline(main_run["prof"], main_run["ms_prof"], peaks, _traffic_db())
    block_tflop = (4 * LAYERS * layer_flops(LQ, LKV) + LAYERS * layer_flops(LQ, LQ)) / 1e12 * (args.layers / LAYERS)
    if pp_mode:
        par = (f"ONE stream on {world} GPUs, DiT layers sharded {LAYERS}/{world} per GPU (BASELINE configs[2]): residual "
               f"stream handed GPU i -> i+1 with one NCCL send/recv per pass (47.9 MB), head output broadcast; stages run "
               f"one after another, so this is the capacity configuration, not a latency one; VAE decode on rank 0")
    elif sp_mode:
        how = ("the rows<->heads exchange is done by the kernels over NVLink peer memory" if main_run.get("exchange") == "p2p"
               else f"the rows<->heads exchange falls back to NCCL all-to-all ({main_run.get('exchange_note')})")
        par = (f"ONE stream on {world} GPUs: token rows sharded for all token-wise kernels, heads sharded for "
               f"self-attention; {how} (realtime_video_b200/parallel.py); VAE decode on rank 0")
    else:
        par = "1 GPU" if world == 1 else f"{world} independent replicas (no data-path collective)"
    line = {
        "metric": "frames_per_second_832x480_4step_t2v", "value": value, "unit": "frames/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True,
        "scaling": "strong" if sp_mode else "weak", "vs_baseline": (value / 11.0) if world == 1 else None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": WORKLOAD, "dims": "Wan2.1-T2V-14B (40 layers, d 5120, ffn 13824, 40 heads)"
                   if args.layers == LAYERS else f"DEBUG {args.layers} layers",
                   "resolution": "832x480", "denoise_steps": 4, "kv_cache_num_frames": 3, "frames_per_step": 12,
                   "passes_per_step": "1-frame VAE encode + 1 KV recompute + 4 denoise DiT passes + VAE decode (fp16)",
                   "first_frame": "re-encoded from the oldest cached pixel frame once the window slides "
                                  "(reference default keep_first_frame=False, release_server.py:571-576)",
                   "parallelism": par,
                   "l2": "weights (28 GB/pass) and KV cache exceed the 126 MB L2 every step; no flush needed",
                   "cuda_graphs": "each DiT pass replayed as a CUDA graph (captured on its 2nd occurrence)" if use_graphs
                                  else "off (eager launches)",
                   "block_fwd": "one kr_dit_block_fwd call per DiT block" if args.block_fwd == "on" else "per-op calls",
                   "dit_tflop_per_step": block_tflop},
        "egress_rgb8": egress,
        "egress_jpeg": egress_jpeg,
        "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": e2e_run["h2d"],
                "d2h_bytes_per_step": e2e_run["d2h"], "ms_per_step": e2e_run["ms"] / K},
        "gpu_launches": main_run["launches"],
        "clocks": main_run["clocks"],
        "roofline": roofline,
        "cpu_baseline": cpu,
        "baseline_note": "vs_baseline = value / 11 fps (reference README.md:31: 11 fps on 1x B200, 4 steps); null for N>1 (nothing published)",
    }
    if secondary is not None:
        line[secondary["mode"]] = secondary
    if fp8_line is not None:
        line["fp8"] = fp8_line
    return line


def run_vae_workload(args, dev, rank, world, barrier, max_over_ranks):
    """BASELINE configs[4]: VAE-decode-only throughput at 832x480.  One step = one steady block (3 latent frames ->
    12 pixel frames) of a running stream (warm feature cache); N > 1 = N independent streams (the decoder is one
    causal stream; nothing to exchange)."""
    from realtime_video_b200 import factory, ops
    K, W = args.steps, max(3, args.warmup)
    vae = factory.synthetic_vae_decoder(device=dev)
    g = torch.Generator(device=dev).manual_seed(7 + rank)
    zs = [torch.randn(1, 3, 16, 60, 104, device=dev, dtype=torch.float16, generator=g) for _ in range(W + K + 1)]
    host_z = [z.cpu().pin_memory() for z in zs]
    host_px = torch.empty(1, 12, 3, 480, 832, dtype=torch.float32).pin_memory()
    cache = [None] * 55
    with torch.inference_mode():
        for i in range(W):
            px, cache = vae(zs[i], *cache)
        barrier()
        clocks = Clocks(dev.index)
        if rank == 0:
            clocks.start()
        n0 = ops.launch_count
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(W, W + K):
            px, cache = vae(zs[i], *cache)
        e1.record()
        barrier()
        launches = ops.launch_count - n0
        clk = clocks.stop() if rank == 0 else None
        ms = max_over_ranks(e0.elapsed_time(e1))
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, {"frames": px.float().cpu()})
        # one profiled step (per-launch events) for the conv family's TF/s
        ops.profile_begin()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        px, cache = vae(zs[W + K], *cache)
        p1.record()
        torch.cuda.synchronize()
        prof = ops.profile_end()
        ms_prof = p0.elapsed_time(p1)
        # end to end: latents from pinned host memory, fp32 frames back to pinned host memory
        cache2 = [None] * 55
        zdev = torch.empty_like(zs[0])
        for i in range(W):
            px, cache2 = vae(zs[i], *cache2)
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for i in range(W, W + K):
            zdev.copy_(host_z[i], non_blocking=True)
            px, cache2 = vae(zdev, *cache2)
            host_px.copy_(px, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        t1.record()
        barrier()
        ms_e2e = max_over_ranks(t0.elapsed_time(t1))
    assert px.shape == (1, 12, 3, 480, 832)
    if rank != 0:
        return
    peaks = measured_peaks()
    vcv = prof.get("vae_conv", {"flops": 0.0, "ms": 0.0, "n": 0})
    conv_tf = vcv["flops"] / (vcv["ms"] * 1e-3) / 1e12 if vcv["ms"] > 0 else None
    # SURVEY.md §8d: >= 24.1 GB of conv input+output (fp16) per steady block if nothing is fused; irreducible
    # (fully fused) = feature-cache read+write 3.8 GB + pixels 57.5 MB + weights 146.6 MB = 4.0 GB
    ALG_UNFUSED, ALG_FUSED = 24.1e9, 4.0e9
    gbs = ALG_UNFUSED / (ms / K * 1e-3) / 1e9
    vt = {}
    tp = ROOT / "profiles" / "r02_vae_traffic.json"
    if tp.exists():
        try:
            vt = json.loads(tp.read_text())
        except Exception:  # noqa: BLE001
            vt = {}
    line = {"metric": "vae_decode_frames_per_second_832x480", "value": world * K * 12 / (ms / 1e3), "unit": "frames/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {"workload": "vae_decode_832x480_block12f", "latent": "[1,3,16,60,104] fp16 per step, warm feature cache",
                       "parallelism": "1 GPU" if world == 1 else f"{world} independent decoder streams",
                       "l2": "each layer's activations (0.9 GB at 480x832) exceed the 126 MB L2; no flush needed"},
            "e2e": {"value": world * K * 12 / (ms_e2e / 1e3), "unit": "frames/s", "ms_per_step": ms_e2e / K,
                    "h2d_bytes_per_step": host_z[0].numel() * 2, "d2h_bytes_per_step": host_px.numel() * 4},
            "gpu_launches": launches, "clocks": clk,
            "roofline": {"bound": "tensor", "kernel": "conv_halo_kernel / conv_igemm_kernel (implicit-GEMM causal conv3d)",
                         "achieved": conv_tf, "peak": peaks["tensor"], "unit": "TFLOP/s",
                         "frac": conv_tf / peaks["tensor"] if conv_tf else None, "peak_source": peaks["source"],
                         "share_of_step": vcv["ms"] / ms_prof if ms_prof > 0 else None, "launches_timed": vcv["n"],
                         "traffic": vt.get("dram_bytes_per_block"),
                         "hbm": {"algorithmic_gb_per_block_unfused": ALG_UNFUSED / 1e9,
                                 "algorithmic_gb_per_block_fully_fused": ALG_FUSED / 1e9,
                                 "achieved_gbs_vs_unfused_bytes": gbs, "peak_gbs": peaks["hbm"],
                                 "frac_of_hbm_peak": gbs / peaks["hbm"],
                                 "measured_dram_gb_per_block": (vt.get("dram_bytes_per_block") or 0) / 1e9 or None}},
            "cpu_baseline": None}
    emit(line)


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--parallel", default="sp", choices=["replicas", "sp", "pp"],
                    help="N>1 headline: ONE stream sequence-parallel over all GPUs (default, strong scaling; "
                         "realtime_video_b200/parallel.py), N independent replicas (weak scaling), or pp = ONE stream "
                         "with the DiT layers sharded over the GPUs (BASELINE configs[2]: capacity, not latency)")
    ap.add_argument("--workload", default="block", choices=["block", "vae_decode"])
    ap.add_argument("--layers", type=int, default=LAYERS, help=argparse.SUPPRESS)      # debugging only
    ap.add_argument("--no-cpu-baseline", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--no-egress", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--no-secondary", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--no-fp8", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--graphs", default="off", choices=["on", "off"],
                    help="replay each DiT pass as a CUDA graph (validated on one GPU, tests/test_server_loop_gpu.py; "
                         "NOT with the multi-GPU exchange inside the capture: an 8-GPU run with it on hung)")
    ap.add_argument("--block-fwd", default="off", choices=["on", "off"],
                    help="issue every DiT block as ONE C-ABI call (kr_dit_block_fwd; same launches, less host work; "
                         "single-GPU bf16 passes with a warm prompt cache)")
    ap.add_argument("--watchdog-s", type=int, default=600, help=argparse.SUPPRESS)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last timed step's outputs as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1 and args.watchdog_s > 0:
        # a multi-rank run that stops making progress (a rank died, a peer never arrived at a barrier) must not sit
        # on N GPUs until an outer limit fires: hard exit after watchdog_s
        def _bail():
            sys.stderr.write(f"bench.py: watchdog fired after {args.watchdog_s} s on rank {rank}; exiting\n")
            sys.stderr.flush()
            os._exit(3)
        _wd = threading.Timer(args.watchdog_s, _bail)
        _wd.daemon = True
        _wd.start()
    if world > 1:
        import torch.distributed as dist
        # stdout carries exactly ONE JSON line: keep NCCL's "NCCL version ..." banner off it
        # (the image exports NCCL_DEBUG; NCCL writes its banner/diagnostics to stdout unless redirected)
        os.environ.setdefault("NCCL_DEBUG_FILE", os.path.join(tempfile.gettempdir(), "nccl_bench.%h.%p.log"))
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        import torch.distributed as dist
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    if args.workload == "vae_decode":
        run_vae_workload(args, dev, rank, world, barrier, max_over_ranks)
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
            dist.destroy_process_group()
        return

    import harness
    from harness import GenerateParams, GenerationSession
    from realtime_video_b200 import factory, ops
    K, W = args.steps, args.warmup
    transformer = factory.synthetic_transformer("14B", device=dev, num_layers=args.layers, seed=0)
    vae = factory.synthetic_vae_decoder(device=dev)
    vae_enc = factory.synthetic_vae_encoder(device=dev)
    models = harness.build_models(transformer, vae_decoder=vae, device=dev, vae_encoder=vae_enc)
    pe = factory.synthetic_prompt_embeds(device=dev)
    sp_mode = world > 1 and args.parallel in ("sp", "pp")      # ONE stream on all GPUs (sequence- or layer-sharded)
    pp_mode = world > 1 and args.parallel == "pp"
    use_graphs = args.graphs == "on"
    transformer.model.use_block_fwd = args.block_fwd == "on"

    def measure(sp: bool, steps: int, seed: int, profile_step: bool, keep_outputs: bool = False):
        """W warm-up blocks, then ``steps`` timed blocks (CUDA events, barrier + synchronize on both sides, max over
        ranks); optionally ONE more block with per-launch events for the kernel split.  ``keep_outputs``: copy what
        the last timed block returned to the host, as ``out["outputs"]``."""
        if sp and pp_mode:
            from realtime_video_b200.parallel import LayerPipeline
            if transformer.model.pp is None:
                transformer.model.pp = LayerPipeline()
        elif sp:
            from realtime_video_b200.parallel import SequenceParallel
            if transformer.model.sp is None:
                transformer.model.sp = SequenceParallel()
        else:
            transformer.model.sp = transformer.model.pp = None
        decode = (not sp) or rank == 0              # one stream -> one VAE decode (rank 0)
        transformer.use_cuda_graphs = use_graphs and sp == sp_mode
        transformer._graphs = {}
        sess = GenerationSession(GenerateParams(num_blocks=W + steps + 1, seed=seed + (0 if sp else rank)), models,
                                 prompt_embeds=pe, device=dev, decode=decode)
        out = {"decode": decode}
        with torch.inference_mode():
            for _ in range(W):
                sess.generate_block()
            barrier()
            clocks = Clocks(local)
            if rank == 0:
                clocks.start()
            n0 = ops.launch_count
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                px = sess.generate_block()
            e1.record()
            barrier()
            if sp and not pp_mode:
                out["exchange"] = transformer.model.sp.exchange
                out["exchange_note"] = transformer.model.sp.fallback_reason
            out["launches"] = ops.launch_count - n0
            out["clocks"] = clocks.stop() if rank == 0 else None
            out["ms"] = max_over_ranks(e0.elapsed_time(e1))
            if decode:
                assert px.shape == (1, 12, 3, 480, 832) and px.dtype == torch.float32
            if keep_outputs and decode and rank == 0:
                out["outputs"] = {"frames": px.float().cpu(), "latents": sess.last_pred.float().cpu()}
            if profile_step:
                barrier()
                ops.profile_begin()
                p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                p0.record()
                sess.generate_block()
                p1.record()
                barrier()
                out["prof"], out["ms_prof"] = ops.profile_end(), p0.elapsed_time(p1)
        return out

    def measure_e2e(sp: bool, steps: int, seed: int, rgb8: bool = False, jpeg: bool = False):
        """Same loop through the same public API with HOST buffers: the block's noise from pinned host memory every
        step and the decoded frames back to pinned host memory inside the timed region."""
        decode = (not sp) or rank == 0
        sess = GenerationSession(GenerateParams(num_blocks=W + steps, seed=seed + (0 if sp else rank)), models,
                                 prompt_embeds=pe, device=dev, decode=decode)
        nf = 3
        host_noise = sess.noise.cpu().pin_memory()
        jpeg_bytes = 0
        if jpeg:
            jcap = 480 * 832 * 3
            host_out = torch.empty(12, jcap, dtype=torch.uint8).pin_memory()
            host_sizes = torch.empty(12, dtype=torch.int32).pin_memory()
            dev_jpg = torch.empty(12, jcap, dtype=torch.uint8, device=dev)
            dev_sizes = torch.empty(12, dtype=torch.int32, device=dev)
        elif rgb8:
            host_out = torch.empty(1, 12, 480, 832, 3, dtype=torch.uint8).pin_memory()
            dev_rgb = torch.empty(1, 12, 480, 832, 3, dtype=torch.uint8, device=dev)
        else:
            host_out = torch.empty(1, 12, 3, 480, 832, dtype=torch.float32).pin_memory()
        with torch.inference_mode():
            for _ in range(W):
                sess.generate_block()
            barrier()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            for _ in range(steps):
                s0 = sess.current_start_frame
                sess.noise[:, s0:s0 + nf].copy_(host_noise[:, s0:s0 + nf], non_blocking=True)      # H2D
                px = sess.generate_block()
                if decode:
                    if jpeg:
                        # the reference's per-frame JPEG (release_server.py:973) encoded on the device: first the 12
                        # file sizes, then only the used bytes of every file cross PCIe
                        ops.frames_to_jpeg(px, 90, cap=jcap, out=dev_jpg, sizes=dev_sizes)
                        host_sizes.copy_(dev_sizes, non_blocking=True)
                        torch.cuda.current_stream().synchronize()
                        for f, nb in enumerate(host_sizes.tolist()):
                            assert nb > 0, "JPEG file did not fit its buffer"
                            host_out[f, :nb].copy_(dev_jpg[f, :nb], non_blocking=True)
                            jpeg_bytes += nb
                    elif rgb8:
                        ops.frames_to_rgb8(px, out=dev_rgb)
                        host_out.copy_(dev_rgb, non_blocking=True)
                    else:
                        host_out.copy_(px, non_blocking=True)                                   # D2H
                torch.cuda.current_stream().synchronize()                                       # frames usable on host
            t1.record()
            barrier()
            host_ref_ms = None
            if jpeg and decode:
                host_ref_ms = _reference_host_egress_ms(px)
        return {"ms": max_over_ranks(t0.elapsed_time(t1)), "host_ref_ms": host_ref_ms,
                "h2d": host_noise[:, :nf].numel() * host_noise.element_size(),
                "d2h": (jpeg_bytes // max(1, steps) + 48) if jpeg else host_out.numel() * host_out.element_size()}

    streams = 1 if sp_mode else world           # independent video streams in flight
    main_run = measure(sp_mode, K, 42, profile_step=True, keep_outputs=args.dump_outputs is not None)
    if "outputs" in main_run:
        dump_outputs(args.dump_outputs, main_run.pop("outputs"))
    e2e_run = measure_e2e(sp_mode, K, 1042)

    # same end-to-end loop with the byte egress kernel (SURVEY.md 8f.2): kr_frames_to_rgb8 does the reference's
    # host-side normalise + to_pil_image conversion on the device, so uint8 [12,H,W,3] (14.4 MB) instead of fp32
    # (57.5 MB) crosses PCIe.  Reported next to `e2e`, which keeps the reference's own fp32 download.
    egress = None
    if not sp_mode and not args.no_egress:
        r = measure_e2e(False, K, 2042, rgb8=True)
        egress = {"value": streams * K * FRAMES_PER_STEP / (r["ms"] / 1e3), "unit": "frames/s",
                  "d2h_bytes_per_step": r["d2h"], "ms_per_step": r["ms"] / K,
                  "what": "e2e loop with kr_frames_to_rgb8 on the device and a uint8 [12,480,832,3] download"}

    # and with the whole egress on the device (SURVEY.md 8f.2, second half): kr_frames_to_jpeg writes the files the
    # reference produces with Pillow in a 24-thread pool (byte-identical, tests/test_zz_jpeg_gpu.py); ~1-3 MB of JPEG
    # bytes per block cross PCIe.  Never allowed to take the headline line down with it.
    egress_jpeg = None
    if world == 1 and not args.no_egress:          # one rank only: a caught failure must not desynchronise barriers
        try:
            r = measure_e2e(False, K, 2542, jpeg=True)
            egress_jpeg = {"value": streams * K * FRAMES_PER_STEP / (r["ms"] / 1e3), "unit": "frames/s",
                           "d2h_bytes_per_step": r["d2h"], "ms_per_step": r["ms"] / K, "quality": 90,
                           "reference_host_egress_ms_per_step": r["host_ref_ms"], "host_threads": 24,
                           "what": "e2e loop with kr_frames_to_jpeg on the device (4 launches per block) and a download "
                                   "of the 12 JPEG files' used bytes; files byte-identical to Pillow quality=90; "
                                   "reference_host_egress_ms_per_step = the reference's own egress of one block (fp32 "
                                   "download + normalise + Pillow in a 24-thread pool) timed on this box's host cores"}
        except Exception as ex:  # noqa: BLE001
            egress_jpeg = {"value": None, "error": f"{type(ex).__name__}: {ex}"[:200]}

    # FP8 tier (SURVEY.md 8f.4; the reference's `enable_fp8: true`): same loop with the DiT block linears on the
    # kind::f8f6f4 GEMM + dynamic per-tensor activation casts.  Reported beside the bf16 headline, never instead of it.
    fp8_line = None
    if world == 1 and not args.no_fp8:
        from realtime_video_b200 import fp8 as fp8mod
        fp8mod.quantize_(transformer)
        try:
            r8 = measure(False, max(2, K // 2), 4042, profile_step=True)
            p8 = r8["prof"].get("gemm_fp8", {"flops": 0.0, "ms": 0.0, "n": 0})
            fp8_line = {"value": max(2, K // 2) * FRAMES_PER_STEP / (r8["ms"] / 1e3), "unit": "frames/s",
                        "ms_per_step": r8["ms"] / max(2, K // 2), "steps": max(2, K // 2),
                        "gemm_fp8_tflops": p8["flops"] / (p8["ms"] * 1e-3) / 1e12 if p8["ms"] > 0 else None,
                        "gemm_fp8_share": p8["ms"] / r8["ms_prof"] if r8["ms_prof"] > 0 else None,
                        "what": "DiT block linears in e4m3 (per-tensor dynamic activation scale, static weight scale = "
                                "torchao Float8DynamicActivationFloat8WeightConfig(PerTensor), release_server.py:179-182); "
                                "attention, norms, VAE unchanged; separate numerics tier (tests/test_fp8_gpu.py)"}
        finally:
            fp8mod.dequantize_(transformer)

    # N > 1: the other way to use the box (N independent replicas, no data-path collective), same run
    secondary = None
    if world > 1 and not args.no_secondary:
        other = measure(not sp_mode, max(2, K // 2), 3042, profile_step=False)
        n_streams = world if sp_mode else 1
        secondary = {"mode": "replicas" if sp_mode else "sp", "scaling": "weak" if sp_mode else "strong",
                     "value": n_streams * max(2, K // 2) * FRAMES_PER_STEP / (other["ms"] / 1e3), "unit": "frames/s",
                     "ms_per_step": other["ms"] / max(2, K // 2), "steps": max(2, K // 2)}

    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    cpu = None
    if not args.no_cpu_baseline:
        try:
            cpu = cpu_reference_sample()
        except Exception as ex:  # noqa: BLE001
            cpu = {"value": None, "unit": "frames/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {ex}"}
    line = assemble_line(args, world, sp_mode, pp_mode, use_graphs, main_run, e2e_run, egress, egress_jpeg, fp8_line,
                         secondary, cpu)
    emit(line)


if __name__ == "__main__":
    main()
