#!/usr/bin/env python
"""Benchmark of the BiSinger synthesis hot path on B200 (contract: see the task brief / DESIGN.md §7).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision bf16x3|bf16] [--dump-outputs DIR]

Metric (BASELINE.json): seconds of audio synthesised per wall-second, diffusion mel (K=100 DiffNet sampler) + HiFi-GAN/NSF
vocoder.  Workload at every N: cfg3 = one batch of 32 x 10 s phrases (T = 1875 mel frames, 24 kHz, hop 128) per rank per
step, random-init models of the named architecture and synthetic conditioner outputs (cond / fs2_mel / f0); the FastSpeech2
conditioner is outside the hot path (SURVEY.md §8) and is not run.  Ranks are independent replicas (weak scaling, no
collective on the data path); time = max over ranks of the CUDA-event time of the K timed steps.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SR, HOP, MEL, HID = 24000, 128, 80, 256
K_STEP, MAX_BETA = 100, 0.06
BATCH, FRAMES = 32, 1875                      # cfg3: 32 phrases x 10 s
FLOPS_DIFFNET_FRAME_STEP = 26_427_392         # SURVEY.md §8d (2*MAC, what the reference computes)
FLOPS_GATE_GEMM_FRAME = 2 * (3 * 256) * 512           # dilated conv k=3 256->512 per frame per layer (the step-invariant
#   conditioner 1x1 is hoisted out of the K loop and evaluated once per batch: SURVEY.md §8d allows exactly this)
FLOPS_RES_GEMM_FRAME = 2 * 256 * 256                  # residual half of the 1x1 output projection per frame per layer
FLOPS_COND_ONCE_FRAME = 20 * 2 * 256 * 512            # 5 242 880 per frame, once
FLOPS_DIFFNET_FRAME_STEP_HOISTED = FLOPS_DIFFNET_FRAME_STEP - FLOPS_COND_ONCE_FRAME   # 21 184 512
FLOPS_HIFIGAN_FRAME = 375_734_272
CONTRACTION_NOTE = {
    "fp16x2": " (per-layer GEMMs, one fused kernel per ResidualBlock: fp16 activations x fp16 weights + a weight-rounding correction "
              "term -- e4m3 x e5m2 on the fp8 pipe in the dilated-conv GEMM, a second fp16 MMA in the residual / skip-sum GEMMs -- "
              "fp32 accumulate; once-per-step GEMMs bf16x3; vocoder bf16)",
    "bf16x3": " (3 tensor-core MMAs per product: hi*hi + lo*hi + hi*lo)",
    "bf16": " (single bf16 MMA per product; fails the 100-step mel tolerance on random-init weights)",
}
MMAS_PER_PRODUCT = {"fp16x2": 2, "bf16x3": 3, "bf16": 1}
METRIC = "audio_seconds_per_second"
UNIT = "audio-s/s"


def read_traffic(kernel: str, B: int, T: int):
    """roofline.traffic = dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed summary of an
    `ncu --set full` capture (profiles/traffic.json, written by tools/ncu_summary.py from the .ncu-rep of the named command); null when
    no capture exists for this kernel and shape -- DRAM counters cannot be read live from inside a timed run."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        for e in json.load(open(p)):
            if e["kernel"] == kernel and e["B"] == B and e["T"] == T:
                return float(e["dram_bytes_per_launch"]), e.get("source", "profiles/traffic.json")
    except Exception:
        pass
    return None, None


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tflops=float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1394.9))), hbm=float(d.get("hbm_gbs", 6549.8)),
                    source="MEASURED_PEAKS.json (sustained bf16 cuBLAS)")
    return dict(tflops=1400.0, hbm=6650.0, source="fallback of B200_PROFILING.md (sustained ~1.4 PFLOP/s)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                    if r[col].lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


DUMP_BYTES = 60 << 20


def dump_outputs(d, arrays):
    """Writes each array as d/<name>.npy in float32.  When they hold more than DUMP_BYTES in all, each one is cut to a sample of its
    elements (its share of the budget, flat indices drawn with a fixed seed and sorted), so that runs with the same arguments write
    the same elements and two builds can be compared output for output."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    total = sum(a.size * 4 for a in arrays.values())
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float32)
        if total > DUMP_BYTES:
            idx = np.random.default_rng(0).choice(a.size, a.size * DUMP_BYTES // total, replace=False)
            a = a.reshape(-1)[np.sort(idx)]
        np.save(os.path.join(d, name + ".npy"), a)


def build_models(dev, precision):
    import torch
    from bisinger_b200 import synthetic as synth   # seeded random-init weights of the named architecture (no checkpoints reachable)
    from bisinger_b200 import B200DiffNet, B200GaussianDiffusion
    from bisinger_b200.diffusion import linear_beta_schedule
    from bisinger_b200.vocoder import B200HifiGanGenerator
    net = B200DiffNet(MEL)
    net.load_state_dict(synth.diffnet_state(1234), strict=True)
    gd = B200GaussianDiffusion(None, MEL, net, timesteps=K_STEP, K_step=K_STEP, betas=linear_beta_schedule(K_STEP, MAX_BETA),
                               spec_min=synth.SPEC_MIN, spec_max=synth.SPEC_MAX, precision=precision,
                               hparams=dict(hidden_size=HID, residual_layers=20, residual_channels=256, dilation_cycle_length=4,
                                            keep_bins=MEL, gaussian_start=False))
    gd.to(dev)
    gd.build_plan()
    gen = B200HifiGanGenerator(synth.HIFIGAN_CONFIG)
    gen.load_folded_state_dict(synth.hifigan_state(4321), strict=True)
    gen.to(dev)
    gen.build_plan(dev)
    return gd, gen, synth


def build_pitch_extractor(dev, synth):
    from bisinger_b200.pitch import B200PitchExtractor
    pe = B200PitchExtractor().eval()
    pe.load_state_dict(synth.pe_state(777, 2), strict=True)
    pe.build_plan(dev)
    return pe


def host_inputs(synth, B, T, seed):
    import torch
    k = synth.kernel_inputs(seed, B, T, 1)
    v = synth.vocoder_inputs(seed + 1, B, T)
    return k["cond"].contiguous(), k["fs2_mel"].contiguous(), v["f0"].contiguous()


def run_ours(args):
    import torch
    import torch.distributed as dist
    from bisinger_b200 import launch_count
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU path for the product arm)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    gd, gen, synth = build_models(dev, args.precision)
    B, T = args.batch, args.frames
    audio_s = B * T * HOP / SR
    cond_h, mel_h, f0_h = host_inputs(synth, B, T, 1000 + rank)
    cond_p, mel_p, f0_p = cond_h.pin_memory(), mel_h.pin_memory(), f0_h.pin_memory()
    wav_p = torch.empty((B, T * HOP), dtype=torch.float32).pin_memory()
    cond_d, mel_d, f0_d = cond_p.to(dev), mel_p.to(dev), f0_p.to(dev)
    stream = torch.cuda.current_stream(dev)

    def step_resident(i):
        mel = gd.sample(cond_d, mel_d, seed=i)                          # [B,T,80]
        return mel, gen(mel.transpose(1, 2).contiguous(), f0_d, seed=i)  # [B,1,T*hop]

    def step_e2e(i):
        c = cond_p.to(dev, non_blocking=True); m = mel_p.to(dev, non_blocking=True); f = f0_p.to(dev, non_blocking=True)
        mel = gd.sample(c, m, seed=i)
        wav = gen(mel.transpose(1, 2).contiguous(), f, seed=i)
        wav_p.copy_(wav[:, 0], non_blocking=True)
        return wav

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps, sample_clocks=False):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        cs = ClockSampler(local) if sample_clocks else None
        if cs:
            cs.start()
        n0 = launch_count()
        e0.record(stream)
        for i in range(steps - 1):
            fn(i)
        out = fn(steps - 1)                 # only the last step's result is held, as a caller of the path would hold it
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        clocks = cs.stop() if cs else None
        n1 = launch_count()
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, n1 - n0, clocks, out

    for i in range(args.warmup):
        step_resident(i)
    ms, launches, clocks, last = timed(step_resident, args.steps, sample_clocks=True)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"mel": last[0].cpu().numpy(), "wav": last[1].cpu().numpy()})
    del last
    for i in range(max(1, args.warmup // 2)):
        step_e2e(i)
    ms_e2e, _, _, _ = timed(step_e2e, args.steps)

    value = world * args.steps * audio_s / (ms / 1e3)
    e2e = world * args.steps * audio_s / (ms_e2e / 1e3)

    line = {
        "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp16" if args.precision == "fp16x2" else "bf16", "data": "synthetic",
        "config": {"workload": f"cfg3: full hot path, batch {B} x {T * HOP / SR:.0f} s phrases (T={T}) per GPU per step, K={K_STEP} "
                               f"DiffNet sampler (20x256, CUDA-graph captured) + HiFi-GAN/NSF vocoder (hop 128, 512 ch); random-init "
                               f"weights, synthetic cond/fs2_mel/f0 (FastSpeech2 conditioner not part of the path)",
                   "global_batch": B * world, "frames": T, "k_step": K_STEP, "parallelism": f"replicas x{world}",
                   "contraction": args.precision + CONTRACTION_NOTE[args.precision],
                   "l2": "per-step working set ~6 GB >> 126 MB L2, no flush needed"},
        "e2e": {"value": round(e2e, 2), "unit": UNIT, "h2d_bytes_per_step": int(cond_p.numel() + mel_p.numel() + f0_p.numel()) * 4,
                "d2h_bytes_per_step": int(wav_p.numel()) * 4},
        "gpu_launches": int(launches), "clocks": clocks,
    }
    if rank == 0:
        peaks = read_peaks()
        reps = 200
        fused = args.precision == "fp16x2"
        try:
            # 4 = all 20 ResidualBlocks in one launch (what a step runs): time per layer, launch = 20 layers
            k_ms = gd.plan.time_kernel(4, B, T, reps) if fused else None
        except RuntimeError:
            fused, k_ms = False, None
        if fused:
            # dominant kernel: one fused ResidualBlock (dilated-conv gate GEMM of both channel halves + residual GEMM + both epilogues)
            layer_flops = (FLOPS_GATE_GEMM_FRAME + FLOPS_RES_GEMM_FRAME) * B * T
            achieved = layer_flops / (k_ms * 1e-3) / 1e12
            n_layers = 20
            line["roofline"] = {
                "bound": "tensor", "kernel": "diffnet_layer_kernel (the 20 fused ResidualBlocks of a step in one launch; per block and 256-row tile: "
                                             "dilated-conv GEMM k=3 256->512 with fp16 + fp8-correction MMAs, gate epilogue, residual GEMM 256->256, "
                                             "residual epilogue)",
                "achieved": round(achieved, 1), "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": round(achieved / peaks["tflops"], 4),
                "traffic": read_traffic("diffnet_layer_kernel", B, T)[0], "traffic_source": read_traffic("diffnet_layer_kernel", B, T)[1],
                "avg_launch_ms": round(k_ms * n_layers, 4), "algorithmic_flops_per_launch": layer_flops * n_layers,
                "ms_per_layer": round(k_ms, 4),
                "issued_mma_flops_per_algorithmic_flop": 2,
                "issued_note": "per product one fp16 MMA + one correction MMA; the gate GEMM's correction runs at the fp8 rate (2x) => 1.5 fp16-MMA "
                               "equivalents there; the kernel is bound by operand bytes into the SM (~1.3 MB per 256-row tile and CTA), see DESIGN.md",
                "peak_source": peaks["source"] + ", of measured",
                "share_of_step": round(n_layers * K_STEP * k_ms / (ms / args.steps), 3),
            }
            r_ms = 0.0
        else:
            k_ms = gd.plan.time_kernel(0, B, T, reps)
            gate_flops = FLOPS_GATE_GEMM_FRAME * B * T
            achieved = gate_flops / (k_ms * 1e-3) / 1e12
            line["roofline"] = {
                "bound": "tensor", "kernel": "conv_gemm_kernel<256,%d,EPI_GATE,pair> (dilated-conv GEMM k=3 256->512, conditioner add + sigmoid*tanh gate epilogue)" % MMAS_PER_PRODUCT[args.precision],
                "achieved": round(achieved, 1), "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": round(achieved / peaks["tflops"], 4),
                "traffic": None, "avg_launch_ms": round(k_ms, 4), "algorithmic_flops_per_launch": gate_flops,
                "issued_mma_flops_per_algorithmic_flop": MMAS_PER_PRODUCT[args.precision],
                "peak_source": peaks["source"] + ", of measured",
                "share_of_step": round(20 * K_STEP * k_ms / (ms / args.steps), 3),
            }
            r_ms = gd.plan.time_kernel(1, B, T, reps)
        s_ms = gd.plan.time_kernel(2, B, T, 50)
        # sampler / vocoder split of a step inside a sustained loop (power-capped clocks as in the timed region): 3 back-to-back steps
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(7)]
        ev[0].record(stream)
        for j in range(3):
            mel_t = gd.sample(cond_d, mel_d, seed=99 + j); ev[2 * j + 1].record(stream)
            gen(mel_t.transpose(1, 2).contiguous(), f0_d, seed=99 + j); ev[2 * j + 2].record(stream)
        torch.cuda.synchronize(dev)
        samp_ms = sum(ev[2 * j].elapsed_time(ev[2 * j + 1]) for j in range(3)) / 3
        voc_ms = sum(ev[2 * j + 1].elapsed_time(ev[2 * j + 2]) for j in range(3)) / 3
        line["breakdown_ms"] = {"sampler": round(samp_ms, 2), "vocoder": round(voc_ms, 2),
                                # sum of the sampler's hot kernels timed in isolation (burst clocks): K x (L fused layers + skip-sum GEMM);
                                # the rest of a step is the input projection, the output projection / posterior and clock droop
                                "sampler_kernel_sum": round(K_STEP * (20 * (k_ms + r_ms) + s_ms), 2),
                                ("fused_layer_launch" if fused else "gate_gemm_launch"): round(k_ms, 4), "resskip_gemm_launch": round(r_ms, 4),
                                "skipsum_gemm_launch": round(s_ms, 4),
                                "layer_gemms_share_of_sampler": round(20 * K_STEP * (k_ms + r_ms) / samp_ms, 3)}
        # the stage the reference runs between the two when hparams['pe_enable'] (mel -> f0, SURVEY.md section 8f-2); reported beside the
        # step, not part of it: the metric's workload feeds the vocoder a synthetic f0
        pe = build_pitch_extractor(dev, synth)
        for _ in range(2):
            pe(mel_t)
        e3, e4 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e3.record(stream); pe(mel_t); e4.record(stream)
        torch.cuda.synchronize(dev)
        line["breakdown_ms"]["pitch_extractor_not_in_step"] = round(e3.elapsed_time(e4), 3)
        # the conditioner's mel-rate handoff (FastSpeech FFT decoder + mel_out, SURVEY.md section 8f-3): once per batch, before the sampler;
        # reported beside the step like the PitchExtractor (the metric's workload feeds the sampler a synthetic fs2_mel / cond)
        try:
            from bisinger_b200.fft import B200FastspeechDecoder
            fsd = synth.fft_state(555)
            dec = B200FastspeechDecoder(hparams=dict(hidden_size=HID, dec_layers=4, num_heads=2, dec_ffn_kernel_size=9)).eval()
            dec.load_state_dict({k: v for k, v in fsd.items() if not k.startswith("mel_out.")}, strict=True)
            mo = torch.nn.Linear(HID, MEL)
            mo.load_state_dict({"weight": fsd["mel_out.weight"], "bias": fsd["mel_out.bias"]})
            dec, mo = dec.to(dev), mo.to(dev)
            tgt = torch.ones((B, T), device=dev)
            for _ in range(2):
                dec.run_decoder(cond_d, tgt, mo)
            e5, e6 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e5.record(stream); dec.run_decoder(cond_d, tgt, mo); e6.record(stream)
            torch.cuda.synchronize(dev)
            line["breakdown_ms"]["fft_decoder_handoff_not_in_step"] = round(e5.elapsed_time(e6), 3)
            del dec, mo
        except Exception as e:
            line["breakdown_ms"]["fft_decoder_handoff_not_in_step"] = "unavailable: " + repr(e)[:120]
        line["pipeline_algorithmic_tflops"] = round((FLOPS_DIFFNET_FRAME_STEP_HOISTED * K_STEP + FLOPS_COND_ONCE_FRAME + FLOPS_HIFIGAN_FRAME) * B * T * world * args.steps / (ms * 1e-3) / 1e12, 1)
        if world == 1:
            line["plms_shipped_config"] = plms_shipped(dev, synth, cond_d, args.precision, B, T)
        if world == 1 and not args.no_eager_baseline:
            line["gpu_eager_baseline"] = gpu_eager_reference(dev, B, T)
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_reference(steps=3, warmup=1)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_cfg5(args):
    """BASELINE.json cfg5: a batch-sharded throughput sweep of 4096 synthetic phrases (128 batches of 32 x 10 s) over the ranks --
    STRONG scaling: the job is fixed, batches go round-robin to the replicas (bisinger_b200.shard.shard_batches), no collective on the
    data path; every batch goes host -> device -> sampler -> vocoder -> host like a real job (pinned buffers, H2D / D2H inside the
    timed region).  value = 40 960 audio-seconds / max-over-ranks time.  Run with  --workload cfg5 [--phrases N]."""
    import torch
    import torch.distributed as dist
    from bisinger_b200 import launch_count
    from bisinger_b200.shard import shard_batches
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU path for the product arm)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    gd, gen, synth = build_models(dev, args.precision)
    B, T = args.batch, args.frames
    mine = shard_batches(args.phrases, B, rank, world)
    # four distinct pinned host batches, cycled (generating 128 x 80 MB of synthetic conditioner output on the host would time the host)
    pool = []
    for j in range(4):
        c, m, f = host_inputs(synth, B, T, 5000 + 17 * rank + j)
        pool.append((c.pin_memory(), m.pin_memory(), f.pin_memory()))
    wav_p = torch.empty((B, T * HOP), dtype=torch.float32).pin_memory()
    stream = torch.cuda.current_stream(dev)

    def one(i, n_rows):
        c, m, f = pool[i % 4]
        cd, md, fd = c[:n_rows].to(dev, non_blocking=True), m[:n_rows].to(dev, non_blocking=True), f[:n_rows].to(dev, non_blocking=True)
        mel = gd.sample(cd, md, seed=i)
        wav = gen(mel.transpose(1, 2).contiguous(), fd, seed=i)
        wav_p[:n_rows].copy_(wav[:, 0], non_blocking=True)

    for i in range(max(3, args.warmup)):
        one(i, B)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    cs = ClockSampler(local)
    cs.start()
    n0 = launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i, (lo, hi) in enumerate(mine):
        one(i, hi - lo)
    e1.record(stream)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1)
    clocks = cs.stop()
    launches = launch_count() - n0
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    audio = args.phrases * T * HOP / SR
    if rank == 0:
        v = audio / (ms / 1e3)
        print(json.dumps({
            "metric": METRIC, "value": round(v, 2), "unit": UNIT, "n_gpus": world, "steps": len(mine), "warmup": max(3, args.warmup),
            "ms_per_step": round(ms / max(1, len(mine)), 3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "fp16" if args.precision == "fp16x2" else "bf16", "data": "synthetic",
            "config": {"workload": f"cfg5: {args.phrases} phrases x {T * HOP / SR:.0f} s in batches of {B}, round-robin over {world} replica(s) "
                                   f"(rank 0 ran {len(mine)} batches), K={K_STEP} sampler + HiFi-GAN/NSF vocoder per batch, host buffers in / out",
                       "global_batch": B, "frames": T, "k_step": K_STEP, "parallelism": f"replicas x{world}, batches round-robin",
                       "l2": "per-batch working set ~6 GB >> 126 MB L2, no flush needed"},
            "e2e": {"value": round(v, 2), "unit": UNIT, "h2d_bytes_per_step": int(sum(t.numel() for t in pool[0])) * 4,
                    "d2h_bytes_per_step": int(wav_p.numel()) * 4},
            "job_seconds": round(ms / 1e3, 3), "gpu_launches": int(launches), "clocks": clocks}), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def plms_shipped(dev, synth, cond_d, precision, B: int, T: int):
    """Beside the K = 100 line: the sampler as BiSinger ships it (usr/configs/lang-esm-style-ori-shift/diff.yaml:16-23: timesteps =
    K_step = 1000, max_beta 0.02, pndm_speedup 5, gaussian_start => 200 PLMS iterations, 201 denoiser evaluations), same batch, CUDA
    graph replay; sampler only (the vocoder is the same as in the step above)."""
    import torch
    from bisinger_b200 import B200DiffNet, B200GaussianDiffusion
    from bisinger_b200.diffusion import linear_beta_schedule
    try:
        net = B200DiffNet(MEL)
        net.load_state_dict(synth.diffnet_state(1234), strict=True)
        gd = B200GaussianDiffusion(None, MEL, net, timesteps=1000, K_step=1000, betas=linear_beta_schedule(1000, 0.02),
                                   spec_min=synth.SPEC_MIN, spec_max=synth.SPEC_MAX, precision=precision,
                                   hparams=dict(hidden_size=HID, residual_layers=20, residual_channels=256, dilation_cycle_length=4,
                                                keep_bins=MEL, gaussian_start=True, pndm_speedup=5)).to(dev)
        gd.sample(cond_d, None, seed=1)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(2):
            gd.sample(cond_d, None, seed=2 + i)
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / 2
        del gd
        torch.cuda.empty_cache()
        return {"sampler_ms_per_batch": round(ms, 1), "denoiser_evaluations": 201, "sampler_audio_s_per_s": round(B * T * HOP / SR / (ms / 1e3), 1),
                "unit": UNIT, "note": "timesteps = K_step = 1000, max_beta 0.02, pndm_speedup 5, gaussian_start; sampler only, graph replay"}
    except Exception as e:
        return {"unavailable": repr(e)[:200]}


def gpu_eager_reference(dev, B: int, T: int):
    """The honest incumbent (SURVEY.md section 8d, BASELINE.md section 4.4): the reference ALGORITHM as eager PyTorch on the same GPU --
    the oracle restatement (pinned to the executed reference) with every tensor on the device, on the same cfg3 batch -- in torch's
    default fp32 (cuDNN convolutions may use TF32) and under bf16 autocast.  A reported leg like cpu_baseline: measured after the
    product's timed region, one warm-up + one timed batch each; nothing of it is on the product path."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import torch

    import svs_oracle as O
    import synth
    to = lambda d: {k: v.to(dev) for k, v in d.items()}
    sd, vsd = to(synth.diffnet_state(1234)), to(synth.hifigan_state(4321))
    sched = to(O.schedule_buffers(O.linear_beta_schedule(K_STEP, MAX_BETA)))
    smin, smax = torch.tensor(synth.SPEC_MIN, device=dev), torch.tensor(synth.SPEC_MAX, device=dev)
    inp = to(synth.kernel_inputs(1000, B, T, 1))
    vin = to(synth.vocoder_inputs(1001, B, T))
    step_noise = torch.randn((K_STEP, B, 1, MEL, T), device=dev)
    audio = B * T * HOP / SR

    def one():
        with torch.no_grad():
            mel = O.diffusion_infer(sd, sched, smin, smax, inp["cond"], K_STEP, step_noise, inp["fs2_mel"], inp["start_noise"])
            return O.hifigan_forward(vsd, synth.HIFIGAN_CONFIG, mel.transpose(1, 2), vin["f0"], vin["rand_ini"], vin["src_noise"])

    def timed():
        one()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); one(); e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1)

    out = {"unit": UNIT, "kind": "oracle modules as eager PyTorch on the same GPU (torch %s)" % torch.__version__,
           "sample": f"1 warm-up + 1 timed batch of cfg3 ({B} x T={T}, K={K_STEP} sampler + vocoder) per mode"}
    try:
        ms32 = timed()
        with torch.autocast("cuda", dtype=torch.bfloat16):
            ms16 = timed()
        out.update({"fp32_default": round(audio / (ms32 / 1e3), 1), "bf16_autocast": round(audio / (ms16 / 1e3), 1),
                    "ms_per_step_fp32": round(ms32, 1), "ms_per_step_bf16": round(ms16, 1)})
    except Exception as e:   # e.g. out of memory next to the product's workspaces: report, do not fail the bench
        out["unavailable"] = repr(e)[:200]
    del sd, vsd, inp, vin, step_noise
    torch.cuda.empty_cache()
    return out


def cpu_reference(steps: int, warmup: int, phrases: int = 1):
    """The reference algorithm on the host cores: the oracle port (oracle/svs_oracle.py, a restatement pinned against the
    executed reference) -- the reference tree itself does not travel to the GPU box.  Bounded sample of the cfg3 workload: ONE
    of the 32 phrases (B=1, T=1875, K=100 sampler + vocoder), all host threads."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import torch

    import svs_oracle as O
    import synth
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    B, T = phrases, FRAMES
    sd, vsd = synth.diffnet_state(1234), synth.hifigan_state(4321)
    sched = O.schedule_buffers(O.linear_beta_schedule(K_STEP, MAX_BETA))
    smin, smax = torch.tensor(synth.SPEC_MIN), torch.tensor(synth.SPEC_MAX)
    inp = synth.kernel_inputs(1000, B, T, K_STEP)
    vin = synth.vocoder_inputs(1001, B, T)

    def one():
        with torch.no_grad():
            mel = O.diffusion_infer(sd, sched, smin, smax, inp["cond"], K_STEP, inp["step_noise"], inp["fs2_mel"], inp["start_noise"])
            return O.hifigan_forward(vsd, synth.HIFIGAN_CONFIG, mel.transpose(1, 2), vin["f0"], vin["rand_ini"], vin["src_noise"])

    for _ in range(warmup):
        one()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    dt = time.perf_counter() - t0
    audio = steps * B * T * HOP / SR
    return {"value": round(audio / dt, 4), "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{steps} x ({B} of the 32 phrases of 10 s, T={T}, K={K_STEP} sampler + vocoder), fp32 torch CPU, {cores} threads",
            "seconds": round(dt, 2)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    base = cpu_reference(steps=args.steps, warmup=min(args.warmup, 1), phrases=2)
    ms = base["seconds"] * 1e3
    line = {
        "impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": int(os.environ.get("WORLD_SIZE", "1")),
        "steps": args.steps, "warmup": min(args.warmup, 1), "ms_per_step": round(ms / args.steps, 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "cfg3 hot path (K=100 DiffNet sampler + HiFi-GAN/NSF vocoder) -- reference algorithm on the host CPU; each "
                               "step is a bounded sample: 2 of the 32 phrases (10 s each, T=1875)", "parallelism": "host threads"},
        "cpu_baseline": base,
        "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default 5); cfg5 times its share of the --phrases batches instead and rejects --steps")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="fp16x2", choices=["fp16x2", "bf16x3", "bf16"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--frames", type=int, default=FRAMES)
    ap.add_argument("--workload", default="cfg3", choices=["cfg3", "cfg5"],
                    help="cfg3 (default): one 32 x 10 s batch per rank and step, weak scaling; cfg5: 4096 phrases sharded over the ranks, strong scaling")
    ap.add_argument("--phrases", type=int, default=4096)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the mel [B,T,80] and waveform [B,1,T*hop] of the last timed step (cfg3, rank 0) as DIR/mel.npy and "
                         "DIR/wav.npy, float32; past 60 MiB in all a fixed seeded sample of each")
    args = ap.parse_args()
    if args.workload == "cfg5" and args.steps is not None:
        ap.error("--steps does not apply to --workload cfg5: it times every batch of --phrases")
    args.steps = 5 if args.steps is None else args.steps
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "cfg3"):
        ap.error("--dump-outputs needs --impl ours and --workload cfg3")
    if args.impl == "reference":
        run_reference(args)
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world == 1:
        # convenience: re-launch under torchrun as the driver would
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    if args.workload == "cfg5":
        run_cfg5(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
