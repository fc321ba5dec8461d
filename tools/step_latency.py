"""Latency of one step call (``DiffusionPlan.p_sample``, conditioner projections reused through the cond tag) beside one step of
``sample()`` (its whole time / K_step, CUDA-graph path), at B=1, T=938 and at B=32, T=1875; at B=32 also with a different step per
batch row (the per-row kernel variants).  CUDA events on the current stream.  Synthetic weights, fp16x2.  The card's name and power
limit (a read-only nvidia-smi query) are printed with the timings: they are part of the numbers."""
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bisinger_b200 import synthetic as synth  # noqa: E402
from bisinger_b200 import B200DiffNet, DiffusionPlan  # noqa: E402
from bisinger_b200.diffusion import _schedule_buffers, linear_beta_schedule  # noqa: E402

K = 100
dev = torch.device("cuda", 0)


def timeit(fn, n):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


net = B200DiffNet(80)
net.load_state_dict(synth.diffnet_state(1234), strict=True)
plan = DiffusionPlan(net, _schedule_buffers(linear_beta_schedule(K, 0.06)), K, K, synth.SPEC_MIN, synth.SPEC_MAX, device=dev)
try:
    power = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip() or "unknown"
except (OSError, subprocess.SubprocessError):
    power = "unknown"
print(f"{torch.cuda.get_device_name(dev)}, power limit {power}; precision {plan.precision}, K_step {K}")
for B, T in ((1, 938), (32, 1875)):
    inp = synth.kernel_inputs(5, B, T, 1)
    cond_btH, fs2 = inp["cond"].to(dev), inp["fs2_mel"].to(dev)
    cond = cond_btH.transpose(1, 2)
    x = inp["start_noise"].to(dev)
    n = 20 if B == 1 else 5
    ms_sample = timeit(lambda: plan.sample(cond_btH, fs2, seed=1), n) / K
    ms_step = timeit(lambda: plan.p_sample(x, torch.full((B,), 50), cond, seed=1), 5 * n)
    line = f"B={B} T={T}: sample() {ms_sample:.3f} ms/step | p_sample uniform t {ms_step:.3f} ms"
    if B > 1:
        mixed = torch.arange(B) * (K - 1) // (B - 1)
        line += f" | p_sample mixed t {timeit(lambda: plan.p_sample(x, mixed, cond, seed=1), 5 * n):.3f} ms"
    print(line, flush=True)
