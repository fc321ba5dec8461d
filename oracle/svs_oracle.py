"""CPU oracle for the BiSinger synthesis hot path (TEST INFRASTRUCTURE ONLY).

This file is a plain-PyTorch fp32 *restatement* of the reference algorithm for the
path named in BASELINE.json (shallow-diffusion reverse loop over DiffNet + HiFi-GAN/NSF
generator forward).  It is the checker for the CUDA path: only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline / ``--impl reference`` legs
may import it.  The product package ``bisinger_b200`` never imports anything from
``oracle/`` and has no CPU fallback.

Pinning: the reference ships no tests or golden vectors for this path (SURVEY.md §4), so
"parity unpinned" by reference-owned tests.  Instead the restatement is pinned against
the *executed reference modules* (``oracle/ref_shim.py`` imports them unmodified from
/root/reference in the build container): ``oracle/make_golden.py`` writes
``tests/golden/*.npz`` from the real reference and ``tests/test_oracle.py`` checks this
file against those fixtures (and, when /root/reference is present, against the live
reference modules).

Every function cites the reference file:line it follows; paths are relative to
/root/reference/train_bisinger/.

Optional ``operand`` argument: None = exact fp32 (the oracle proper).  "bf16"/"fp16"
rounds the *operands* of every contraction to that type and accumulates in fp32 -- a model
of what a tensor-core path computes, used by tests to tell precision effects from bugs.
"fp16x2" models the sampler's default mode: fp16 activations x fp16 hi/lo-split weights.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch
import torch.nn.functional as F

Tensor = torch.Tensor
LRELU_SLOPE = 0.1  # modules/hifigan/hifigan.py:11


def _rnd(x: Tensor, operand: Optional[str]) -> Tensor:
    """Activation operand of a contraction as the emulated tensor-core path sees it."""
    if operand is None:
        return x
    dt = {"bf16": torch.bfloat16, "fp16": torch.float16, "fp16x2": torch.float16}[operand]
    return x.to(dt).to(torch.float32)


def _rnd_side(x: Tensor, operand: Optional[str]) -> Tensor:
    """Activation operand of the once-per-step / once-per-batch GEMMs (conditioner projection, input projection,
    skip_projection, output_projection): the "fp16x2" mode runs those as bf16x3 (~16 bits, modelled as hi + lo)."""
    if operand == "fp16x2":
        hi = x.to(torch.bfloat16).to(torch.float32)
        return hi + (x - hi).to(torch.bfloat16).to(torch.float32)
    return _rnd(x, operand)


def _rnd_w(w: Tensor, operand: Optional[str]) -> Tensor:
    """Weight operand: "fp16x2" carries weights as an fp16 hi/lo pair (~21 bits), modelled as hi + lo."""
    if operand == "fp16x2":
        hi = w.to(torch.float16).to(torch.float32)
        return hi + (w - hi).to(torch.float16).to(torch.float32)
    return _rnd(w, operand)


# --------------------------------------------------------------------------------------
# DiffNet (usr/diff/net.py)
# --------------------------------------------------------------------------------------

def sinusoidal_pos_emb(t: Tensor, dim: int) -> Tensor:
    """usr/diff/net.py:32-44 -- emb = [sin(t*w_j), cos(t*w_j)], w_j = exp(-j ln(1e4)/(dim/2-1))."""
    half = dim // 2
    w = torch.exp(torch.arange(half, dtype=torch.float32) * -(math.log(10000) / (half - 1))).to(t.device)
    e = t.to(torch.float32)[:, None] * w[None, :]
    return torch.cat((e.sin(), e.cos()), dim=-1)


def mish(x: Tensor) -> Tensor:
    """usr/diff/diffusion.py:68-70."""
    return x * torch.tanh(F.softplus(x))


def step_embedding(p: Dict[str, Tensor], t: Tensor, C: int) -> Tensor:
    """usr/diff/net.py:119-120 -- SinusoidalPosEmb -> Linear -> Mish -> Linear.  [B] -> [B, C]."""
    e = sinusoidal_pos_emb(t, C)
    e = F.linear(e, p["mlp.0.weight"], p["mlp.0.bias"])
    e = mish(e)
    return F.linear(e, p["mlp.2.weight"], p["mlp.2.bias"])


def n_residual_layers(p: Dict[str, Tensor]) -> int:
    n = 0
    while f"residual_layers.{n}.dilated_conv.weight" in p:
        n += 1
    return n


def residual_block(p: Dict[str, Tensor], i: int, dilation: int, x: Tensor, cond: Tensor,
                   step: Tensor, operand: Optional[str] = None):
    """usr/diff/net.py:66-78.  x [B,C,T], cond [B,H,T], step [B,C] -> (x', skip)."""
    pre = f"residual_layers.{i}."
    d = F.linear(step, p[pre + "diffusion_projection.weight"], p[pre + "diffusion_projection.bias"])
    c = F.conv1d(_rnd_side(cond, operand), _rnd_w(p[pre + "conditioner_projection.weight"], operand),
                 p[pre + "conditioner_projection.bias"])
    y = x + d[:, :, None]
    y = F.conv1d(_rnd(y, operand), _rnd_w(p[pre + "dilated_conv.weight"], operand),
                 p[pre + "dilated_conv.bias"], padding=dilation, dilation=dilation) + c
    gate, filt = torch.chunk(y, 2, dim=1)
    y = torch.sigmoid(gate) * torch.tanh(filt)
    y = F.conv1d(_rnd(y, operand), _rnd_w(p[pre + "output_projection.weight"], operand),
                 p[pre + "output_projection.bias"])
    residual, skip = torch.chunk(y, 2, dim=1)
    return (x + residual) / math.sqrt(2.0), skip


def diffnet_forward(p: Dict[str, Tensor], spec: Tensor, t: Tensor, cond: Tensor,
                    dilation_cycle: int = 4, operand: Optional[str] = None) -> Tensor:
    """usr/diff/net.py:107-130.  spec [B,1,M,T], t [B] int, cond [B,H,T] -> [B,1,M,T]."""
    C = p["input_projection.weight"].shape[0]
    L = n_residual_layers(p)
    x = spec[:, 0]
    x = F.conv1d(_rnd_side(x, operand), _rnd_w(p["input_projection.weight"], operand), p["input_projection.bias"])
    x = F.relu(x)
    step = step_embedding(p, t, C)
    skip_sum = None
    for i in range(L):
        x, s = residual_block(p, i, 2 ** (i % dilation_cycle), x, cond, step, operand)
        skip_sum = s if skip_sum is None else skip_sum + s
    x = skip_sum / math.sqrt(L)
    x = F.conv1d(_rnd_side(x, operand), _rnd_w(p["skip_projection.weight"], operand), p["skip_projection.bias"])
    x = F.relu(x)
    x = F.conv1d(_rnd_side(x, operand), _rnd_w(p["output_projection.weight"], operand), p["output_projection.bias"])
    return x[:, None]


# --------------------------------------------------------------------------------------
# Gaussian diffusion schedule + ancestral sampler (usr/diff/shallow_diffusion_tts.py)
# --------------------------------------------------------------------------------------

def linear_beta_schedule(timesteps: int, max_beta: float) -> np.ndarray:
    """usr/diff/shallow_diffusion_tts.py:44-49 (float64 numpy)."""
    return np.linspace(1e-4, max_beta, timesteps)


def cosine_beta_schedule(timesteps: int, s: float = 0.008) -> np.ndarray:
    """usr/diff/shallow_diffusion_tts.py:52-62."""
    steps = timesteps + 1
    x = np.linspace(0, steps, steps)
    ac = np.cos(((x / steps) + s) / (1 + s) * np.pi * 0.5) ** 2
    ac = ac / ac[0]
    betas = 1 - (ac[1:] / ac[:-1])
    return np.clip(betas, a_min=0, a_max=0.999)


def schedule_buffers(betas: np.ndarray) -> Dict[str, Tensor]:
    """usr/diff/shallow_diffusion_tts.py:89-123 -- float64 math, buffers cast to fp32."""
    betas = np.asarray(betas, dtype=np.float64)
    alphas = 1. - betas
    ac = np.cumprod(alphas, axis=0)
    ac_prev = np.append(1., ac[:-1])
    pv = betas * (1. - ac_prev) / (1. - ac)
    f32 = lambda a: torch.tensor(a, dtype=torch.float32)
    return {
        "betas": f32(betas),
        "alphas_cumprod": f32(ac),
        "alphas_cumprod_prev": f32(ac_prev),
        "sqrt_alphas_cumprod": f32(np.sqrt(ac)),
        "sqrt_one_minus_alphas_cumprod": f32(np.sqrt(1. - ac)),
        "log_one_minus_alphas_cumprod": f32(np.log(1. - ac)),
        "sqrt_recip_alphas_cumprod": f32(np.sqrt(1. / ac)),
        "sqrt_recipm1_alphas_cumprod": f32(np.sqrt(1. / ac - 1)),
        "posterior_variance": f32(pv),
        "posterior_log_variance_clipped": f32(np.log(np.maximum(pv, 1e-20))),
        "posterior_mean_coef1": f32(betas * np.sqrt(ac_prev) / (1. - ac)),
        "posterior_mean_coef2": f32((1. - ac_prev) * np.sqrt(alphas) / (1. - ac)),
    }


def norm_spec(x: Tensor, spec_min: Tensor, spec_max: Tensor) -> Tensor:
    """usr/diff/shallow_diffusion_tts.py:275-276."""
    return (x - spec_min) / (spec_max - spec_min) * 2 - 1


def denorm_spec(x: Tensor, spec_min: Tensor, spec_max: Tensor) -> Tensor:
    """usr/diff/shallow_diffusion_tts.py:278-279."""
    return (x + 1) / 2 * (spec_max - spec_min) + spec_min


def q_sample(sched: Dict[str, Tensor], x_start: Tensor, t: int, noise: Tensor) -> Tensor:
    """usr/diff/shallow_diffusion_tts.py:203-208 (t broadcast over batch as at :252)."""
    return sched["sqrt_alphas_cumprod"][t] * x_start + sched["sqrt_one_minus_alphas_cumprod"][t] * noise


def p_sample(p: Dict[str, Tensor], sched: Dict[str, Tensor], x: Tensor, t: int, cond: Tensor,
             noise: Tensor, dilation_cycle: int = 4, operand: Optional[str] = None,
             clip_denoised: bool = True) -> Tensor:
    """usr/diff/shallow_diffusion_tts.py:149-166 (+ :134-147).  One ancestral step with
    injected noise z (the reference draws randn(x.shape) every step, also at t == 0)."""
    B = x.shape[0]
    tt = torch.full((B,), t, dtype=torch.long, device=x.device)
    eps = diffnet_forward(p, x, tt, cond, dilation_cycle, operand)
    x_recon = sched["sqrt_recip_alphas_cumprod"][t] * x - sched["sqrt_recipm1_alphas_cumprod"][t] * eps
    if clip_denoised:
        x_recon = x_recon.clamp(-1., 1.)
    mean = sched["posterior_mean_coef1"][t] * x_recon + sched["posterior_mean_coef2"][t] * x
    nonzero = 0.0 if t == 0 else 1.0
    return mean + nonzero * (0.5 * sched["posterior_log_variance_clipped"][t]).exp() * noise


def diffusion_infer(p: Dict[str, Tensor], sched: Dict[str, Tensor], spec_min: Tensor, spec_max: Tensor,
                    cond_btH: Tensor, K_step: int, step_noise: Tensor,
                    fs2_mel: Optional[Tensor] = None, start_noise: Optional[Tensor] = None,
                    mel2ph: Optional[Tensor] = None, gaussian_start: bool = False,
                    dilation_cycle: int = 4, operand: Optional[str] = None,
                    return_trace: bool = False):
    """Infer branch of GaussianDiffusion.forward, usr/diff/shallow_diffusion_tts.py:235,245-272.

    cond_btH   [B,T,H]   = ret['decoder_inp'] (transposed to [B,H,T] at :235)
    fs2_mel    [B,T,M]   = ret['mel_out'] of the FastSpeech2 decoder (shallow start, :246-252)
    start_noise[B,1,M,T] = the randn_like of q_sample (:204) or the randn of gaussian_start (:256)
    step_noise [K,B,1,M,T], index k is the k-th *executed* step, i.e. t = K_step-1-k (:266-267)
    returns mel_out [B,T,M] (de-normalised, masked by mel2ph>0 as at :269-272)
    """
    cond = cond_btH.transpose(1, 2)
    if gaussian_start:
        x = start_noise
    else:
        xs = norm_spec(fs2_mel, spec_min, spec_max).transpose(1, 2)[:, None]
        x = q_sample(sched, xs, K_step - 1, start_noise)
    trace = []
    for k, t in enumerate(reversed(range(K_step))):
        x = p_sample(p, sched, x, t, cond, step_noise[k], dilation_cycle, operand)
        if return_trace:
            trace.append(x.clone())
    out = denorm_spec(x[:, 0].transpose(1, 2), spec_min, spec_max)
    if mel2ph is not None:
        out = out * (mel2ph > 0).float()[:, :, None]
    return (out, x, trace) if return_trace else out


def plms_x_pred(sched: Dict[str, Tensor], x: Tensor, noise_t: Tensor, t: int, interval: int) -> Tensor:
    """get_x_pred of p_sample_plms, usr/diff/shallow_diffusion_tts.py:174-183 (fp32 buffers, fp32 arithmetic)."""
    a_t = sched["alphas_cumprod"][t]
    a_prev = sched["alphas_cumprod"][max(t - interval, 0)]
    a_t_sq, a_prev_sq = a_t.sqrt(), a_prev.sqrt()
    x_delta = (a_prev - a_t) * ((1 / (a_t_sq * (a_t_sq + a_prev_sq))) * x
                                - 1 / (a_t_sq * (((1 - a_prev) * a_t).sqrt() + ((1 - a_t) * a_prev).sqrt())) * noise_t)
    return x + x_delta


def diffusion_infer_plms(p: Dict[str, Tensor], sched: Dict[str, Tensor], spec_min: Tensor, spec_max: Tensor,
                         cond_btH: Tensor, K_step: int, interval: int, fs2_mel: Optional[Tensor] = None,
                         start_noise: Optional[Tensor] = None, mel2ph: Optional[Tensor] = None,
                         gaussian_start: bool = False, dilation_cycle: int = 4, operand: Optional[str] = None,
                         return_x: bool = False):
    """Infer branch of GaussianDiffusion.forward with hparams['pndm_speedup'] = interval: the PLMS / PNDM sampler,
    usr/diff/shallow_diffusion_tts.py:168-201 (p_sample_plms) and :258-264 (the loop over reversed(range(0, K_step, interval))).
    Deterministic after the start: no noise is drawn.  The reference evaluates max(t - interval, 0) on a [B] tensor, which only
    works for B = 1 (SURVEY.md §9.2); the step index is the same for all rows, so this restatement (and the CUDA path) take it
    as a scalar and accept any B."""
    cond = cond_btH.transpose(1, 2)
    if gaussian_start:
        x = start_noise
    else:
        xs = norm_spec(fs2_mel, spec_min, spec_max).transpose(1, 2)[:, None]
        x = q_sample(sched, xs, K_step - 1, start_noise)
    B = x.shape[0]
    noise_list = []                                                      # deque(maxlen=4), :259
    for t in reversed(range(0, K_step, interval)):
        noise_pred = diffnet_forward(p, x, torch.full((B,), t, dtype=torch.long, device=x.device), cond, dilation_cycle, operand)
        if len(noise_list) == 0:                                         # :188-191
            x_pred = plms_x_pred(sched, x, noise_pred, t, interval)
            noise_pred_prev = diffnet_forward(p, x_pred, torch.full((B,), max(t - interval, 0), dtype=torch.long, device=x.device), cond,
                                              dilation_cycle, operand)
            prime = (noise_pred + noise_pred_prev) / 2
        elif len(noise_list) == 1:                                       # :192-193
            prime = (3 * noise_pred - noise_list[-1]) / 2
        elif len(noise_list) == 2:                                       # :194-195
            prime = (23 * noise_pred - 16 * noise_list[-1] + 5 * noise_list[-2]) / 12
        else:                                                            # :196-197
            prime = (55 * noise_pred - 59 * noise_list[-1] + 37 * noise_list[-2] - 9 * noise_list[-3]) / 24
        x = plms_x_pred(sched, x, prime, t, interval)                    # :199
        noise_list.append(noise_pred)
        noise_list = noise_list[-4:]
    out = denorm_spec(x[:, 0].transpose(1, 2), spec_min, spec_max)
    if mel2ph is not None:
        out = out * (mel2ph > 0).float()[:, :, None]
    return (out, x) if return_x else out


# --------------------------------------------------------------------------------------
# NSF harmonic source (modules/parallel_wavegan/models/source.py)
# --------------------------------------------------------------------------------------

def sinegen(f0_up: Tensor, rand_ini: Tensor, noise: Tensor, sampling_rate: int, harmonic_num: int = 8,
            sine_amp: float = 0.1, noise_std: float = 0.003, voiced_threshold: float = 0.0):
    """SineGen.forward/_f02sine, source.py:45-74,105-138 (flag_for_pulse False).

    f0_up [B,L,1]; rand_ini [B,dim] (column 0 forced to 0 as at :56); noise [B,L,dim] ~ N(0,1).
    returns (sine_waves [B,L,dim], uv [B,L,1])
    """
    dim = harmonic_num + 1
    mult = torch.arange(1, dim + 1, dtype=torch.float32).to(f0_up.device)
    f0_buf = f0_up[:, :, :1] * mult[None, None, :]                      # :112-118
    rad = (f0_buf / sampling_rate) % 1                                   # :51
    ri = rand_ini.clone()
    ri[:, 0] = 0                                                         # :56
    rad = rad.clone()
    rad[:, 0, :] = rad[:, 0, :] + ri                                     # :57
    tmp_over_one = torch.cumsum(rad, 1) % 1                              # :67
    over_idx = (tmp_over_one[:, 1:, :] - tmp_over_one[:, :-1, :]) < 0    # :68-69
    shift = torch.zeros_like(rad)
    shift[:, 1:, :] = over_idx * -1.0                                    # :70-71
    sines = torch.sin(torch.cumsum(rad + shift, dim=1) * 2 * np.pi)      # :73-74
    sine_waves = sines * sine_amp                                        # :121
    uv = torch.ones_like(f0_up) * (f0_up > voiced_threshold)             # :38-43,126
    noise_amp = uv * noise_std + (1 - uv) * sine_amp / 3                 # :131
    sine_waves = sine_waves * uv + noise_amp * noise                     # :133-137
    return sine_waves, uv


def nsf_source(p: Dict[str, Tensor], f0: Tensor, hop: int, rand_ini: Tensor, noise: Tensor,
               sampling_rate: int, harmonic_num: int = 8) -> Tensor:
    """hifigan.py:147-149 + SourceModuleHnNSF.forward source.py:386-399.
    f0 [B,T] -> har_source [B,1,L] (nearest up-sample x hop, sines, Linear 9->1, tanh)."""
    f0_up = f0[:, :, None].repeat_interleave(hop, dim=1)                 # nn.Upsample(nearest)
    sine_wavs, _uv = sinegen(f0_up, rand_ini, noise, sampling_rate, harmonic_num)
    merged = torch.tanh(F.linear(sine_wavs, p["m_source.l_linear.weight"], p["m_source.l_linear.bias"]))
    return merged.transpose(1, 2)


# --------------------------------------------------------------------------------------
# HiFi-GAN generator (modules/hifigan/hifigan.py), weight-norm already folded
# --------------------------------------------------------------------------------------

def resblock1(p: Dict[str, Tensor], pre: str, x: Tensor, k: int, dilations: Sequence[int],
              operand: Optional[str] = None) -> Tensor:
    """ResBlock1.forward, hifigan.py:54-61."""
    for m, d in enumerate(dilations):
        xt = F.leaky_relu(x, LRELU_SLOPE)
        xt = F.conv1d(_rnd(xt, operand), _rnd_w(p[f"{pre}convs1.{m}.weight"], operand), p[f"{pre}convs1.{m}.bias"],
                      dilation=d, padding=(k * d - d) // 2)
        xt = F.leaky_relu(xt, LRELU_SLOPE)
        xt = F.conv1d(_rnd(xt, operand), _rnd_w(p[f"{pre}convs2.{m}.weight"], operand), p[f"{pre}convs2.{m}.bias"],
                      dilation=1, padding=(k - 1) // 2)
        x = xt + x
    return x


def hifigan_forward(p: Dict[str, Tensor], h: dict, mel: Tensor, f0: Optional[Tensor],
                    rand_ini: Optional[Tensor] = None, src_noise: Optional[Tensor] = None,
                    operand: Optional[str] = None, return_source: bool = False):
    """HifiGanGenerator.forward, hifigan.py:144-173.  mel [B,80,T], f0 [B,T] -> wav [B,1,T*hop]."""
    rates = list(h["upsample_rates"])
    ksz = list(h["upsample_kernel_sizes"])
    rk = list(h["resblock_kernel_sizes"])
    rd = list(h["resblock_dilation_sizes"])
    hop = int(np.prod(rates))
    har = None
    if f0 is not None:
        har = nsf_source(p, f0, hop, rand_ini, src_noise, h["audio_sample_rate"])
    x = F.conv1d(_rnd(mel, operand), _rnd_w(p["conv_pre.weight"], operand), p["conv_pre.bias"], padding=3)
    for i, (u, k) in enumerate(zip(rates, ksz)):
        x = F.leaky_relu(x, LRELU_SLOPE)
        x = F.conv_transpose1d(_rnd(x, operand), _rnd_w(p[f"ups.{i}.weight"], operand), p[f"ups.{i}.bias"],
                               stride=u, padding=(k - u) // 2)
        if har is not None:
            if i + 1 < len(rates):
                s = int(np.prod(rates[i + 1:]))
                xs = F.conv1d(har, p[f"noise_convs.{i}.weight"], p[f"noise_convs.{i}.bias"], stride=s, padding=s // 2)
            else:
                xs = F.conv1d(har, p[f"noise_convs.{i}.weight"], p[f"noise_convs.{i}.bias"])
            xs = F.relu(xs)
            C = xs.shape[1]
            xs = F.layer_norm(xs.transpose(1, -1), (C,)).transpose(1, -1)
            x = x + xs
        acc = None
        for j in range(len(rk)):
            r = resblock1(p, f"resblocks.{i * len(rk) + j}.", x, rk[j], rd[j], operand)
            acc = r if acc is None else acc + r
        x = acc / len(rk)
    x = F.leaky_relu(x)            # default slope 0.01, hifigan.py:169
    x = F.conv1d(x, p["conv_post.weight"], p["conv_post.bias"], padding=3)
    x = torch.tanh(x)
    return (x, har) if return_source else x


# --------------------------------------------------------------------------------------
# PitchExtractor (SURVEY.md section 8f-2): mel -> f0 between the sampler and the vocoder
# --------------------------------------------------------------------------------------

PE_HPARAMS = dict(predictor_hidden=-1, ffn_padding="SAME", predictor_kernel=5, pitch_type="frame", use_uv=True,
                  pitch_norm="log", f0_mean=0.0, f0_std=1.0)   # configs/tts/fs2.yaml:13-14,23,33, configs/tts/base.yaml:64, usr/configs/base.yaml:2


def pe_conv_layers(p: Dict[str, Tensor]) -> int:
    n = 0
    while f"mel_encoder.conv.{n}.conv.conv.weight" in p:
        n += 1
    return n


def pe_positions(x0: Tensor) -> Tensor:
    """utils/__init__.py:146-158 make_positions(tensor, padding_idx=0) on the float tensor xs[..., 0]
    (modules/fastspeech/tts_modules.py:230): position = running count of non-zero entries, 0 where the entry is zero."""
    mask = x0.ne(0).int()
    return (torch.cumsum(mask, dim=1).type_as(mask) * mask).long()


def pe_pos_table(n: int, dim: int) -> Tensor:
    """modules/commons/common_layers.py:123-144 get_embedding(n, dim, padding_idx=0)."""
    half = dim // 2
    emb = math.log(10000) / (half - 1)
    emb = torch.exp(torch.arange(half, dtype=torch.float) * -emb)
    emb = torch.arange(n, dtype=torch.float).unsqueeze(1) * emb.unsqueeze(0)
    emb = torch.cat([torch.sin(emb), torch.cos(emb)], dim=1).view(n, -1)
    emb[0, :] = 0
    return emb


def pe_forward(p: Dict[str, Tensor], mel: Tensor, hp: Optional[dict] = None) -> Dict[str, Tensor]:
    """PitchExtractor.forward in eval mode (modules/fastspeech/pe.py:138-150): mel [B,T,80] ->
    {'pitch_pred' [B,T,2], 'f0_denorm_pred' [B,T]}."""
    hp = {**PE_HPARAMS, **(hp or {})}
    # ---- Prenet (pe.py:24-42): 3 x [conv k5 -> ReLU -> BatchNorm1d(eval)] * nonpadding, Linear, * nonpadding
    nonpad = 1 - mel.abs().sum(-1).eq(0).float()[:, None, :]          # [B,1,T]
    x = mel.transpose(1, 2)
    i = 0
    while f"mel_prenet.layers.{i}.0.weight" in p:
        pre = f"mel_prenet.layers.{i}."
        k = p[pre + "0.weight"].shape[-1]
        x = F.conv1d(x, p[pre + "0.weight"], p[pre + "0.bias"], padding=k // 2)
        x = F.relu(x)
        x = F.batch_norm(x, p[pre + "2.running_mean"], p[pre + "2.running_var"], p[pre + "2.weight"], p[pre + "2.bias"],
                         training=False, eps=1e-5)
        x = x * nonpad
        i += 1
    x = F.linear(x.transpose(1, 2), p["mel_prenet.out_proj.weight"], p["mel_prenet.out_proj.bias"])
    x = x * nonpad.transpose(1, 2)
    # ---- ConvStacks (pe.py:83-117), ConvBlock norm='gn' (:45-78): Linear, n x [x + ReLU(GroupNorm(C/16 groups)(conv k5))], Linear
    n_enc = pe_conv_layers(p)
    if n_enc > 0:
        x = F.linear(x, p["mel_encoder.in_proj.weight"], p["mel_encoder.in_proj.bias"]).transpose(1, 2)
        for j in range(n_enc):
            pre = f"mel_encoder.conv.{j}."
            w = p[pre + "conv.conv.weight"]
            y = F.conv1d(x, w, p[pre + "conv.conv.bias"], padding=(w.shape[-1] - 1) // 2)    # ConvNorm, common_layers.py:56-58
            y = F.group_norm(y, w.shape[0] // 16, p[pre + "norm.weight"], p[pre + "norm.bias"], eps=1e-5)
            x = x + F.relu(y)
        x = F.linear(x.transpose(1, 2), p["mel_encoder.out_proj.weight"], p["mel_encoder.out_proj.bias"])
    # ---- PitchPredictor (tts_modules.py:224-237): + alpha * sinusoidal positions, 5 x [pad, conv k, ReLU, LayerNorm(C, eps 1e-12)], Linear -> 2
    pos = pe_positions(x[..., 0])
    table = pe_pos_table(max(4096, 1 + x.shape[1]), x.shape[-1])          # init_size=4096, grown to padding_idx+1+T (:151-158)
    x = x + p["pitch_predictor.pos_embed_alpha"] * table[pos]
    x = x.transpose(1, 2)
    i = 0
    while f"pitch_predictor.conv.{i}.1.weight" in p:
        pre = f"pitch_predictor.conv.{i}."
        k = p[pre + "1.weight"].shape[-1]
        pad = ((k - 1) // 2, (k - 1) // 2) if hp["ffn_padding"] == "SAME" else (k - 1, 0)
        x = F.conv1d(F.pad(x, pad), p[pre + "1.weight"], p[pre + "1.bias"])
        x = F.relu(x)
        x = F.layer_norm(x.transpose(1, 2), (x.shape[1],), p[pre + "3.weight"], p[pre + "3.bias"], eps=1e-12).transpose(1, 2)
        i += 1
    pred = F.linear(x.transpose(1, 2), p["pitch_predictor.linear.weight"], p["pitch_predictor.linear.bias"])
    # ---- denorm_f0 (utils/pitch_utils.py:63-76) as called at pe.py:144-149
    f0 = pred[:, :, 0]
    if hp["pitch_norm"] == "standard":
        f0 = f0 * hp["f0_std"] + hp["f0_mean"]
    if hp["pitch_norm"] == "log":
        f0 = 2 ** f0
    f0 = f0.clone()
    if hp["pitch_type"] == "frame" and hp["use_uv"]:
        f0[pred[:, :, 1] > 0] = 0
    f0[mel.abs().sum(-1) == 0] = 0
    return {"pitch_pred": pred, "f0_denorm_pred": f0}


# --------------------------------------------------------------------------------------
# Metrics used by the parity tests
# --------------------------------------------------------------------------------------

# --------------------------------------------------------------------------------------
# FastSpeech FFT blocks: the mel-rate decoder + mel_out (SURVEY.md section 8f-3)
# --------------------------------------------------------------------------------------
FFT_HPARAMS = dict(hidden_size=256, dec_layers=4, num_heads=2, dec_ffn_kernel_size=9, ffn_act="gelu", use_pos_embed=True)


def fft_n_layers(p: Dict[str, Tensor]) -> int:
    n = 0
    while f"layers.{n}.op.layer_norm1.weight" in p:
        n += 1
    return n


def fft_decoder_forward(p: Dict[str, Tensor], x: Tensor, hp: Optional[dict] = None, mel_out: Optional[Dict[str, Tensor]] = None,
                        tgt_nonpad: Optional[Tensor] = None, padding_mask: Optional[Tensor] = None):
    """FastspeechDecoder.forward in eval mode (modules/fastspeech/tts_modules.py:286-310 FFTBlocks.forward, :340-347) over
    TransformerEncoderLayer -> EncSALayer (modules/commons/common_layers.py:696-731): x [B,T,C] -> hidden [B,T,C]; with
    ``mel_out`` = {'weight','bias'} also the projection and mask of FastSpeech2.run_decoder (modules/fastspeech/fs2.py:236-240).
    The attention is MultiheadAttention(self_attention=True, bias=False) -> F.multi_head_attention_forward (:321-345): no biases,
    q scaled by head_dim^-0.5, key_padding_mask = the padding frames, softmax over the keys.
    ``padding_mask`` [B,T] bool = FFTBlocks.forward's explicit mask (the encoder passes txt_tokens.eq(0), :333-335)."""
    hp = {**FFT_HPARAMS, **(hp or {})}
    B, T, C = x.shape
    H = hp["num_heads"]
    d = C // H
    k = hp["dec_ffn_kernel_size"]
    pad = x.abs().sum(-1).eq(0) if padding_mask is None else padding_mask.bool()      # tts_modules.py:291
    nonpad = (~pad).float()[:, :, None]                                # :292 (as [B,T,1]; the reference works in [T,B,C])
    if hp["use_pos_embed"]:                                            # :293-296
        pos = pe_positions(x[..., 0])
        table = pe_pos_table(int(pos.max()) + 2, C).to(x.device)
        x = x + p["pos_embed_alpha"] * table[pos]
    x = x * nonpad                                                     # :298
    for i in range(fft_n_layers(p)):
        pre = f"layers.{i}.op."
        res = x                                                        # common_layers.py:703-714
        h = F.layer_norm(x, (C,), p[pre + "layer_norm1.weight"], p[pre + "layer_norm1.bias"], 1e-5)
        qkv = F.linear(h, p[pre + "self_attn.in_proj_weight"])
        q, kk, v = qkv.chunk(3, dim=-1)
        q = q * d ** -0.5
        heads = lambda t: t.reshape(B, T, H, d).transpose(1, 2)       # [B,H,T,d]
        sc = heads(q) @ heads(kk).transpose(-1, -2)                    # [B,H,T,T]
        sc = sc.masked_fill(pad[:, None, None, :], float("-inf"))
        o = (torch.softmax(sc, dim=-1) @ heads(v)).transpose(1, 2).reshape(B, T, C)
        x = (res + F.linear(o, p[pre + "self_attn.out_proj.weight"])) * nonpad
        res = x                                                        # :716-722, :626-644
        h = F.layer_norm(x, (C,), p[pre + "layer_norm2.weight"], p[pre + "layer_norm2.bias"], 1e-5)
        h = F.conv1d(h.transpose(1, 2), p[pre + "ffn.ffn_1.weight"], p[pre + "ffn.ffn_1.bias"], padding=k // 2).transpose(1, 2)
        h = h * k ** -0.5
        h = F.gelu(h) if hp["ffn_act"] == "gelu" else F.relu(h)
        x = (res + F.linear(h, p[pre + "ffn.ffn_2.weight"], p[pre + "ffn.ffn_2.bias"])) * nonpad
    x = F.layer_norm(x, (C,), p["layer_norm.weight"], p["layer_norm.bias"], 1e-5) * nonpad    # tts_modules.py:303-304
    if mel_out is None:
        return x
    m = F.linear(x, mel_out["weight"], mel_out["bias"])                # fs2.py:238-240
    if tgt_nonpad is not None:
        m = m * tgt_nonpad[:, :, None]
    return x, m


def fft_encoder_forward(p: Dict[str, Tensor], txt_tokens: Tensor, hp: Optional[dict] = None) -> Tensor:
    """FastspeechEncoder.forward in eval mode (modules/fastspeech/tts_modules.py:327-346): x = sqrt(C) * embed_tokens(txt) +
    SinusoidalPositionalEmbedding(txt_tokens) (positions count the non-padding tokens, padding_idx 0), then the FFT blocks with
    use_pos_embed = False and the explicit padding mask txt_tokens.eq(0).  txt_tokens [B,T] int64 -> [B,T,C]."""
    hp = {**FFT_HPARAMS, **(hp or {})}
    w = p["embed_tokens.weight"]
    C = w.shape[1]
    x = math.sqrt(C) * F.embedding(txt_tokens, w, padding_idx=0)       # :340
    if hp.get("use_pos_embed", True):                                  # :341-343 (hparams['use_pos_embed'], not the FFTBlocks flag)
        pos = pe_positions(txt_tokens)
        x = x + pe_pos_table(int(pos.max()) + 2, C).to(x.device)[pos]
    blocks = {**hp, "use_pos_embed": False, "dec_ffn_kernel_size": hp.get("enc_ffn_kernel_size", hp["dec_ffn_kernel_size"])}
    return fft_decoder_forward(p, x, blocks, padding_mask=txt_tokens.eq(0))


def snr_db(ref: Tensor, out: Tensor) -> float:
    ref = ref.double().flatten()
    out = out.double().flatten()
    num = (ref * ref).sum()
    den = ((ref - out) ** 2).sum().clamp_min(1e-300)
    return float(10.0 * torch.log10(num / den))


def frame_snr_db(ref: Tensor, out: Tensor, hop: int = 128) -> float:
    """Local counterpart of snr_db for one utterance: the mean signal power of the whole of ``ref`` over the error energy of
    the worst ``hop``-sample frame, in dB (float64).  A defect confined to a few frames is diluted in the global SNR but not
    here.  Frames are measured against the utterance's power, not their own: quiet and unvoiced frames would make a
    per-frame ratio unstable.  A ragged last frame is averaged over the samples it has."""
    ref = ref.double().flatten()
    out = out.double().flatten()
    assert ref.shape == out.shape and ref.numel() > 0
    err = (ref - out) ** 2
    n = err.numel() // hop * hop
    frames = err[:n].reshape(-1, hop).mean(1)
    if n < err.numel():
        frames = torch.cat([frames, err[n:].mean()[None]])
    return float(10.0 * torch.log10((ref * ref).mean() / frames.max().clamp_min(1e-300)))


def wav_rows_db(ref: Tensor, out: Tensor, hop: int = 128) -> List[tuple]:
    """(snr_db, frame_snr_db) of every batch row of a waveform [B, L] or [B, 1, L]: each row is its own utterance."""
    assert ref.shape == out.shape
    ref, out = ref.reshape(ref.shape[0], -1), out.reshape(out.shape[0], -1)
    return [(snr_db(r, o), frame_snr_db(r, o, hop)) for r, o in zip(ref, out)]


def assert_wav_rows(ref: Tensor, out: Tensor, snr_min_db: float, frame_min_db: float, hop: int = 128) -> None:
    """Every batch row meets both bounds.  The figures of all rows are printed first (pytest -s shows them), so a failure
    reports the rows that passed as well."""
    rows = wav_rows_db(torch.as_tensor(ref), torch.as_tensor(out), hop)
    print("wav rows (SNR dB, worst-frame dB):", ", ".join(f"({s:.1f}, {f:.1f})" for s, f in rows))
    for b, (s, f) in enumerate(rows):
        assert s >= snr_min_db and f >= frame_min_db, \
            f"batch row {b}: SNR {s:.1f} dB (>= {snr_min_db}), worst frame {f:.1f} dB (>= {frame_min_db})"
