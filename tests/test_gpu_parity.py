"""GPU parity tests (-m gpu): the CUDA path through the C-ABI against the fp32 oracle and the committed golden vectors.

Tolerances are BASELINE.json's: mel max-abs error <= 1e-2 (de-normalised log-mel), waveform SNR >= 40 dB, both versus the
fp32 reference with identical weights, inputs and injected noise."""
import ctypes as C

import numpy as np
import pytest
import torch

import svs_oracle as O
import synth
from make_golden import DIFF_CASES, EPS_CASES, K_STEP, MAX_BETA, VOC_CASES

pytestmark = pytest.mark.gpu

MEL_TOL = 1e-2      # north_star: mel max-abs error
SNR_TOL_DB = 40.0   # north_star: waveform SNR
FRAME_TOL_DB = 33.0  # worst 128-sample frame per batch row (O.frame_snr_db); measured values: tests/test_gpu_vocoder_frames.py


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda", 0)


# fp16x2 is the default contraction mode of the sampler, bf16x3 the alternative; both must meet the north-star tolerance
@pytest.fixture(scope="module", params=["fp16x2", "bf16x3"])
def diff(dev, request):
    from bisinger_b200 import B200DiffNet, DiffusionPlan
    sd = synth.diffnet_state(1234)
    net = B200DiffNet(80)
    net.load_state_dict(sd, strict=True)
    sched = O.schedule_buffers(O.linear_beta_schedule(K_STEP, MAX_BETA))
    plan = DiffusionPlan(net, sched, K_STEP, K_STEP, synth.SPEC_MIN, synth.SPEC_MAX, precision=request.param, device=dev)
    return sd, sched, plan


@pytest.fixture(scope="module")
def voc(dev):
    from bisinger_b200.vocoder import B200HifiGanGenerator
    sd = synth.hifigan_state(4321)
    gen = B200HifiGanGenerator(synth.HIFIGAN_CONFIG)
    gen.load_folded_state_dict(sd, strict=True)
    gen.build_plan(dev)
    return sd, gen


def _conv_ref(a, w, bias, shifts):
    B, L, _ = a.shape
    out = bias.double()[None, None, :].repeat(B, L, 1)
    for tp, s in enumerate(shifts):
        sh = torch.zeros_like(a, dtype=torch.float64)
        lo, hi = max(0, -s), min(L, L - s)
        if hi > lo:
            sh[:, lo:hi] = a[:, lo + s:hi + s].double()
        out += sh @ w[:, tp, :].double().t()
    return out


@pytest.mark.parametrize("case", [
    (1, 128, 64, 128, [0], 128, 0), (1, 128, 256, 256, [0], 256, 0), (2, 300, 256, 512, [-2, 0, 2], 256, 0),
    (2, 300, 256, 512, [-8, 0, 8], 256, 1), (3, 77, 80, 256, [0], 256, 1), (2, 200, 64, 64, [-1, 0, 1], 64, 0),
    (2, 200, 32, 32, [-3, 0, 3], 32, 0), (1, 1, 64, 128, [0], 128, 0), (1, 129, 64, 128, [-25, 0, 25], 128, 0),
    (1, 1000, 128, 128, [-5, -4, -3, -2, -1, 0, 1, 2, 3, 4, 5], 128, 0),
    (2, 300, 256, 512, [-8, 0, 8], 256, 2), (1, 1875, 256, 256, [0], 128, 2), (3, 77, 256, 256, [-1, 0, 1], 256, 2),
    (2, 300, 256, 512, [-8, 0, 8], 256, 2 | 0x100), (4, 1000, 512, 256, [0], 256, 2 | 0x100),          # fp16x2, also on 2-CTA tiles
    (2, 300, 256, 512, [-2, 0, 2], 256, 1 | 0x100), (1, 1875, 256, 256, [0], 128, 1 | 0x100),          # bf16x3 on 2-CTA tiles
    (2, 300, 256, 512, [-8, 0, 8], 256, 2 | 0x200), (5, 600, 256, 512, [-4, 0, 4], 256, 1 | 0x200),    # 4-CTA clusters, multicast weights
    (3, 77, 256, 256, [-1, 0, 1], 256, 0 | 0x200),                                                     # (odd number of row tiles)
])
def test_conv_kernel_selftest(dev, case):
    """The tcgen05 implicit-GEMM kernel alone: taps as row shifts with zero padding, ragged L, channel tails (80, 32)."""
    from bisinger_b200 import _lib
    B, L, Cin, N, shifts, n_tile, prec = case
    g = torch.Generator().manual_seed(sum(case[:4]))
    a = torch.randn(B, L, Cin, generator=g).to(dev)
    w = (torch.randn(N, len(shifts), Cin, generator=g) / (Cin * len(shifts)) ** 0.5).contiguous()
    bias = torch.randn(N, generator=g)
    out = torch.full((B, L, N), float("nan"), device=dev)
    sh = (C.c_int * len(shifts))(*shifts)
    _lib.check(_lib.lib().bsg_selftest_conv(_lib.dev_ptr(a), _lib.fptr(w), _lib.fptr(bias), B, L, Cin, N, len(shifts), sh, n_tile, prec,
                                            _lib.dev_ptr(out), None))
    if prec & 0xff == 0:   # bf16 operands: compare with the exactly-rounded operands (fp32 accumulate => ~1e-6)
        ref = _conv_ref(a.bfloat16().float(), w.bfloat16().float().to(dev), bias.to(dev), shifts)
        tol = 2e-5
    elif prec & 0xff == 2:  # fp16x2: fp16 activations (exactly-rounded reference) x ~21-bit split weights
        ref = _conv_ref(a.half().float(), w.to(dev), bias.to(dev), shifts)
        tol = 2e-5
    else:           # bf16x3: ~16 mantissa bits against the unrounded operands
        ref = _conv_ref(a, w.to(dev), bias.to(dev), shifts)
        tol = 2e-4
    assert float((out.double() - ref).abs().max()) < tol


@pytest.mark.parametrize("i", range(len(EPS_CASES)))
def test_diffnet_forward_vs_golden(golden, diff, dev, i):
    sd, sched, plan = diff
    c = EPS_CASES[i]
    inp = synth.kernel_inputs(c["seed"], c["B"], c["T"], 1)
    eps = plan.denoise(inp["start_noise"].to(dev), c["t"], inp["cond"].to(dev)).cpu().numpy()
    # single evaluation, eps rms ~0.9; fp16x2 rounds the activations to 11 significant bits
    assert np.abs(eps - golden[f"eps.{i}"]).max() < (5e-4 if plan.precision == "bf16x3" else 4e-3)


@pytest.mark.parametrize("i", range(len(DIFF_CASES)))
def test_sampler_vs_golden(golden, diff, dev, i):
    sd, sched, plan = diff
    c = DIFF_CASES[i]
    inp = synth.kernel_inputs(c["seed"], c["B"], c["T"], c["K"])
    mel, x0 = plan.sample(inp["cond"].to(dev), inp["fs2_mel"].to(dev), inp["start_noise"].to(dev), inp["step_noise"].to(dev),
                          return_x=True)
    assert np.abs(mel.cpu().numpy() - golden[f"mel.{i}"]).max() <= MEL_TOL
    assert np.abs(x0.cpu().numpy() - golden[f"x0.{i}"]).max() <= MEL_TOL / 2.5


@pytest.mark.parametrize("B,T", [(1, 1), (1, 127), (2, 129), (3, 300), (1, 938)])
def test_sampler_vs_oracle_ragged(diff, dev, B, T):
    """Edge shapes: a single frame, one-less / one-more than a 128-row tile, several tiles, and cfg1's T=938."""
    sd, sched, plan = diff
    inp = synth.kernel_inputs(100 + T, B, T, K_STEP)
    with torch.no_grad():
        ref = O.diffusion_infer(sd, sched, torch.tensor(synth.SPEC_MIN), torch.tensor(synth.SPEC_MAX), inp["cond"], K_STEP,
                                inp["step_noise"], inp["fs2_mel"], inp["start_noise"])
    mel = plan.sample(inp["cond"].to(dev), inp["fs2_mel"].to(dev), inp["start_noise"].to(dev), inp["step_noise"].to(dev)).cpu()
    assert float((mel - ref).abs().max()) <= MEL_TOL


def test_sampler_multi_tile_is_deterministic(diff, dev):
    """Several 256-row tiles per item, a ragged last tile and more than one item: the fused layer kernel hands rows from tile to
    tile (halo rows of the neighbours, z rows read back by TMA, shared-memory boxes recycled by TMA) -- any ordering hole
    there shows up as run-to-run differences near the 128-row block edges (two such races were found and fixed)."""
    sd, sched, plan = diff
    B, T = 3, 700
    inp = synth.kernel_inputs(77, B, T, K_STEP)
    with torch.no_grad():
        ref = O.diffusion_infer(sd, sched, torch.tensor(synth.SPEC_MIN), torch.tensor(synth.SPEC_MAX), inp["cond"], K_STEP,
                                inp["step_noise"], inp["fs2_mel"], inp["start_noise"])
    args = [inp[k].to(dev) for k in ("cond", "fs2_mel", "start_noise", "step_noise")]
    runs = [plan.sample(*args).cpu() for _ in range(4)]
    assert float((runs[0] - ref).abs().max()) <= MEL_TOL
    for r in runs[1:]:
        assert torch.equal(r, runs[0])


@pytest.mark.parametrize("env", [{"BSG_LAYER_STACK": "0"}, {"BSG_LAYER_MC": "1"}, {"BSG_LAYER_STACK": "0", "BSG_LAYER_MC": "1"},
                                 {"BSG_NO_FUSE": "1"}])
def test_layer_kernel_variants(dev, monkeypatch, env):
    """The fused ResidualBlock kernel one launch per layer / on 4-CTA multicast clusters computes bit-identically to the
    default (all layers in one launch on CTA pairs); the unfused two-launch path (different arithmetic) meets the tolerance."""
    from bisinger_b200 import B200DiffNet, DiffusionPlan
    sd = synth.diffnet_state(1234)
    net = B200DiffNet(80)
    net.load_state_dict(sd, strict=True)
    sched = O.schedule_buffers(O.linear_beta_schedule(K_STEP, MAX_BETA))
    B, T = 2, 300
    inp = synth.kernel_inputs(55, B, T, K_STEP)
    args = [inp[k].to(dev) for k in ("cond", "fs2_mel", "start_noise", "step_noise")]
    base = DiffusionPlan(net, sched, K_STEP, K_STEP, synth.SPEC_MIN, synth.SPEC_MAX, precision="fp16x2", device=dev).sample(*args).cpu()
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    var = DiffusionPlan(net, sched, K_STEP, K_STEP, synth.SPEC_MIN, synth.SPEC_MAX, precision="fp16x2", device=dev).sample(*args).cpu()
    with torch.no_grad():
        ref = O.diffusion_infer(sd, sched, torch.tensor(synth.SPEC_MIN), torch.tensor(synth.SPEC_MAX), inp["cond"], K_STEP,
                                inp["step_noise"], inp["fs2_mel"], inp["start_noise"])
    assert float((base - ref).abs().max()) <= MEL_TOL
    assert float((var - ref).abs().max()) <= MEL_TOL
    if "BSG_NO_FUSE" not in env:
        assert torch.equal(var, base)


@pytest.mark.parametrize("B,T,interval", [(1, 60, 5), (3, 300, 5), (2, 90, 10), (1, 40, 1)])
def test_plms_sampler_vs_oracle(diff, dev, B, T, interval):
    """PLMS / PNDM sampler (p_sample_plms, shallow_diffusion_tts.py:168-201): CUDA path vs the oracle (which is pinned to the executed
    reference for B = 1); the first case is also a committed golden fixture of the reference itself."""
    import os
    sd, sched, plan = diff
    seed = 61 if (B, T, interval) == (1, 60, 5) else 200 + T
    inp = synth.kernel_inputs(seed, B, T, 1)
    mel2ph = torch.ones(B, T, dtype=torch.long)
    mel2ph[-1, T - 7:] = 0
    with torch.no_grad():
        ref = O.diffusion_infer_plms(sd, sched, torch.tensor(synth.SPEC_MIN), torch.tensor(synth.SPEC_MAX), inp["cond"], K_STEP, interval,
                                     inp["fs2_mel"], inp["start_noise"], mel2ph=mel2ph)
    mel = plan.sample_plms(inp["cond"].to(dev), inp["fs2_mel"].to(dev), inp["start_noise"].to(dev), interval=interval,
                           mel2ph=mel2ph.to(dev)).cpu()
    assert float((mel - ref).abs().max()) <= MEL_TOL
    assert float(mel[-1, T - 7:].abs().max()) == 0.0
    if (B, T, interval) == (1, 60, 5):
        g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "plms_golden.npz"))
        unmasked = plan.sample_plms(inp["cond"].to(dev), inp["fs2_mel"].to(dev), inp["start_noise"].to(dev), interval=interval).cpu()
        assert np.abs(unmasked.numpy() - g["mel.0"]).max() <= MEL_TOL


def test_sampler_mel2ph_mask_and_gaussian_start(diff, dev):
    sd, sched, plan = diff
    B, T = 2, 90
    inp = synth.kernel_inputs(31, B, T, K_STEP)
    mel2ph = torch.ones(B, T, dtype=torch.long)
    mel2ph[1, 60:] = 0   # padded tail of the second utterance
    with torch.no_grad():
        ref = O.diffusion_infer(sd, sched, torch.tensor(synth.SPEC_MIN), torch.tensor(synth.SPEC_MAX), inp["cond"], K_STEP,
                                inp["step_noise"], None, inp["start_noise"], mel2ph=mel2ph, gaussian_start=True)
    mel = plan.sample(inp["cond"].to(dev), None, inp["start_noise"].to(dev), inp["step_noise"].to(dev), mel2ph=mel2ph.to(dev)).cpu()
    assert float((mel - ref).abs().max()) <= MEL_TOL
    assert float(mel[1, 60:].abs().max()) == 0.0


def test_sampler_graph_path_properties(diff, dev):
    """Device-RNG / CUDA-graph path: deterministic per seed, seed-sensitive, finite, inside the mel range, and batch rows are
    independent (a row's result does not depend on what else is in the batch -- the property the replicas rely on)."""
    sd, sched, plan = diff
    inp = synth.kernel_inputs(41, 3, 200, 1)
    cond, fs2 = inp["cond"].to(dev), inp["fs2_mel"].to(dev)
    a = plan.sample(cond, fs2, seed=5)
    b = plan.sample(cond, fs2, seed=5)
    c = plan.sample(cond, fs2, seed=6)
    assert torch.equal(a, b) and not torch.equal(a, c)
    assert bool(torch.isfinite(a).all())
    smin, smax = torch.tensor(synth.SPEC_MIN, device=dev), torch.tensor(synth.SPEC_MAX, device=dev)
    assert bool((a >= smin - 1e-4).all()) and bool((a <= smax + 1e-4).all())   # clamp(-1,1) at the last step
    # injected-noise runs: row 0 alone == row 0 inside the batch
    K = K_STEP
    full = synth.kernel_inputs(43, 2, 100, K)
    m2 = plan.sample(full["cond"].to(dev), full["fs2_mel"].to(dev), full["start_noise"].to(dev), full["step_noise"].to(dev))
    m1 = plan.sample(full["cond"][:1].to(dev), full["fs2_mel"][:1].to(dev), full["start_noise"][:1].to(dev),
                     full["step_noise"][:, :1].contiguous().to(dev))
    assert torch.equal(m1[0], m2[0])


@pytest.mark.parametrize("i", range(len(VOC_CASES)))
def test_vocoder_vs_golden(golden, voc, dev, i):
    sd, gen = voc
    c = VOC_CASES[i]
    inp = synth.vocoder_inputs(c["seed"], c["B"], c["T"])
    har = gen.plan.source(inp["f0"], inp["rand_ini"], inp["src_noise"]).cpu().numpy()
    assert np.abs(har - golden[f"har.{i}"][:, 0]).max() < 1e-4
    wav = gen(inp["mel"].to(dev), inp["f0"].to(dev), inp["rand_ini"].to(dev), inp["src_noise"].to(dev)).cpu()
    O.assert_wav_rows(torch.from_numpy(golden[f"wav.{i}"]), wav, SNR_TOL_DB, FRAME_TOL_DB)
    wav2 = gen(inp["mel"].to(dev), None).cpu()
    O.assert_wav_rows(torch.from_numpy(golden[f"wav_nof0.{i}"]), wav2, SNR_TOL_DB, FRAME_TOL_DB)


@pytest.mark.parametrize("B,T", [(1, 1), (2, 9), (1, 257), (1, 938)])
def test_vocoder_vs_oracle_ragged(voc, dev, B, T):
    sd, gen = voc
    inp = synth.vocoder_inputs(200 + T, B, T)
    with torch.no_grad():
        ref, har = O.hifigan_forward(sd, synth.HIFIGAN_CONFIG, inp["mel"], inp["f0"], inp["rand_ini"], inp["src_noise"], return_source=True)
    out = gen(inp["mel"].to(dev), inp["f0"].to(dev), inp["rand_ini"].to(dev), inp["src_noise"].to(dev)).cpu()
    assert out.shape == ref.shape
    O.assert_wav_rows(ref, out, SNR_TOL_DB, FRAME_TOL_DB)
    hs = gen.plan.source(inp["f0"], inp["rand_ini"], inp["src_noise"]).cpu()
    assert float((hs - har[:, 0]).abs().max()) < 1e-4


def test_vocoder_long_source_phase(voc, dev):
    """60 s segment (cfg4 length): the NSF phase accumulation must not drift (fp64 frame scan) -- compared with a float64
    evaluation of the reference formula, which is what the reference approximates in fp32."""
    sd, gen = voc
    B, T = 1, 11250
    inp = synth.vocoder_inputs(77, B, T)
    hs = gen.plan.source(inp["f0"], inp["rand_ini"], torch.zeros_like(inp["src_noise"])).cpu().double()
    f0_up = inp["f0"][:, :, None].repeat_interleave(128, dim=1)
    mult = torch.arange(1, 10, dtype=torch.float32)
    rad = ((f0_up * mult) / 24000) % 1
    rad = rad.double()
    ri = inp["rand_ini"].double().clone()
    ri[:, 0] = 0
    rad[:, 0, :] += ri
    ph = torch.cumsum(rad, 1) % 1
    uv = (f0_up > 0).double()
    sines = torch.sin(ph * 2 * np.pi) * 0.1 * uv
    ref = torch.tanh(sines @ sd["m_source.l_linear.weight"].double().t() + sd["m_source.l_linear.bias"].double())[..., 0]
    assert float((hs - ref).abs().max()) < 1e-4


def test_full_pipeline_cfg_shapes_properties(diff, voc, dev):
    """BASELINE cfg3-sized row count (reduced batch to keep the test short): finite outputs, waveform in (-1, 1), mel in range."""
    sd, sched, plan = diff
    vsd, gen = voc
    B, T = 4, 1875
    inp = synth.kernel_inputs(55, B, T, 1)
    mel = plan.sample(inp["cond"].to(dev), inp["fs2_mel"].to(dev), seed=1)
    assert mel.shape == (B, T, 80) and bool(torch.isfinite(mel).all())
    vin = synth.vocoder_inputs(56, B, T)
    wav = gen(mel.transpose(1, 2).contiguous(), vin["f0"].to(dev), seed=2)
    assert wav.shape == (B, 1, T * 128) and bool(torch.isfinite(wav).all()) and float(wav.abs().max()) <= 1.0


def test_drop_in_module_surface(dev):
    """B200GaussianDiffusion.forward(infer=True) returns the reference's dict keys given a stand-in conditioner."""
    from bisinger_b200 import B200DiffNet, B200GaussianDiffusion
    sd = synth.diffnet_state(1234)
    net = B200DiffNet(80)
    net.load_state_dict(sd, strict=True)
    inp = synth.kernel_inputs(61, 2, 64, K_STEP)

    class FakeFs2(torch.nn.Module):
        def forward(self, txt_tokens, mel2ph, spk_embed, ref_mels, f0, uv, energy, skip_decoder=False, infer=True, **kw):
            return {"decoder_inp": inp["cond"].to(dev), "mel_out": inp["fs2_mel"].to(dev), "mel2ph": None}

    gd = B200GaussianDiffusion(None, 80, net, timesteps=K_STEP, K_step=K_STEP, betas=O.linear_beta_schedule(K_STEP, MAX_BETA),
                               spec_min=synth.SPEC_MIN, spec_max=synth.SPEC_MAX, fs2=FakeFs2())
    ret = gd(torch.zeros(2, 8, dtype=torch.long), infer=True, start_noise=inp["start_noise"], step_noise=inp["step_noise"])
    assert {"mel_out", "fs2_mel", "decoder_inp"} <= set(ret)
    sched = O.schedule_buffers(O.linear_beta_schedule(K_STEP, MAX_BETA))
    with torch.no_grad():
        ref = O.diffusion_infer(sd, sched, torch.tensor(synth.SPEC_MIN), torch.tensor(synth.SPEC_MAX), inp["cond"], K_STEP,
                                inp["step_noise"], inp["fs2_mel"], inp["start_noise"])
    assert float((ret["mel_out"].cpu() - ref).abs().max()) <= MEL_TOL
    # B200DiffNet.forward signature == DiffNet.forward(spec, diffusion_step, cond[B,H,T])
    eps = net.to(dev)(inp["start_noise"].to(dev), torch.full((2,), 10, device=dev), inp["cond"].to(dev).transpose(1, 2))
    with torch.no_grad():
        eref = O.diffnet_forward(sd, inp["start_noise"], torch.full((2,), 10), inp["cond"].transpose(1, 2))
    assert float((eps.cpu() - eref).abs().max()) < 4e-3    # default fp16x2 contraction, single evaluation


def test_vocoder_graph_replay_matches_plain_launches(voc, dev, monkeypatch):
    """Production path (no injected noise): one captured CUDA graph per shape, replayed with new inputs through the plan-owned
    staging buffers -- bit-identical to the plain launches (BSG_VOC_GRAPH=0), with and without the NSF branch."""
    from bisinger_b200.vocoder import B200HifiGanGenerator
    vsd, gen = voc
    monkeypatch.setenv("BSG_VOC_GRAPH", "0")
    plain = B200HifiGanGenerator(synth.HIFIGAN_CONFIG)
    plain.load_folded_state_dict(vsd, strict=True)
    plain.build_plan(dev)
    for seed in (201, 202, 203):       # first call captures, the next replay with other inputs
        vin = synth.vocoder_inputs(seed, 2, 70)
        mel, f0 = vin["mel"].to(dev), vin["f0"].to(dev)
        a, b = gen(mel, f0, seed=seed), plain(mel, f0, seed=seed)
        assert torch.equal(a, b)
        assert torch.equal(gen(mel, None, seed=seed), plain(mel, None, seed=seed))
    # the replay leaves the injected-noise path intact
    vin = synth.vocoder_inputs(204, 2, 70)
    w1 = gen(vin["mel"].to(dev), vin["f0"].to(dev), vin["rand_ini"].to(dev), vin["src_noise"].to(dev))
    w2 = plain(vin["mel"].to(dev), vin["f0"].to(dev), vin["rand_ini"].to(dev), vin["src_noise"].to(dev))
    assert torch.equal(w1, w2)


def test_batch_rows_are_independent(diff, voc, dev):
    """What the replica sharding rests on (SURVEY.md section 8e): an utterance's result does not depend on which batch it is in.
    Sampler (injected noise) and vocoder (injected source noise): a batch of 3 against the three single-utterance calls."""
    sd, sched, plan = diff
    vsd, gen = voc
    B, T = 3, 140
    inp = synth.kernel_inputs(401, B, T, K_STEP)
    cond, fs2, sn, zn = (inp[k].to(dev) for k in ("cond", "fs2_mel", "start_noise", "step_noise"))
    mel = plan.sample(cond, fs2, sn, zn)
    for b in range(B):
        one = plan.sample(cond[b:b + 1].contiguous(), fs2[b:b + 1].contiguous(), sn[b:b + 1].contiguous(), zn[:, b:b + 1].contiguous())
        assert float((one[0] - mel[b]).abs().max()) <= 1e-5
    vin = synth.vocoder_inputs(402, B, T)
    m, f0, ri, nz = (vin[k].to(dev) for k in ("mel", "f0", "rand_ini", "src_noise"))
    wav = gen(m, f0, ri, nz)
    for b in range(B):
        one = gen(m[b:b + 1].contiguous(), f0[b:b + 1].contiguous(), ri[b:b + 1].contiguous(), nz[b:b + 1].contiguous())
        assert float((one[0] - wav[b]).abs().max()) <= 1e-6


def test_vocoder_small_kernel_variants(voc, dev, monkeypatch):
    """The row-group noise-branch kernel (default) against its predecessor (BSG_VOC_NOISE_V2=0) and the oracle; lengths that leave
    partial row groups.  The two differ in the summation order of the LayerNorm statistics, which the bf16 operand rounding of the
    following convolutions amplifies, so they are compared by SNR, not bit for bit."""
    from bisinger_b200.vocoder import B200HifiGanGenerator
    vsd, gen = voc
    monkeypatch.setenv("BSG_VOC_NOISE_V2", "0")
    old = B200HifiGanGenerator(synth.HIFIGAN_CONFIG)
    old.load_folded_state_dict(vsd, strict=True)
    old.build_plan(dev)
    for B, T in ((1, 3), (2, 37), (3, 101)):
        vin = synth.vocoder_inputs(600 + T, B, T)
        args = [vin[k].to(dev) for k in ("mel", "f0", "rand_ini", "src_noise")]
        a, b = gen(*args).cpu(), old(*args).cpu()
        with torch.no_grad():
            ref = O.hifigan_forward(vsd, synth.HIFIGAN_CONFIG, vin["mel"], vin["f0"], vin["rand_ini"], vin["src_noise"])
        O.assert_wav_rows(ref, a, SNR_TOL_DB, FRAME_TOL_DB)
        O.assert_wav_rows(ref, b, SNR_TOL_DB, FRAME_TOL_DB)
        assert O.snr_db(b, a) >= SNR_TOL_DB
        a0, b0 = gen(args[0], None).cpu(), old(args[0], None).cpu()      # no NSF branch: the kernel only adds 0 and applies lrelu
        assert torch.equal(a0, b0)


def test_row_per_thread_epilogue_matches_transposing_epilogue(voc, dev, monkeypatch):
    """The row-per-thread epilogues with 256-bit global accesses (default) against the transposing epilogue (BSG_ROWS_EPI=0): vocoder
    (full and partial tiles, 2-CTA tiles from 4096 rows up) and PitchExtractor (write-only epilogues: bit-identical)."""
    from bisinger_b200.pitch import B200PitchExtractor
    from bisinger_b200.vocoder import B200HifiGanGenerator
    vsd, gen = voc
    psd = synth.pe_state(777, 2)
    pe = B200PitchExtractor().eval()
    pe.load_state_dict(psd, strict=True)
    pe.build_plan(dev)
    monkeypatch.setenv("BSG_ROWS_EPI", "0")
    old = B200HifiGanGenerator(synth.HIFIGAN_CONFIG)
    old.load_folded_state_dict(vsd, strict=True)
    old.build_plan(dev)
    pe_old = B200PitchExtractor().eval()
    pe_old.load_state_dict(psd, strict=True)
    pe_old.build_plan(dev)
    for B, T in ((1, 5), (2, 77), (1, 600)):
        vin = synth.vocoder_inputs(700 + T, B, T)
        args = [vin[k].to(dev) for k in ("mel", "f0", "rand_ini", "src_noise")]
        a, b = gen(*args).cpu(), old(*args).cpu()
        # the read-modify-write epilogues use explicit mul / add where the transposing epilogue leaves the contraction to the compiler
        assert O.snr_db(b, a) >= 60.0
        with torch.no_grad():
            ref = O.hifigan_forward(vsd, synth.HIFIGAN_CONFIG, vin["mel"], vin["f0"], vin["rand_ini"], vin["src_noise"])
        O.assert_wav_rows(ref, a, SNR_TOL_DB, FRAME_TOL_DB)
        O.assert_wav_rows(ref, b, SNR_TOL_DB, FRAME_TOL_DB)
    for B, T in ((2, 45), (3, 1500)):
        mel = synth.pe_inputs(710 + T, B, T, pad_tail=7).to(dev)
        a, b = pe(mel), pe_old(mel)
        assert torch.equal(a["pitch_pred"], b["pitch_pred"]) and torch.equal(a["f0_denorm_pred"], b["f0_denorm_pred"])


def test_workspace_cache_evicts_least_recently_used_shape(diff, voc, dev):
    """ADVICE r1: utterance lengths vary from call to call; the per-(B, T) workspaces (buffers + captured graphs) are evicted one at a time,
    least recently used first (6 sampler / 3 vocoder shapes) -- more shapes than the cache holds, revisiting the first: same results."""
    sd, sched, plan = diff
    vsd, gen = voc
    inp = synth.kernel_inputs(301, 1, 64, 1)
    first = plan.sample(inp["cond"].to(dev), inp["fs2_mel"].to(dev), seed=9)
    for T in (65, 70, 80, 96, 100, 110, 120, 130):
        i2 = synth.kernel_inputs(300 + T, 1, T, 1)
        assert bool(torch.isfinite(plan.sample(i2["cond"].to(dev), i2["fs2_mel"].to(dev), seed=9)).all())
    assert torch.equal(plan.sample(inp["cond"].to(dev), inp["fs2_mel"].to(dev), seed=9), first)
    vin = synth.vocoder_inputs(302, 1, 40)
    w0 = gen(vin["mel"].to(dev), vin["f0"].to(dev), seed=3)
    for T in (41, 50, 60, 70, 33):
        v2 = synth.vocoder_inputs(300 + T, 1, T)
        assert bool(torch.isfinite(gen(v2["mel"].to(dev), v2["f0"].to(dev), seed=3)).all())
    assert torch.equal(gen(vin["mel"].to(dev), vin["f0"].to(dev), seed=3), w0)
