"""CPU tests: the oracle restatement (oracle/svs_oracle.py) against the golden vectors written by the executed
reference (oracle/make_golden.py) and -- when /root/reference is present -- against the live reference modules."""
import numpy as np
import pytest
import torch

import svs_oracle as O
import synth
from make_golden import DIFF_CASES, EPS_CASES, K_STEP, MAX_BETA, VOC_CASES

torch.set_num_threads(8)


@pytest.fixture(scope="module")
def sd_diff():
    return synth.diffnet_state(1234)


@pytest.fixture(scope="module")
def sd_voc():
    return synth.hifigan_state(4321)


def test_schedule_buffers_bit_exact(golden):
    s = O.schedule_buffers(O.linear_beta_schedule(K_STEP, MAX_BETA))
    for k in ("betas", "sqrt_alphas_cumprod", "sqrt_one_minus_alphas_cumprod", "sqrt_recip_alphas_cumprod",
              "sqrt_recipm1_alphas_cumprod", "posterior_mean_coef1", "posterior_mean_coef2", "posterior_log_variance_clipped"):
        assert np.array_equal(s[k].numpy(), golden["sched." + k]), k


def test_schedule_known_answers():
    # SURVEY.md §9.2 (probe of the reference, timesteps=100, linear, max_beta=0.06)
    s = O.schedule_buffers(O.linear_beta_schedule(100, 0.06))
    assert abs(s["sqrt_recip_alphas_cumprod"][99].item() - 4.635046) < 1e-5
    assert abs(s["sqrt_recipm1_alphas_cumprod"][50].item() - 1.09157) < 1e-5
    assert abs(s["posterior_mean_coef1"][1].item() - 0.875817) < 1e-6
    assert abs(s["posterior_log_variance_clipped"][0].item() - (-46.051701)) < 1e-4
    assert s["posterior_mean_coef2"][0].item() == 0.0


@pytest.mark.parametrize("i", range(len(EPS_CASES)))
def test_diffnet_forward_vs_golden(golden, sd_diff, i):
    c = EPS_CASES[i]
    inp = synth.kernel_inputs(c["seed"], c["B"], c["T"], 1)
    with torch.no_grad():
        eps = O.diffnet_forward(sd_diff, inp["start_noise"], torch.full((c["B"],), c["t"]), inp["cond"].transpose(1, 2))
    # identical arithmetic up to the order of the skip summation (the reference stacks then sums, net.py:126)
    assert np.abs(eps.numpy() - golden[f"eps.{i}"]).max() < 2e-5


@pytest.mark.parametrize("i", range(len(DIFF_CASES)))
def test_sampler_vs_golden(golden, sd_diff, i):
    c = DIFF_CASES[i]
    inp = synth.kernel_inputs(c["seed"], c["B"], c["T"], c["K"])
    sched = O.schedule_buffers(O.linear_beta_schedule(K_STEP, MAX_BETA))
    smin, smax = torch.tensor(synth.SPEC_MIN), torch.tensor(synth.SPEC_MAX)
    with torch.no_grad():
        mel, x0, _ = O.diffusion_infer(sd_diff, sched, smin, smax, inp["cond"], K_STEP, inp["step_noise"], inp["fs2_mel"],
                                       inp["start_noise"], return_trace=True)
    assert np.abs(mel.numpy() - golden[f"mel.{i}"]).max() < 1e-4
    assert np.abs(x0.numpy() - golden[f"x0.{i}"]).max() < 1e-4


@pytest.mark.parametrize("i", range(len(VOC_CASES)))
def test_vocoder_vs_golden(golden, sd_voc, i):
    c = VOC_CASES[i]
    inp = synth.vocoder_inputs(c["seed"], c["B"], c["T"])
    with torch.no_grad():
        wav, har = O.hifigan_forward(sd_voc, synth.HIFIGAN_CONFIG, inp["mel"], inp["f0"], inp["rand_ini"], inp["src_noise"],
                                     return_source=True)
        wav2 = O.hifigan_forward(sd_voc, synth.HIFIGAN_CONFIG, inp["mel"], None)
    assert np.abs(har.numpy() - golden[f"har.{i}"]).max() < 1e-6
    assert np.abs(wav.numpy() - golden[f"wav.{i}"]).max() < 1e-5
    assert np.abs(wav2.numpy() - golden[f"wav_nof0.{i}"]).max() < 1e-5


def test_zero_init_trap_documented(sd_diff):
    """The reference zero-initialises DiffNet.output_projection.weight (net.py:105): eps would then be independent of the
    input and any parity test vacuous.  The synthetic factory must NOT reproduce that."""
    assert float(sd_diff["output_projection.weight"].abs().max()) > 0


def test_operand_rounding_model_orders(sd_diff):
    """bf16 operand rounding must be much worse than the bf16x3 split (DESIGN.md §5) -- guards the emulation used by the
    GPU tests to separate precision effects from bugs."""
    inp = synth.kernel_inputs(5, 1, 64, 1)
    t = torch.full((1,), 37)
    with torch.no_grad():
        ref = O.diffnet_forward(sd_diff, inp["start_noise"], t, inp["cond"].transpose(1, 2))
        bf = O.diffnet_forward(sd_diff, inp["start_noise"], t, inp["cond"].transpose(1, 2), operand="bf16")
    e = float((bf - ref).abs().max())
    assert 1e-3 < e < 0.2


def test_fp16x2_model_meets_mel_tolerance(sd_diff):
    """The contraction mode the CUDA sampler runs by default (fp16 activations x split fp16 weights, DESIGN.md §5), emulated on
    the oracle over all 100 steps: inside the north-star tolerance with margin, while plain bf16 operands are far outside."""
    K = 100
    sched = O.schedule_buffers(O.linear_beta_schedule(K, 0.06))
    smin, smax = torch.tensor(synth.SPEC_MIN), torch.tensor(synth.SPEC_MAX)
    inp = synth.kernel_inputs(8, 1, 48, K)
    with torch.no_grad():
        run = lambda op: O.diffusion_infer(sd_diff, sched, smin, smax, inp["cond"], K, inp["step_noise"], inp["fs2_mel"],
                                           inp["start_noise"], operand=op)
        ref, f16, bf = run(None), run("fp16x2"), run("bf16")
    assert float((f16 - ref).abs().max()) < 5e-3
    assert float((bf - ref).abs().max()) > 2e-2


reference_present = __import__("ref_shim").available()


@pytest.mark.skipif(not reference_present, reason="needs the original BiSinger source tree (set BISINGER_REFERENCE)")
def test_live_reference_matches_oracle(sd_diff):
    """Build container only: run the unmodified reference DiffNet on fresh inputs and compare with the restatement."""
    import ref_shim
    ns = ref_shim.load()
    net = ns.DiffNet(80)
    net.load_state_dict(sd_diff, strict=True)
    inp = synth.kernel_inputs(99, 2, 70, 1)
    t = torch.full((2,), 63)
    with torch.no_grad():
        a = net(inp["start_noise"], t, inp["cond"].transpose(1, 2))
        b = O.diffnet_forward(sd_diff, inp["start_noise"], t, inp["cond"].transpose(1, 2))
    assert float((a - b).abs().max()) < 2e-5


def test_plms_sampler_vs_golden(sd_diff):
    """oracle.diffusion_infer_plms against the executed reference's p_sample_plms loop (oracle/make_golden_plms.py)."""
    import os
    from make_golden_plms import PLMS_CASES
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "plms_golden.npz"))
    sched = O.schedule_buffers(O.linear_beta_schedule(K_STEP, MAX_BETA))
    smin, smax = torch.tensor(synth.SPEC_MIN), torch.tensor(synth.SPEC_MAX)
    for i, c in enumerate(PLMS_CASES):
        inp = synth.kernel_inputs(c["seed"], c["B"], c["T"], 1)
        with torch.no_grad():
            mel, x0 = O.diffusion_infer_plms(sd_diff, sched, smin, smax, inp["cond"], K_STEP, c["interval"], inp["fs2_mel"],
                                             inp["start_noise"], return_x=True)
        assert np.abs(mel.numpy() - g[f"mel.{i}"]).max() < 1e-4
        assert np.abs(x0.numpy() - g[f"x0.{i}"]).max() < 5e-5


def _fwd_tol(ref):
    """Tolerance of a forward-golden case: the north-star 1e-2 on a mel range of spec_max - spec_min ~ 6.2, scaled to the range the
    reference output really has.  Case 1 (1000-step PLMS from a Gaussian start, no clamp in p_sample_plms) leaves the mel range by
    orders of magnitude on a random-init denoiser (|mel| ~ 2e3): errors are amplified with the signal, so the bound is relative."""
    return 1e-2 * max(1.0, float(np.abs(ref).max()) / 6.2)


def test_forward_golden_vs_oracle(sd_diff):
    """The restatement against the executed reference's public entry point GaussianDiffusion.forward(infer=True)
    (oracle/make_golden_forward.py): the K = 100 ancestral sampler with a mel2ph mask, and BiSinger's shipped configuration
    (timesteps = K_step = 1000, max_beta 0.02, pndm_speedup 5, gaussian_start; diff.yaml:16-23)."""
    import os
    from make_golden_forward import FWD_CASES, forward_inputs, forward_noise
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "forward_golden.npz"))
    smin, smax = torch.tensor(synth.SPEC_MIN), torch.tensor(synth.SPEC_MAX)
    for i, c in enumerate(FWD_CASES):
        sched = O.schedule_buffers(O.linear_beta_schedule(c["timesteps"], c["max_beta"]))
        cond, fs2_mel, mel2ph = forward_inputs(c)
        start, steps = forward_noise(c)
        with torch.no_grad():
            if c["pndm_speedup"]:
                mel = O.diffusion_infer_plms(sd_diff, sched, smin, smax, cond, c["K_step"], c["pndm_speedup"], fs2_mel, start,
                                             mel2ph=mel2ph, gaussian_start=c["gaussian_start"])
            else:
                mel = O.diffusion_infer(sd_diff, sched, smin, smax, cond, c["K_step"], steps, fs2_mel, start, mel2ph=mel2ph,
                                        gaussian_start=c["gaussian_start"])
        ref = g[f"mel.{i}"]
        assert np.abs(mel.numpy() - ref).max() < 0.05 * _fwd_tol(ref), i
        if c["pad_tail"]:
            assert float(np.abs(ref[-1, c["T"] - c["pad_tail"]:]).max()) == 0.0


@pytest.mark.skipif(not reference_present, reason="needs the original BiSinger source tree (set BISINGER_REFERENCE)")
def test_from_reference_wraps_the_live_module_and_delegates_training(sd_diff):
    """B200GaussianDiffusion.from_reference(ref): denoiser weights, schedule buffers and spec_min/max are taken over from the live
    reference module (strict load), ``fs2`` is shared, and ``forward(infer=False)`` -- the training branch,
    shallow_diffusion_tts.py:237-242 -- runs in the reference and returns its ``diff_loss``."""
    import ref_shim
    from bisinger_b200 import B200GaussianDiffusion
    ns = ref_shim.load()
    gd = ns.gd
    inp = synth.kernel_inputs(81, 2, 24, 1)

    class StubFs2(torch.nn.Module):
        def forward(self, txt_tokens, mel2ph, spk_embed, ref_mels, f0, uv, energy, skip_decoder=False, infer=True, **kw):
            return {"decoder_inp": inp["cond"], "mel_out": inp["fs2_mel"]}

    gd.FastSpeech2 = lambda *a, **k: StubFs2()
    net = ns.DiffNet(80)
    net.load_state_dict(sd_diff, strict=True)
    ref = gd.GaussianDiffusion(None, 80, net, timesteps=K_STEP, K_step=K_STEP, loss_type="l1",
                               betas=gd.linear_beta_schedule(K_STEP, max_beta=MAX_BETA), spec_min=synth.SPEC_MIN, spec_max=synth.SPEC_MAX)
    ref.posterior_mean_coef1[3] = 0.123            # as if a checkpoint had overwritten a schedule buffer
    model = B200GaussianDiffusion.from_reference(ref, hparams=dict(ns.hparams))
    assert model.fs2 is ref.fs2 and model.reference is ref
    assert float(model.posterior_mean_coef1[3]) == pytest.approx(0.123)
    for k, v in ref.denoise_fn.state_dict().items():
        assert torch.equal(model.denoise_fn.state_dict()[k], v)
    assert "reference" not in dict(model.named_children())          # the reference's parameters stay its own
    torch.manual_seed(3)
    out = model(torch.zeros(2, 8, dtype=torch.long), ref_mels=inp["fs2_mel"], infer=False)
    torch.manual_seed(3)
    want = ref(torch.zeros(2, 8, dtype=torch.long), ref_mels=inp["fs2_mel"], infer=False)
    assert "diff_loss" in out and torch.equal(out["diff_loss"], want["diff_loss"]) and out["diff_loss"].requires_grad
    assert model._ref_dirty                                          # weights are re-read before the next inference call
    with pytest.raises(NotImplementedError):
        B200GaussianDiffusion(None, 80, model.denoise_fn, timesteps=K_STEP, K_step=K_STEP, betas=O.linear_beta_schedule(K_STEP, MAX_BETA),
                              spec_min=synth.SPEC_MIN, spec_max=synth.SPEC_MAX)(torch.zeros(1, 4, dtype=torch.long), infer=False)
