"""PitchExtractor (SURVEY.md section 8f-2).  CPU: the oracle restatement against the golden vectors of the executed reference
module (oracle/make_golden_pe.py) and against the live reference where /root/reference exists; the drop-in's state-dict layout.
GPU (-m gpu): bsg_pe_forward through the drop-in against the fp32 oracle.

Tolerance (written here; north_star states none for f0): |pitch_pred - ref| <= 2e-3 in the log2-f0 / uv-logit domain
(= 2.4 cents), f0 relative error <= 2e-3 on frames whose voicing decision is not within the tolerance of the threshold,
identical voiced/unvoiced decisions everywhere else, padding frames exactly 0."""
import numpy as np
import pytest
import torch

import ref_shim
import svs_oracle as O
import synth
from make_golden_pe import PE_CASES

PRED_TOL = 2e-3
F0_RTOL = 2e-3


@pytest.fixture(scope="module")
def pe_golden():
    import os
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pe_golden.npz"))


@pytest.mark.parametrize("i", range(len(PE_CASES)))
def test_oracle_vs_golden(pe_golden, i):
    c = PE_CASES[i]
    sd = synth.pe_state(777, c["conv_layers"])
    mel = synth.pe_inputs(c["seed"], c["B"], c["T"], pad_tail=c["pad_tail"])
    with torch.no_grad():
        r = O.pe_forward(sd, mel)
    assert np.abs(r["pitch_pred"].numpy() - pe_golden[f"pitch_pred.{i}"]).max() < 1e-5
    f0, g = r["f0_denorm_pred"].numpy(), pe_golden[f"f0.{i}"]
    assert np.array_equal(f0 == 0, g == 0)
    assert np.abs(f0 - g).max() < 1e-2 * 1e-2          # Hz
    if c["pad_tail"]:
        assert np.all(g[1::2, c["T"] - c["pad_tail"]:] == 0)     # padding frames (pe.py:145)
    assert 0.05 < float((g > 0).mean()) < 0.95                    # both voicing decisions occur


@pytest.mark.skipif(not ref_shim.available(), reason="needs the original BiSinger source tree (set BISINGER_REFERENCE)")
def test_oracle_vs_live_reference():
    from make_golden_pe import build_reference_pe
    ns = ref_shim.load()
    pe = build_reference_pe(ns, 2)
    mel = synth.pe_inputs(91, 2, 77, pad_tail=9)
    with torch.no_grad():
        ref = pe(mel)
        r = O.pe_forward(synth.pe_state(777, 2), mel)
    assert torch.allclose(ref["pitch_pred"], r["pitch_pred"], atol=1e-5)
    assert torch.allclose(ref["f0_denorm_pred"], r["f0_denorm_pred"], atol=1e-3)


def test_oracle_left_padding_and_standard_norm():
    """hparams branches of the reference: ffn_padding != 'SAME' pads (k-1, 0) (tts_modules.py:212-214); pitch_norm 'standard'
    (pitch_utils.py:64-65); use_uv False leaves unvoiced frames un-zeroed (:72)."""
    sd = synth.pe_state(777, 2)
    mel = synth.pe_inputs(92, 1, 40)
    with torch.no_grad():
        a = O.pe_forward(sd, mel)
        b = O.pe_forward(sd, mel, dict(ffn_padding="LEFT"))
        c = O.pe_forward(sd, mel, dict(pitch_norm="standard", f0_mean=200.0, f0_std=50.0, use_uv=False))
    assert not torch.allclose(a["pitch_pred"], b["pitch_pred"])
    assert torch.allclose(c["f0_denorm_pred"], a["pitch_pred"][:, :, 0] * 50.0 + 200.0)


def test_drop_in_state_dict_layout():
    from bisinger_b200.pitch import B200PitchExtractor
    for cl, n in ((2, 3257219), (0, 2468739)):
        sd = synth.pe_state(777, cl)
        pe = B200PitchExtractor(conv_layers=cl).eval()
        res = pe.load_state_dict(sd, strict=True)
        assert not res.missing_keys and not res.unexpected_keys
        assert set(pe.state_dict()) == set(sd)
        assert pe.flat_weights().numel() == n
    with pytest.raises(RuntimeError):
        pe.train()


def test_drop_in_no_cpu_fallback():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from bisinger_b200.pitch import B200PitchExtractor
    pe = B200PitchExtractor().eval()
    with pytest.raises(RuntimeError):
        pe(torch.zeros(1, 8, 80))


# ---------------------------------------------------------------------------------------------------------------------
def _check(out, ref, mel):
    pred, f0 = out["pitch_pred"].cpu(), out["f0_denorm_pred"].cpu()
    rp, rf = ref["pitch_pred"], ref["f0_denorm_pred"]
    assert bool(torch.isfinite(pred).all()) and bool(torch.isfinite(f0).all())
    err = float((pred - rp).abs().max())
    assert err <= PRED_TOL, f"pitch_pred max-abs error {err}"
    pad = mel.abs().sum(-1) == 0
    assert bool((f0[pad] == 0).all())
    sure = (rp[:, :, 1].abs() > PRED_TOL) | pad            # voicing decision not within the tolerance of the threshold
    assert bool(((f0 == 0) == (rf == 0))[sure].all())
    v = sure & (rf > 0)
    if bool(v.any()):
        rel = float(((f0[v] - rf[v]).abs() / rf[v]).max())
        assert rel <= F0_RTOL, f"f0 relative error {rel}"
    return err


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda", 0)


def _pe(dev, conv_layers=2, hp=None):
    from bisinger_b200.pitch import B200PitchExtractor
    sd = synth.pe_state(777, conv_layers)
    pe = B200PitchExtractor(conv_layers=conv_layers, hparams=hp).eval()
    pe.load_state_dict(sd, strict=True)
    pe.build_plan(dev)
    return sd, pe


@pytest.mark.gpu
@pytest.mark.parametrize("i", range(len(PE_CASES)))
def test_gpu_vs_golden(pe_golden, dev, i):
    c = PE_CASES[i]
    sd, pe = _pe(dev, c["conv_layers"])
    mel = synth.pe_inputs(c["seed"], c["B"], c["T"], pad_tail=c["pad_tail"])
    ref = dict(pitch_pred=torch.from_numpy(pe_golden[f"pitch_pred.{i}"]), f0_denorm_pred=torch.from_numpy(pe_golden[f"f0.{i}"]))
    _check(pe(mel.to(dev)), ref, mel)


@pytest.mark.gpu
@pytest.mark.parametrize("B,T,pad", [(1, 1, 0), (1, 127, 0), (2, 129, 30), (3, 1500, 100), (1, 5000, 0)])
def test_gpu_vs_oracle_ragged(dev, B, T, pad):
    """single frame, tile-edge lengths, the 2-CTA tile path (>= 4096 rows), more than one GroupNorm chunk and more than one block
    of the position scan."""
    sd, pe = _pe(dev)
    mel = synth.pe_inputs(100 + T, B, T, pad_tail=pad)
    with torch.no_grad():
        ref = O.pe_forward(sd, mel)
    _check(pe(mel.to(dev)), ref, mel)


@pytest.mark.gpu
def test_gpu_hparam_branches(dev):
    hp = dict(ffn_padding="LEFT", pitch_norm="standard", f0_mean=200.0, f0_std=50.0, use_uv=False)
    sd, pe = _pe(dev, 2, hp)
    mel = synth.pe_inputs(93, 2, 90, pad_tail=11)
    with torch.no_grad():
        ref = O.pe_forward(sd, mel, hp)
    out = pe(mel.to(dev))
    assert float((out["pitch_pred"].cpu() - ref["pitch_pred"]).abs().max()) <= PRED_TOL
    assert float((out["f0_denorm_pred"].cpu() - ref["f0_denorm_pred"]).abs().max()) <= 50.0 * PRED_TOL * 1.01


@pytest.mark.gpu
def test_gpu_single_cta_tiles_and_determinism(dev, monkeypatch):
    mel = synth.pe_inputs(94, 3, 1500, pad_tail=50)
    sd, pe = _pe(dev)
    a = pe(mel.to(dev))
    b = pe(mel.to(dev))
    assert torch.equal(a["pitch_pred"], b["pitch_pred"]) and torch.equal(a["f0_denorm_pred"], b["f0_denorm_pred"])
    monkeypatch.setenv("BSG_PE_PAIR", "0")
    monkeypatch.setenv("BSG_PE_GRAPH", "0")
    sd, pe1 = _pe(dev)
    c = pe1(mel.to(dev))
    with torch.no_grad():
        ref = O.pe_forward(sd, mel)
    _check(c, ref, mel)


@pytest.mark.gpu
def test_gpu_mel_to_wav_chain(dev):
    """The chain the reference runs (a-lang-esm-style-ori-shift.py:628-632): mel -> pe -> f0 -> vocoder, against the oracle's
    chain with the reference-precision f0: waveform SNR >= 40 dB (north_star) with the PitchExtractor in the loop."""
    from bisinger_b200.vocoder import B200HifiGanGenerator
    sd, pe = _pe(dev)
    vsd = synth.hifigan_state(4321)
    gen = B200HifiGanGenerator(synth.HIFIGAN_CONFIG)
    gen.load_folded_state_dict(vsd, strict=True)
    gen.build_plan(dev)
    B, T = 2, 200
    vin = synth.vocoder_inputs(95, B, T)
    mel = vin["mel"].transpose(1, 2).contiguous()
    with torch.no_grad():
        rf0 = O.pe_forward(sd, mel)["f0_denorm_pred"]
        wref = O.hifigan_forward(vsd, synth.HIFIGAN_CONFIG, vin["mel"], rf0, vin["rand_ini"], vin["src_noise"])
    f0 = pe(mel.to(dev))["f0_denorm_pred"]
    flips = (f0.cpu() == 0) != (rf0 == 0)
    if bool(flips.any()):
        pytest.skip("a voicing logit within rounding of 0 flipped; the chain comparison needs identical decisions")
    from bisinger_b200 import mel_to_wav
    wav = mel_to_wav(mel.to(dev), gen, pe, rand_ini=vin["rand_ini"].to(dev), src_noise=vin["src_noise"].to(dev)).cpu()
    O.assert_wav_rows(wref[:, 0], wav, 40.0, 33.0)    # waveform SNR and worst-frame bound of tests/test_gpu_vocoder_frames.py, per row
    assert mel_to_wav(mel.to(dev), gen, pe, seed=3).shape == (B, T * 128)        # production path: device-drawn source noise


@pytest.mark.gpu
def test_gpu_graph_replay_matches_plain_launches(dev, monkeypatch):
    """forward replays one captured CUDA graph per shape through plan-owned staging buffers: bit-identical to plain launches
    (BSG_PE_GRAPH=0), also on the second and third call with other inputs."""
    sd, pe = _pe(dev)
    monkeypatch.setenv("BSG_PE_GRAPH", "0")
    sd, plain = _pe(dev)
    for seed in (301, 302, 303):
        mel = synth.pe_inputs(seed, 2, 150, pad_tail=seed % 7).to(dev)
        a, b = pe(mel), plain(mel)
        assert torch.equal(a["pitch_pred"], b["pitch_pred"]) and torch.equal(a["f0_denorm_pred"], b["f0_denorm_pred"])


@pytest.mark.gpu
def test_gpu_batch_rows_are_independent_and_long_segment(dev):
    """GroupNorm statistics, the position scan and the padding mask are per utterance: a batch of 3 equals the three single calls;
    and a 60 s segment (cfg4 length, T = 11250: 88 GroupNorm chunks, 11 blocks of the position scan) agrees with the oracle."""
    sd, pe = _pe(dev)
    mel = synth.pe_inputs(501, 3, 260, pad_tail=13).to(dev)
    out = pe(mel)
    for b in range(3):
        one = pe(mel[b:b + 1].contiguous())
        assert float((one["pitch_pred"][0] - out["pitch_pred"][b]).abs().max()) <= 1e-6
        assert torch.equal(one["f0_denorm_pred"][0] == 0, out["f0_denorm_pred"][b] == 0)
    long_mel = synth.pe_inputs(502, 1, 11250)
    with torch.no_grad():
        ref = O.pe_forward(sd, long_mel)
    _check(pe(long_mel.to(dev)), ref, long_mel)
