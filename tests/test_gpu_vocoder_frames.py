"""Vocoder waveform checks that a pooled SNR cannot make, and the vocoder paths no other test reaches.

Every vocoder comparison with the fp32 oracle asserts two things per batch row (O.assert_wav_rows): the waveform SNR >= 40 dB
(BASELINE.json north_star) and a local bound, O.frame_snr_db >= FRAME_TOL_DB: the worst 128-sample frame's error energy
against the utterance's mean power.  Precision noise is spread evenly over the frames, so its worst frame sits a few dB
below the global SNR; a defect confined to a tile, a row group or a tail moves the worst frame by tens of dB while the
global SNR of a long utterance hardly notices it.

The shipped synthetic weights (synth.hifigan_state(4321)) drive most samples into tanh saturation (|wav| > 0.9 where the
slope of tanh is below 0.19), which damps an error before the final tanh 5-50x.  The linear-range state scales conv_post by
0.1 (RMS ~0.23, |wav| < 0.5), so an error anywhere in the generator reaches the waveform undamped.  The golden fixtures were
generated from the unscaled state and keep it.

The CPU tests (no marker) show each check detects what it is meant to detect; the GPU tests (-m gpu) run the linear-range
weights on the shapes of the existing vocoder tests, on the plan variants selected by environment at plan build, on lengths
where a fused stage's last ResBlock tile is full or nearly empty, and on MRF configurations with one and two ResBlocks."""
import math

import pytest
import torch

import svs_oracle as O
import synth

SNR_TOL_DB = 40.0
# Worst-frame bound, per batch row.  Measured on a B200 (1000 W limit) over every vocoder comparison of the suite, in dB
# (profiles/r03_a_vocoder_frame_snr.log has each case and row):
#   shipped weights, default plan: golden fixtures 47.7-51.9 (no-f0 path 47.7-47.9), oracle shapes 48.2-55.3, cfg4 length
#     48.5, cfg3 rows 49.2-49.8, mel -> pe -> wav chain 48.9-49.2; global SNR 49.4-55.6
#   linear-range weights: ragged 49.2-53.3, cfg4 length 48.6, cfg3 rows 49.0-49.1, default / BSG_VOC_PAIR=0 / BSG_ROWS_RMW=0
#     49.0-49.6, BSG_VOC_FUSE=0 46.5-47.1, fused tile tails 49.1-53.3; global SNR 48.4-53.3
#   resblock_kernel_sizes [3, 7]: 45.6-46.0 (SNR 47.2-47.3); [3]: 41.4-42.0 (SNR 43.0-43.2), the lowest figure
# The bound sits 8.4 dB below the lowest worst frame.  A frame off by 0.3 x RMS measures ~10.5 dB.
FRAME_TOL_DB = 33.0

H = synth.HIFIGAN_CONFIG
TILE_M = 128          # rows of the fused ResBlock kernel's intermediate tile (kTileM in conv_gemm.cuh)

torch.set_num_threads(8)


def linear_range_state(h=None):
    """synth.hifigan_state(4321, h) with conv_post.weight / .bias scaled by 0.1: the waveform stays out of tanh saturation."""
    sd = synth.hifigan_state(4321, h)
    return {k: v * 0.1 if k.startswith("conv_post.") else v for k, v in sd.items()}


def _oracle(sd, h, inp):
    with torch.no_grad():
        return O.hifigan_forward(sd, h, inp["mel"], inp["f0"], inp["rand_ini"], inp["src_noise"])


def _fused_tail_lengths(h, tile=TILE_M):
    """Utterance lengths T at which the last tile of a fused ResBlock launch is full, or holds as few rows as any T can make it.
    A fused stage (32, 64 or 128 channels) runs ResBlocks of kernel size k on tiles of V = tile - (k - 1) output rows, over the
    T * prod(upsample_rates[:i + 1]) rows of an utterance; the last tile holds (rows mod V) of them (V when that is 0).  The
    fewest rows is gcd(rate, V): 2 for the shipped configuration, whose row counts and V are all even."""
    out = set()
    C0, rate = h["upsample_initial_channel"], 1
    for i, u in enumerate(h["upsample_rates"]):
        rate *= u
        if C0 // 2 ** (i + 1) not in (32, 64, 128):
            continue
        for k in h["resblock_kernel_sizes"]:
            V = tile - (k - 1)
            for rem in (0, math.gcd(rate, V)):
                out.add(next(T for T in range(1, V + 1) if T * rate % V == rem))
    return sorted(out)


# ------------------------------------------------------------------ CPU: the checks and the fixture do what they are for

@pytest.fixture(scope="module")
def lin_938():
    inp = synth.vocoder_inputs(200 + 938, 1, 938)
    return inp, _oracle(linear_range_state(), H, inp)


def test_frame_bound_catches_a_one_frame_defect_the_snr_misses(lin_938):
    inp, ref = lin_938
    rms = float(ref.pow(2).mean().sqrt())
    bad = ref.clone()
    f = 938 // 2
    bad.view(-1)[f * 128:(f + 1) * 128] += 0.3 * rms * torch.randn(128, generator=torch.Generator().manual_seed(1))
    assert O.snr_db(ref, bad) >= SNR_TOL_DB               # the pooled SNR passes a frame that is off by 0.3 x RMS
    assert O.frame_snr_db(ref, bad) < FRAME_TOL_DB        # ... the frame bound does not
    assert O.frame_snr_db(ref, bad) < 15.0
    assert O.frame_snr_db(ref, ref) > 200.0


def test_frame_snr_measures_against_the_utterance_power():
    ref = torch.ones(1000, dtype=torch.float64)
    out = ref.clone()
    out[-1] += 0.1                                         # ragged last frame (1000 = 7 * 128 + 104): error 0.01 / 104 per sample
    assert abs(O.frame_snr_db(ref, out) - 10 * math.log10(104 / 0.01)) < 1e-9
    assert abs(O.snr_db(ref, out) - 10 * math.log10(1000 / 0.01)) < 1e-9
    rows = O.wav_rows_db(torch.stack([ref, out])[:, None], torch.stack([out, out])[:, None])
    assert rows[1][0] > 300 and abs(rows[0][1] - 10 * math.log10(104 / 0.01)) < 1e-9


@pytest.mark.parametrize("operand", [None, "bf16"])
def test_bf16_precision_oracle_meets_both_bounds(lin_938, operand):
    """Precision noise of the kind the CUDA path makes passes both bounds with room: bf16-rounded weights (operand None), and
    bf16 rounding of every convolution's operands (the two-launch ResBlock path's arithmetic)."""
    inp, ref = lin_938
    sd = linear_range_state()
    if operand is None:
        sd = {k: v.bfloat16().float() for k, v in sd.items()}
    with torch.no_grad():
        emu = O.hifigan_forward(sd, H, inp["mel"], inp["f0"], inp["rand_ini"], inp["src_noise"], operand=operand)
    O.assert_wav_rows(ref, emu, SNR_TOL_DB + 5.0, FRAME_TOL_DB + 8.0)


def test_linear_range_state_keeps_the_waveform_off_tanh_saturation(lin_938):
    inp, ref = lin_938
    assert float(ref.abs().max()) < 0.9
    with torch.no_grad():
        nof0 = O.hifigan_forward(linear_range_state(), H, inp["mel"], None)
        shipped = _oracle(synth.hifigan_state(4321), H, inp)
    assert float(nof0.abs().max()) < 0.9
    assert float((shipped.abs() > 0.9).double().mean()) > 0.5       # what the scaling is for
    for ks in ([3], [3, 7]):
        h = dict(H, resblock_kernel_sizes=ks, resblock_dilation_sizes=[[1, 3, 5]] * len(ks))
        v = synth.vocoder_inputs(5, 1, 77)
        assert float(_oracle(linear_range_state(h), h, v).abs().max()) < 0.9


def test_fused_tail_lengths_follow_the_tile_rule():
    Ts = _fused_tail_lengths(H)
    rates = [32, 64, 128]                                  # rows per mel frame in the fused stages (128, 64, 32 channels)
    for k in H["resblock_kernel_sizes"]:
        V = TILE_M - (k - 1)
        assert any(T * r % V == 0 for T in Ts for r in rates)
        assert any(T * r % V == 2 for T in Ts for r in rates)
    assert all(T * r % 2 == 0 for T in range(1, 64) for r in rates)    # an odd remainder (one row) cannot occur here


# ------------------------------------------------------------------ GPU

@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda", 0)


def _gen(dev, sd, h=H):
    from bisinger_b200.vocoder import B200HifiGanGenerator
    gen = B200HifiGanGenerator(h)
    gen.load_folded_state_dict(sd, strict=True)
    gen.build_plan(dev)
    return gen


@pytest.fixture(scope="module")
def voc_lin(dev):
    sd = linear_range_state()
    return sd, _gen(dev, sd)


def _run(gen, inp, dev):
    return gen(*(inp[k].to(dev) for k in ("mel", "f0", "rand_ini", "src_noise"))).cpu()


@pytest.mark.gpu
@pytest.mark.parametrize("B,T", [(1, 1), (2, 9), (1, 257), (1, 938)])
def test_vocoder_linear_range_vs_oracle_ragged(voc_lin, dev, B, T):
    """The shapes of test_vocoder_vs_oracle_ragged with the linear-range weights."""
    sd, gen = voc_lin
    inp = synth.vocoder_inputs(200 + T, B, T)
    O.assert_wav_rows(_oracle(sd, H, inp), _run(gen, inp, dev), SNR_TOL_DB, FRAME_TOL_DB)


@pytest.mark.gpu
def test_vocoder_linear_range_cfg4_length_vs_oracle(voc_lin, dev):
    """B = 1, T = 11 250 (60 s) with the linear-range weights: a defect in one tile of thousands shows in its frames."""
    sd, gen = voc_lin
    inp = synth.vocoder_inputs(9200, 1, 11250)
    O.assert_wav_rows(_oracle(sd, H, inp), _run(gen, inp, dev), SNR_TOL_DB, FRAME_TOL_DB)


@pytest.mark.gpu
def test_vocoder_linear_range_cfg3_batch_rows_vs_oracle(voc_lin, dev):
    """cfg3 batch (32 x 1875) with the linear-range weights: two CPU-seeded rows among device-drawn ones against the oracle."""
    sd, gen = voc_lin
    B, T, rows = 32, 1875, (3, 31)
    g = torch.Generator(device=dev)
    g.manual_seed(9300)
    base = synth.vocoder_inputs(9301, 1, T)
    mel = base["mel"].to(dev).repeat(B, 1, 1) + 0.05 * torch.randn((B, 80, T), generator=g, device=dev)
    f0 = base["f0"].to(dev).repeat(B, 1)
    ri = torch.rand((B, 9), generator=g, device=dev)
    nz = torch.randn((B, T * 128, 9), generator=g, device=dev)
    cpu = synth.vocoder_inputs(9302, len(rows), T)
    for j, r in enumerate(rows):
        mel[r], f0[r], ri[r], nz[r] = cpu["mel"][j].to(dev), cpu["f0"][j].to(dev), cpu["rand_ini"][j].to(dev), cpu["src_noise"][j].to(dev)
    out = gen(mel, f0, ri, nz)[list(rows)].cpu()
    O.assert_wav_rows(_oracle(sd, H, cpu), out, SNR_TOL_DB, FRAME_TOL_DB)


@pytest.fixture(scope="module")
def variant_cases():
    """(inputs, linear-range oracle) per shape, shared by the plan variants.  3 x 1500 = 4500 conv_pre rows: 2-CTA tiles on
    every stage of >= 128 channels; 2 x 37 leaves partial tiles and row groups."""
    sd = linear_range_state()
    cases = []
    for B, T in ((3, 1500), (2, 37)):
        inp = synth.vocoder_inputs(800 + T, B, T)
        cases.append((inp, _oracle(sd, H, inp)))
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{}, {"BSG_VOC_FUSE": "0"}, {"BSG_VOC_PAIR": "0"}, {"BSG_ROWS_RMW": "0"}],
                         ids=["default", "fuse0", "pair0", "rows_rmw0"])
def test_vocoder_plan_variants_vs_oracle(dev, monkeypatch, variant_cases, env):
    """Paths chosen when the plan is built: the default, the two-launch fp32-stream ResBlock path on every stage followed by
    conv_post_kernel<false> (BSG_VOC_FUSE=0), single-CTA tiles everywhere (BSG_VOC_PAIR=0), and the transposing epilogue for
    the read-modify-write epilogues (BSG_ROWS_RMW=0)."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    gen = _gen(dev, linear_range_state())
    for inp, ref in variant_cases:
        O.assert_wav_rows(ref, _run(gen, inp, dev), SNR_TOL_DB, FRAME_TOL_DB)


@pytest.mark.gpu
@pytest.mark.parametrize("T", _fused_tail_lengths(H))
def test_vocoder_fused_tile_tails_vs_oracle(voc_lin, dev, T):
    """Lengths at which the last tile of a fused ResBlock launch is full, or holds the fewest rows possible (_fused_tail_lengths);
    two utterances, so a tail tile is followed by the next utterance's first tile."""
    sd, gen = voc_lin
    inp = synth.vocoder_inputs(900 + T, 2, T)
    O.assert_wav_rows(_oracle(sd, H, inp), _run(gen, inp, dev), SNR_TOL_DB, FRAME_TOL_DB)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel_sizes", [[3], [3, 7]], ids=["k3", "k3_7"])
def test_vocoder_resblock_kernel_subsets_vs_oracle(dev, kernel_sizes):
    """MRF with one ResBlock (its only iteration writes the stage output without an MRF sum to add to) and with two (the sum is
    started and finished without ever being accumulated into): shipped upsampling and dilations, linear-range conv_post."""
    h = dict(H, resblock_kernel_sizes=kernel_sizes, resblock_dilation_sizes=[[1, 3, 5]] * len(kernel_sizes))
    sd = linear_range_state(h)
    gen = _gen(dev, sd, h)
    for B, T in ((2, 77), (1, 300)):
        inp = synth.vocoder_inputs(1000 + T, B, T)
        O.assert_wav_rows(_oracle(sd, h, inp), _run(gen, inp, dev), SNR_TOL_DB, FRAME_TOL_DB)
