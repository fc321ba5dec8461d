"""FastSpeech FFT encoder (SURVEY.md section 8f-3, the phoneme-rate side): the oracle restatement against fixtures written by the
executed reference FastspeechEncoder and by FFTBlocks.forward(x, padding_mask) called on it (oracle/make_golden_fft.py), the
drop-in's parameter names, and -- on the GPU -- the CUDA path (bsg_fft_forward_masked: the decoder's kernels with the caller's
padding mask and no positional term) against both.

Tolerance as for the decoder (tests/test_fft_decoder.py): |hidden - ref| <= 5e-3 on values of O(1) .. O(5); padding positions exactly 0."""
import os

import numpy as np
import pytest
import torch

import svs_oracle as O
import synth
from make_golden_fft import ENC_CASES

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fft_encoder_golden.npz")
TOL = 5e-3


def test_encoder_oracle_vs_reference_golden():
    g = np.load(GOLDEN)
    sd = synth.fft_encoder_state(777)
    for i, c in enumerate(ENC_CASES):
        tok = synth.fft_tokens(c["seed"], c["B"], c["T"], pad_tail=c["pad_tail"])
        x = synth.fft_inputs(c["seed"] + 100, c["B"], c["T"])
        with torch.no_grad():
            e = O.fft_encoder_forward(sd, tok)
            b = O.fft_decoder_forward(sd, x, dict(use_pos_embed=False), padding_mask=tok.eq(0))
        assert np.abs(e.numpy() - g[f"enc.{i}"]).max() < 2e-5
        assert np.abs(b.numpy() - g[f"blocks.{i}"]).max() < 2e-5
        if c["pad_tail"]:
            assert float(e[1, c["T"] - c["pad_tail"]:].abs().max()) == 0.0
            assert float(b[1, c["T"] - c["pad_tail"]:].abs().max()) == 0.0


def _encoder(dev=None):
    from bisinger_b200.fft import B200FastspeechEncoder
    sd = synth.fft_encoder_state(777)
    emb = torch.nn.Embedding(sd["embed_tokens.weight"].shape[0], 256, padding_idx=0)
    enc = B200FastspeechEncoder(emb, 256, 4, 9, num_heads=2).eval()
    r = enc.load_state_dict(sd, strict=True)
    assert not r.missing_keys and not r.unexpected_keys
    return sd, (enc if dev is None else enc.to(dev))


def test_encoder_drop_in_state_dict_and_embedding():
    """Names as FastspeechEncoder's state dict (no pos_embed_alpha: FFTBlocks(use_pos_embed=False)); forward_embedding -- torch ops,
    runnable on the CPU -- equals the oracle's embedding sum bit for bit up to sin/cos rounding; no CPU forward exists."""
    sd, enc = _encoder()
    assert set(enc.state_dict().keys()) == set(sd.keys())
    assert "pos_embed_alpha" not in enc.state_dict()
    tok = synth.fft_tokens(41, 2, 37, pad_tail=5)
    x = enc.forward_embedding(tok)
    pos = O.pe_positions(tok)
    ref = 16.0 * torch.nn.functional.embedding(tok, sd["embed_tokens.weight"]) + O.pe_pos_table(int(pos.max()) + 2, 256)[pos]
    assert float((x - ref).abs().max()) < 1e-5
    assert float(x[1, 32:].abs().max()) == 0.0
    n = 1 + 128 + 4 * (2 * 256 + 768 * 256 + 256 * 256 + 2 * 256 + 1024 * 256 * 9 + 1024 + 256 * 1024 + 256) + 2 * 256
    assert enc.flat_weights().numel() == n
    with pytest.raises((RuntimeError, AssertionError, OSError)):          # no CPU fallback
        enc(tok)


@pytest.fixture(scope="module")
def enc_gpu():
    assert torch.cuda.is_available()
    dev = torch.device("cuda", 0)
    sd, enc = _encoder(dev)
    return sd, enc, dev


@pytest.mark.gpu
@pytest.mark.parametrize("i", range(len(ENC_CASES)))
def test_gpu_encoder_vs_reference_golden(enc_gpu, i):
    sd, enc, dev = enc_gpu
    g = np.load(GOLDEN)
    c = ENC_CASES[i]
    tok = synth.fft_tokens(c["seed"], c["B"], c["T"], pad_tail=c["pad_tail"])
    e = enc(tok.to(dev)).cpu()
    x = synth.fft_inputs(c["seed"] + 100, c["B"], c["T"])
    b = enc.forward_blocks(x.to(dev), tok.eq(0).to(dev)).cpu()
    assert np.abs(e.numpy() - g[f"enc.{i}"]).max() <= TOL
    assert np.abs(b.numpy() - g[f"blocks.{i}"]).max() <= TOL
    if c["pad_tail"]:
        assert float(e[1, c["T"] - c["pad_tail"]:].abs().max()) == 0.0 and float(b[1, c["T"] - c["pad_tail"]:].abs().max()) == 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("B,T,pad", [(1, 1, 0), (2, 7, 3), (3, 129, 64), (32, 120, 50), (2, 1000, 333)])
def test_gpu_encoder_vs_oracle_shapes(enc_gpu, B, T, pad):
    """A single token, phrases shorter than one attention tile, one more than a 128-query tile, a cfg3-sized batch of phoneme
    sequences, a long sequence; padded tails on the odd rows; a mask that differs from the all-zero-frame rule (the masked rows of x
    are NOT zero on input)."""
    sd, enc, dev = enc_gpu
    tok = synth.fft_tokens(1200 + T, B, T, pad_tail=pad)
    with torch.no_grad():
        ref = O.fft_encoder_forward(sd, tok)
    out = enc(tok.to(dev)).cpu()
    assert float((out - ref).abs().max()) <= TOL
    assert torch.equal(enc(tok.to(dev)).cpu(), out)                     # deterministic
    x = synth.fft_inputs(1300 + T, B, T)
    with torch.no_grad():
        bref = O.fft_decoder_forward(sd, x, dict(use_pos_embed=False), padding_mask=tok.eq(0))
    bout = enc.forward_blocks(x.to(dev), tok.eq(0).to(dev)).cpu()
    assert float((bout - bref).abs().max()) <= TOL
    if pad and B > 1:
        assert float(bout[1, T - pad:].abs().max()) == 0.0


@pytest.mark.gpu
def test_gpu_blocks_mask_argument_on_the_decoder(enc_gpu):
    """FFTBlocks.forward(x, padding_mask) on a stack WITH the positional term (the decoder's class): the explicit mask replaces
    the all-zero-frame rule, the positions still come from x[..., 0] (tts_modules.py:291-296)."""
    from bisinger_b200.fft import B200FastspeechDecoder
    _, _, dev = enc_gpu
    sd = synth.fft_state(555)
    dec = B200FastspeechDecoder(hparams=dict(hidden_size=256, dec_layers=4, num_heads=2, dec_ffn_kernel_size=9)).eval()
    dec.load_state_dict({k: v for k, v in sd.items() if not k.startswith("mel_out.")}, strict=True)
    dec = dec.to(dev)
    x = synth.fft_inputs(77, 2, 90)
    mask = torch.zeros(2, 90, dtype=torch.bool)
    mask[1, 70:] = True
    with torch.no_grad():
        ref = O.fft_decoder_forward(sd, x, padding_mask=mask)
    out = dec(x.to(dev), padding_mask=mask.to(dev)).cpu()
    assert float((out - ref).abs().max()) <= TOL
    assert float(out[1, 70:].abs().max()) == 0.0


def test_from_reference_copies_a_live_encoder_block_stack():
    """B200FFTBlocks.from_reference on the executed reference's FastspeechEncoder (build container only): geometry and every
    block weight taken over by name, no positional term (the encoder's stack is FFTBlocks(use_pos_embed=False))."""
    import ref_shim
    if not ref_shim.available():
        pytest.skip("needs the original BiSinger source tree (set BISINGER_REFERENCE)")
    from make_golden_fft import FFT_HP
    ns = ref_shim.load()
    ns.hparams.update(FFT_HP)
    from modules.commons.common_layers import Embedding  # type: ignore
    from modules.fastspeech.tts_modules import FastspeechDecoder, FastspeechEncoder  # type: ignore
    from bisinger_b200.fft import B200FFTBlocks
    sd = synth.fft_encoder_state(777)
    ref = FastspeechEncoder(Embedding(62, 256, 0), 256, 4, 9, num_heads=2).eval()
    ref.load_state_dict(sd, strict=True)
    twin = B200FFTBlocks.from_reference(ref)
    assert (twin.hidden_size, twin.num_layers, twin.kernel_size, twin.num_heads, twin.use_pos_embed) == (256, 4, 9, 2, False)
    for n, v in twin.state_dict().items():
        assert torch.equal(v, sd[n]), n
    assert not any(n.startswith("embed_tokens") for n in twin.state_dict())
    dsd = {k: v for k, v in synth.fft_state(555).items() if not k.startswith("mel_out.")}
    dref = FastspeechDecoder().eval()
    dref.load_state_dict(dsd, strict=True)
    dtwin = B200FFTBlocks.from_reference(dref)
    assert dtwin.use_pos_embed and float(dtwin.pos_embed_alpha) == pytest.approx(0.9)
    from bisinger_b200 import B200FastspeechDecoder
    own = B200FastspeechDecoder(hparams=FFT_HP)
    own.load_state_dict(dsd, strict=True)
    assert torch.equal(dtwin.flat_weights(), own.flat_weights())         # the same device blob either way


def test_device_blocks_encoder_is_the_reference_midi_encoder_with_the_block_stack_rerouted(monkeypatch):
    """device_blocks_encoder(FastspeechMIDIEncoder) on the executed reference (build container only), BiSinger's shipped
    positional setting (rel_pos: true): same state-dict keys as the reference class, the training-mode forward is the reference's,
    and the eval-mode forward hands (forward_embedding(...), txt_tokens.eq(0)) to forward_blocks -- checked numerically by answering
    that call with the oracle's FFT blocks and comparing with the reference encoder's own eval forward."""
    import ref_shim
    if not ref_shim.available():
        pytest.skip("needs the original BiSinger source tree (set BISINGER_REFERENCE)")
    from make_golden_fft import FFT_HP
    ns = ref_shim.load()
    ns.hparams.update({**FFT_HP, "rel_pos": True})
    try:
        from modules.commons.common_layers import ESM, Embedding  # type: ignore
        from modules.diffsinger_midi.fs2 import FastspeechMIDIEncoder  # type: ignore
        from bisinger_b200.fft import B200FFTBlocks, device_blocks_encoder
        torch.manual_seed(3)
        esm = ESM(d_model=256, nhead=8)
        ref = FastspeechMIDIEncoder(esm, Embedding(62, 256, 0), 256, 4, 9, num_heads=2).eval()
        cls = device_blocks_encoder(FastspeechMIDIEncoder)
        assert cls.__name__ == "B200FastspeechMIDIEncoder" and issubclass(cls, FastspeechMIDIEncoder)
        own = cls(esm, Embedding(62, 256, 0), 256, 4, 9, num_heads=2).eval()
        own.load_state_dict(ref.state_dict(), strict=True)
        assert list(own.state_dict().keys()) == list(ref.state_dict().keys())
        B, T = 2, 23
        tok = synth.fft_tokens(51, B, T, pad_tail=6)
        g = torch.Generator().manual_seed(52)
        emb = [0.1 * torch.randn((B, T, 256), generator=g) for _ in range(4)]     # midi, midi_dur, slur, lang embeddings
        with torch.no_grad():
            want = ref(tok, *emb)
        seen = {}

        def oracle_blocks(self, x, padding_mask=None):
            seen["mask"] = padding_mask
            sd = {k: v for k, v in self.state_dict().items()}
            return O.fft_decoder_forward(sd, x, dict(use_pos_embed=False), padding_mask=padding_mask)

        monkeypatch.setattr(B200FFTBlocks, "forward_blocks", oracle_blocks)
        with torch.no_grad():
            got = own(tok, *emb)
        assert torch.equal(seen["mask"], tok.eq(0))
        assert float((got - want).abs().max()) < 2e-5
        assert list(own.state_dict().keys()) == list(ref.state_dict().keys())      # the twin did not join the module tree
        twin = own._b200_blocks()
        own.load_state_dict(ref.state_dict(), strict=True)
        assert own._b200_blocks() is not twin                                       # rebuilt after the weights changed
        own.train()
        torch.manual_seed(9)
        a = own(tok, *emb)
        torch.manual_seed(9)
        b = ref.train()(tok, *emb)
        assert torch.equal(a, b)                                                    # training forward = the reference's, dropout included
    finally:
        ns.hparams.pop("rel_pos", None)
