"""GPU tests (-m gpu) of the fused layer kernel's row tiling: 128-row slabs numbered across the batch, pair tile u = slabs 2u and
2u + 1, so the two CTAs of a pair may work on two items (and, with a step per item, at two diffusion steps), and the last pair
tile of an odd slab count has an empty half.

Shapes: T < 128; T % 256 in (0, 128] (the last slab of every item ends inside the item's last 256 rows); an odd slab count;
pairs straddling two items.  Every output row goes through the same MMAs and epilogue whichever slab it shares a pair with,
so besides the oracle tolerance each batch row must equal, bit for bit, the same row sampled alone, and the variants of the
kernel (4-CTA multicast clusters, one launch per layer) must equal the default bit for bit."""
import pytest
import torch

import svs_oracle as O
import synth
from make_golden import K_STEP, MAX_BETA

pytestmark = pytest.mark.gpu

MEL_TOL = 1e-2
EPS_TOL = 4e-3   # one fp16x2 DiffNet evaluation against the fp32 oracle (test_diffnet_forward_vs_golden)

# (B, T): slabs per item, pair tiles
SHAPES = [
    (1, 100),    # 1 slab: one pair tile with an empty second half
    (2, 340),    # 3 slabs per item (340 % 256 = 84): pair tile 1 = last slab of item 0 + first slab of item 1
    (1, 300),    # 3 slabs: odd slab count, the second pair tile's second half is empty
    (3, 1875),   # 15 slabs per item (the bench's T): 45 slabs, pair tile 7 straddles items 0 / 1, pair tile 22 is half empty
]


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def sd():
    return synth.diffnet_state(1234)


@pytest.fixture(scope="module")
def sched():
    return O.schedule_buffers(O.linear_beta_schedule(K_STEP, MAX_BETA))


def _plan(dev, sd, sched):
    from bisinger_b200 import B200DiffNet, DiffusionPlan
    net = B200DiffNet(80)
    net.load_state_dict(sd, strict=True)
    return DiffusionPlan(net, sched, K_STEP, K_STEP, synth.SPEC_MIN, synth.SPEC_MAX, precision="fp16x2", device=dev)


@pytest.fixture(scope="module")
def plan(dev, sd, sched):
    return _plan(dev, sd, sched)


def _sample_args(B, T, dev):
    inp = synth.kernel_inputs(4000 + 7 * B + T, B, T, K_STEP)
    return inp, [inp[k].to(dev) for k in ("cond", "fs2_mel", "start_noise", "step_noise")]


@pytest.mark.parametrize("B,T", SHAPES)
def test_slab_shapes_vs_oracle_and_rows_alone(plan, sd, sched, dev, B, T):
    inp, args = _sample_args(B, T, dev)
    mel = plan.sample(*args).cpu()
    with torch.no_grad():
        ref = O.diffusion_infer(sd, sched, torch.tensor(synth.SPEC_MIN), torch.tensor(synth.SPEC_MAX), inp["cond"], K_STEP,
                                inp["step_noise"], inp["fs2_mel"], inp["start_noise"])
    err = float((mel - ref).abs().max())
    assert err <= MEL_TOL, f"mel max-abs error {err} at B={B}, T={T}"
    if B > 1:
        for b in range(B):
            one = plan.sample(args[0][b:b + 1], args[1][b:b + 1], args[2][b:b + 1], args[3][:, b:b + 1]).cpu()
            assert torch.equal(one[0], mel[b]), f"row {b} of B={B}, T={T} differs from the same row sampled alone"


@pytest.mark.parametrize("B,T", [(2, 340), (3, 300), (3, 1875)])
def test_mixed_steps_on_straddling_pairs(plan, sd, dev, B, T):
    """A step per item, so the two slabs of a straddling pair tile are at different steps (each CTA's residual epilogue reads its
    own item's step embedding): the oracle at each row's step, and the batch in reverse order (other slab pairings) bit-equal."""
    inp = synth.kernel_inputs(500 + T, B, T, 1)
    cond = inp["cond"].transpose(1, 2)
    x = torch.randn((B, 1, 80, T), generator=torch.Generator().manual_seed(501 + T))
    t = torch.tensor([0, 99, 37][:B])
    eps = plan.denoise_steps(x.to(dev), t, cond.to(dev)).cpu()
    with torch.no_grad():
        ref = O.diffnet_forward(sd, x, t, cond)
    assert float((eps - ref).abs().max()) < EPS_TOL
    rev = torch.arange(B - 1, -1, -1)
    eps_rev = plan.denoise_steps(x[rev].contiguous().to(dev), t[rev], cond[rev].contiguous().to(dev)).cpu()
    assert torch.equal(eps_rev[rev], eps)


@pytest.mark.parametrize("env", [{"BSG_LAYER_MC": "1"}, {"BSG_LAYER_STACK": "0"}, {"BSG_LAYER_STACK": "0", "BSG_LAYER_MC": "1"}])
def test_layer_variants_bit_equal_on_slabs(plan, sd, sched, dev, monkeypatch, env):
    """4-CTA clusters (two pair tiles per unit; with 5 pair tiles the last unit's second pair has no slab) and one launch per layer
    give the default's mel bit for bit."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    var = _plan(dev, sd, sched)
    for B, T in [(3, 300), (2, 340), (3, 1875)]:
        _, args = _sample_args(B, T, dev)
        assert torch.equal(var.sample(*args), plan.sample(*args)), (B, T, env)
