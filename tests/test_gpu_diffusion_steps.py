"""Step calls of the sampler with a diffusion step per batch row: ``q_sample`` / ``p_sample`` / ``p_sample_plms`` of the drop-in
(shallow_diffusion_tts.py:149-208), ``B200DiffNet.forward`` with mixed steps, and the C-ABI entry points behind them.

CPU part: a per-row restatement of q_sample, p_sample and the PLMS step (the reference gathers its coefficients row by row with
``extract``), checked against the scalar oracle and, where BISINGER_REFERENCE points at the original tree, against the live
reference methods with injected noise.  GPU part (-m gpu): the device path against that restatement and ``O.diffnet_forward``,
row independence against the existing uniform-step path, the reference's own loops through the drop-in reproducing
``sample`` / ``sample_plms`` bit for bit, and the reuse rule of the conditioner projections."""
import gc
import weakref
from collections import deque

import pytest
import torch

import svs_oracle as O
import synth
from make_golden import K_STEP, MAX_BETA

MEL_TOL = 1e-2
MIXED_T = [0, 37, 99, 64]
SHAPES = [(1, 1), (2, 129), (3, 300), (4, 1000)]
SMIN, SMAX = torch.tensor(synth.SPEC_MIN), torch.tensor(synth.SPEC_MAX)


# ------------------------------------------------------------------------------------------------
# per-row restatement (t is a [B] long tensor, coefficients gathered per row as extract() does)
# ------------------------------------------------------------------------------------------------
def _ext(buf, t):
    return buf[t].reshape(-1, 1, 1, 1)


def ref_q_sample(sched, x_start, t, noise):
    """shallow_diffusion_tts.py:203-208."""
    return _ext(sched["sqrt_alphas_cumprod"], t) * x_start + _ext(sched["sqrt_one_minus_alphas_cumprod"], t) * noise


def ref_p_sample(sd, sched, x, t, cond, noise, clip_denoised=True):
    """:149-166 with :134-147; cond [B,H,T]; no noise where t == 0 (nonzero_mask, :165)."""
    eps = O.diffnet_forward(sd, x, t, cond)
    x_recon = _ext(sched["sqrt_recip_alphas_cumprod"], t) * x - _ext(sched["sqrt_recipm1_alphas_cumprod"], t) * eps
    if clip_denoised:
        x_recon = x_recon.clamp(-1., 1.)
    mean = _ext(sched["posterior_mean_coef1"], t) * x_recon + _ext(sched["posterior_mean_coef2"], t) * x
    nonzero = (1 - (t == 0).float()).reshape(-1, 1, 1, 1)
    return mean + nonzero * (0.5 * _ext(sched["posterior_log_variance_clipped"], t)).exp() * noise


def ref_x_pred(sched, x, noise_t, t, interval):
    """get_x_pred (:174-183) with a_prev at max(t - interval, 0) per row."""
    a_t = _ext(sched["alphas_cumprod"], t)
    a_prev = _ext(sched["alphas_cumprod"], torch.clamp(t - interval, min=0))
    a_t_sq, a_prev_sq = a_t.sqrt(), a_prev.sqrt()
    x_delta = (a_prev - a_t) * ((1 / (a_t_sq * (a_t_sq + a_prev_sq))) * x
                                - 1 / (a_t_sq * (((1 - a_prev) * a_t).sqrt() + ((1 - a_t) * a_prev).sqrt())) * noise_t)
    return x + x_delta


def ref_p_sample_plms(sd, sched, x, t, interval, cond, noise_list):
    """:168-201 (the history is the caller's list, appended to as the reference appends to self.noise_list)."""
    noise_pred = O.diffnet_forward(sd, x, t, cond)
    if len(noise_list) == 0:
        x_pred = ref_x_pred(sched, x, noise_pred, t, interval)
        noise_pred_prev = O.diffnet_forward(sd, x_pred, torch.clamp(t - interval, min=0), cond)
        prime = (noise_pred + noise_pred_prev) / 2
    elif len(noise_list) == 1:
        prime = (3 * noise_pred - noise_list[-1]) / 2
    elif len(noise_list) == 2:
        prime = (23 * noise_pred - 16 * noise_list[-1] + 5 * noise_list[-2]) / 12
    else:
        prime = (55 * noise_pred - 59 * noise_list[-1] + 37 * noise_list[-2] - 9 * noise_list[-3]) / 24
    noise_list.append(noise_pred)
    return ref_x_pred(sched, x, prime, t, interval)


@pytest.fixture(scope="module")
def sd():
    return synth.diffnet_state(1234)


@pytest.fixture(scope="module")
def sched():
    return O.schedule_buffers(O.linear_beta_schedule(K_STEP, MAX_BETA))


def _inputs(seed, B, T):
    inp = synth.kernel_inputs(seed, B, T, 1)
    x = torch.randn((B, 1, 80, T), generator=torch.Generator().manual_seed(seed + 1))
    return inp["cond"], x, inp["start_noise"]


def test_restatement_matches_scalar_oracle_row_by_row(sd, sched):
    """Each row of the per-row restatement equals the scalar oracle (q_sample, p_sample, get_x_pred) at that row's step."""
    B, T = 3, 12
    cond_btH, x, z = _inputs(5, B, T)
    cond = cond_btH.transpose(1, 2)
    t = torch.tensor([0, 37, 99])
    q = ref_q_sample(sched, x, t, z)
    with torch.no_grad():
        p = ref_p_sample(sd, sched, x, t, cond, z)
        pu = ref_p_sample(sd, sched, x, t, cond, z, clip_denoised=False)
    for b in range(B):
        tb = int(t[b])
        assert torch.equal(q[b:b + 1], O.q_sample(sched, x[b:b + 1], tb, z[b:b + 1]))
        with torch.no_grad():
            assert torch.allclose(p[b:b + 1], O.p_sample(sd, sched, x[b:b + 1], tb, cond[b:b + 1], z[b:b + 1]), atol=1e-5)
            assert torch.allclose(pu[b:b + 1], O.p_sample(sd, sched, x[b:b + 1], tb, cond[b:b + 1], z[b:b + 1], clip_denoised=False),
                                  atol=1e-5)
        xp = ref_x_pred(sched, x, z, t, 5)
        assert torch.allclose(xp[b:b + 1], O.plms_x_pred(sched, x[b:b + 1], z[b:b + 1], tb, 5), atol=1e-6)
    assert torch.equal(p[0], ref_p_sample(sd, sched, x, t, cond, 2 * z)[0])   # t == 0: no noise


reference_present = __import__("ref_shim").available()


@pytest.mark.skipif(not reference_present, reason="needs the original BiSinger source tree (set BISINGER_REFERENCE)")
def test_restatement_matches_live_reference(sd, sched, monkeypatch):
    """The restatement against the live reference's q_sample / p_sample (mixed t, injected noise) and p_sample_plms (B = 1, which is
    all the reference's max(t - interval, 0) supports)."""
    import ref_shim
    ns = ref_shim.load()
    gd = ns.gd
    net = ns.DiffNet(80)
    net.load_state_dict(sd, strict=True)
    ref = gd.GaussianDiffusion(None, 80, net, timesteps=K_STEP, K_step=K_STEP, loss_type="l1",
                               betas=gd.linear_beta_schedule(K_STEP, max_beta=MAX_BETA), spec_min=synth.SPEC_MIN, spec_max=synth.SPEC_MAX)
    B, T = 3, 16
    cond_btH, x, z = _inputs(7, B, T)
    cond = cond_btH.transpose(1, 2)
    t = torch.tensor([0, 37, 99])
    assert torch.allclose(ref.q_sample(x, t, noise=z), ref_q_sample(sched, x, t, z), atol=1e-6)
    monkeypatch.setattr(gd, "noise_like", lambda shape, device, repeat=False: z.to(device))
    with torch.no_grad():
        assert torch.allclose(ref.p_sample(x, t, cond), ref_p_sample(sd, sched, x, t, cond, z), atol=1e-5)
        ref.noise_list = deque(maxlen=4)
        mine = []
        x1 = x[:1]
        for tt in (99, 94, 89, 84, 79):
            tb = torch.tensor([tt])
            want = ref_p_sample_plms(sd, sched, x1, tb, 5, cond[:1], mine)
            x1 = ref.p_sample_plms(x1, tb, 5, cond[:1])
            assert torch.allclose(x1, want, atol=1e-5)


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda", 0)


def _plan(dev, sd, sched, precision="fp16x2"):
    from bisinger_b200 import B200DiffNet, DiffusionPlan
    net = B200DiffNet(80)
    net.load_state_dict(sd, strict=True)
    return DiffusionPlan(net, sched, K_STEP, K_STEP, synth.SPEC_MIN, synth.SPEC_MAX, precision=precision, device=dev)


def _model(dev, sd, interval=None):
    from bisinger_b200 import B200DiffNet, B200GaussianDiffusion
    net = B200DiffNet(80)
    net.load_state_dict(sd, strict=True)
    hp = dict(hidden_size=256, residual_layers=20, residual_channels=256, dilation_cycle_length=4, keep_bins=80)
    if interval:
        hp["pndm_speedup"] = interval
    m = B200GaussianDiffusion(None, 80, net, timesteps=K_STEP, K_step=K_STEP, betas=O.linear_beta_schedule(K_STEP, MAX_BETA),
                              spec_min=synth.SPEC_MIN, spec_max=synth.SPEC_MAX, hparams=hp)
    return m.to(dev)


MODES = [("fp16x2", {}), ("fp16x2", {"BSG_LAYER_STACK": "0"}), ("fp16x2", {"BSG_NO_FUSE": "1"}), ("bf16x3", {})]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", range(len(MODES)), ids=["fused", "layer_stack0", "no_fuse", "bf16x3"])
def test_diffnet_mixed_steps_vs_oracle(dev, sd, sched, monkeypatch, mode):
    """DiffNet.forward with a different step per row against O.diffnet_forward, tolerances of test_diffnet_forward_vs_golden; every
    row against the same utterance alone through the uniform-step path (the bound of test_batch_rows_are_independent)."""
    precision, env = MODES[mode]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    plan = _plan(dev, sd, sched, precision)
    tol = 5e-4 if plan.precision == "bf16x3" else 4e-3
    for B, T in SHAPES:
        cond_btH, x, _ = _inputs(300 + T, B, T)
        t = torch.tensor(MIXED_T[:B])
        eps = plan.denoise_steps(x.to(dev), t, cond_btH.to(dev).transpose(1, 2)).cpu()
        with torch.no_grad():
            ref = O.diffnet_forward(sd, x, t, cond_btH.transpose(1, 2))
        assert float((eps - ref).abs().max()) < tol, (B, T)
        for b in range(B):
            one = plan.denoise(x[b:b + 1].to(dev), int(t[b]), cond_btH[b:b + 1].to(dev)).cpu()
            assert float((one[0] - eps[b]).abs().max()) <= 1e-5, (B, T, b)


@pytest.mark.gpu
def test_b200diffnet_forward_accepts_mixed_steps(dev, sd):
    from bisinger_b200 import B200DiffNet
    net = B200DiffNet(80).to(dev)
    net.load_state_dict(sd, strict=True)
    cond_btH, x, _ = _inputs(11, 3, 140)
    t = torch.tensor([0, 500, 999])
    eps = net(x.to(dev), t.to(dev), cond_btH.to(dev).transpose(1, 2)).cpu()
    with torch.no_grad():
        ref = O.diffnet_forward(sd, x, t, cond_btH.transpose(1, 2))
    assert float((eps - ref).abs().max()) < 4e-3


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp16x2", "bf16x3"])
def test_p_sample_mixed_steps_vs_oracle(dev, sd, sched, precision):
    """p_sample with mixed t and injected noise, clamped and not; rows at t == 0 get no noise; q_sample per row."""
    plan = _plan(dev, sd, sched, precision)
    B, T = 4, 300
    cond_btH, x, z = _inputs(21, B, T)
    cond = cond_btH.to(dev).transpose(1, 2)
    t = torch.tensor(MIXED_T)
    for clip in (True, False):
        got = plan.p_sample(x.to(dev), t, cond, clip, noise=z.to(dev)).cpu()
        with torch.no_grad():
            ref = ref_p_sample(sd, sched, x, t, cond_btH.transpose(1, 2), z, clip)
        assert float((got - ref).abs().max()) < 2e-3, clip
    again = plan.p_sample(x.to(dev), t, cond, True, noise=(3 * z).to(dev)).cpu()
    base = plan.p_sample(x.to(dev), t, cond, True, noise=z.to(dev)).cpu()
    assert torch.equal(again[0], base[0]) and not torch.equal(again[1], base[1])
    q = plan.q_sample(x.to(dev), t, z.to(dev)).cpu()
    assert float((q - ref_q_sample(sched, x, t, z)).abs().max()) < 1e-6


@pytest.mark.gpu
def test_reference_loop_reproduces_sample_bit_for_bit(dev, sd):
    """The reference's infer loop (:246-267) driven through the drop-in's step methods: q_sample(t = K-1) and K p_sample calls give
    plan.sample's x_0 bit for bit, with injected noise and with device noise from the same seed."""
    m = _model(dev, sd)
    B, T = 2, 200
    inp = synth.kernel_inputs(31, B, T, K_STEP)
    cond_btH, fs2, sn, zn = (inp[k].to(dev) for k in ("cond", "fs2_mel", "start_noise", "step_noise"))
    cond = cond_btH.transpose(1, 2)
    x_start = m.norm_spec(fs2).transpose(1, 2)[:, None]
    for injected in (True, False):
        kw = dict(start_noise=sn, step_noise=zn) if injected else dict(seed=77)
        _, x0 = m.plan.sample(cond_btH, fs2, return_x=True, **kw)
        x = m.q_sample(x_start, torch.full((B,), K_STEP - 1, dtype=torch.long, device=dev), noise=sn if injected else None,
                       seed=None if injected else 77)
        for k, i in enumerate(reversed(range(K_STEP))):
            tt = torch.full((B,), i, dtype=torch.long, device=dev)
            x = m.p_sample(x, tt, cond, noise=zn[k] if injected else None, seed=None if injected else 77)
        assert torch.equal(x, x0), injected


@pytest.mark.gpu
def test_reference_plms_loop_reproduces_sample_plms_bit_for_bit(dev, sd):
    m = _model(dev, sd, interval=5)
    B, T = 2, 150
    inp = synth.kernel_inputs(41, B, T, 1)
    cond_btH, fs2, sn = (inp[k].to(dev) for k in ("cond", "fs2_mel", "start_noise"))
    cond = cond_btH.transpose(1, 2)
    _, x0 = m.plan.sample_plms(cond_btH, fs2, sn, 5, return_x=True)
    x = m.q_sample(m.norm_spec(fs2).transpose(1, 2)[:, None], torch.full((B,), K_STEP - 1, dtype=torch.long), noise=sn)
    m.noise_list = deque(maxlen=4)
    for i in reversed(range(0, K_STEP, 5)):
        x = m.p_sample_plms(x, torch.full((B,), i, dtype=torch.long, device=dev), 5, cond)
    assert torch.equal(x, x0)


@pytest.mark.gpu
def test_p_sample_plms_mixed_steps_vs_oracle(dev, sd, sched):
    """p_sample_plms with a different t per row through every history length, and over a whole loop (mel <= 1e-2 at B = 3).  The per-row
    max(t_b - interval, 0) is exercised where one row's t_b - interval < 0 and the others' is not: in the second evaluation of a first
    step, and in get_x_pred at the end of the loop (the last row reaches t_b = 3 while the others are at 25 and 15)."""
    m = _model(dev, sd, interval=5)
    B, T = 3, 120
    cond_btH, x, _ = _inputs(51, B, T)
    cond = cond_btH.transpose(1, 2)
    t = torch.tensor([3, 50, 97])
    m.noise_list = deque(maxlen=4)
    first = m.p_sample_plms(x.to(dev), t.to(dev), 5, cond.to(dev)).cpu()
    with torch.no_grad():
        want = ref_p_sample_plms(sd, sched, x, t, 5, cond, [])
    assert float((first - want).abs().max()) < 2e-3
    offs = torch.tensor([0, 10, 22])
    m.noise_list = deque(maxlen=4)
    mine = []
    xg, xr = x.to(dev), x.clone()
    for step, i in enumerate(reversed(range(25, K_STEP, 5))):   # 15 steps: histories 0, 1, 2, 3, 3, ...
        t = torch.full((B,), i) - offs
        xg = m.p_sample_plms(xg, t.to(dev), 5, cond.to(dev))
        with torch.no_grad():
            xr = ref_p_sample_plms(sd, sched, xr, t, 5, cond, mine)
        if step < 4:
            assert float((xg.cpu() - xr).abs().max()) < 2e-3, step
    mel = m.denorm_spec(xg[:, 0].transpose(1, 2)).cpu()
    ref = O.denorm_spec(xr[:, 0].transpose(1, 2), SMIN, SMAX)
    assert float((mel - ref).abs().max()) <= MEL_TOL


@pytest.mark.gpu
def test_cond_reuse_survives_interleaving_and_eviction(dev, sd, sched, monkeypatch):
    """A step call whose cond tag is stored on the workspace, after sample() on the same shape (which overwrote the projections) and
    after the workspace was evicted, still matches the oracle; in-place writes to cond are seen.  Bad arguments raise."""
    plan = _plan(dev, sd, sched)
    B, T = 2, 100
    cond_btH, x, z = _inputs(61, B, T)
    cond = cond_btH.to(dev).transpose(1, 2)
    t = torch.tensor([10, 90])
    with torch.no_grad():
        want = ref_p_sample(sd, sched, x, t, cond_btH.transpose(1, 2), z)
    from bisinger_b200 import launch_count
    check = lambda: float((plan.p_sample(x.to(dev), t, cond, noise=z.to(dev)).cpu() - want).abs().max()) < 2e-3
    n0 = launch_count()
    assert check()
    n1 = launch_count()
    assert check()                                                   # second call reuses the projections: no split, no 20 GEMMs
    assert launch_count() - n1 == (n1 - n0) - 21
    other = synth.kernel_inputs(62, B, T, K_STEP)
    plan.sample(other["cond"].to(dev), other["fs2_mel"].to(dev), other["start_noise"].to(dev), other["step_noise"].to(dev))
    assert check()
    plan.denoise(x.to(dev), 5, other["cond"].to(dev))
    assert check()
    for i in range(8):                                               # more shapes than the plan keeps: (B, T) is evicted
        plan.denoise(x[:1, :, :, :8 + i].contiguous().to(dev), 5, cond_btH[:1, :8 + i].contiguous().to(dev))
    assert check()
    cond.mul_(1.0).add_(0.0)                                          # an in-place write bumps the version: a new tag
    assert check()
    cond.add_(1.0)
    with torch.no_grad():
        moved = ref_p_sample(sd, sched, x, t, cond.cpu(), z)
    assert float((plan.p_sample(x.to(dev), t, cond, noise=z.to(dev)).cpu() - moved).abs().max()) < 2e-3
    with pytest.raises(RuntimeError, match="outside"):
        plan.p_sample(x.to(dev), torch.tensor([0, K_STEP]), cond, noise=z.to(dev))
    with pytest.raises(RuntimeError, match="outside"):
        plan.denoise_steps(x.to(dev), torch.tensor([-1, 3]), cond)
    with pytest.raises(RuntimeError, match="steps for a batch"):
        plan.p_sample(x.to(dev), torch.tensor([1, 2, 3]), cond)
    with pytest.raises(RuntimeError, match="cond must be"):
        plan.p_sample(x.to(dev), t, cond[:, :, :50])
    m = _model(dev, sd)
    with pytest.raises(NotImplementedError):
        m.p_sample(x.to(dev), t, cond, repeat_noise=True)


@pytest.mark.gpu
def test_cond_identity_is_bounded_and_keeps_nothing_alive(dev, sd, sched):
    """Step calls over more lengths than the plan keeps workspaces: the remembered cond identities stay bounded, no cond tensor is kept
    alive by the plan, and every result matches the oracle -- also after a shape fell out of both caches and its cond was replaced by a
    new tensor (which may take the old one's memory)."""
    plan = _plan(dev, sd, sched)
    t = torch.tensor([42])
    for rnd in range(2):
        for i in range(9):
            T = 20 + i
            cond_btH, x, z = _inputs(700 + 10 * rnd + i, 1, T)
            cond = cond_btH.to(dev).transpose(1, 2)
            ref_alive = weakref.ref(cond)
            got = plan.p_sample(x.to(dev), t, cond, noise=z.to(dev)).cpu()
            with torch.no_grad():
                want = ref_p_sample(sd, sched, x, t, cond_btH.transpose(1, 2), z)
            assert float((got - want).abs().max()) < 2e-3, (rnd, T)
            assert len(plan._cond_seen) <= plan.COND_SHAPES
            del cond
            gc.collect()
            assert ref_alive() is None, "the plan must not keep the caller's cond alive"


@pytest.mark.gpu
def test_noise_and_history_shapes_must_match_x(dev, sd):
    """noise / eps tensors are indexed with x's geometry: any other shape raises -- e.g. a noise_list left over from an utterance of
    another length, where the reference raises a shape error too."""
    m = _model(dev, sd, interval=5)
    cond_btH, x, z = _inputs(81, 1, 50)
    m.noise_list = deque(maxlen=4)
    m.p_sample_plms(x.to(dev), torch.tensor([60]), 5, cond_btH.to(dev).transpose(1, 2))
    cond2, x2, z2 = _inputs(82, 1, 60)
    with pytest.raises(RuntimeError, match="eps"):
        m.p_sample_plms(x2.to(dev), torch.tensor([55]), 5, cond2.to(dev).transpose(1, 2))
    with pytest.raises(RuntimeError, match="noise"):
        m.p_sample(x2.to(dev), torch.tensor([55]), cond2.to(dev).transpose(1, 2), noise=z.to(dev))
    with pytest.raises(RuntimeError, match="noise"):
        m.q_sample(x2.to(dev), torch.tensor([55]), noise=z.to(dev))
    with pytest.raises(RuntimeError, match="noise predictions"):
        m.plan.plms_update(x2.to(dev), torch.tensor([55]), 5, 2, [x2.to(dev)])
