"""`dl_sampler_step` (the guided-model samplers' fused guidance + step) against a torch fp32 restatement with the
kernel's op order: every coefficient pattern the schedules produce, with and without classifier-free guidance, clamp
on and off, x0_prev and noise null and non-null, a size that is not a multiple of the 256-thread block, operands inside
NaN-filled buffers (nothing past the end is read into a result or written), and the argument checks."""
import pytest
import torch

pytestmark = pytest.mark.gpu

NAMES = ["euler", "euler_a", "ddim", "dpmpp_2m", "dpmpp_2m_karras"]
N = 4 * (3 * 256 + 5)             # not a multiple of the block's 1024 elements


@pytest.fixture(scope="module")
def lib():
    from dreamlab_b200 import lib as L
    L.load()
    return L


def _f(v):
    return torch.tensor(float(v), dtype=torch.float32)


def reference(u, t, gs, x, x0_prev, z, coeffs, clip):
    """The kernel's arithmetic in torch fp32, one rounded op at a time."""
    a_x, a_e, c_x, c_e, c_0, c_1, c_n = (_f(c) for c in coeffs)
    e = u if t is None else u + _f(gs) * (t - u)
    x0 = a_x * x + a_e * e
    if clip is not None:
        x0 = x0.clamp(-clip, clip)
    v = c_x * x + c_e * e
    v = v + c_0 * x0
    if x0_prev is not None:
        v = v + c_1 * x0_prev
    if z is not None:
        v = v + c_n * z
    return v, x0


def _in_nan(t):
    """t copied into the front of a NaN-filled device buffer 64 elements longer."""
    if t is None:
        return None
    b = torch.full((t.numel() + 64,), float("nan"), device="cuda")
    b[:t.numel()] = t.reshape(-1).cuda()
    return b[:t.numel()]


def _run(lib, u, t, gs, x, p, z, coeffs, clip):
    xn = torch.full((N + 64,), float("nan"), device="cuda")
    x0 = torch.full((N + 64,), float("nan"), device="cuda")
    lib.sampler_step(_in_nan(u), _in_nan(t), gs, _in_nan(x), _in_nan(p), _in_nan(z), xn[:N], x0[:N], coeffs, clip)
    torch.cuda.synchronize()
    assert torch.isnan(xn[N:]).all() and torch.isnan(x0[N:]).all(), "guard elements written"
    return xn[:N].cpu(), x0[:N].cpu()


def _check(got, want, what):
    g, w = got
    rn, r0 = want
    assert not torch.isnan(g).any() and not torch.isnan(w).any(), what
    # the restatement rounds every op as the kernel does: equal up to the last bit of the largest value
    tol_n = 2 ** -22 * max(rn.abs().max().item(), 1.0)
    tol_0 = 2 ** -22 * max(r0.abs().max().item(), 1.0)
    assert (g - rn).abs().max().item() <= tol_n, (what, (g - rn).abs().max().item())
    assert (w - r0).abs().max().item() <= tol_0, (what, (w - r0).abs().max().item())


def _operands(seed):
    g = torch.Generator().manual_seed(seed)
    return [1.5 * torch.randn(N, generator=g) for _ in range(5)]


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("pred", ["epsilon", "v_prediction", "sample"])
@pytest.mark.parametrize("cfg", [None, 7.5])
def test_schedule_coefficients(lib, name, pred, cfg):
    """Each step's coefficients of a 6-step schedule (first, second-order, last; Euler ancestral's noise term; DDIM's
    clamp), as the engine passes them."""
    from dreamlab_b200.scheduler import SchedulerConfig, sampler_schedule
    d = {"prediction_type": pred, "clip_sample": True, "clip_sample_range": 1.0}
    if pred != "epsilon":
        d.update(rescale_betas_zero_snr=True, timestep_spacing="trailing")
    sched = sampler_schedule(name, 6, SchedulerConfig.from_dict(d))
    for i in range(6):
        u, t, x, p, z = _operands(100 + i)
        t = None if cfg is None else t
        p = p if sched.uses_prev_x0(i) else None
        z = z if sched.has_noise(i) else None
        got = _run(lib, u, t, cfg or 1.0, x, p, z, sched.coeffs(i), sched.clip_range)
        _check(got, reference(u, t, cfg or 1.0, x, p, z, sched.coeffs(i), sched.clip_range), (name, pred, i))


@pytest.mark.parametrize("cfg", [None, 3.0])
@pytest.mark.parametrize("clip", [None, 0.5])
@pytest.mark.parametrize("prev", [False, True])
@pytest.mark.parametrize("noise", [False, True])
def test_every_operand_pattern(lib, cfg, clip, prev, noise):
    coeffs = (0.75, -1.25, 0.5, 0.3125, -0.625, 0.21875 if prev else 0.0, 1.5 if noise else 0.0)
    u, t, x, p, z = _operands(7)
    t = t if cfg is not None else None
    p = p if prev else None
    z = z if noise else None
    got = _run(lib, u, t, cfg or 1.0, x, p, z, coeffs, clip)
    want = reference(u, t, cfg or 1.0, x, p, z, coeffs, clip)
    _check(got, want, (cfg, clip, prev, noise))
    if clip is not None:
        assert got[1].abs().max().item() <= clip and (want[1].abs() == clip).any()   # the clamp bit


def test_guidance_matches_cfg_combine_bit_for_bit(lib):
    """With a_x = 0, a_e = 1 the x0 output is the guided output itself: the same bits as dl_cfg_combine."""
    u, t, x, _, _ = (v.cuda() for v in _operands(11))
    want = torch.empty_like(u)
    lib.cfg_combine(u, t, 7.5, want)
    xn, x0 = torch.empty_like(u), torch.empty_like(u)
    lib.sampler_step(u, t, 7.5, x, None, None, xn, x0, (0.0, 1.0, 0.0, 0.0, 1.0, 0.0, 0.0))
    torch.cuda.synchronize()
    assert torch.equal(x0.view(torch.int32), want.view(torch.int32))
    assert torch.equal(xn.view(torch.int32), want.view(torch.int32))


def test_argument_checks(lib):
    x = torch.zeros(16, device="cuda")
    with pytest.raises(RuntimeError, match="x0_prev"):
        lib.sampler_step(x, None, 1.0, x, None, None, x.clone(), x.clone(), (1, 0, 0, 0, 1, 0.5, 0))
    with pytest.raises(RuntimeError, match="noise"):
        lib.sampler_step(x, None, 1.0, x, None, None, x.clone(), x.clone(), (1, 0, 0, 0, 1, 0, 0.5))
    with pytest.raises(RuntimeError, match="aligned"):
        b = torch.zeros(24, device="cuda")
        lib.sampler_step(b[1:17], None, 1.0, x, None, None, x.clone(), x.clone(), (1, 0, 0, 0, 1, 0, 0))
    with pytest.raises(RuntimeError, match="multiple of 4"):
        y = torch.zeros(6, device="cuda")
        lib.sampler_step(y, None, 1.0, y, None, None, y.clone(), y.clone(), (1, 0, 0, 0, 1, 0, 0))
    with pytest.raises(RuntimeError, match="x0_prev"):
        lib.sampler_step(x, None, 1.0, x, torch.zeros(8, device="cuda"), None, x.clone(), x.clone(),
                         (1, 0, 0, 0, 1, 0, 0))
