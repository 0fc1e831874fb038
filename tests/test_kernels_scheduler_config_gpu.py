"""`dl_lcm_step_ex` and `dl_lcm_step_inpaint_ex` bit for bit against the oracle's `LCMScheduler.step` of a configured
scheduler, for every prediction type x clamp on / off x last / non-last step; `dl_lcm_step` and
`dl_lcm_step_inpaint` unchanged (equal to the epsilon instantiation and to the oracle).  Operands sit inside
NaN-filled buffers: nothing outside them is read or written."""
import pytest
import torch

pytestmark = pytest.mark.gpu

PREDS = ["epsilon", "v_prediction", "sample"]


@pytest.fixture(scope="module")
def lib():
    from dreamlab_b200 import lib as L
    L.load()
    return L


def _config(pred, clip):
    d = {"prediction_type": pred}
    if pred != "epsilon":
        d["rescale_betas_zero_snr"] = True          # covers a_t = 0 at t = 999
    if clip is not None:
        d.update(clip_sample=True, clip_sample_range=clip)
    return d


def _padded(t):
    if t is None:
        return None
    b = torch.full((t.numel() + 32,), float("nan"), device="cuda")
    b[:t.numel()] = t.reshape(-1).cuda()
    return b[:t.numel()].view(t.shape)


def _out(shape):
    n = 1
    for s in shape:
        n *= s
    return torch.full((n + 8,), float("nan"), device="cuda"), n


@pytest.mark.parametrize("pred", PREDS)
@pytest.mark.parametrize("clip", [None, 1.0])
@pytest.mark.parametrize("steps", [1, 4])
def test_lcm_step_ex_bit_exact_vs_oracle(lib, pred, clip, steps):
    from dreamlab_b200.scheduler import LCMSchedule, SchedulerConfig
    from oracle.lcm_config import OracleLCMSchedulerConfigured
    d = _config(pred, clip)
    osch = OracleLCMSchedulerConfigured.from_config(d)
    ts = osch.set_timesteps(steps)
    sch = LCMSchedule(steps, config=SchedulerConfig.from_dict(d))
    assert sch.timesteps == ts.tolist()
    shape = (2, 4, 24, 40)
    x = 1.5 * torch.randn(*shape, generator=torch.Generator().manual_seed(5))
    clamped = 0
    for i, t in enumerate(ts):
        mo = 1.5 * torch.randn(*shape, generator=torch.Generator().manual_seed(10 + i))
        z = torch.randn(*shape, generator=torch.Generator().manual_seed(20 + i)) if i < steps - 1 else None
        ref_prev, ref_den = osch.step(mo, int(t), x, noise=z)
        xn, N = _out(shape)
        dn, _ = _out(shape)
        lib.lcm_step_ex(_padded(mo), _padded(x), _padded(z), xn[:N].view(shape), dn[:N].view(shape), sch.coeffs(i),
                        sch.prediction_type, sch.clip_range)
        torch.cuda.synchronize()
        got_prev, got_den = xn[:N].view(shape).cpu(), dn[:N].view(shape).cpu()
        assert not torch.isnan(got_prev).any() and not torch.isnan(got_den).any()
        assert torch.equal(got_prev, ref_prev), f"prev_sample {pred} clip={clip} i={i}"
        assert torch.equal(got_den, ref_den), f"denoised {pred} clip={clip} i={i}"
        assert torch.isnan(xn[N:]).all() and torch.isnan(dn[N:]).all()
        if clip is not None:           # the clamp must have bitten, or this case tests nothing
            free = OracleLCMSchedulerConfigured.from_config({**d, "clip_sample": False})
            free.set_timesteps(steps)
            free.set_begin_index(i)
            clamped += int(not torch.equal(free.step(mo, int(t), x, noise=z)[1], ref_den))
        if pred == "epsilon" and clip is None:
            xo, do = torch.empty(shape, device="cuda"), torch.empty(shape, device="cuda")
            lib.lcm_step(mo.cuda(), x.cuda(), None if z is None else z.cuda(), xo, do, sch.coeffs(i))
            torch.cuda.synchronize()
            assert torch.equal(xo.cpu(), ref_prev) and torch.equal(do.cpu(), ref_den)
        x = ref_prev
    if clip is not None:
        assert clamped == steps


def test_lcm_step_unchanged_and_equal_to_epsilon_ex(lib):
    """dl_lcm_step on the default schedule: the same bits as its epsilon instantiation through dl_lcm_step_ex."""
    from dreamlab_b200.scheduler import LCMSchedule
    sch = LCMSchedule(4)
    g = torch.Generator().manual_seed(3)
    eps, x, z = (torch.randn(3, 64, 64, 4, generator=g).cuda() for _ in range(3))
    for i in range(4):
        zi = z if sch.has_noise(i) else None
        a, b, c, d = (torch.empty_like(x) for _ in range(4))
        lib.lcm_step(eps, x, zi, a, b, sch.coeffs(i))
        lib.lcm_step_ex(eps, x, zi, c, d, sch.coeffs(i), "epsilon", None)
        torch.cuda.synchronize()
        assert torch.equal(a.view(torch.int32), c.view(torch.int32)) and torch.equal(b.view(torch.int32),
                                                                                    d.view(torch.int32))


def test_lcm_step_ex_refuses_unknown_prediction_type(lib):
    x = torch.zeros(16, device="cuda")
    with pytest.raises(RuntimeError, match="prediction_type"):
        lib.lcm_step_ex(x, x, None, x.clone(), x.clone(), (1, 0, 0, 1, 1, 0), "flow")


@pytest.mark.parametrize("pred", PREDS)
@pytest.mark.parametrize("clip", [None, 1.0])
@pytest.mark.parametrize("step", [0, 3])
def test_lcm_step_inpaint_ex_bit_exact_vs_oracle(lib, pred, clip, step):
    """The oracle's configured step, then the 4-channel blend with the pipeline's op order (`run_pipeline_inpaint`):
    (1 - m) * add_noise(image_latents, noise0, t_{i+1}) + m * prev; image_latents itself after the last step."""
    from dreamlab_b200.scheduler import LCMSchedule, SchedulerConfig
    from oracle.lcm_config import OracleLCMSchedulerConfigured
    d = _config(pred, clip)
    sched = LCMSchedule(4, 1.0, truncate=True, config=SchedulerConfig.from_dict(d))
    osch = OracleLCMSchedulerConfigured.from_config(d)
    ts = osch.set_timesteps(4)
    osch.set_begin_index(step)
    last = step == len(sched.timesteps) - 1
    n, h, w = 2, 8, 6
    g = torch.Generator().manual_seed(10 + step)
    mo, x, z, img, z0 = (1.5 * torch.randn(n, h, w, 4, generator=g) for _ in range(5))
    m = (torch.rand(n, h, w, generator=g) > 0.5).float()
    m[0] = torch.rand(h, w, generator=g)                     # fractional mask values in one image
    z = None if last else z
    ref_prev, ref_den = osch.step(mo, int(ts[step]), x, noise=z)
    proper = img if last else osch.add_noise(img, z0, ts[step + 1])
    want = (1 - m[..., None]) * proper + m[..., None] * ref_prev
    an = (1.0, 0.0) if last else sched.add_noise_coeffs(sched.timesteps[step + 1])
    xn, N = _out((n, h, w, 4))
    den, _ = _out((n, h, w, 4))
    lib.lcm_step_inpaint_ex(_padded(mo), _padded(x), _padded(z), _padded(img), None if last else _padded(z0),
                            _padded(m), xn[:N].view(n, h, w, 4), den[:N].view(n, h, w, 4), sched.coeffs(step), an,
                            last, sched.prediction_type, sched.clip_range)
    torch.cuda.synchronize()
    got = xn[:N].view(n, h, w, 4).cpu()
    assert not torch.isnan(got).any()
    assert torch.equal(got, want)
    assert torch.equal(den[:N].view(n, h, w, 4).cpu(), ref_den)
    assert torch.isnan(xn[N:]).all() and torch.isnan(den[N:]).all()
    if pred == "epsilon" and clip is None:                   # dl_lcm_step_inpaint: the same bits
        a, b = torch.empty(N, device="cuda"), torch.empty(N, device="cuda")
        lib.lcm_step_inpaint(mo.cuda(), x.cuda(), None if z is None else z.cuda(), img.cuda(),
                             None if last else z0.cuda(), m.cuda(), a.view(n, h, w, 4), b.view(n, h, w, 4),
                             sched.coeffs(step), an, last)
        torch.cuda.synchronize()
        assert torch.equal(a.view(n, h, w, 4).cpu(), got) and torch.equal(b.view(n, h, w, 4).cpu(), ref_den)
