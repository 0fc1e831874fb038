"""Inpainting side kernels, bit for bit: `dl_pack_image_im2col_masked` / `dl_pack_image_im2col_masked_f32` against
`dl_pack_image_im2col` of the same image with the masked taps zeroed on the host, `dl_inpaint_latent_mask` against
F.interpolate(nearest) of the binarised mask, `dl_pack_latent_inpaint` / `dl_pack_latent_inpaint_f32` against the host
concat, and `dl_lcm_step_inpaint` against the
same sequence of fp32 roundings on the host.  Operands sit inside NaN-filled buffers: nothing outside them is read
(a NaN would reach the result) or written (the sentinels would change)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib():
    from dreamlab_b200 import lib as L
    L.load()
    return L


def _masks(n, h, w, seed=0):
    g = np.random.default_rng(seed)
    cb = np.where((np.add.outer(np.arange(h), np.arange(w)) % 2) == 0, 127, 128).astype(np.uint8)
    return {"zero": np.zeros((n, h, w), np.uint8), "full": np.full((n, h, w), 255, np.uint8),
            "random": g.integers(0, 256, size=(n, h, w), dtype=np.uint8), "checker": np.stack([cb] * n)}


def _host_masked_cols(cols, mask):
    """Zero the im2col entries (k < 27) whose source pixel is masked (m >= 128); cols [n*h*w, 64]."""
    n, h, w = mask.shape
    m = torch.from_numpy(mask >= 128)
    mp = F.pad(m, (1, 1, 1, 1))                                   # out-of-window taps are zero padding anyway
    out = cols.clone().view(n, h, w, 64)
    for tap in range(9):
        dy, dx = tap // 3, tap % 3
        hit = mp[:, dy:dy + h, dx:dx + w].to(out.device)
        for c in range(3):
            out[..., tap * 3 + c][hit] = 0
    return out.view(n * h * w, 64)


@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("kind", ["zero", "full", "random", "checker"])
def test_masked_im2col_matches_host_masked(lib, dt, kind):
    n, h, w = 2, 24, 40
    img = torch.from_numpy(np.random.default_rng(1).integers(0, 256, size=(n, h, w, 3), dtype=np.uint8)).cuda()
    mask = _masks(n, h, w)[kind]
    plain = torch.empty(n * h * w, 64, device="cuda", dtype=dt)
    lib.pack_image_im2col(img, plain)
    buf = torch.full((n * h * w + 5, 64), float("nan"), device="cuda", dtype=dt)
    lib.pack_image_im2col(img, buf[:n * h * w], mask=torch.from_numpy(mask).cuda())
    torch.cuda.synchronize()
    want = _host_masked_cols(plain, mask)
    got = buf[:n * h * w]
    assert torch.equal(got.float().view(torch.int32), want.float().view(torch.int32)), kind
    assert torch.isnan(buf[n * h * w:].float()).all()
    if kind == "zero":
        assert torch.equal(got, plain)


@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float32])
def test_masked_im2col_tile_window_in_place(lib, dt):
    """A tile window of the canvas and of the mask, read in place at the canvas' strides (tiled encode)."""
    n, H, W = 2, 48, 64
    g = np.random.default_rng(3)
    canvas = torch.from_numpy(g.integers(0, 256, size=(n, H, W, 3), dtype=np.uint8)).cuda()
    mcanvas = torch.from_numpy(_masks(n, H, W, seed=4)["random"]).cuda()
    win, mwin = canvas[:, 8:32, 16:56], mcanvas[:, 8:32, 16:56]
    h, w = 24, 40
    a = torch.empty(n * h * w, 64, device="cuda", dtype=dt)
    b = torch.empty_like(a)
    plain = torch.empty_like(a)
    lib.pack_image_im2col(win, a, mask=mwin)
    lib.pack_image_im2col(win.contiguous(), b, mask=mwin.contiguous())
    lib.pack_image_im2col(win.contiguous(), plain)
    torch.cuda.synchronize()
    assert torch.equal(a, b)
    want = _host_masked_cols(plain, mwin.cpu().numpy())
    assert torch.equal(a.float().view(torch.int32), want.float().view(torch.int32))


def test_masked_im2col_refuses_bad_mask(lib):
    img = torch.zeros(1, 16, 16, 3, device="cuda", dtype=torch.uint8)
    out = torch.empty(256, 64, device="cuda", dtype=torch.bfloat16)
    with pytest.raises(RuntimeError, match="mask"):
        lib.pack_image_im2col(img, out, mask=torch.zeros(1, 16, 8, device="cuda", dtype=torch.uint8))
    with pytest.raises(RuntimeError, match="mask"):
        lib.pack_image_im2col(img, out, mask=torch.zeros(1, 16, 16, device="cuda", dtype=torch.float32))


def test_inpaint_latent_mask_is_nearest_of_binarised(lib):
    n, h, w = 3, 8, 6
    for kind, m in _masks(n, 8 * h, 8 * w, seed=7).items():
        mt = torch.from_numpy(m).cuda()
        buf = torch.full((n * h * w + 9,), float("nan"), device="cuda")
        lib.inpaint_latent_mask(mt, buf[:n * h * w].view(n, h, w))
        torch.cuda.synchronize()
        x = torch.from_numpy(m).float() / 255.0
        b = torch.where(x < 0.5, torch.zeros_like(x), torch.ones_like(x))[:, None]
        want = F.interpolate(b, size=(h, w))[:, 0]
        assert torch.equal(buf[:n * h * w].view(n, h, w).cpu(), want), kind
        assert torch.isnan(buf[n * h * w:]).all()


@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("repeat", [1, 2])
def test_pack_latent_inpaint(lib, dt, repeat):
    n, h, w = 2, 8, 6
    g = torch.Generator().manual_seed(5)
    lat = torch.randn(n, h, w, 4, generator=g)
    mask = (torch.rand(n, h, w, generator=g) > 0.5).float()
    masked = torch.randn(n, h, w, 4, generator=g)
    npix = n * h * w

    def padded(t):          # operand followed by NaNs
        b = torch.full((t.numel() + 16,), float("nan"), device="cuda")
        b[:t.numel()] = t.reshape(-1).cuda()
        return b[:t.numel()].view(t.shape)
    out = torch.full((repeat * npix + 3, 64), float("nan"), device="cuda", dtype=dt)
    lib.pack_latent_inpaint(padded(lat), padded(mask), padded(masked), out[:repeat * npix], repeat=repeat)
    torch.cuda.synchronize()
    one = torch.cat([lat, mask[..., None], masked, torch.zeros(n, h, w, 55)], -1).reshape(npix, 64)
    want = torch.cat([one] * repeat).to(dt)
    got = out[:repeat * npix].cpu()
    assert torch.equal(got.float().view(torch.int32), want.float().view(torch.int32))
    assert torch.isnan(out[repeat * npix:].float()).all()


def _host_step(eps, x, z, img, z0, m, k, an, last):
    """The kernel's sequence of fp32 roundings, op by op on fp32 tensors."""
    f = lambda v: torch.tensor(v, dtype=torch.float32)               # noqa: E731
    sa_t, sb_t, c_skip, c_out, sa_p, sb_p = (f(v) for v in k)
    x0 = (x - sb_t * eps) / sa_t
    d = c_out * x0 + c_skip * x
    prev = sa_p * d + sb_p * z if z is not None else d
    proper = img if last else f(an[0]) * img + f(an[1]) * z0
    return (f(1.0) - m[..., None]) * proper + m[..., None] * prev, d


@pytest.mark.parametrize("step", [0, 1, 3])
@pytest.mark.parametrize("binary", [True, False])
def test_lcm_step_inpaint_bit_exact(lib, step, binary):
    from dreamlab_b200.scheduler import LCMSchedule
    sched = LCMSchedule(4, 1.0, truncate=True)
    last = step == len(sched.timesteps) - 1
    n, h, w = 2, 8, 6
    g = torch.Generator().manual_seed(10 + step)
    eps, x, z, img, z0 = (torch.randn(n, h, w, 4, generator=g) for _ in range(5))
    m = torch.rand(n, h, w, generator=g)
    if binary:
        m = (m > 0.5).float()
    z = None if last else z
    an = (1.0, 0.0) if last else sched.add_noise_coeffs(sched.timesteps[step + 1])

    def padded(t):
        if t is None:
            return None
        b = torch.full((t.numel() + 32,), float("nan"), device="cuda")
        b[:t.numel()] = t.reshape(-1).cuda()
        return b[:t.numel()].view(t.shape)
    xn = torch.full((n * h * w * 4 + 8,), float("nan"), device="cuda")
    den = torch.full_like(xn, float("nan"))
    N = n * h * w * 4
    lib.lcm_step_inpaint(padded(eps), padded(x), padded(z), padded(img), None if last else padded(z0), padded(m),
                         xn[:N].view(n, h, w, 4), den[:N].view(n, h, w, 4), sched.coeffs(step), an, last)
    torch.cuda.synchronize()
    want, want_d = _host_step(eps, x, z, img, z0, m, sched.coeffs(step), an, last)
    got = xn[:N].view(n, h, w, 4).cpu()
    assert not torch.isnan(got).any()
    assert torch.equal(got, want)                        # == : equal up to the sign of zero
    assert torch.equal(den[:N].view(n, h, w, 4).cpu(), want_d)
    assert torch.isnan(xn[N:]).all() and torch.isnan(den[N:]).all()
    if binary:
        # m = 0: the noised image latents (image_latents itself after the last step); m = 1: the plain LCM step
        out_plain, d_plain = torch.empty_like(xn[:N]), torch.empty_like(xn[:N])
        lib.lcm_step(eps.cuda(), x.cuda(), None if z is None else z.cuda(), out_plain, d_plain, sched.coeffs(step))
        torch.cuda.synchronize()
        keep = m == 1
        assert torch.equal(got[keep], out_plain.view(n, h, w, 4).cpu()[keep])
