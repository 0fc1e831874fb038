"""Kernel-level parity of the image-to-image entry points (csrc/img2img.cu, the pad-0 stride-2 im2col) against
numpy / torch restatements on the same inputs.  NaN sentinels around the outputs (and, for the image, canvas
pixels outside the tile window) show that nothing outside the described operands is read or written.
The fp32 outputs reach `dl_pack_image_im2col_f32` and `dl_im2col_s2_pad01_f32` through the dtype-dispatching
bindings, the bf16 ones `dl_pack_image_im2col` and `dl_im2col_s2_pad01`."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda"
NAN = float("nan")


def L():
    import dreamlab_b200.lib as lib
    lib.load()
    return lib


def image_im2col_ref(img):
    """numpy restatement: u8 [n,h,w,3] -> fp32 [n*h*w, 64], K = (ky*3+kx)*3 + c, 2*(u/255)-1, zero padding."""
    n, h, w, _ = img.shape
    x = (2.0 * (img.astype(np.float32) / np.float32(255.0)) - np.float32(1.0)).astype(np.float32)
    xp = np.zeros((n, h + 2, w + 2, 3), np.float32)
    xp[:, 1:h + 1, 1:w + 1] = x
    out = np.zeros((n, h, w, 64), np.float32)
    for ky in range(3):
        for kx in range(3):
            t = ky * 3 + kx
            out[..., 3 * t:3 * t + 3] = xp[:, ky:ky + h, kx:kx + w]
    return out.reshape(n * h * w, 64)


def _sentinel_out(rows, dtype):
    buf = torch.full((rows + 2, 64), NAN, device=DEV, dtype=dtype)
    return buf, buf[1:rows + 1]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("n,h,w", [(2, 16, 24), (1, 9, 5), (3, 1, 1)])
def test_pack_image_im2col_whole_image(dtype, n, h, w):
    lib = L()
    g = np.random.default_rng(h * 100 + w)
    img = g.integers(0, 256, size=(n, h, w, 3), dtype=np.uint8)
    img[0, 0, 0] = (0, 255, 128)                                   # the extremes of the range
    ref = torch.from_numpy(image_im2col_ref(img))
    buf, out = _sentinel_out(n * h * w, dtype)
    lib.pack_image_im2col(torch.from_numpy(img).to(DEV), out)
    torch.cuda.synchronize()
    assert torch.isnan(buf[0]).all() and torch.isnan(buf[-1]).all()
    want = ref if dtype == torch.float32 else ref.to(torch.bfloat16)           # round to nearest even
    assert torch.equal(out.cpu(), want)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_pack_image_im2col_tile_window(dtype):
    """A tile window inside a larger canvas, read in place: its border taps are zero, not the canvas' pixels."""
    lib = L()
    g = np.random.default_rng(7)
    canvas = g.integers(0, 256, size=(2, 40, 48, 3), dtype=np.uint8)
    y0, x0, th, tw = 8, 16, 24, 16
    tile = np.ascontiguousarray(canvas[:, y0:y0 + th, x0:x0 + tw])
    ref = torch.from_numpy(image_im2col_ref(tile))
    dev = torch.from_numpy(canvas).to(DEV)
    buf, out = _sentinel_out(2 * th * tw, dtype)
    lib.pack_image_im2col(dev[:, y0:y0 + th, x0:x0 + tw], out)
    torch.cuda.synchronize()
    assert torch.isnan(buf[0]).all() and torch.isnan(buf[-1]).all()
    want = ref if dtype == torch.float32 else ref.to(torch.bfloat16)
    assert torch.equal(out.cpu(), want)
    # the first pixel's up-left tap is zero although the canvas has a pixel there (2*(u/255)-1 != 0 for any u8)
    assert float(out[0, 0]) == 0.0


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("n,h,w,c", [(2, 8, 12, 16), (1, 6, 4, 64), (1, 2, 2, 8)])
def test_im2col_s2_pad01_bit_exact(dtype, n, h, w, c):
    """F.pad(x, (0,1,0,1)) + unfold(3, stride 2): the last row and column of taps read the zero pad."""
    lib = L()
    if dtype == torch.float32 and c % 4 or dtype == torch.bfloat16 and c % 8:
        pytest.skip("channel vector width")
    x = torch.randn(n, h, w, c, generator=torch.Generator().manual_seed(c)).to(dtype)
    xp = F.pad(x.float().permute(0, 3, 1, 2), (0, 1, 0, 1))
    u = F.unfold(xp, 3, stride=2)                                   # [n, c*9, L], index c*9 + tap
    ho, wo = h // 2, w // 2
    ref = u.view(n, c, 9, ho * wo).permute(0, 3, 2, 1).reshape(n * ho * wo, 9 * c).to(dtype)
    buf = torch.full((n * ho * wo + 2, 9 * c), NAN, device=DEV, dtype=dtype)
    cols = buf[1:-1]
    lib.im2col_s2_pad01(x.to(DEV), cols, nimg=n, h=h, w=w)
    torch.cuda.synchronize()
    assert torch.isnan(buf[0]).all() and torch.isnan(buf[-1]).all()
    assert torch.equal(cols.cpu(), ref)
    # the UNet's symmetric-pad form is a different gather on the same input
    cols1 = torch.empty_like(cols)
    lib.im2col_s2(x.to(DEV), cols1, nimg=n, h=h, w=w)
    torch.cuda.synchronize()
    assert not torch.equal(cols1, cols)


def _sample_inputs(n, h, w, seed, lv_scale=3.0):
    g = torch.Generator().manual_seed(seed)
    mom = torch.randn(n, h, w, 8, generator=g)
    mom[..., 4:] *= lv_scale
    return mom, torch.randn(n, 4, h, w, generator=g), torch.randn(n, 4, h, w, generator=g)


def _sample_ref(mom, es, en, sf, sa, sb):
    mean = mom[..., :4].permute(0, 3, 1, 2)
    lv = torch.clamp(mom[..., 4:].permute(0, 3, 1, 2), -30.0, 20.0)
    std = torch.exp(0.5 * lv)
    x0 = sf * (mean + std * es)
    return (sa * x0 + sb * en).permute(0, 2, 3, 1)


def _run_sample(mom, es, en, sf, sa, sb, with_mean=True):
    lib = L()
    n, h, w, _ = mom.shape
    buf = torch.full((n * h * w * 4 + 2,), NAN, device=DEV)
    out = buf[1:-1].view(n, h, w, 4)
    mbuf = torch.full((n * h * w * 4 + 2,), NAN, device=DEV)
    mean = mbuf[1:-1].view(n, h, w, 4)
    lib.vae_sample_latents(mom.to(DEV), es.to(DEV), en.to(DEV), out, scaling_factor=sf, sqrt_alpha=sa,
                           sqrt_one_minus_alpha=sb, mean_out=mean if with_mean else None)
    torch.cuda.synchronize()
    assert torch.isnan(buf[0]) and torch.isnan(buf[-1]) and torch.isnan(mbuf[0]) and torch.isnan(mbuf[-1])
    return out.cpu(), mean.cpu()


def test_vae_sample_latents_bit_exact_without_posterior_noise():
    from dreamlab_b200.scheduler import LCMSchedule
    mom, _, en = _sample_inputs(2, 8, 12, 1)
    es = torch.zeros(2, 4, 8, 12)
    sa, sb = LCMSchedule(4, 0.5).add_noise_coeffs()
    got, mean = _run_sample(mom, es, en, 0.18215, sa, sb)
    assert torch.equal(got, _sample_ref(mom, es, en, 0.18215, sa, sb))
    assert torch.equal(mean, mom[..., :4])


def test_vae_sample_latents_against_float64():
    mom, es, en = _sample_inputs(3, 16, 8, 2)
    sa, sb = 0.5269435048103333, 0.8499003052711487
    got, _ = _run_sample(mom, es, en, 0.13025, sa, sb, with_mean=False)
    ref = _sample_ref(mom.double(), es.double(), en.double(), 0.13025, sa, sb)
    err = (got.double() - ref).abs().max().item()
    bar = 1e-6 * ref.abs().max().item()
    print(f"vae_sample_latents vs float64: max|d| {err:.3e} (bar {bar:.3e})")
    assert err <= bar


def test_vae_sample_latents_clamps_logvar():
    mom, es, en = _sample_inputs(1, 4, 4, 3)
    mom[..., 4:6] = 80.0                       # above 20: std = exp(10)
    mom[..., 6:8] = -500.0                     # below -30: std = exp(-15)
    got, _ = _run_sample(mom, es, en, 1.0, 1.0, 0.0)
    ref = _sample_ref(mom.double(), es.double(), en.double(), 1.0, 1.0, 0.0)
    assert torch.isfinite(got).all()
    assert ((got.double() - ref).abs().max() / ref.abs().max()).item() <= 1e-6
    hi = mom[..., 0] + np.exp(10.0) * es[:, 0]
    assert torch.allclose(got[..., 0].double(), hi.double(), rtol=1e-6)
