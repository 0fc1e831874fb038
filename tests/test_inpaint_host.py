"""Inpainting, host side: the truncated schedule (`get_timesteps` on the full `set_timesteps(n)` schedule), the
per-request draw order of the worker, the pool's batch key, mask parsing, single-file `in_channels`, and the
parameter count of the 9-channel SD1.5 UNet."""
import io
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from dreamlab_b200 import single_file as sf
from dreamlab_b200 import synthetic as syn
from dreamlab_b200.scheduler import LCMSchedule, lcm_timesteps


def _oracle_coeffs(n, strength):
    """(timesteps, coefficient tuples) of the oracle's full schedule stepped from its begin index."""
    from oracle.inpaint import OracleLCMSchedulerInpaint, get_timesteps
    s = OracleLCMSchedulerInpaint()
    full = s.set_timesteps(n)
    ts, k = get_timesteps(s, n, strength)
    if k < 1:
        raise ValueError("no step")
    out = []
    for i, t in enumerate(ts.tolist()):
        j = s._step_index + i
        prev = int(full[j + 1]) if j + 1 < n else t
        a_t, a_p = s.alphas_cumprod[t], s.alphas_cumprod[prev]
        c_skip, c_out = s.boundary_scalings(t)
        out.append((a_t.sqrt().item(), (1 - a_t).sqrt().item(), c_skip.item(), c_out.item(), a_p.sqrt().item(),
                    (1 - a_p).sqrt().item()))
    return ts.tolist(), out, n - k


@pytest.mark.parametrize("n", [1, 2, 4, 8])
@pytest.mark.parametrize("strength", [1.0, 0.8, 0.5, 0.3])
def test_truncated_schedule_matches_oracle(n, strength):
    if int(n * strength) == 0:                       # diffusers: "num_inference_steps < 1" -> ValueError
        with pytest.raises(ValueError):
            LCMSchedule(n, strength, truncate=True)
        with pytest.raises(ValueError):
            _oracle_coeffs(n, strength)
        return
    ts, coeffs, t_start = _oracle_coeffs(n, strength)
    s = LCMSchedule(n, strength, truncate=True)
    assert s.timesteps == ts == lcm_timesteps(n)[t_start:]
    assert s.begin_index == t_start
    assert [s.coeffs(i) for i in range(len(ts))] == coeffs
    # a noise draw at every step but the last one (full index n - 1)
    assert [s.has_noise(i) for i in range(len(ts))] == [True] * (len(ts) - 1) + [False]
    for t in ts:
        from oracle.inpaint import OracleLCMSchedulerInpaint
        a = OracleLCMSchedulerInpaint().alphas_cumprod[t]
        assert s.add_noise_coeffs(t) == ((a ** 0.5).item(), ((1 - a) ** 0.5).item())
    assert s.add_noise_coeffs() == s.add_noise_coeffs(ts[0])


def test_truncated_schedule_examples_and_full_strength():
    assert LCMSchedule(4, 0.5, truncate=True).timesteps == [499, 259]
    assert LCMSchedule(8, 0.3, truncate=True).timesteps == [259, 139]
    with pytest.raises(ValueError):
        LCMSchedule(4, 0.2, truncate=True)                      # int(0.8) = 0
    for n in (1, 4, 8, 50):                                      # strength 1: the text-to-image schedule
        a, b = LCMSchedule(n), LCMSchedule(n, 1.0, truncate=True)
        assert a.timesteps == b.timesteps and [a.coeffs(i) for i in range(n)] == [b.coeffs(i) for i in range(n)]


def _worker(in_channels):
    from backends.b200_worker import B200Worker
    w = object.__new__(B200Worker)
    w.device, w.dtype = "cpu", torch.float32
    w.pipe = SimpleNamespace(unet=SimpleNamespace(cfg=SimpleNamespace(in_channels=in_channels)))
    return w


@pytest.mark.parametrize("in_channels,strength,want_posterior,want_steps", [
    (4, 1.0, True, 4), (4, 0.5, True, 2), (9, 1.0, False, 4), (9, 0.5, True, 2)])
def test_draw_order(in_channels, strength, want_posterior, want_steps):
    """diffusers' order with one generator per request: the image's posterior draw (only where the image is encoded),
    the latents / add_noise draw, the masked image's posterior draw (always), one draw per non-final step of the
    truncated schedule."""
    w = _worker(in_channels)
    k, posterior = w._inpaint_plan(4, strength)
    assert (k, posterior) == (want_steps, want_posterior)
    lat, noise, eps_s, eps_m = w._draw(7, 2, 3, k, posterior=posterior, masked=True)
    g = torch.Generator().manual_seed(7)
    seq = [torch.randn(1, 4, 2, 3, generator=g) for _ in range(2 + int(posterior) + k - 1)]
    want = ([seq.pop(0)] if posterior else [None]) + seq
    assert (eps_s is None) == (not posterior)
    if posterior:
        assert torch.equal(eps_s, want[0])
    assert torch.equal(lat, want[1]) and torch.equal(eps_m, want[2])
    assert len(noise) == k - 1 and all(torch.equal(a, b) for a, b in zip(noise, want[3:]))


def test_draw_order_without_mask_is_unchanged():
    w = _worker(4)
    g = torch.Generator().manual_seed(3)
    seq = [torch.randn(1, 4, 2, 2, generator=g) for _ in range(4)]
    lat, noise, eps_s = w._draw(3, 2, 2, 3, posterior=True)
    assert torch.equal(eps_s, seq[0]) and torch.equal(lat, seq[1]) and all(torch.equal(a, b) for a, b in zip(noise, seq[2:]))


def test_batch_key_separates_inpainting():
    from backends.worker_pool import _batch_key

    def j(**kw):
        return SimpleNamespace(req=SimpleNamespace(prompt="p", size="512x512", num_inference_steps=4,
                                                   guidance_scale=1.0, **kw))
    t2i = _batch_key(j())
    i2i = _batch_key(j(init_image=b"png", strength=0.5))
    a = _batch_key(j(init_image=b"png", mask_image=b"m", strength=0.5))
    assert a == t2i + (("inpaint", 0.5),) and a != i2i
    assert _batch_key(j(init_image=b"png", mask_image=b"m")) == t2i + (("inpaint", 1.0),)     # default strength 1.0
    assert _batch_key(j(init_image=b"x", mask_image=b"other", strength=0.5)) == a
    assert _batch_key(j(init_image=b"png", mask_image=b"m", strength=0.6)) != a
    assert _batch_key(j(init_image=b"png", mask_image=b"m", strength=0.5), same_guidance=True) == a + (1.0,)


def test_genspec_and_mask_parsing():
    from PIL import Image
    from backends.b200_worker import B200Worker
    from backends.base import GenSpec
    assert GenSpec(prompt="p", size="64x64", steps=4, cfg=1.0).mask_image is None
    g = GenSpec(prompt="p", size="64x64", steps=4, cfg=1.0, init_image=b"i", mask_image=b"m", strength=0.5)
    assert g.mask_image == b"m" and g.init_image == b"i" and g.strength == 0.5
    m = (np.arange(16 * 24).reshape(16, 24) % 256).astype(np.uint8)
    buf = io.BytesIO()
    Image.fromarray(m).save(buf, format="PNG")
    assert np.array_equal(B200Worker._mask_image(buf.getvalue(), 24, 16), m)
    assert np.array_equal(B200Worker._mask_image(m, 24, 16), m)
    rgb = np.stack([m] * 3, -1)
    buf = io.BytesIO()
    Image.fromarray(rgb).save(buf, format="PNG")
    assert np.array_equal(B200Worker._mask_image(buf.getvalue(), 24, 16), m)        # RGB bytes -> "L"
    with pytest.raises(RuntimeError, match="not resized"):
        B200Worker._mask_image(m, 16, 24)
    with pytest.raises(RuntimeError, match="uint8"):
        B200Worker._mask_image(m.astype(np.float32), 24, 16)
    with pytest.raises(RuntimeError, match="uint8"):
        B200Worker._mask_image(rgb, 24, 16)


def test_sdxl_worker_refuses_inpainting():
    from backends.b200_worker import B200SDXLWorker
    with pytest.raises(RuntimeError, match="SDXL"):
        object.__new__(B200SDXLWorker)._check_inpaint()


def test_load_single_file_reads_in_channels(tmp_path):
    """A 9-channel inpainting checkpoint (all other tensors shrunk: only the probed shapes matter to the loader)."""
    from safetensors.torch import save_file
    from test_single_file import _invert, _ns
    for cin in (4, 9):
        ucfg = {**sf.SD15_UNET, "in_channels": cin}
        shapes = syn.unet_shapes(_ns(ucfg))
        um = sf.unet_module_map(ucfg)
        out = {}
        for k, s in shapes.items():
            keep = k == "conv_in.weight" or k.endswith("attn2.to_k.weight")
            out[_invert(k, um, sf._RESNET, sf.UNET_PREFIX)] = torch.zeros(s if keep else (1,), dtype=torch.float16)
        p = str(tmp_path / f"sd15_{cin}.safetensors")
        save_file(out, p)
        got = sf.load_single_file(p)
        assert got["unet"][0]["in_channels"] == cin
        assert tuple(got["unet"][1]["conv_in.weight"].shape) == (320, cin, 3, 3)


def test_nine_channel_sd15_unet_parameter_count():
    """4-channel count + 5 * 320 * 9 for conv_in (meta device: no memory)."""
    from oracle.unet import OracleUNet, UNetConfig
    with torch.device("meta"):
        plain = OracleUNet(UNetConfig(in_channels=9, time_cond_proj_dim=None))
        lcm = OracleUNet(UNetConfig(in_channels=9))
        four = OracleUNet(UNetConfig(time_cond_proj_dim=None))
    n = lambda m: sum(p.numel() for p in m.parameters())       # noqa: E731
    assert n(plain) == 859_535_364 and n(lcm) == 859_617_284
    assert n(plain) - n(four) == 5 * 320 * 9
    assert {k: tuple(v.shape) for k, v in plain.state_dict().items()} == \
        syn.unet_shapes(SimpleNamespace(**{**syn.sd15_lcm_unet_cfg().__dict__, "in_channels": 9, "time_cond_proj_dim": None}))


def test_oracle_mask_preprocessing():
    from oracle.inpaint import preprocess_mask
    import torch.nn.functional as F
    m = np.array([[[0, 127, 128, 255] * 4] * 16], dtype=np.uint8)          # [1, 16, 16]
    p = preprocess_mask(m)
    assert p.shape == (1, 1, 16, 16) and p.unique().tolist() == [0.0, 1.0]
    assert p[0, 0, 0, :4].tolist() == [0.0, 0.0, 1.0, 1.0]
    # nearest downsample takes pixel (8i, 8j)
    assert F.interpolate(p, size=(2, 2))[0, 0].tolist() == [[0.0, 0.0], [0.0, 0.0]]
    m[0, 8, 8] = 200
    assert F.interpolate(preprocess_mask(m), size=(2, 2))[0, 0].tolist() == [[0.0, 0.0], [0.0, 1.0]]
