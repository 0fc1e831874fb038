"""Inpainting on the device against the fp32 oracle (`oracle/inpaint.py`): 4- and 9-channel UNets teacher-forced per
step (with and without classifier-free guidance, untiled and tiled), the exact invariants of the 4-channel blend, CUDA
graph against eager, batches against single runs, and the b200 worker / pool behaviour for requests that carry a
mask."""
import io
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from test_img2img_gpu import BF16_TOL, FP32_TOL, _bar, _image, _png, job
from test_pipeline_gpu import guided_tol, max_rel_err, psnr_u8, teacher_inputs

pytestmark = pytest.mark.gpu

torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False


def _mask(n, h, w, seed=0):
    """A box to repaint per image, ragged edges of 127 / 128 values and a few stray pixels."""
    g = np.random.default_rng(seed)
    out = np.zeros((n, h, w), np.uint8)
    for i in range(n):
        y0, x0 = g.integers(0, h // 2), g.integers(0, w // 2)
        out[i, y0:y0 + h // 2, x0:x0 + w // 2] = 255
        out[i, y0, x0:x0 + w // 2] = 128
        out[i, y0 + h // 2 - 1, x0:x0 + w // 2] = 127
        out[i][g.random((h, w)) < 0.02] = 200
    return out


def _models(in_channels, lcm=True, full=False, vae_cfg=None):
    from oracle.img2img import build_random_init_img2img
    from oracle.unet import UNetConfig
    from oracle.vae import VAEConfig
    ucfg = UNetConfig(in_channels=in_channels) if full else UNetConfig.tiny()
    ucfg.in_channels = in_channels
    if not lcm:
        ucfg.time_cond_proj_dim = None
    return build_random_init_img2img(ucfg, vae_cfg or VAEConfig.tiny(), seed=0)


def _pipe(unet, vae, enc, precision="bf16", tiling=False):
    from dreamlab_b200.engine import LCMPipelineB200
    return LCMPipelineB200(unet.state_dict(), unet.cfg, {**vae.state_dict(), **enc.state_dict()}, vae.cfg, "cuda:0",
                           vae_tiling=tiling, precision=precision)


def _inputs(unet, B, H, W, steps, strength, seed=3000):
    from dreamlab_b200.scheduler import LCMSchedule
    from oracle.pipeline import synthetic_inputs
    k = len(LCMSchedule(steps, strength, truncate=True).timesteps)
    pe, _, _ = synthetic_inputs(B, H, W, steps, ctx_dim=unet.cfg.cross_attention_dim)
    es, en, em, noise = [], [], [], []
    for i in range(B):
        g = torch.Generator().manual_seed(seed + i)
        es.append(torch.randn(1, 4, H // 8, W // 8, generator=g))
        en.append(torch.randn(1, 4, H // 8, W // 8, generator=g))
        em.append(torch.randn(1, 4, H // 8, W // 8, generator=g))
        noise.append(torch.stack([torch.randn(1, 4, H // 8, W // 8, generator=g) for _ in range(k - 1)])
                     if k > 1 else torch.zeros(1, 1, 4, H // 8, W // 8))
    return pe, torch.cat(es), torch.cat(en), torch.cat(em), torch.cat(noise, 1), _image(B, H, W, seed=11), \
        _mask(B, H, W, seed=12)


def _kw(img, mask, es, em, strength):
    return dict(init_images=torch.from_numpy(img), mask_images=torch.from_numpy(mask), strength=strength,
                posterior_noise=es, masked_posterior_noise=em)


def _parity(unet, vae, enc, B, H, W, steps, strength, precision, gs=1.0, tiling=False):
    from oracle.inpaint import run_pipeline_inpaint
    pipe = _pipe(unet, vae, enc, precision, tiling)
    pe, es, en, em, noise, img, mask = _inputs(unet, B, H, W, steps, strength)
    rec_o, rec_c = {}, {}
    ref = run_pipeline_inpaint(unet, vae, enc, pe, img, mask, es, en, em, noise, steps, strength, gs, tiling=tiling,
                               record=rec_o)
    teacher = teacher_inputs(rec_o["init_latents"], rec_o["latents"])
    kw = _kw(img, mask, es, em, strength)
    pipe.generate(pe, en, noise, steps, gs, record=rec_c, teacher_latents=teacher, **kw)
    out = pipe.generate(pe, en, noise, steps, gs, **kw)
    torch.cuda.synchronize()
    assert torch.equal(rec_c["mask"].cpu(), rec_o["mask"])
    lat_errs = {k: max_rel_err(rec_c[k].cpu(), rec_o[k]) for k in ("init_latents", "image_latents",
                                                                   "masked_image_latents") if k in rec_c}
    errs = [max_rel_err(c.cpu(), o) for c, o in zip(rec_c["noise_pred"], rec_o["noise_pred"])]
    raw = [max_rel_err(c.cpu(), o) for c, o in zip(rec_c.get("noise_pred_raw", []), rec_o["noise_pred_raw"])]
    p = psnr_u8(out.cpu().numpy(), ref)
    return pipe, (pe, es, en, em, noise, img, mask), lat_errs, errs, raw, p, _bar(precision, enc, img, tiling)


@pytest.mark.parametrize("in_channels", [4, 9])
@pytest.mark.parametrize("precision,bar", [("bf16", BF16_TOL), ("fp32", FP32_TOL)])
def test_tiny_inpaint_parity(in_channels, precision, bar):
    unet, vae, enc = _models(in_channels)
    strength = 0.5 if in_channels == 4 else 1.0
    pipe, inp, lat, errs, _, p, mbar = _parity(unet, vae, enc, 2, 128, 128, 4, strength, precision)
    print(f"tiny inpaint {in_channels}ch {precision}: latents {lat} (bar {mbar:.2e}), teacher-forced noise_pred "
          f"{['%.2e' % e for e in errs]}, PSNR {p:.1f} dB")
    assert ("image_latents" in lat) == (in_channels == 4) and ("masked_image_latents" in lat) == (in_channels == 9)
    assert max(lat.values()) <= mbar and max(errs) <= bar and p >= 35.0
    if precision == "fp32":
        return
    # graph replay == eager, byte for byte; a batch equals its single runs; a batch of 3 pads to the 4-bucket
    pe, es, en, em, noise, img, mask = inp
    kw = _kw(img, mask, es, em, strength)
    eager = pipe.generate(pe, en, noise, 4, 1.0, **kw).clone()
    g = pipe.generate(pe, en, noise, 4, 1.0, use_graph=True, **kw).clone()
    torch.cuda.synchronize()
    assert torch.equal(g, eager)
    for i in range(2):
        one = pipe.generate(pe[i:i + 1], en[i:i + 1], noise[:, i:i + 1], 4, 1.0, use_graph=True,
                            **_kw(img[i:i + 1], mask[i:i + 1], es[i:i + 1], em[i:i + 1], strength)).clone()
        torch.cuda.synchronize()
        assert (one[0].int() - g[i].int()).abs().max() <= 1
    three = lambda t, d=0: torch.cat([t, t.narrow(d, 0, 1)], d)                 # noqa: E731
    img3, mask3 = np.concatenate([img, img[:1]]), np.concatenate([mask, mask[:1]])
    g3 = pipe.generate(three(pe), three(en), three(noise, 1), 4, 1.0, use_graph=True,
                       **_kw(img3, mask3, three(es), three(em), strength)).clone()
    torch.cuda.synchronize()
    assert g3.shape[0] == 3 and (g3[:2].int() - g[:2].int()).abs().max() <= 1
    other = pipe.generate(pe, en, noise, 4, 1.0, use_graph=True,
                          **_kw(img, 255 - mask, es, em, strength)).clone()
    torch.cuda.synchronize()
    assert not torch.equal(other, g)


def test_tiny_nine_channel_cfg_parity():
    """A 9-channel UNet without the LCM guidance embedding: classifier-free guidance at gs 4 on the doubled batch."""
    unet, vae, enc = _models(9, lcm=False)
    _, _, lat, errs, raw, p, mbar = _parity(unet, vae, enc, 2, 128, 128, 4, 0.5, "bf16", gs=4.0)
    print(f"tiny inpaint 9ch CFG 4: latents {lat}, raw noise_pred {['%.2e' % e for e in raw]}, guided "
          f"{['%.2e' % e for e in errs]}, PSNR {p:.1f} dB")
    assert max(lat.values()) <= mbar and max(raw) <= BF16_TOL and max(errs) <= guided_tol(4.0) and p >= 35.0


def test_tiny_four_channel_cfg_parity():
    unet, vae, enc = _models(4, lcm=False)
    _, _, lat, errs, raw, p, mbar = _parity(unet, vae, enc, 1, 128, 128, 4, 1.0, "bf16", gs=4.0)
    print(f"tiny inpaint 4ch CFG 4: latents {lat}, raw noise_pred {['%.2e' % e for e in raw]}, PSNR {p:.1f} dB")
    assert max(lat.values()) <= mbar and max(raw) <= BF16_TOL and max(errs) <= guided_tol(4.0) and p >= 35.0


def test_full_sd15_nine_channel_256_parity():
    from oracle.vae import VAEConfig
    unet, vae, enc = _models(9, full=True, vae_cfg=VAEConfig())
    _, _, lat, errs, _, p, _ = _parity(unet, vae, enc, 1, 256, 256, 2, 1.0, "bf16")
    print(f"full SD1.5 9ch inpaint 256^2 bf16: latents {lat}, teacher-forced noise_pred {['%.2e' % e for e in errs]}, "
          f"PSNR {p:.1f} dB")
    assert max(lat.values()) <= BF16_TOL and max(errs) <= BF16_TOL and p >= 35.0


@pytest.mark.parametrize("in_channels", [4, 9])
def test_tiled_inpaint_parity(in_channels):
    """Tiny VAE with sample_size 128: 192 x 256 encodes as tiles, the mask windows read in place."""
    unet, vae, enc = _models(in_channels)
    _, _, lat, errs, _, p, mbar = _parity(unet, vae, enc, 1, 192, 256, 4, 0.5, "bf16", tiling=True)
    print(f"tiled tiny inpaint {in_channels}ch 256x192: latents {lat} (bar {mbar:.2e}), noise_pred "
          f"{['%.2e' % e for e in errs]}, PSNR {p:.1f} dB")
    assert max(lat.values()) <= mbar and max(errs) <= BF16_TOL and p >= 35.0


def test_four_channel_blend_invariants():
    unet, vae, enc = _models(4)
    pipe = _pipe(unet, vae, enc)
    pe, es, en, em, noise, img, _ = _inputs(unet, 2, 128, 128, 4, 1.0)
    zero = np.zeros((2, 128, 128), np.uint8)
    rec = {}
    _, lat = pipe.generate(pe, en, noise, 4, 1.0, record=rec, return_latents=True, **_kw(img, zero, es, em, 1.0))
    torch.cuda.synchronize()
    # nothing to repaint: the final latents are the engine's own image latents, bit for bit
    assert torch.equal(lat.permute(0, 3, 1, 2).cpu(), rec["image_latents"].cpu())
    # everything repainted at strength 1: the text-to-image pass with the same latents and step noise
    full = np.full((2, 128, 128), 255, np.uint8)
    a = pipe.generate(pe, en, noise, 4, 1.0, **_kw(img, full, es, em, 1.0)).clone()
    b = pipe.generate(pe, en, noise, 4, 1.0).clone()
    torch.cuda.synchronize()
    assert torch.equal(a, b)


def test_default_strength_is_one():
    unet, vae, enc = _models(9)
    pipe = _pipe(unet, vae, enc)
    pe, es, en, em, noise, img, mask = _inputs(unet, 1, 64, 64, 2, 1.0)
    kw = _kw(img, mask, es, em, 1.0)
    a = pipe.generate(pe, en, noise, 2, 1.0, **kw).clone()
    kw.pop("strength")
    b = pipe.generate(pe, en, noise, 2, 1.0, **kw).clone()
    torch.cuda.synchronize()
    assert torch.equal(a, b)


def test_pipeline_refusals():
    from dreamlab_b200.engine import LCMPipelineB200
    unet, vae, enc = _models(9)
    pe, es, en, em, noise, img, mask = _inputs(unet, 1, 64, 64, 2, 1.0)
    pipe = LCMPipelineB200(unet.state_dict(), unet.cfg, vae.state_dict(), vae.cfg, "cuda:0")
    with pytest.raises(RuntimeError, match="encoder"):
        pipe.generate(pe, en, noise, 2, 1.0, **_kw(img, mask, es, em, 1.0))
    pipe = _pipe(unet, vae, enc)
    with pytest.raises(RuntimeError, match="in_channels=9"):                     # text-to-image on an inpainting UNet
        pipe.generate(pe, en, noise, 2, 1.0)
    with pytest.raises(RuntimeError, match="in_channels=9"):                     # image-to-image without a mask
        pipe.generate(pe, en, noise, 2, 1.0, init_images=torch.from_numpy(img), strength=0.5, posterior_noise=es)
    with pytest.raises(RuntimeError, match="init_images"):
        pipe.generate(pe, en, noise, 2, 1.0, mask_images=torch.from_numpy(mask), masked_posterior_noise=em)
    with pytest.raises(RuntimeError, match="mask_images"):
        pipe.generate(pe, en, noise, 2, 1.0, **_kw(img, mask[:, :32], es, em, 1.0))
    with pytest.raises(RuntimeError, match="mask_images"):
        pipe.generate(pe, en, noise, 2, 1.0, **_kw(img, mask.astype(np.int32), es, em, 1.0))
    with pytest.raises(RuntimeError, match="masked_posterior_noise"):
        pipe.generate(pe, en, noise, 2, 1.0, **{**_kw(img, mask, es, em, 1.0), "masked_posterior_noise": None})
    with pytest.raises(ValueError):
        pipe.generate(pe, en, noise, 4, 1.0, **_kw(img, mask, es, em, 0.2))
    with pytest.raises(RuntimeError, match="patch parallel"):
        x = torch.zeros(1, 8, 8, 4, device="cuda")
        pipe.unet.forward(x, None, None, comm=SimpleNamespace(), inpaint_cond=(x[..., 0], x))


# ------------------------------------------------------------------------------------------------ worker / pool
def _make_worker(root, name, in_channels, vae_encoder=True):
    from dreamlab_b200 import synthetic as S
    from oracle.unet import UNetConfig
    from oracle.vae import VAEConfig
    ucfg = UNetConfig.tiny()
    ucfg.cross_attention_dim = 768
    ucfg.in_channels = in_channels
    S.write_model_dir(str(root / name), ucfg, VAEConfig.tiny(), vae_encoder=vae_encoder)
    os.environ["MODEL_ROOT"], os.environ["MODEL"] = str(root), name
    os.environ.pop("CUDA_DEVICE", None)
    from backends.b200_worker import B200Worker
    return B200Worker(0)


@pytest.fixture(scope="module")
def workers(tmp_path_factory):
    root = tmp_path_factory.mktemp("models")
    return _make_worker(root, "tiny-inp4", 4), _make_worker(root, "tiny-inp9", 9)


def _mask_png(m):
    from PIL import Image
    buf = io.BytesIO()
    Image.fromarray(m).save(buf, format="PNG")
    return buf.getvalue()


@pytest.mark.parametrize("which", [0, 1])
def test_worker_inpaint(workers, which):
    from PIL import Image
    w = workers[which]
    init = _image(1, 128, 128, seed=21)[0]
    m = _mask(1, 128, 128, seed=22)[0]
    png, seed = w.run_job(job(seed=42, init_image=_png(init), mask_image=_mask_png(m), strength=0.5))
    assert png[:8] == b"\x89PNG\r\n\x1a\n" and seed == 42
    assert Image.open(io.BytesIO(png)).size == (128, 128)
    assert w.run_job(job(seed=42, init_image=init, mask_image=m, strength=0.5))[0] == png       # array forms
    assert w.run_job(job(seed=42, init_image=init, mask_image=m, strength=1.0))[0] != png       # another strength
    assert w.run_job(job(seed=42, init_image=init, mask_image=255 - m, strength=0.5))[0] != png  # another mask
    arr, _ = w.run_job_array(job(seed=42, init_image=init, mask_image=m, strength=0.5))
    assert np.array_equal(np.asarray(Image.open(io.BytesIO(png))), arr)
    png2, _, lat = w.run_job_with_latents(job(seed=42, init_image=init, mask_image=m, strength=0.5))
    assert png2 == png and len(lat) == 512
    lat_only, _ = w.run_job_latents(job(seed=42, init_image=init, mask_image=m, strength=0.5))
    assert lat_only.shape == (4, 16, 16)
    assert w.run_job(job(seed=42, init_image=init, mask_image=m))[0] == \
        w.run_job(job(seed=42, init_image=init, mask_image=m, strength=1.0))[0]                  # default 1.0


def test_worker_inpaint_refusals(workers, tmp_path):
    w4, w9 = workers
    init = _image(1, 128, 128)[0]
    m = _mask(1, 128, 128)[0]
    with pytest.raises(RuntimeError, match="init_image"):
        w4.run_job(job(mask_image=m))
    with pytest.raises(RuntimeError, match="not resized"):
        w4.run_job(job(init_image=init, mask_image=m[:64]))
    with pytest.raises(RuntimeError, match="uint8"):
        w4.run_job(job(init_image=init, mask_image=m.astype(np.float32)))
    with pytest.raises(RuntimeError, match="in_channels=9"):           # a 9-channel model refuses text-to-image
        w9.run_job(job())
    with pytest.raises(RuntimeError, match="in_channels=9"):
        w9.run_job(job(init_image=init))
    with pytest.raises(RuntimeError, match="share a batch"):
        w4.run_batch([job(init_image=init, mask_image=m), job(init_image=init)])
    w_noenc = _make_worker(tmp_path, "tiny-noenc", 4, vae_encoder=False)
    with pytest.raises(RuntimeError, match="encoder"):
        w_noenc.run_job(job(init_image=init, mask_image=m))


def test_pool_mixes_text_to_image_img2img_and_inpaint(workers):
    from unittest.mock import Mock
    from PIL import Image
    from backends.worker_pool import GenerationJob, WorkerPool
    w, _ = workers
    init = _image(1, 128, 128, seed=4)[0]
    m = _mask(1, 128, 128, seed=5)[0]
    kinds = [{}, {"init_image": init, "strength": 0.5}, {"init_image": init, "mask_image": m},
             {"init_image": init, "mask_image": m, "strength": 0.5}]
    jobs = [job(prompt=f"p{i}", seed=500 + i, **kinds[i % 4]) for i in range(8)]
    singles = [w.run_job(j) for j in jobs]
    cfg = Mock()
    cfg.config.model_root = os.environ["MODEL_ROOT"]
    cfg.get_mode.return_value = Mock(model=os.environ["MODEL"], model_path="x", loras=[])
    cfg.get_default_mode.return_value = "tiny"
    reg = Mock()
    reg.get_used_vram.return_value = 0
    pool = WorkerPool(queue_max=16, worker_factory=lambda worker_id: w, mode_config=cfg, registry=reg,
                      num_workers=1, max_batch=4)
    futs = [pool.submit_job(GenerationJob(req=j.req)) for j in jobs]
    res = [f.result(timeout=300) for f in futs]
    pool._workers = []
    pool.shutdown()
    for (pr, sr), (ps, ss) in zip(res, singles):
        assert sr == ss
        a = np.asarray(Image.open(io.BytesIO(pr))).astype(int)
        b = np.asarray(Image.open(io.BytesIO(ps))).astype(int)
        assert np.abs(a - b).max() <= 1
