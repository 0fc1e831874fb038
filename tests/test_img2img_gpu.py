"""Image-to-image on the device against the fp32 oracle (`oracle/img2img.py`): encoder moments (untiled and
tiled), the whole LCM img2img pass teacher-forced per step, CUDA graph against eager, batches against single
runs, and the b200 worker / pool behaviour for requests that carry an init image."""
import copy
import io
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from test_pipeline_gpu import max_rel_err, psnr_u8

pytestmark = pytest.mark.gpu

torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False

BF16_TOL, FP32_TOL = 2e-2, 1e-4
# The bf16 path stores every conv / linear / GroupNorm output in bf16.  For the narrow test topology
# (64/64/128/128 channels) that storage alone moves the fp32 oracle's moments by 1.5-2.7e-2 (max|d| / max|ref|,
# depending on the image), while the full SD1.5 encoder stays near 1.4e-2.  So the bf16 bar is BF16_TOL, widened
# only where the oracle with those storage points emulated is itself further off: by at most STORAGE_MARGIN x
# that error, which leaves room for the accumulation order and nothing else.
STORAGE_MARGIN = 1.5


def _image(n, h, w, seed=0):
    """A smooth RGB u8 test picture (gradients + blobs) with some noise: an encoder sees structure, not only noise."""
    g = np.random.default_rng(seed)
    yy, xx = np.meshgrid(np.linspace(0, 1, h), np.linspace(0, 1, w), indexing="ij")
    out = []
    for i in range(n):
        f = g.uniform(1, 4, size=3)
        base = np.stack([np.sin(f[0] * np.pi * xx + i), np.cos(f[1] * np.pi * yy), np.sin(f[2] * np.pi * (xx + yy))], -1)
        img = 127.5 + 100 * base + g.normal(0, 12, size=(h, w, 3))
        out.append(np.clip(np.round(img), 0, 255).astype(np.uint8))
    return np.stack(out)


def _models(vae_cfg=None, unet_cfg=None, full_unet=False):
    from oracle.img2img import build_random_init_img2img
    from oracle.unet import UNetConfig
    from oracle.vae import VAEConfig
    return build_random_init_img2img(unet_cfg or (UNetConfig() if full_unet else UNetConfig.tiny()),
                                     vae_cfg or VAEConfig.tiny(), seed=0)


def _encoder(enc, precision="bf16"):
    from dreamlab_b200.engine import VAEEncoderB200
    return VAEEncoderB200(enc.state_dict(), enc.cfg, "cuda:0", precision)


def _bf16_storage_err(enc, img, tiling=False):
    """max|d| / max|ref| of the fp32 oracle encoder against itself with the bf16 path's storage emulated: GEMM
    weights, the normalised image and every conv / linear / GroupNorm output rounded to bf16 (conv_out and
    quant_conv write fp32 moments, as on the device)."""
    from oracle.img2img import preprocess
    bf = lambda t: t.to(torch.bfloat16).float()                      # noqa: E731
    e = copy.deepcopy(enc).cpu()
    with torch.no_grad():
        for m in e.modules():
            if isinstance(m, (torch.nn.Conv2d, torch.nn.Linear)) and m is not e.quant_conv:
                m.weight.copy_(bf(m.weight))
        for name, m in e.named_modules():
            if (isinstance(m, (torch.nn.Conv2d, torch.nn.Linear, torch.nn.GroupNorm))
                    and name not in ("encoder.conv_out", "quant_conv")):
                m.register_forward_hook(lambda mod, i, o: bf(o))
        x = preprocess(img)
        return max_rel_err(e(bf(x), tiling=tiling), enc.cpu()(x, tiling=tiling))


def _bar(precision, enc, img, tiling=False):
    if precision == "fp32":
        return FP32_TOL
    return max(BF16_TOL, STORAGE_MARGIN * _bf16_storage_err(enc, img, tiling))


def _moments_err(enc, img, precision, tiling=False, oracle_device="cpu"):
    from oracle.img2img import preprocess
    eng = _encoder(enc, precision)
    got = eng.moments(torch.from_numpy(img).cuda(), tiling=tiling).permute(0, 3, 1, 2).cpu()
    torch.cuda.synchronize()
    with torch.no_grad():
        ref = enc.to(oracle_device)(preprocess(img).to(oracle_device), tiling=tiling).cpu()
    enc.to("cpu")
    assert got.shape == ref.shape
    return max_rel_err(got, ref)


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_encoder_moments_tiny(precision):
    _, _, enc = _models()
    for size in ((64, 64), (128, 96)):
        img = _image(2, *size)
        e, bar = _moments_err(enc, img, precision), _bar(precision, enc, img)
        print(f"tiny encoder {size} {precision}: moments max-rel-err {e:.3e} (bar {bar:.2e})")
        assert e <= bar


@pytest.mark.parametrize("precision,bar", [("bf16", BF16_TOL), ("fp32", FP32_TOL)])
def test_encoder_moments_full_sd15_vae_256(precision, bar):
    """The full SD1.5 encoder is held to the plain bars."""
    from oracle.img2img import build_random_init_encoder
    enc = build_random_init_encoder(None, seed=0)
    e = _moments_err(enc, _image(1, 256, 256, 3), precision, oracle_device="cuda")
    print(f"SD1.5 VAE encoder 256^2 {precision}: moments max-rel-err {e:.3e} (bar {bar:.0e})")
    assert e <= bar


@pytest.mark.parametrize("size", [(192, 192), (256, 256), (256, 192)])
def test_tiled_encode_against_oracle(size):
    """Tiny VAE with sample_size 128: 128-pixel tiles at stride 96, ragged last tiles, moment-space blending."""
    _, _, enc = _models()
    assert enc.cfg.sample_size == 128
    img = _image(1, *size, seed=5)
    e = _moments_err(enc, img, "bf16", tiling=True)
    e32 = _moments_err(enc, img, "fp32", tiling=True)
    bar = _bar("bf16", enc, img, tiling=True)
    print(f"tiled encode {size}: moments max-rel-err bf16 {e:.3e} (bar {bar:.2e}), fp32 {e32:.3e}")
    assert e <= bar and e32 <= FP32_TOL


def _draws(B, h, w, steps, seed=2000):
    es, en, noise = [], [], []
    for i in range(B):
        g = torch.Generator().manual_seed(seed + i)
        es.append(torch.randn(1, 4, h, w, generator=g))
        en.append(torch.randn(1, 4, h, w, generator=g))
        noise.append(torch.stack([torch.randn(1, 4, h, w, generator=g) for _ in range(steps - 1)])
                     if steps > 1 else torch.zeros(1, 1, 4, h, w))
    return torch.cat(es), torch.cat(en), torch.cat(noise, 1)


def _pipeline_parity(unet, vae, enc, B, H, W, steps, strength, precision, tiling=False):
    from oracle.img2img import run_pipeline_img2img
    from oracle.pipeline import synthetic_inputs
    from dreamlab_b200.engine import LCMPipelineB200
    from test_pipeline_gpu import teacher_inputs
    sd = {**vae.state_dict(), **enc.state_dict()}
    pipe = LCMPipelineB200(unet.state_dict(), unet.cfg, sd, vae.cfg, "cuda:0", vae_tiling=tiling, precision=precision)
    pe, _, _ = synthetic_inputs(B, H, W, steps, ctx_dim=unet.cfg.cross_attention_dim)
    es, en, noise = _draws(B, H // 8, W // 8, steps)
    img = _image(B, H, W, seed=11)
    rec_o, rec_c = {}, {}
    ref = run_pipeline_img2img(unet, vae, enc, pe, img, es, en, noise, steps, strength, 1.0, tiling=tiling,
                               record=rec_o)
    teacher = teacher_inputs(rec_o["init_latents"], rec_o["latents"])
    pipe.generate(pe, en, noise, steps, 1.0, record=rec_c, teacher_latents=teacher,
                  init_images=torch.from_numpy(img), strength=strength, posterior_noise=es)
    out = pipe.generate(pe, en, noise, steps, 1.0, init_images=torch.from_numpy(img), strength=strength,
                        posterior_noise=es)
    torch.cuda.synchronize()
    e_mom = max_rel_err(rec_c["moments"].cpu(), rec_o["moments"])
    e_init = max_rel_err(rec_c["init_latents"].cpu(), rec_o["init_latents"])
    errs = [max_rel_err(c.cpu(), o) for c, o in zip(rec_c["noise_pred"], rec_o["noise_pred"])]
    p = psnr_u8(out.cpu().numpy(), ref)
    # the moments' bar (and that of the latents sampled from them); the UNet's noise_pred keeps the plain bar
    mbar = _bar(precision, enc, img, tiling)
    return pipe, (pe, en, noise, es, img), e_mom, e_init, errs, p, mbar


@pytest.mark.parametrize("precision,bar", [("bf16", BF16_TOL), ("fp32", FP32_TOL)])
def test_tiny_img2img_pipeline_parity(precision, bar):
    unet, vae, enc = _models()
    pipe, inp, e_mom, e_init, errs, p, mbar = _pipeline_parity(unet, vae, enc, 2, 128, 128, 4, 0.5, precision)
    print(f"tiny img2img {precision}: moments {e_mom:.2e}, init latents {e_init:.2e} (bar {mbar:.2e}), teacher-forced "
          f"noise_pred {['%.2e' % e for e in errs]}, PSNR {p:.1f} dB")
    assert e_mom <= mbar and e_init <= mbar and max(errs) <= bar and p >= 35.0
    # graph replay == eager, byte for byte; a batch equals its single runs
    pe, en, noise, es, img = inp
    eager = pipe.generate(pe, en, noise, 4, 1.0, init_images=torch.from_numpy(img), strength=0.5,
                          posterior_noise=es).clone()
    g = pipe.generate(pe, en, noise, 4, 1.0, init_images=torch.from_numpy(img), strength=0.5,
                      posterior_noise=es, use_graph=True).clone()
    torch.cuda.synchronize()
    assert torch.equal(g, eager)
    for i in range(2):
        one = pipe.generate(pe[i:i + 1], en[i:i + 1], noise[:, i:i + 1], 4, 1.0,
                            init_images=torch.from_numpy(img[i:i + 1]), strength=0.5,
                            posterior_noise=es[i:i + 1], use_graph=True).clone()
        torch.cuda.synchronize()
        assert (one[0].int() - g[i].int()).abs().max() <= 1       # same tolerance as the text-to-image batch test
    other = pipe.generate(pe, en, noise, 4, 1.0, init_images=torch.from_numpy(img), strength=0.8,
                          posterior_noise=es, use_graph=True).clone()
    torch.cuda.synchronize()
    assert not torch.equal(other, g)


def test_full_arch_img2img_256_parity():
    from oracle.vae import VAEConfig
    unet, vae, enc = _models(VAEConfig(), full_unet=True)
    _, _, e_mom, e_init, errs, p, _ = _pipeline_parity(unet, vae, enc, 1, 256, 256, 2, 0.5, "bf16")
    print(f"full-arch img2img 256^2 bf16: moments {e_mom:.2e}, init latents {e_init:.2e}, teacher-forced noise_pred "
          f"{['%.2e' % e for e in errs]}, PSNR {p:.1f} dB")
    assert e_mom <= BF16_TOL and e_init <= BF16_TOL and max(errs) <= BF16_TOL and p >= 35.0


def test_tiled_img2img_pipeline_parity():
    unet, vae, enc = _models()
    _, _, e_mom, e_init, errs, p, mbar = _pipeline_parity(unet, vae, enc, 1, 192, 256, 2, 0.8, "bf16", tiling=True)
    print(f"tiled tiny img2img 256x192: moments {e_mom:.2e} (bar {mbar:.2e}), noise_pred {['%.2e' % e for e in errs]}, "
          f"PSNR {p:.1f} dB")
    assert e_mom <= mbar and max(errs) <= BF16_TOL and p >= 35.0


def test_pipeline_refusals():
    from dreamlab_b200.engine import LCMPipelineB200
    unet, vae, enc = _models()
    pipe = LCMPipelineB200(unet.state_dict(), unet.cfg, vae.state_dict(), vae.cfg, "cuda:0")
    assert pipe.vae_encoder is None
    pe = torch.randn(1, 77, unet.cfg.cross_attention_dim)
    z = torch.randn(1, 4, 8, 8)
    img = torch.from_numpy(_image(1, 64, 64))
    with pytest.raises(RuntimeError, match="encoder"):
        pipe.generate(pe, z, torch.randn(1, 1, 4, 8, 8), 2, 1.0, init_images=img, strength=0.5, posterior_noise=z)
    pipe = LCMPipelineB200(unet.state_dict(), unet.cfg, {**vae.state_dict(), **enc.state_dict()}, vae.cfg, "cuda:0")
    with pytest.raises(RuntimeError, match="init_images"):
        pipe.generate(pe, z, torch.randn(1, 1, 4, 8, 8), 2, 1.0, init_images=img[:, :32], strength=0.5,
                      posterior_noise=z)
    with pytest.raises(ValueError):
        pipe.generate(pe, z, torch.randn(3, 1, 4, 8, 8), 4, 1.0, init_images=img, strength=0.05, posterior_noise=z)


# ------------------------------------------------------------------------------------------------ worker / pool
class Req(SimpleNamespace):
    pass


def job(prompt="a cat", size="128x128", steps=2, gs=1.0, seed=42, **kw):
    return SimpleNamespace(req=Req(prompt=prompt, size=size, num_inference_steps=steps, guidance_scale=gs,
                                   seed=seed, **kw))


def _png(arr):
    from PIL import Image
    buf = io.BytesIO()
    Image.fromarray(arr).save(buf, format="PNG")
    return buf.getvalue()


def _make_worker(root, name, vae_encoder, ucfg=None):
    from dreamlab_b200 import synthetic as S
    from oracle.unet import UNetConfig
    from oracle.vae import VAEConfig
    if ucfg is None:
        ucfg = UNetConfig.tiny()
        ucfg.cross_attention_dim = 768
    S.write_model_dir(str(root / name), ucfg, VAEConfig.tiny(), vae_encoder=vae_encoder)
    os.environ["MODEL_ROOT"], os.environ["MODEL"] = str(root), name
    os.environ.pop("CUDA_DEVICE", None)
    from backends.b200_worker import B200Worker
    return B200Worker(0)


@pytest.fixture(scope="module")
def workers(tmp_path_factory):
    root = tmp_path_factory.mktemp("models")
    return _make_worker(root, "tiny-i2i", True), _make_worker(root, "tiny-t2i", False)


def test_worker_img2img(workers):
    from PIL import Image
    w, _ = workers
    init = _image(1, 128, 128, seed=21)[0]
    png, seed = w.run_job(job(seed=42, init_image=_png(init), strength=0.5))
    assert png[:8] == b"\x89PNG\r\n\x1a\n" and seed == 42
    assert Image.open(io.BytesIO(png)).size == (128, 128)
    assert w.run_job(job(seed=42, init_image=_png(init), strength=0.5))[0] == png       # same seed + image
    assert w.run_job(job(seed=42, init_image=init, strength=0.5))[0] == png             # array form
    assert w.run_job(job(seed=42, init_image=_png(init), strength=0.8))[0] != png       # another strength
    assert w.run_job(job(seed=42))[0] != png                                             # text-to-image
    arr, _ = w.run_job_array(job(seed=42, init_image=init, strength=0.5))
    assert np.array_equal(np.asarray(Image.open(io.BytesIO(png))), arr)
    png2, _, lat = w.run_job_with_latents(job(seed=42, init_image=init, strength=0.5))
    assert png2 == png and len(lat) == 512
    lat_only, _ = w.run_job_latents(job(seed=42, init_image=init, strength=0.5))
    assert lat_only.shape == (4, 16, 16)
    # default strength 0.8
    assert w.run_job(job(seed=42, init_image=init))[0] == w.run_job(job(seed=42, init_image=init, strength=0.8))[0]


def test_worker_img2img_refusals(workers, tmp_path):
    w, w_noenc = workers
    init = _image(1, 128, 128)[0]
    with pytest.raises(RuntimeError, match="not resized"):
        w.run_job(job(size="128x64", init_image=init))
    with pytest.raises(RuntimeError, match="encoder"):
        w_noenc.run_job(job(init_image=init))
    with pytest.raises(RuntimeError, match="uint8"):
        w.run_job(job(init_image=init.astype(np.float32)))
    from backends.b200_worker import B200SDXLWorker
    sdxl = object.__new__(B200SDXLWorker)
    with pytest.raises(RuntimeError, match="SDXL"):
        sdxl._check_img2img()
    from oracle.unet import UNetConfig
    ucfg = UNetConfig.tiny()
    ucfg.cross_attention_dim = 768
    ucfg.time_cond_proj_dim = None
    w_cfg = _make_worker(tmp_path, "tiny-cfg", True, ucfg)
    with pytest.raises(RuntimeError, match="time_cond_proj_dim"):
        w_cfg.run_job(job(init_image=init))


def test_text_to_image_unchanged_by_encoder_weights(workers):
    a, b = workers
    for s in (7, 8):
        assert a.run_job(job(seed=s))[0] == b.run_job(job(seed=s))[0]


def test_pool_mixes_text_to_image_and_img2img(workers):
    from unittest.mock import Mock
    from backends.worker_pool import GenerationJob, WorkerPool
    w, _ = workers
    init = _image(1, 128, 128, seed=4)[0]
    jobs = [job(prompt=f"p{i}", seed=300 + i, **({"init_image": init, "strength": (0.5, 0.8)[i % 2]} if i % 3 else {}))
            for i in range(6)]
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
    from PIL import Image
    for (pr, sr), (ps, ss) in zip(res, singles):
        assert sr == ss
        a = np.asarray(Image.open(io.BytesIO(pr))).astype(int)
        b = np.asarray(Image.open(io.BytesIO(ps))).astype(int)
        assert np.abs(a - b).max() <= 1
