"""Guided-model samplers end to end on the device against the fp32 oracle (`oracle/samplers.py`), and through the
worker and the pool.

- Teacher-forced per-step UNet outputs (both CFG halves) for every sampler, on a tiny SD1.5-topology UNet without the
  LCM guidance embedding and on the tiny SDXL UNet, epsilon and v_prediction configs: <= 2e-2 in bf16, <= 1e-4 in the
  fp32 mode.  The fp32 mode's free-running final latents within 1e-4 of the oracle's.
- Euler ancestral through the worker consumes the per-request Philox stream in the documented order (latents, then
  one draw per step).
- Workers: sampler None / "lcm" are today's bytes; every sampler through every entry point, same-seed determinism,
  batches equal to singles, B200_PNG=gpu, the SDXL worker, and the refusals."""
import io
import os

import numpy as np
import pytest
import torch

from test_img2img_gpu import job
from test_pipeline_gpu import NOISE_PRED_TOL, max_rel_err, teacher_inputs

pytestmark = pytest.mark.gpu

torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False

NAMES = ["euler", "euler_a", "ddim", "dpmpp_2m", "dpmpp_2m_karras"]
FP32_TOL = 1e-4
SD15 = {"_class_name": "PNDMScheduler", "beta_end": 0.012, "beta_schedule": "scaled_linear", "beta_start": 0.00085,
        "num_train_timesteps": 1000, "set_alpha_to_one": False, "skip_prk_steps": True, "steps_offset": 1,
        "trained_betas": None, "clip_sample": False}
CONFIGS = {"epsilon": SD15,
           "v_prediction": dict(SD15, prediction_type="v_prediction", rescale_betas_zero_snr=True,
                                timestep_spacing="trailing")}


def _cfg_unet(kind):
    from oracle.unet import UNetConfig
    if kind == "sdxl":
        return UNetConfig.tiny_sdxl()
    u = UNetConfig.tiny()
    u.time_cond_proj_dim = None            # a vanilla SD1.5-class UNet: classifier-free guidance
    return u


def _case(kind, sampler, pred, precision, steps=4, B=2, size=64, gs=7.5):
    from dreamlab_b200.engine import LCMPipelineB200
    from dreamlab_b200.scheduler import SchedulerConfig
    from oracle.pipeline import build_random_init, synthetic_inputs
    from oracle.samplers import noise_draws, run_pipeline_sampler
    from oracle.vae import VAEConfig
    ucfg = _cfg_unet(kind)
    unet, vae = build_random_init(ucfg, VAEConfig.tiny(), seed=0)
    conf = CONFIGS[pred]
    pipe = LCMPipelineB200(unet.state_dict(), unet.cfg, vae.state_dict(), vae.cfg, "cuda:0", precision=precision,
                           scheduler_config=SchedulerConfig.from_dict(conf))
    pe, lat, _ = synthetic_inputs(B, size, size, 1, ctx_dim=ucfg.cross_attention_dim)
    nd = noise_draws(sampler, steps)
    noise = torch.randn(max(nd, 1), B, 4, size // 8, size // 8, generator=torch.Generator().manual_seed(9))
    kw = {}
    if kind == "sdxl":
        pdim = ucfg.projection_class_embeddings_input_dim - 6 * ucfg.addition_time_embed_dim
        kw = dict(pooled_embeds=torch.randn(B, pdim, generator=torch.Generator().manual_seed(2)))
    rec_o = {}
    ref = run_pipeline_sampler(unet, vae, pe, lat, noise, sampler, steps, gs, conf, height=size, width=size,
                               output_type="latent", record=rec_o, **kw)
    teacher = teacher_inputs(rec_o["init_latents"], rec_o["latents"])
    return pipe, pe, lat, noise if nd else None, kw, rec_o, ref, teacher


@pytest.mark.parametrize("kind", ["sd15_cfg", "sdxl"])
@pytest.mark.parametrize("pred", ["epsilon", "v_prediction"])
@pytest.mark.parametrize("sampler", NAMES)
@pytest.mark.parametrize("precision,bar", [("bf16", NOISE_PRED_TOL), ("fp32", FP32_TOL)])
def test_teacher_forced_parity(kind, pred, sampler, precision, bar):
    steps, gs = 4, 7.5
    pipe, pe, lat, noise, kw, rec_o, ref, teacher = _case(kind, sampler, pred, precision, steps=steps, gs=gs)
    B = lat.shape[0]
    rec_t = {}
    pipe.generate(pe, lat, noise, steps, gs, record=rec_t, teacher_latents=teacher, sampler=sampler, **kw)
    torch.cuda.synchronize()
    assert [float(t) for t in rec_o["timesteps"]] == [float(t) for t in pipe.schedule(steps, sampler=sampler).timesteps]
    halves = [(max_rel_err(c[:B].cpu(), o[:B]), max_rel_err(c[B:].cpu(), o[B:]))
              for c, o in zip(rec_t["noise_pred_raw"], rec_o["noise_pred_raw"])]
    print(f"{kind} {pred} {sampler} {precision}: teacher-forced halves {[('%.2e' % a, '%.2e' % b) for a, b in halves]}")
    assert max(max(h) for h in halves) <= bar, halves
    if precision == "fp32":
        _, final = pipe.generate(pe, lat, noise, steps, gs, return_latents=True, decode=False, sampler=sampler, **kw)
        torch.cuda.synchronize()
        err = max_rel_err(final.permute(0, 3, 1, 2).cpu(), ref)
        print(f"  free-running final latents {err:.2e}")
        assert err <= FP32_TOL, err


@pytest.mark.parametrize("sampler", NAMES)
def test_graph_replay_equals_eager(sampler):
    pipe, pe, lat, noise, kw, _, _, _ = _case("sd15_cfg", sampler, "epsilon", "bf16")
    eager = pipe.generate(pe, lat, noise, 4, 7.5, sampler=sampler)
    graph = pipe.generate(pe, lat, noise, 4, 7.5, sampler=sampler, use_graph=True)
    lcm = pipe.generate(pe, lat, torch.randn(3, *lat.shape), 4, 7.5, use_graph=True)
    torch.cuda.synchronize()
    assert torch.equal(eager, graph)
    assert not torch.equal(graph, lcm)
    assert len({k for k in pipe._graphs if "sampler" in k}) == 1


def test_engine_refuses_samplers_on_img2img_and_unknown_names():
    from dreamlab_b200.engine import LCMPipelineB200
    from oracle.pipeline import build_random_init
    from oracle.unet import UNetConfig
    from oracle.vae import VAEConfig
    unet, vae = build_random_init(UNetConfig.tiny(), VAEConfig.tiny(), seed=0)
    pipe = LCMPipelineB200(unet.state_dict(), unet.cfg, vae.state_dict(), vae.cfg, "cuda:0")
    lat = torch.zeros(1, 4, 8, 8)
    pe = torch.zeros(1, 77, unet.cfg.cross_attention_dim)
    with pytest.raises(RuntimeError, match="LCM sampler only"):
        pipe.generate(pe, lat, None, 2, 1.0, init_images=torch.zeros(1, 64, 64, 3, dtype=torch.uint8),
                      posterior_noise=lat, sampler="ddim")
    with pytest.raises(RuntimeError, match="euler_a"):
        pipe.generate(pe, lat, None, 2, 1.0, sampler="heun")
    with pytest.raises(RuntimeError, match="LCM sampler only"):
        pipe.schedule(4, 0.5, sampler="euler")


# ------------------------------------------------------------------------------------------------ worker
def _model_dir(root, name, ucfg, scheduler=None):
    import json
    from dreamlab_b200 import synthetic as S
    from oracle.vae import VAEConfig
    d = os.path.join(str(root), name)
    S.write_model_dir(d, ucfg, VAEConfig.tiny())
    if scheduler is not None:
        os.makedirs(os.path.join(d, "scheduler"), exist_ok=True)
        with open(os.path.join(d, "scheduler", "scheduler_config.json"), "w") as f:
            json.dump(scheduler, f)
    return d


def _worker(root, name, cls=None):
    os.environ["MODEL_ROOT"], os.environ["MODEL"] = str(root), name
    os.environ.pop("CUDA_DEVICE", None)
    from backends.b200_worker import B200Worker
    return (cls or B200Worker)(0)


@pytest.fixture(scope="module")
def cfg_worker(tmp_path_factory):
    root = tmp_path_factory.mktemp("samplers")
    ucfg = _cfg_unet("sd15_cfg")
    ucfg.cross_attention_dim = 768
    _model_dir(root, "tiny-cfg", ucfg, SD15)
    return _worker(root, "tiny-cfg")


def _u8(png):
    from PIL import Image
    return np.asarray(Image.open(io.BytesIO(png)).convert("RGB"))


def test_worker_default_sampler_is_unchanged(cfg_worker):
    w = cfg_worker
    base = [w.run_job(job(seed=s, steps=3, gs=5.0))[0] for s in (1, 2)]
    assert [w.run_job(job(seed=s, steps=3, gs=5.0, sampler=None))[0] for s in (1, 2)] == base
    assert [w.run_job(job(seed=s, steps=3, gs=5.0, sampler="lcm"))[0] for s in (1, 2)] == base


@pytest.mark.parametrize("sampler", NAMES)
def test_worker_every_sampler_every_entry_point(cfg_worker, sampler, monkeypatch):
    w = cfg_worker
    kw = dict(steps=4, gs=5.0, sampler=sampler)
    png, seed = w.run_job(job(seed=5, **kw))
    assert png[:8] == b"\x89PNG\r\n\x1a\n" and seed == 5
    assert w.run_job(job(seed=5, **kw))[0] == png                        # same seed, same bytes
    assert w.run_job(job(seed=6, **kw))[0] != png
    assert w.run_job(job(seed=5, steps=4, gs=5.0))[0] != png             # not the LCM image
    singles = [_u8(w.run_job(job(seed=s, **kw))[0]) for s in (5, 6, 7)]
    batch = w.run_batch([job(seed=s, **kw) for s in (5, 6, 7)])
    for (p, s), one in zip(batch, singles):
        assert np.abs(_u8(p).astype(int) - one.astype(int)).max() <= 1, s
    p2, s2, lat8 = w.run_job_with_latents(job(seed=5, **kw))
    assert p2 == png and s2 == 5 and len(lat8) == 512
    arr, s3 = w.run_job_array(job(seed=5, **kw))
    assert s3 == 5 and np.array_equal(arr, _u8(png))
    lat, s4 = w.run_job_latents(job(seed=5, **kw))
    assert s4 == 5 and lat.shape == (4, 16, 16) and np.isfinite(lat).all()
    monkeypatch.setenv("B200_PNG", "gpu")
    g, _ = w.run_job(job(seed=5, **kw))
    assert np.array_equal(_u8(g), _u8(png))


def test_worker_euler_a_draw_order(cfg_worker):
    """The worker's euler_a pass equals the pipeline fed the per-request Philox stream drawn as documented: the
    latents, then one draw per step (the last step's too), each through the noise dtype."""
    w = cfg_worker
    steps, seed = 4, 11
    lat_w, _ = w.run_job_latents(job(seed=seed, steps=steps, gs=5.0, sampler="euler_a"))
    gen = torch.Generator(device=w.device)
    gen.manual_seed(seed)
    draws = [torch.randn(1, 4, 16, 16, generator=gen, device=w.device) for _ in range(1 + steps)]
    lat = draws[0].to(w.dtype).float()
    noise = torch.stack(draws[1:]).to(w.dtype).float()
    pe = w._text.encode(["a cat"])
    neg = w._negative(1)
    _, final = w.pipe.generate(pe, lat, noise, steps, torch.tensor([5.0]), return_latents=True, decode=False,
                               negative_prompt_embeds=neg, sampler="euler_a")
    torch.cuda.synchronize()
    assert np.array_equal(final.permute(0, 3, 1, 2)[0].cpu().numpy(), lat_w)
    _, rolled = w.pipe.generate(pe, lat, noise.roll(1, 0), steps, torch.tensor([5.0]), return_latents=True,
                                decode=False, negative_prompt_embeds=neg, sampler="euler_a")
    torch.cuda.synchronize()
    assert not np.array_equal(rolled.permute(0, 3, 1, 2)[0].cpu().numpy(), lat_w)    # the order matters


def test_worker_refusals(cfg_worker):
    w = cfg_worker
    with pytest.raises(RuntimeError, match="dpmpp_2m"):
        w.run_job(job(sampler="heun"))
    with pytest.raises(RuntimeError, match="LCM sampler only"):
        w.run_job(job(sampler="ddim", init_image=np.zeros((128, 128, 3), np.uint8)))
    with pytest.raises(RuntimeError, match="share the sampler"):
        w.run_batch([job(seed=1, sampler="ddim"), job(seed=2, sampler="euler")])


@pytest.mark.parametrize("sampler", ["euler", "dpmpp_2m_karras"])
def test_sdxl_worker_samplers(tmp_path, sampler):
    from backends.b200_worker import B200SDXLWorker
    ucfg = _cfg_unet("sdxl")
    sdxl = dict(SD15, _class_name="EulerDiscreteScheduler", timestep_spacing="leading", use_karras_sigmas=False)
    _model_dir(tmp_path, "tiny-xl", ucfg, sdxl)
    w = _worker(tmp_path, "tiny-xl", B200SDXLWorker)
    png, _ = w.run_job(job(seed=3, steps=5, gs=7.5, sampler=sampler))
    assert png == w.run_job(job(seed=3, steps=5, gs=7.5, sampler=sampler))[0]
    assert png != w.run_job(job(seed=3, steps=5, gs=7.5))[0]
    assert w.run_job(job(seed=3, steps=5, gs=7.5, sampler="lcm"))[0] == w.run_job(job(seed=3, steps=5, gs=7.5))[0]
