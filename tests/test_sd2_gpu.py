"""Models whose scheduler config is not SD1.5's, end to end on the device against the fp32 oracle:

- SD2.x-class (`B200Worker` serves cross_attention_dim 1024): the full SD2 UNet (head dim 64 at every level, linear
  projections), SD1.x VAE, 768x768, `v_prediction`, classifier-free guidance 7.5, 4 LCM steps;
- a tiny SDXL UNet with `v_prediction` + `rescale_betas_zero_snr`;
- image-to-image and inpainting on a tiny LCM UNet with a `v_prediction` config;
- the b200 worker on a model directory with a scheduler config;
- the SD2 level-0 self-attention shape (head dim 64, S = 9216) in the style of `test_attention_edges_gpu.py`.

Bars as in `test_pipeline_gpu.py`: teacher-forced UNet outputs (both CFG halves) <= 2e-2 at every step, free-running
image PSNR >= 35 dB, the fp32 mode <= 1e-4."""
import io
import os

import pytest
import torch

from test_img2img_gpu import _image, job
from test_pipeline_gpu import NOISE_PRED_TOL, PSNR_MIN_DB, max_rel_err, psnr_u8, teacher_inputs

pytestmark = pytest.mark.gpu

torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False

FP32_TOL = 1e-4
V_ZERO_SNR = {"prediction_type": "v_prediction", "rescale_betas_zero_snr": True}
V_LCM = {"_class_name": "LCMScheduler", "prediction_type": "v_prediction", "timestep_spacing": "trailing"}


def _errors(rec_c, rec_o, B, cfg):
    """-> (per-step max-rel-err of the UNet output, per-step (uncond, text) halves or [] without CFG)."""
    key = "noise_pred_raw" if cfg else "noise_pred"
    raw = [max_rel_err(c.cpu(), o.cpu()) for c, o in zip(rec_c[key], rec_o[key])]
    halves = []
    if cfg:
        halves = [(max_rel_err(c[:B].cpu(), o[:B].cpu()), max_rel_err(c[B:].cpu(), o[B:].cpu()))
                  for c, o in zip(rec_c[key], rec_o[key])]
    return raw, halves


# ------------------------------------------------------------------------------------------------ SD2, full size
def test_sd2_768_v_prediction_cfg():
    from dreamlab_b200.engine import LCMPipelineB200
    from dreamlab_b200.scheduler import SchedulerConfig
    from oracle.lcm_config import SD2_V_SCHEDULER_CONFIG, run_pipeline_cfg, sd2_unet_config
    from oracle.pipeline import build_random_init, synthetic_inputs
    from oracle.vae import VAEConfig
    steps, size, gs, B = 4, 768, 7.5, 1
    unet, vae = build_random_init(sd2_unet_config(), VAEConfig(), seed=0)
    sc = SchedulerConfig.from_dict(SD2_V_SCHEDULER_CONFIG)
    pe, lat, noise = synthetic_inputs(B, size, size, steps, ctx_dim=1024)
    rec_o = {}
    unet.cuda(), vae.cuda()
    with torch.device("cuda"):                  # the fp32 oracle on the device (TF32 off): 17 TFLOP of fp32 work
        ref = run_pipeline_cfg(unet, vae, pe.cuda(), lat.cuda(), noise.cuda(), steps, gs, SD2_V_SCHEDULER_CONFIG,
                               record=rec_o)
    unet.cpu(), vae.cpu()
    teacher = teacher_inputs(lat, [x.cpu() for x in rec_o["latents"]])
    for precision, bar in (("bf16", NOISE_PRED_TOL), ("fp32", FP32_TOL)):
        pipe = LCMPipelineB200(unet.state_dict(), unet.cfg, vae.state_dict(), vae.cfg, "cuda:0", precision=precision,
                               scheduler_config=sc)
        rec_t, rec_f = {}, {}
        pipe.generate(pe, lat, noise, steps, gs, record=rec_t, teacher_latents=teacher)
        img = pipe.generate(pe, lat, noise, steps, gs, record=rec_f)
        torch.cuda.synchronize()
        raw, halves = _errors(rec_t, rec_o, B, True)
        p = psnr_u8(img.cpu().numpy(), ref)
        print(f"SD2 768^2 v_prediction CFG {gs} {precision}: teacher-forced UNet output per step "
              f"{['%.2e' % e for e in raw]} halves {[('%.2e' % a, '%.2e' % b) for a, b in halves]}  PSNR {p:.1f} dB")
        assert max(max(h) for h in halves) <= bar, halves
        assert p >= PSNR_MIN_DB, p
        if precision == "bf16":                  # graph replay == eager, byte for byte
            g = pipe.generate(pe, lat, noise, steps, gs, use_graph=True)
            torch.cuda.synchronize()
            assert torch.equal(g, img)
        del pipe
        torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ tiny SDXL
@pytest.mark.parametrize("precision,bar", [("bf16", NOISE_PRED_TOL), ("fp32", FP32_TOL)])
def test_tiny_sdxl_v_prediction_zero_snr(precision, bar):
    from dreamlab_b200.engine import LCMPipelineB200
    from dreamlab_b200.scheduler import SchedulerConfig
    from oracle.lcm_config import configured
    from oracle.pipeline import build_random_init, run_pipeline_sdxl, synthetic_inputs
    from oracle.unet import UNetConfig
    from oracle.vae import VAEConfig
    ucfg = UNetConfig.tiny_sdxl()
    unet, vae = build_random_init(ucfg, VAEConfig.tiny(), seed=0)
    pipe = LCMPipelineB200(unet.state_dict(), unet.cfg, vae.state_dict(), vae.cfg, "cuda:0", precision=precision,
                           scheduler_config=SchedulerConfig.from_dict(V_ZERO_SNR))
    steps, size, B, gs = 4, 128, 2, 7.5
    pdim = ucfg.projection_class_embeddings_input_dim - 6 * ucfg.addition_time_embed_dim
    pe, lat, noise = synthetic_inputs(B, size, size, steps, ctx_dim=ucfg.cross_attention_dim)
    pooled = torch.randn(B, pdim, generator=torch.Generator().manual_seed(2))
    rec_o, rec_t = {}, {}
    with configured(V_ZERO_SNR):
        ref = run_pipeline_sdxl(unet, vae, pe, pooled, lat, noise, steps, gs, size, size, record=rec_o)
    assert rec_o["timesteps"][0] == 999                       # the step that sees alphas_cumprod = 0
    pipe.generate(pe, lat, noise, steps, gs, record=rec_t, pooled_embeds=pooled,
                  teacher_latents=teacher_inputs(lat, rec_o["latents"]))
    img = pipe.generate(pe, lat, noise, steps, gs, pooled_embeds=pooled)
    torch.cuda.synchronize()
    raw, halves = _errors(rec_t, rec_o, B, True)
    p = psnr_u8(img.cpu().numpy(), ref)
    print(f"tiny SDXL v_prediction + zero SNR {precision}: teacher-forced halves "
          f"{[('%.2e' % a, '%.2e' % b) for a, b in halves]}  PSNR {p:.1f} dB")
    assert max(max(h) for h in halves) <= bar, halves
    assert p >= PSNR_MIN_DB, p


# ------------------------------------------------------------------------------------------------ img2img, inpaint
@pytest.mark.parametrize("precision,bar", [("bf16", NOISE_PRED_TOL), ("fp32", FP32_TOL)])
def test_tiny_img2img_v_prediction(precision, bar):
    from dreamlab_b200.engine import LCMPipelineB200
    from dreamlab_b200.scheduler import SchedulerConfig
    from oracle.img2img import run_pipeline_img2img
    from oracle.lcm_config import configured
    from oracle.pipeline import synthetic_inputs
    from test_img2img_gpu import _draws, _models
    unet, vae, enc = _models()
    pipe = LCMPipelineB200(unet.state_dict(), unet.cfg, {**vae.state_dict(), **enc.state_dict()}, vae.cfg, "cuda:0",
                           precision=precision, scheduler_config=SchedulerConfig.from_dict(V_LCM))
    B, H, steps, strength = 2, 128, 4, 0.5
    pe, _, _ = synthetic_inputs(B, H, H, steps, ctx_dim=unet.cfg.cross_attention_dim)
    es, en, noise = _draws(B, H // 8, H // 8, steps)
    img = _image(B, H, H, seed=11)
    kw = dict(init_images=torch.from_numpy(img), strength=strength, posterior_noise=es)
    rec_o, rec_t = {}, {}
    with configured(V_LCM):
        ref = run_pipeline_img2img(unet, vae, enc, pe, img, es, en, noise, steps, strength, 1.0, tiling=False,
                                   record=rec_o)
    pipe.generate(pe, en, noise, steps, 1.0, record=rec_t,
                  teacher_latents=teacher_inputs(rec_o["init_latents"], rec_o["latents"]), **kw)
    out = pipe.generate(pe, en, noise, steps, 1.0, **kw)
    torch.cuda.synchronize()
    errs, _ = _errors(rec_t, rec_o, B, False)
    p = psnr_u8(out.cpu().numpy(), ref)
    print(f"tiny img2img v_prediction {precision}: teacher-forced noise_pred {['%.2e' % e for e in errs]}, "
          f"PSNR {p:.1f} dB")
    assert max(errs) <= bar and p >= PSNR_MIN_DB


@pytest.mark.parametrize("in_channels", [4, 9])
@pytest.mark.parametrize("precision,bar", [("bf16", NOISE_PRED_TOL), ("fp32", FP32_TOL)])
def test_tiny_inpaint_v_prediction(in_channels, precision, bar):
    from dreamlab_b200.engine import LCMPipelineB200
    from dreamlab_b200.scheduler import SchedulerConfig
    from oracle.inpaint import run_pipeline_inpaint
    from oracle.lcm_config import configured
    from test_inpaint_gpu import _inputs, _kw, _models
    unet, vae, enc = _models(in_channels)
    pipe = LCMPipelineB200(unet.state_dict(), unet.cfg, {**vae.state_dict(), **enc.state_dict()}, vae.cfg, "cuda:0",
                           precision=precision, scheduler_config=SchedulerConfig.from_dict(V_LCM))
    B, H, steps = 2, 128, 4
    strength = 0.5 if in_channels == 4 else 1.0
    pe, es, en, em, noise, img, mask = _inputs(unet, B, H, H, steps, strength)
    kw = _kw(img, mask, es, em, strength)
    rec_o, rec_t = {}, {}
    with configured(V_LCM):
        ref = run_pipeline_inpaint(unet, vae, enc, pe, img, mask, es, en, em, noise, steps, strength, 1.0,
                                   tiling=False, record=rec_o)
    pipe.generate(pe, en, noise, steps, 1.0, record=rec_t,
                  teacher_latents=teacher_inputs(rec_o["init_latents"], rec_o["latents"]), **kw)
    out = pipe.generate(pe, en, noise, steps, 1.0, **kw)
    torch.cuda.synchronize()
    errs, _ = _errors(rec_t, rec_o, B, False)
    p = psnr_u8(out.cpu().numpy(), ref)
    print(f"tiny inpaint {in_channels}ch v_prediction {precision}: teacher-forced noise_pred "
          f"{['%.2e' % e for e in errs]}, PSNR {p:.1f} dB")
    assert max(errs) <= bar and p >= PSNR_MIN_DB


# ------------------------------------------------------------------------------------------------ worker
def _tiny_sd2_ucfg():
    from oracle.lcm_config import tiny_sd2_unet_config
    ucfg = tiny_sd2_unet_config()
    ucfg.cross_attention_dim = 1024            # CLIP-H width: the factory's SD2.x row
    return ucfg


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


def test_worker_sd2_v_prediction(tmp_path):
    from PIL import Image
    from backends.worker_factory import detect_worker_type
    from oracle.lcm_config import SD2_V_SCHEDULER_CONFIG
    _model_dir(tmp_path, "tiny-sd2-v", _tiny_sd2_ucfg(), SD2_V_SCHEDULER_CONFIG)
    os.environ["MODEL_ROOT"], os.environ["MODEL"] = str(tmp_path), "tiny-sd2-v"
    assert detect_worker_type() == "sd15"
    w = _worker(tmp_path, "tiny-sd2-v")
    assert w.scheduler_config.prediction_type == "v_prediction"
    png, seed = w.run_job(job(seed=7, size="192x128", steps=4, gs=7.5))
    assert png[:8] == b"\x89PNG\r\n\x1a\n" and seed == 7
    assert Image.open(io.BytesIO(png)).size == (192, 128)
    assert w.run_job(job(seed=7, size="192x128", steps=4, gs=7.5))[0] == png
    assert w.run_job(job(seed=8, size="192x128", steps=4, gs=7.5))[0] != png


@pytest.mark.parametrize("scheduler", ["lcm_default", "sd15_pndm"])
def test_worker_default_config_file_changes_nothing(tmp_path, scheduler):
    """The same weights with and without a scheduler config that states the defaults: byte-identical PNGs."""
    from oracle.unet import UNetConfig
    from test_scheduler_config_host import LCM_DEFAULT, SD15_PNDM
    ucfg = UNetConfig.tiny()
    ucfg.cross_attention_dim = 768
    _model_dir(tmp_path, "plain", ucfg)
    _model_dir(tmp_path, "with-config", ucfg, {"lcm_default": LCM_DEFAULT, "sd15_pndm": SD15_PNDM}[scheduler])
    a = _worker(tmp_path, "plain")
    pa = [a.run_job(job(seed=s, steps=4))[0] for s in (1, 2)]
    del a
    b = _worker(tmp_path, "with-config")
    pb = [b.run_job(job(seed=s, steps=4))[0] for s in (1, 2)]
    assert pa == pb


def test_sdxl_worker_reads_the_config(tmp_path):
    from backends.b200_worker import B200SDXLWorker
    from oracle.unet import UNetConfig
    ucfg = UNetConfig.tiny_sdxl()
    _model_dir(tmp_path, "tiny-xl-v", ucfg, V_ZERO_SNR)
    w = _worker(tmp_path, "tiny-xl-v", B200SDXLWorker)
    assert w.pipe.scheduler_config.rescale_betas_zero_snr and w.pipe.schedule(4).prediction_type == "v_prediction"
    png, _ = w.run_job(job(seed=3, steps=4, gs=7.5))
    assert png == w.run_job(job(seed=3, steps=4, gs=7.5))[0]


# ------------------------------------------------------------------------------------------------ CLIP-H text tower
def test_clip_h_text_tower_vs_transformers():
    """SD2.x's text_encoder: OpenCLIP ViT-H's text tower in `CLIPTextModel` form (hidden 1024, 16 heads, MLP 4096,
    exact GELU) through `clip.py` against `transformers` on the same random-init weights; SD2 conditions on
    last_hidden_state.  3 of its 23 layers, like the CLIP-L / bigG geometries of `test_clip_gpu.py`: at the full
    depth the bf16 tower measured 2.27e-2 on last_hidden_state (1.19e-2 on pooler_output) on a B200, above this bar."""
    from transformers import CLIPTextConfig, CLIPTextModel
    from dreamlab_b200.clip import CLIPTextB200, clip_cfg_from_json
    torch.manual_seed(0)
    cfg = CLIPTextConfig(vocab_size=2000, hidden_size=1024, intermediate_size=4096, num_hidden_layers=3,
                         num_attention_heads=16, max_position_embeddings=77, hidden_act="gelu", projection_dim=512,
                         eos_token_id=1999, bos_token_id=1998)
    ref = CLIPTextModel(cfg).eval()
    ids = torch.randint(0, 1990, (3, 77), generator=torch.Generator().manual_seed(1))
    ids[:, 0] = 1998
    for b, n in enumerate((5, 40, 76)):
        ids[b, n:] = 1999
    with torch.no_grad():
        o = ref(ids)
    got = CLIPTextB200(ref.state_dict(), clip_cfg_from_json(cfg.to_dict()), "cuda:0").forward(ids)
    torch.cuda.synchronize()
    errs = {"last_hidden_state": max_rel_err(got["last_hidden_state"].float().cpu(), o.last_hidden_state),
            "pooler_output": max_rel_err(got["pooler_output"].float().cpu(), o.pooler_output)}
    print("CLIP-H 1024/16h/3L gelu: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    assert max(errs.values()) <= NOISE_PRED_TOL, errs


# ------------------------------------------------------------------------------------------------ attention
SD2_ATTN_CASE = dict(name="sd2_self_96", B=2, sq=9216, skv=9216, H=5, d=64, layout="fused",
                     kernel="attn_tc<1,1,4,128,0>", kt=128)


def attention_child_main():
    """Every input set of `test_attention_edges_gpu.py` on the SD2 level-0 case; exit status 1 on a failure."""
    import sys
    from test_attention_edges_gpu import INPUTS, _case, _report, run_case
    c = SD2_ATTN_CASE
    case = _case(c["name"], c["B"], c["sq"], c["skv"], c["H"], c["d"], c["layout"], c["kernel"], c["kt"])
    failures = []
    for kind in INPUTS:
        try:
            _report(case["name"], kind, *run_case(case, kind, case["kernel"], case["kt"]))
        except AssertionError as e:
            failures.append(str(e))
            print(f"  FAILED {e}", flush=True)
    sys.exit(1 if failures else 0)


def test_attention_sd2_level0_head_dim_64():
    """SD2 at 768^2: level-0 self-attention, 5 heads of 64 over S = 96 * 96 = 9216 keys (SDXL's head dim 64 runs
    up to S = 4096 only; SD1.5 at 768^2 runs head dim 40): random inputs, boundary needles, foreign rows and ramps
    per element against float64, output guards, determinism and the dispatched kernel, as `test_attention_edges_gpu.py`
    checks its cases.  In a child process of its own, like that file's knob variants: the profiler that pins the
    kernel starts there in a fresh process."""
    import subprocess
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    env = {k: v for k, v in os.environ.items() if not k.startswith("DL_ATTN_")}
    code = ("import sys; sys.path[:0] = [%r, %r]; import test_sd2_gpu as t; t.attention_child_main()"
            % (os.path.dirname(here), here))
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
    print(r.stdout, end="")
    assert r.returncode == 0, r.stdout[-6000:] + r.stderr[-6000:]
