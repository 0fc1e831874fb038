"""Image-to-image, host side: the strength schedule (`LCMScheduler.set_timesteps(n, strength)`), the oracle
encoder's architecture and key names, the single-file encoder conversion and the pool's batch key."""
from types import SimpleNamespace

import pytest
import torch

from dreamlab_b200 import single_file as sf
from dreamlab_b200 import synthetic as syn
from dreamlab_b200.scheduler import LCMSchedule, alphas_cumprod, lcm_timesteps


@pytest.mark.parametrize("n,strength,want", [
    (4, 1.0, [999, 759, 499, 259]),
    (4, 0.5, [499, 379, 259, 139]),
    (4, 0.8, [799, 599, 399, 199]),
    (8, 0.3, [299, 279, 239, 199, 159, 119, 79, 39]),
])
def test_strength_tables(n, strength, want):
    from oracle.img2img import OracleLCMSchedulerImg2Img
    assert lcm_timesteps(n, strength) == want
    assert LCMSchedule(n, strength).timesteps == want
    assert OracleLCMSchedulerImg2Img().set_timesteps(n, strength).tolist() == want


@pytest.mark.parametrize("n,strength", [(4, 0.05), (4, 0.0), (4, -0.1), (4, 1.5), (50, 0.9)])
def test_strength_value_errors(n, strength):
    from oracle.img2img import OracleLCMSchedulerImg2Img
    with pytest.raises(ValueError):
        lcm_timesteps(n, strength)
    with pytest.raises(ValueError):
        OracleLCMSchedulerImg2Img().set_timesteps(n, strength)


def test_strength_one_is_todays_schedule():
    for n in range(1, 51):
        assert lcm_timesteps(n, 1.0) == lcm_timesteps(n)
        a, b = LCMSchedule(n), LCMSchedule(n, 1.0)
        assert a.timesteps == b.timesteps
        assert [a.coeffs(i) for i in range(n)] == [b.coeffs(i) for i in range(n)]


def test_truncated_schedule_coefficients_follow_the_list():
    s = LCMSchedule(4, 0.5)
    ac = alphas_cumprod()
    for i, t in enumerate(s.timesteps):
        prev = s.timesteps[i + 1] if i + 1 < 4 else t
        assert s.coeffs(i)[0] == ac[t].sqrt().item()
        assert s.coeffs(i)[4] == ac[prev].sqrt().item()
    sa, sb = s.add_noise_coeffs()
    assert sa == (ac[499] ** 0.5).item() and sb == ((1 - ac[499]) ** 0.5).item()


def test_oracle_encoder_parameter_count_and_names():
    from oracle.img2img import OracleVAEEncoder
    from oracle.vae import OracleVAEDecoder
    enc = OracleVAEEncoder()
    n_enc = sum(p.numel() for p in enc.encoder.parameters())
    n_all = sum(p.numel() for p in enc.parameters())
    n_dec = sum(p.numel() for p in OracleVAEDecoder().parameters())
    assert n_enc == 34_163_592 and n_all == 34_163_664
    assert n_all + n_dec == 83_653_863                       # the published AutoencoderKL (SD1.5) count
    keys = set(enc.state_dict())
    for k in ("encoder.conv_in.weight", "encoder.down_blocks.0.resnets.1.conv2.weight",
              "encoder.down_blocks.1.resnets.0.conv_shortcut.weight", "encoder.down_blocks.2.downsamplers.0.conv.bias",
              "encoder.mid_block.attentions.0.group_norm.weight", "encoder.mid_block.attentions.0.to_out.0.bias",
              "encoder.mid_block.resnets.1.norm2.bias", "encoder.conv_norm_out.weight", "encoder.conv_out.weight",
              "quant_conv.weight"):
        assert k in keys, k
    assert "encoder.down_blocks.3.downsamplers.0.conv.weight" not in keys
    shapes = syn.vae_encoder_shapes(syn.sd_vae_cfg())
    assert {k: tuple(v.shape) for k, v in enc.state_dict().items()} == shapes


def _meta(shapes):
    return {k: torch.empty(s, device="meta") for k, s in shapes.items()}


@pytest.mark.parametrize("cfg", [sf.SD_VAE, sf.SDXL_VAE])
def test_convert_vae_encoder_is_a_bijection(cfg):
    shapes = syn.vae_encoder_shapes(SimpleNamespace(**{**cfg, "block_out_channels": tuple(cfg["block_out_channels"])}))
    modules, attn = sf.vae_encoder_module_map(cfg)
    inv = {v: k for k, v in modules.items()}
    ldm = {}
    for k, s in shapes.items():
        mod = max((m for m in inv if k.startswith(m + ".")), key=len)
        rest = k[len(mod) + 1:]
        table = sf._VAE_ATTN if inv[mod] in attn else sf._VAE_RES
        for a, b in table.items():
            if rest == b or rest.startswith(b + "."):
                rest = a + rest[len(b):]
                break
        if inv[mod] in attn and len(s) == 2:
            s = tuple(s) + (1, 1)
        ldm[sf.VAE_PREFIX + inv[mod] + "." + rest] = s
    assert "first_stage_model.encoder.down.0.block.0.norm1.weight" in ldm      # levels keep their order
    assert "first_stage_model.encoder.down.2.downsample.conv.weight" in ldm
    assert "first_stage_model.encoder.mid.attn_1.q.weight" in ldm
    assert "first_stage_model.encoder.down.1.block.0.nin_shortcut.weight" in ldm
    ldm["first_stage_model.decoder.conv_in.weight"] = (512, 4, 3, 3)           # decoder keys are skipped
    back = sf.convert_vae_encoder(_meta(ldm), cfg)
    assert set(back) == set(shapes)
    for k in shapes:
        assert tuple(back[k].shape) == tuple(shapes[k]), k


def test_batch_key_separates_img2img_by_strength():
    from backends.worker_pool import _batch_key

    def j(**kw):
        return SimpleNamespace(req=SimpleNamespace(prompt="p", size="512x512", num_inference_steps=4,
                                                   guidance_scale=1.0, **kw))
    t2i = _batch_key(j())
    assert t2i == ("512x512", 4, (None, 0))                       # text-to-image keys are unchanged
    assert _batch_key(j(strength=0.5)) == t2i                    # a strength without an image is ignored
    a = _batch_key(j(init_image=b"png", strength=0.5))
    b = _batch_key(j(init_image=b"png", strength=0.6))
    c = _batch_key(j(init_image=b"other", strength=0.5))
    d = _batch_key(j(init_image=b"png"))
    assert a == t2i + (("img2img", 0.5),) and a != b and a == c
    assert d == t2i + (("img2img", 0.8),)
    assert _batch_key(j(init_image=b"png", strength=0.5), same_guidance=True) == a + (1.0,)


def test_genspec_has_optional_img2img_fields():
    from backends.base import GenSpec
    g = GenSpec(prompt="p", size="64x64", steps=4, cfg=1.0)
    assert g.init_image is None and g.strength is None
