"""Random-init weights of the named architectures, keyed like diffusers state dicts.

No checkpoints are available offline (BASELINE.json), so benchmarks and fixture model
directories use random-init weights: PyTorch's default Conv2d/Linear init distribution
(U(+-1/sqrt(fan_in)) for weights and biases), norm scales 1 / shifts 0, from a fixed seed.
Shapes follow SURVEY.md Appendix A.2 / A.3 exactly (the key set and parameter counts are
checked against the oracle modules in tests/test_synthetic.py).
"""
from __future__ import annotations

import json
import os
from types import SimpleNamespace
from typing import Dict, Tuple

import torch


def sd15_lcm_unet_cfg():
    return SimpleNamespace(in_channels=4, out_channels=4, block_out_channels=(320, 640, 1280, 1280),
                           down_attn=(True, True, True, False), layers_per_block=2,
                           cross_attention_dim=768, attention_head_dim=8, norm_num_groups=32,
                           norm_eps=1e-5, time_cond_proj_dim=256)


def sdxl_unet_cfg():
    """SDXL-base UNet (SURVEY.md App. A.2 "SDXL-base"; BASELINE config C5)."""
    return SimpleNamespace(in_channels=4, out_channels=4, block_out_channels=(320, 640, 1280),
                           down_attn=(False, True, True), layers_per_block=2,
                           cross_attention_dim=2048, attention_head_dim=(5, 10, 20),
                           norm_num_groups=32, norm_eps=1e-5, time_cond_proj_dim=None,
                           transformer_layers_per_block=(1, 2, 10), use_linear_projection=True,
                           addition_embed_type="text_time", addition_time_embed_dim=256,
                           projection_class_embeddings_input_dim=2816)


def sdxl_vae_cfg():
    return SimpleNamespace(latent_channels=4, out_channels=3, block_out_channels=(128, 256, 512, 512),
                           layers_per_block=2, norm_num_groups=32, scaling_factor=0.13025,
                           sample_size=1024)


def heads_at(cfg, i: int) -> int:
    a = cfg.attention_head_dim
    return a if isinstance(a, int) else a[i]


def depth_at(cfg, i: int) -> int:
    t = getattr(cfg, "transformer_layers_per_block", None)
    return t[i] if t else 1


def sd_vae_cfg():
    return SimpleNamespace(latent_channels=4, out_channels=3, block_out_channels=(128, 256, 512, 512),
                           layers_per_block=2, norm_num_groups=32, scaling_factor=0.18215,
                           sample_size=512)


def _resnet(s, p, cin, cout, temb):
    s[p + "norm1.weight"] = (cin,); s[p + "norm1.bias"] = (cin,)
    s[p + "conv1.weight"] = (cout, cin, 3, 3); s[p + "conv1.bias"] = (cout,)
    if temb:
        s[p + "time_emb_proj.weight"] = (cout, temb); s[p + "time_emb_proj.bias"] = (cout,)
    s[p + "norm2.weight"] = (cout,); s[p + "norm2.bias"] = (cout,)
    s[p + "conv2.weight"] = (cout, cout, 3, 3); s[p + "conv2.bias"] = (cout,)
    if cin != cout:
        s[p + "conv_shortcut.weight"] = (cout, cin, 1, 1); s[p + "conv_shortcut.bias"] = (cout,)


def _transformer(s, p, c, ctx, depth=1, linear_proj=False):
    proj = (c, c) if linear_proj else (c, c, 1, 1)
    s[p + "norm.weight"] = (c,); s[p + "norm.bias"] = (c,)
    s[p + "proj_in.weight"] = proj; s[p + "proj_in.bias"] = (c,)
    for l in range(depth):
        b = p + f"transformer_blocks.{l}."
        for i in (1, 2, 3):
            s[b + f"norm{i}.weight"] = (c,); s[b + f"norm{i}.bias"] = (c,)
        for a, kd in (("attn1", c), ("attn2", ctx)):
            s[b + f"{a}.to_q.weight"] = (c, c)
            s[b + f"{a}.to_k.weight"] = (c, kd)
            s[b + f"{a}.to_v.weight"] = (c, kd)
            s[b + f"{a}.to_out.0.weight"] = (c, c); s[b + f"{a}.to_out.0.bias"] = (c,)
        s[b + "ff.net.0.proj.weight"] = (8 * c, c); s[b + "ff.net.0.proj.bias"] = (8 * c,)
        s[b + "ff.net.2.weight"] = (c, 4 * c); s[b + "ff.net.2.bias"] = (c,)
    s[p + "proj_out.weight"] = proj; s[p + "proj_out.bias"] = (c,)


def unet_shapes(cfg) -> Dict[str, Tuple[int, ...]]:
    s: Dict[str, Tuple[int, ...]] = {}
    ch = cfg.block_out_channels
    temb = ch[0] * 4
    s["conv_in.weight"] = (ch[0], cfg.in_channels, 3, 3); s["conv_in.bias"] = (ch[0],)
    s["time_embedding.linear_1.weight"] = (temb, ch[0]); s["time_embedding.linear_1.bias"] = (temb,)
    s["time_embedding.linear_2.weight"] = (temb, temb); s["time_embedding.linear_2.bias"] = (temb,)
    if cfg.time_cond_proj_dim:
        s["time_embedding.cond_proj.weight"] = (ch[0], cfg.time_cond_proj_dim)
    if getattr(cfg, "addition_embed_type", None) == "text_time":
        pin = cfg.projection_class_embeddings_input_dim
        s["add_embedding.linear_1.weight"] = (temb, pin); s["add_embedding.linear_1.bias"] = (temb,)
        s["add_embedding.linear_2.weight"] = (temb, temb); s["add_embedding.linear_2.bias"] = (temb,)
    lin = bool(getattr(cfg, "use_linear_projection", False))
    n_lv = len(ch)
    skips = [ch[0]]
    cout = ch[0]
    for i, c in enumerate(ch):
        cin, cout = cout, c
        for j in range(cfg.layers_per_block):
            _resnet(s, f"down_blocks.{i}.resnets.{j}.", cin if j == 0 else cout, cout, temb)
            if cfg.down_attn[i]:
                _transformer(s, f"down_blocks.{i}.attentions.{j}.", cout, cfg.cross_attention_dim,
                             depth_at(cfg, i), lin)
            skips.append(cout)
        if i != len(ch) - 1:
            s[f"down_blocks.{i}.downsamplers.0.conv.weight"] = (cout, cout, 3, 3)
            s[f"down_blocks.{i}.downsamplers.0.conv.bias"] = (cout,)
            skips.append(cout)
    _resnet(s, "mid_block.resnets.0.", ch[-1], ch[-1], temb)
    _transformer(s, "mid_block.attentions.0.", ch[-1], cfg.cross_attention_dim, depth_at(cfg, n_lv - 1), lin)
    _resnet(s, "mid_block.resnets.1.", ch[-1], ch[-1], temb)
    rev, rattn = list(reversed(ch)), list(reversed(cfg.down_attn))
    prev = rev[0]
    for i, c in enumerate(rev):
        for j in range(cfg.layers_per_block + 1):
            _resnet(s, f"up_blocks.{i}.resnets.{j}.", (prev if j == 0 else c) + skips.pop(), c, temb)
            if rattn[i]:
                _transformer(s, f"up_blocks.{i}.attentions.{j}.", c, cfg.cross_attention_dim,
                             depth_at(cfg, n_lv - 1 - i), lin)
        if i != len(ch) - 1:
            s[f"up_blocks.{i}.upsamplers.0.conv.weight"] = (c, c, 3, 3)
            s[f"up_blocks.{i}.upsamplers.0.conv.bias"] = (c,)
        prev = c
    s["conv_norm_out.weight"] = (ch[0],); s["conv_norm_out.bias"] = (ch[0],)
    s["conv_out.weight"] = (cfg.out_channels, ch[0], 3, 3); s["conv_out.bias"] = (cfg.out_channels,)
    return s


def vae_decoder_shapes(cfg) -> Dict[str, Tuple[int, ...]]:
    s: Dict[str, Tuple[int, ...]] = {}
    ch = cfg.block_out_channels
    lc = cfg.latent_channels
    s["post_quant_conv.weight"] = (lc, lc, 1, 1); s["post_quant_conv.bias"] = (lc,)
    d = "decoder."
    top = ch[-1]
    s[d + "conv_in.weight"] = (top, lc, 3, 3); s[d + "conv_in.bias"] = (top,)
    _resnet(s, d + "mid_block.resnets.0.", top, top, 0)
    a = d + "mid_block.attentions.0."
    s[a + "group_norm.weight"] = (top,); s[a + "group_norm.bias"] = (top,)
    for n in ("to_q", "to_k", "to_v", "to_out.0"):
        s[a + n + ".weight"] = (top, top); s[a + n + ".bias"] = (top,)
    _resnet(s, d + "mid_block.resnets.1.", top, top, 0)
    rev = list(reversed(ch))
    prev = rev[0]
    for i, c in enumerate(rev):
        for j in range(cfg.layers_per_block + 1):
            _resnet(s, d + f"up_blocks.{i}.resnets.{j}.", prev if j == 0 else c, c, 0)
        if i != len(ch) - 1:
            s[d + f"up_blocks.{i}.upsamplers.0.conv.weight"] = (c, c, 3, 3)
            s[d + f"up_blocks.{i}.upsamplers.0.conv.bias"] = (c,)
        prev = c
    s[d + "conv_norm_out.weight"] = (ch[0],); s[d + "conv_norm_out.bias"] = (ch[0],)
    s[d + "conv_out.weight"] = (cfg.out_channels, ch[0], 3, 3); s[d + "conv_out.bias"] = (cfg.out_channels,)
    return s


def vae_encoder_shapes(cfg) -> Dict[str, Tuple[int, ...]]:
    """AutoencoderKL encoder (double_z) + quant_conv, diffusers names."""
    s: Dict[str, Tuple[int, ...]] = {}
    ch = cfg.block_out_channels
    m = 2 * cfg.latent_channels
    d = "encoder."
    s[d + "conv_in.weight"] = (ch[0], 3, 3, 3); s[d + "conv_in.bias"] = (ch[0],)
    prev = ch[0]
    for i, c in enumerate(ch):
        for j in range(cfg.layers_per_block):
            _resnet(s, d + f"down_blocks.{i}.resnets.{j}.", prev if j == 0 else c, c, 0)
        if i != len(ch) - 1:
            s[d + f"down_blocks.{i}.downsamplers.0.conv.weight"] = (c, c, 3, 3)
            s[d + f"down_blocks.{i}.downsamplers.0.conv.bias"] = (c,)
        prev = c
    top = ch[-1]
    _resnet(s, d + "mid_block.resnets.0.", top, top, 0)
    a = d + "mid_block.attentions.0."
    s[a + "group_norm.weight"] = (top,); s[a + "group_norm.bias"] = (top,)
    for n in ("to_q", "to_k", "to_v", "to_out.0"):
        s[a + n + ".weight"] = (top, top); s[a + n + ".bias"] = (top,)
    _resnet(s, d + "mid_block.resnets.1.", top, top, 0)
    s[d + "conv_norm_out.weight"] = (top,); s[d + "conv_norm_out.bias"] = (top,)
    s[d + "conv_out.weight"] = (m, top, 3, 3); s[d + "conv_out.bias"] = (m,)
    s["quant_conv.weight"] = (m, m, 1, 1); s["quant_conv.bias"] = (m,)
    return s


def random_state_dict(shapes: Dict[str, Tuple[int, ...]], seed: int = 0,
                      dtype=torch.float32) -> Dict[str, torch.Tensor]:
    g = torch.Generator().manual_seed(seed)
    sd = {}
    fan = {}
    for k, shp in shapes.items():
        if "norm" in k and len(shp) == 1:
            sd[k] = torch.ones(shp, dtype=dtype) if k.endswith("weight") else torch.zeros(shp, dtype=dtype)
            continue
        if k.endswith("weight"):
            fan_in = 1
            for d in shp[1:]:
                fan_in *= d
            fan[k[:-6]] = fan_in
        bound = 1.0 / (fan.get(k[:-6] if k.endswith("weight") else k[:-4], 1) ** 0.5)
        sd[k] = ((torch.rand(shp, generator=g) * 2 - 1) * bound).to(dtype)
    return sd


def synthetic_inputs(batch: int, height: int, width: int, steps: int, ctx_dim: int = 768,
                     seed_base: int = 1000, embed_seed: int = 1):
    """SURVEY.md §8(d) synthetic request batch: prompt embeddings N(0,1); per-sample latents and
    step noise from per-sample generators in the reference's draw order (App. A.5)."""
    g = torch.Generator().manual_seed(embed_seed)
    pe = torch.randn(batch, 77, ctx_dim, generator=g)
    lat, noise = [], []
    h, w = height // 8, width // 8
    for i in range(batch):
        gi = torch.Generator().manual_seed(seed_base + i)
        lat.append(torch.randn(1, 4, h, w, generator=gi))
        noise.append(torch.stack([torch.randn(1, 4, h, w, generator=gi) for _ in range(steps - 1)])
                     if steps > 1 else torch.zeros(1, 1, 4, h, w))
    return pe, torch.cat(lat, 0), torch.cat(noise, 1)


def clip_text_shapes(hidden: int = 768, layers: int = 12, inter: int = 3072, vocab: int = 49408,
                     positions: int = 77) -> Dict[str, Tuple[int, ...]]:
    """State-dict layout of transformers' CLIPTextModel (defaults: CLIP ViT-L/14's text tower, 123 M parameters)."""
    s: Dict[str, Tuple[int, ...]] = {}
    p = "text_model."
    s[p + "embeddings.token_embedding.weight"] = (vocab, hidden)
    s[p + "embeddings.position_embedding.weight"] = (positions, hidden)
    for i in range(layers):
        b = f"{p}encoder.layers.{i}."
        for n in ("q_proj", "k_proj", "v_proj", "out_proj"):
            s[b + f"self_attn.{n}.weight"] = (hidden, hidden)
            s[b + f"self_attn.{n}.bias"] = (hidden,)
        for n in ("layer_norm1", "layer_norm2"):
            s[b + n + ".weight"] = (hidden,)
            s[b + n + ".bias"] = (hidden,)
        s[b + "mlp.fc1.weight"] = (inter, hidden)
        s[b + "mlp.fc1.bias"] = (inter,)
        s[b + "mlp.fc2.weight"] = (hidden, inter)
        s[b + "mlp.fc2.bias"] = (hidden,)
    s[p + "final_layer_norm.weight"] = (hidden,)
    s[p + "final_layer_norm.bias"] = (hidden,)
    return s


def write_text_encoder(model_dir: str, hidden: int = 768, layers: int = 12, heads: int = 12, inter: int = 3072,
                       seed: int = 2, dtype=torch.float16) -> None:
    """`text_encoder/` (transformers layout, random init) under a model dir written by write_model_dir: with it the
    worker runs the prompt through the on-device CLIP tower, as a real checkpoint would.  No tokenizer files are
    written (there is no vocabulary offline): the worker falls back to its hashed stand-in token ids."""
    from safetensors.torch import save_file
    te = os.path.join(model_dir, "text_encoder")
    os.makedirs(te, exist_ok=True)
    with open(os.path.join(te, "config.json"), "w") as f:
        json.dump({"_class_name": "CLIPTextModel", "architectures": ["CLIPTextModel"], "model_type": "clip_text_model",
                   "vocab_size": 49408, "hidden_size": hidden, "intermediate_size": inter, "num_hidden_layers": layers,
                   "num_attention_heads": heads, "max_position_embeddings": 77, "hidden_act": "quick_gelu",
                   "layer_norm_eps": 1e-5, "eos_token_id": 49407, "bos_token_id": 49406, "pad_token_id": 1}, f)
    sd = random_state_dict(clip_text_shapes(hidden, layers, inter), seed, dtype)
    # embeddings at the scale of a trained tower (transformers initialises them N(0, 0.02))
    for k in list(sd):
        if "embedding" in k:
            sd[k] = (sd[k].float() * (0.02 * (3.0 * sd[k].shape[1]) ** 0.5)).to(dtype)
    save_file(sd, os.path.join(te, "model.safetensors"))


def write_model_dir(path: str, unet_cfg=None, vae_cfg=None, seed: int = 0, dtype=torch.float16,
                    vae_encoder: bool = False):
    """A diffusers-layout directory (model_index.json, unet/, vae/) with random-init weights —
    what `MODEL_ROOT/MODEL` points at for offline tests of the b200 worker.  vae_encoder: also write the
    VAE's encoder + quant_conv (image-to-image), from a seed of their own: the decoder weights are the same
    either way."""
    from safetensors.torch import save_file
    unet_cfg = unet_cfg or sd15_lcm_unet_cfg()
    vae_cfg = vae_cfg or sd_vae_cfg()
    os.makedirs(os.path.join(path, "unet"), exist_ok=True)
    os.makedirs(os.path.join(path, "vae"), exist_ok=True)
    with open(os.path.join(path, "model_index.json"), "w") as f:
        sdxl = getattr(unet_cfg, "addition_embed_type", None) == "text_time"
        json.dump({"_class_name": "StableDiffusionXLPipeline" if sdxl else "StableDiffusionPipeline",
                   "unet": ["diffusers", "UNet2DConditionModel"],
                   "vae": ["diffusers", "AutoencoderKL"], "scheduler": ["diffusers", "LCMScheduler"]}, f)
    down = ["CrossAttnDownBlock2D" if a else "DownBlock2D" for a in unet_cfg.down_attn]
    ucj = {"_class_name": "UNet2DConditionModel", "in_channels": unet_cfg.in_channels,
           "out_channels": unet_cfg.out_channels,
           "block_out_channels": list(unet_cfg.block_out_channels), "down_block_types": down,
           "layers_per_block": unet_cfg.layers_per_block,
           "cross_attention_dim": unet_cfg.cross_attention_dim,
           "attention_head_dim": (list(unet_cfg.attention_head_dim)
                                  if isinstance(unet_cfg.attention_head_dim, (tuple, list)) else unet_cfg.attention_head_dim),
           "norm_num_groups": unet_cfg.norm_num_groups, "norm_eps": unet_cfg.norm_eps,
           "time_cond_proj_dim": unet_cfg.time_cond_proj_dim}
    if getattr(unet_cfg, "addition_embed_type", None):          # SDXL-class keys
        ucj.update(transformer_layers_per_block=list(unet_cfg.transformer_layers_per_block),
                   use_linear_projection=bool(unet_cfg.use_linear_projection),
                   addition_embed_type=unet_cfg.addition_embed_type,
                   addition_time_embed_dim=unet_cfg.addition_time_embed_dim,
                   projection_class_embeddings_input_dim=unet_cfg.projection_class_embeddings_input_dim)
    with open(os.path.join(path, "unet", "config.json"), "w") as f:
        json.dump(ucj, f)
    with open(os.path.join(path, "vae", "config.json"), "w") as f:
        json.dump({"_class_name": "AutoencoderKL", "latent_channels": vae_cfg.latent_channels,
                   "out_channels": vae_cfg.out_channels,
                   "block_out_channels": list(vae_cfg.block_out_channels),
                   "layers_per_block": vae_cfg.layers_per_block,
                   "norm_num_groups": vae_cfg.norm_num_groups,
                   "scaling_factor": vae_cfg.scaling_factor, "sample_size": vae_cfg.sample_size}, f)
    save_file(random_state_dict(unet_shapes(unet_cfg), seed, dtype),
              os.path.join(path, "unet", "diffusion_pytorch_model.safetensors"))
    vae_sd = random_state_dict(vae_decoder_shapes(vae_cfg), seed + 1, dtype)
    if vae_encoder:
        vae_sd.update(random_state_dict(vae_encoder_shapes(vae_cfg), seed + 3, dtype))
    save_file(vae_sd, os.path.join(path, "vae", "diffusion_pytorch_model.safetensors"))
    return path
