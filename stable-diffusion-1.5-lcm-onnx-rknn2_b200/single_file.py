"""Single-file checkpoints (`*.safetensors` in the original CompVis / SGM layout) -> diffusers state dicts.

The reference loads such files with `StableDiffusionPipeline.from_single_file` /
`StableDiffusionXLPipeline.from_single_file` (reference `backends/cuda_worker.py:79-85`, `:380`; every model in
its `modes.yaml.example` is one).  diffusers is not a dependency here, so the key renaming it performs
(`convert_ldm_unet_checkpoint` / `convert_ldm_vae_checkpoint` / the text-encoder converters) is restated as
tables generated from the architecture: the b200 engine then packs the result exactly like a diffusers
directory.  Covered: SD1.x (UNet + VAE + CLIP-L text tower) and SDXL-base (UNet + VAE + CLIP-L + OpenCLIP-bigG
text towers).  The VAE's decoder and encoder halves are converted separately (`convert_vae_decoder`,
`convert_vae_encoder`); the encoder serves image-to-image only.
"""
from __future__ import annotations

from typing import Dict, Tuple

import torch

UNET_PREFIX = "model.diffusion_model."
VAE_PREFIX = "first_stage_model."

SD15_UNET = dict(in_channels=4, out_channels=4, block_out_channels=[320, 640, 1280, 1280], layers_per_block=2,
                 down_block_types=["CrossAttnDownBlock2D"] * 3 + ["DownBlock2D"], cross_attention_dim=768,
                 attention_head_dim=8, norm_num_groups=32, norm_eps=1e-5, time_cond_proj_dim=None)
SDXL_UNET = dict(in_channels=4, out_channels=4, block_out_channels=[320, 640, 1280], layers_per_block=2,
                 down_block_types=["DownBlock2D", "CrossAttnDownBlock2D", "CrossAttnDownBlock2D"],
                 cross_attention_dim=2048, attention_head_dim=[5, 10, 20], norm_num_groups=32, norm_eps=1e-5,
                 time_cond_proj_dim=None, transformer_layers_per_block=[1, 2, 10], use_linear_projection=True,
                 addition_embed_type="text_time", addition_time_embed_dim=256,
                 projection_class_embeddings_input_dim=2816)
SD_VAE = dict(latent_channels=4, out_channels=3, block_out_channels=[128, 256, 512, 512], layers_per_block=2,
              norm_num_groups=32, scaling_factor=0.18215, sample_size=512)
SDXL_VAE = dict(SD_VAE, scaling_factor=0.13025, sample_size=1024)
CLIP_L = dict(vocab_size=49408, hidden_size=768, intermediate_size=3072, num_hidden_layers=12,
              num_attention_heads=12, max_position_embeddings=77, hidden_act="quick_gelu", layer_norm_eps=1e-5,
              projection_dim=768)
CLIP_BIGG = dict(vocab_size=49408, hidden_size=1280, intermediate_size=5120, num_hidden_layers=32,
                 num_attention_heads=20, max_position_embeddings=77, hidden_act="gelu", layer_norm_eps=1e-5,
                 projection_dim=1280, architectures=["CLIPTextModelWithProjection"])

_RESNET = {"in_layers.0": "norm1", "in_layers.2": "conv1", "emb_layers.1": "time_emb_proj",
           "out_layers.0": "norm2", "out_layers.3": "conv2", "skip_connection": "conv_shortcut"}


def unet_module_map(cfg: dict) -> Dict[str, str]:
    """LDM module prefix -> diffusers module prefix for a UNet of this config (both without trailing dot).
    Resnet / transformer internals are renamed separately (`_RESNET`; transformer keys are identical)."""
    down_attn = ["CrossAttn" in t for t in cfg["down_block_types"]]
    n, lpb = len(cfg["block_out_channels"]), cfg["layers_per_block"]
    m = {"time_embed.0": "time_embedding.linear_1", "time_embed.2": "time_embedding.linear_2",
         "time_embed.cond_proj": "time_embedding.cond_proj",
         "label_emb.0.0": "add_embedding.linear_1", "label_emb.0.2": "add_embedding.linear_2",
         "input_blocks.0.0": "conv_in", "out.0": "conv_norm_out", "out.2": "conv_out",
         "middle_block.0": "mid_block.resnets.0", "middle_block.1": "mid_block.attentions.0",
         "middle_block.2": "mid_block.resnets.1"}
    idx = 1
    for i in range(n):
        for j in range(lpb):
            m[f"input_blocks.{idx}.0"] = f"down_blocks.{i}.resnets.{j}"
            if down_attn[i]:
                m[f"input_blocks.{idx}.1"] = f"down_blocks.{i}.attentions.{j}"
            idx += 1
        if i != n - 1:
            m[f"input_blocks.{idx}.0.op"] = f"down_blocks.{i}.downsamplers.0.conv"
            idx += 1
    up_attn = list(reversed(down_attn))
    idx = 0
    for i in range(n):
        for j in range(lpb + 1):
            m[f"output_blocks.{idx}.0"] = f"up_blocks.{i}.resnets.{j}"
            k = 1
            if up_attn[i]:
                m[f"output_blocks.{idx}.1"] = f"up_blocks.{i}.attentions.{j}"
                k = 2
            if j == lpb and i != n - 1:
                m[f"output_blocks.{idx}.{k}.conv"] = f"up_blocks.{i}.upsamplers.0.conv"
            idx += 1
    return m


def _rename(key: str, modules: Dict[str, str], inner: Dict[str, str]):
    """Longest module-prefix match, then the in-module rename table."""
    best = None
    for src in modules:
        if (key == src or key.startswith(src + ".")) and (best is None or len(src) > len(best)):
            best = src
    if best is None:
        return None
    rest = key[len(best):].lstrip(".")
    for a, b in inner.items():
        if rest == a or rest.startswith(a + "."):
            rest = b + rest[len(a):]
            break
    return modules[best] + ("." + rest if rest else "")


def convert_unet(sd: Dict[str, torch.Tensor], cfg: dict) -> Dict[str, torch.Tensor]:
    modules = unet_module_map(cfg)
    out = {}
    for k, v in sd.items():
        if not k.startswith(UNET_PREFIX):
            continue
        new = _rename(k[len(UNET_PREFIX):], modules, _RESNET)
        if new is None:
            raise RuntimeError(f"single-file UNet: no diffusers name for '{k}'")
        out[new] = v
    return out


_VAE_RES = {"nin_shortcut": "conv_shortcut"}
_VAE_ATTN = {"norm": "group_norm", "q": "to_q", "k": "to_k", "v": "to_v", "proj_out": "to_out.0"}


def vae_decoder_module_map(cfg: dict) -> Tuple[Dict[str, str], set]:
    n, lpb = len(cfg["block_out_channels"]), cfg["layers_per_block"]
    m = {"post_quant_conv": "post_quant_conv", "decoder.conv_in": "decoder.conv_in",
         "decoder.norm_out": "decoder.conv_norm_out", "decoder.conv_out": "decoder.conv_out",
         "decoder.mid.block_1": "decoder.mid_block.resnets.0", "decoder.mid.block_2": "decoder.mid_block.resnets.1",
         "decoder.mid.attn_1": "decoder.mid_block.attentions.0"}
    for i in range(n):                                   # LDM counts the up levels from the output side
        for j in range(lpb + 1):
            m[f"decoder.up.{n - 1 - i}.block.{j}"] = f"decoder.up_blocks.{i}.resnets.{j}"
        if i != n - 1:
            m[f"decoder.up.{n - 1 - i}.upsample.conv"] = f"decoder.up_blocks.{i}.upsamplers.0.conv"
    return m, {"decoder.mid.attn_1"}


def convert_vae_decoder(sd: Dict[str, torch.Tensor], cfg: dict) -> Dict[str, torch.Tensor]:
    modules, attn = vae_decoder_module_map(cfg)
    out = {}
    for k, v in sd.items():
        if not k.startswith(VAE_PREFIX):
            continue
        k2 = k[len(VAE_PREFIX):]
        if not (k2.startswith("decoder.") or k2.startswith("post_quant_conv.")):
            continue                                     # encoder / quant_conv: not on the path
        src = max((s for s in modules if k2 == s or k2.startswith(s + ".")), key=len, default=None)
        if src is None:
            raise RuntimeError(f"single-file VAE: no diffusers name for '{k}'")
        new = _rename(k2, modules, _VAE_ATTN if src in attn else _VAE_RES)
        if src in attn and v.dim() == 4:                 # 1x1 convs -> Linear weights
            v = v.reshape(v.shape[0], v.shape[1])
        out[new] = v
    return out


def vae_encoder_module_map(cfg: dict) -> Tuple[Dict[str, str], set]:
    """Encoder levels keep their order in LDM (unlike the decoder's up levels)."""
    n, lpb = len(cfg["block_out_channels"]), cfg["layers_per_block"]
    m = {"quant_conv": "quant_conv", "encoder.conv_in": "encoder.conv_in",
         "encoder.norm_out": "encoder.conv_norm_out", "encoder.conv_out": "encoder.conv_out",
         "encoder.mid.block_1": "encoder.mid_block.resnets.0", "encoder.mid.block_2": "encoder.mid_block.resnets.1",
         "encoder.mid.attn_1": "encoder.mid_block.attentions.0"}
    for i in range(n):
        for j in range(lpb):
            m[f"encoder.down.{i}.block.{j}"] = f"encoder.down_blocks.{i}.resnets.{j}"
        if i != n - 1:
            m[f"encoder.down.{i}.downsample.conv"] = f"encoder.down_blocks.{i}.downsamplers.0.conv"
    return m, {"encoder.mid.attn_1"}


def convert_vae_encoder(sd: Dict[str, torch.Tensor], cfg: dict) -> Dict[str, torch.Tensor]:
    """Encoder + quant_conv keys of a single-file checkpoint (empty when it has none)."""
    modules, attn = vae_encoder_module_map(cfg)
    out = {}
    for k, v in sd.items():
        if not k.startswith(VAE_PREFIX):
            continue
        k2 = k[len(VAE_PREFIX):]
        if not (k2.startswith("encoder.") or k2.startswith("quant_conv.")):
            continue
        src = max((s for s in modules if k2 == s or k2.startswith(s + ".")), key=len, default=None)
        if src is None:
            raise RuntimeError(f"single-file VAE: no diffusers name for '{k}'")
        new = _rename(k2, modules, _VAE_ATTN if src in attn else _VAE_RES)
        if src in attn and v.dim() == 4:                 # 1x1 convs -> Linear weights
            v = v.reshape(v.shape[0], v.shape[1])
        out[new] = v
    return out


def convert_clip_hf(sd, prefix: str) -> Dict[str, torch.Tensor]:
    """CLIP-L ships in transformers' own naming under `prefix` (…transformer.)."""
    return {k[len(prefix):]: v for k, v in sd.items()
            if k.startswith(prefix) and not k.endswith("position_ids")}


def convert_openclip(sd, prefix: str, cfg: dict) -> Dict[str, torch.Tensor]:
    """OpenCLIP text tower (SDXL's second encoder, `conditioner.embedders.1.model.`) -> transformers naming."""
    out = {}
    d = cfg["hidden_size"]
    for k, v in sd.items():
        if not k.startswith(prefix):
            continue
        r = k[len(prefix):]
        if r == "token_embedding.weight":
            out["text_model.embeddings.token_embedding.weight"] = v
        elif r == "positional_embedding":
            out["text_model.embeddings.position_embedding.weight"] = v
        elif r.startswith("ln_final."):
            out["text_model.final_layer_norm." + r[len("ln_final."):]] = v
        elif r == "text_projection":
            out["text_projection.weight"] = v.t().contiguous()
        elif r.startswith("transformer.resblocks."):
            parts = r.split(".")
            li, rest = parts[2], ".".join(parts[3:])
            base = f"text_model.encoder.layers.{li}."
            if rest.startswith("attn.in_proj_"):
                kind = rest[len("attn.in_proj_"):]       # weight | bias
                for n_, chunk in zip("qkv", v.reshape(3, d, *v.shape[1:])):
                    out[base + f"self_attn.{n_}_proj.{kind}"] = chunk.contiguous()
            else:
                for a, b in (("ln_1.", "layer_norm1."), ("ln_2.", "layer_norm2."), ("mlp.c_fc.", "mlp.fc1."),
                             ("mlp.c_proj.", "mlp.fc2."), ("attn.out_proj.", "self_attn.out_proj.")):
                    if rest.startswith(a):
                        out[base + b + rest[len(a):]] = v
                        break
                else:
                    raise RuntimeError(f"single-file OpenCLIP: no transformers name for '{k}'")
        elif r in ("logit_scale", "attn_mask"):
            continue
        else:
            raise RuntimeError(f"single-file OpenCLIP: no transformers name for '{k}'")
    return out


def sniff(path: str) -> dict:
    """Header-only look at a single-file checkpoint: {"variant": "sd15" | "sdxl", "cross_attention_dim": int}."""
    from safetensors import safe_open
    with safe_open(path, "pt") as f:
        keys = set(f.keys())
        sdxl = any(k.startswith("conditioner.embedders.1.") for k in keys)
        probe = next((k for k in sorted(keys) if k.startswith(UNET_PREFIX) and k.endswith("attn2.to_k.weight")), None)
        if probe is None:
            raise RuntimeError(f"{path}: not a Stable Diffusion checkpoint (no cross-attention keys)")
        dim = f.get_slice(probe).get_shape()[1]          # Linear weight [out, in]: in = cross_attention_dim
    return {"variant": "sdxl" if sdxl else "sd15", "cross_attention_dim": int(dim)}


def load_single_file(path: str) -> dict:
    """-> {"unet": (config, state dict), "vae": (...), "text_encoder": (...) | None, "text_encoder_2": (...) | None,
    "model_index": {...}} with diffusers / transformers key names."""
    from safetensors.torch import load_file
    sd = load_file(path)
    sdxl = any(k.startswith("conditioner.embedders.1.") for k in sd)
    ucfg = dict(SDXL_UNET if sdxl else SD15_UNET)
    if UNET_PREFIX + "time_embed.cond_proj.weight" in sd:            # LCM-distilled UNet
        ucfg["time_cond_proj_dim"] = sd[UNET_PREFIX + "time_embed.cond_proj.weight"].shape[1]
    probe = next(k for k in sorted(sd) if k.startswith(UNET_PREFIX) and k.endswith("attn2.to_k.weight"))
    ucfg["cross_attention_dim"] = sd[probe].shape[1]
    ucfg["in_channels"] = sd[UNET_PREFIX + "input_blocks.0.0.weight"].shape[1]     # 9: an inpainting UNet
    vcfg = dict(SDXL_VAE if sdxl else SD_VAE)
    out = {"unet": (ucfg, convert_unet(sd, ucfg)),
           "vae": (vcfg, {**convert_vae_decoder(sd, vcfg), **convert_vae_encoder(sd, vcfg)}),
           "text_encoder": None, "text_encoder_2": None,
           "model_index": {"_class_name": "StableDiffusionXLPipeline" if sdxl else "StableDiffusionPipeline",
                           "force_zeros_for_empty_prompt": True}}
    te_prefix = "conditioner.embedders.0.transformer." if sdxl else "cond_stage_model.transformer."
    te = convert_clip_hf(sd, te_prefix)
    if te:
        out["text_encoder"] = (dict(CLIP_L), te)
    if sdxl:
        te2 = convert_openclip(sd, "conditioner.embedders.1.model.", CLIP_BIGG)
        if te2:
            out["text_encoder_2"] = (dict(CLIP_BIGG), te2)
    return out
