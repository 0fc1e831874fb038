"""Oracle image-to-image (test infrastructure).

fp32 PyTorch restatement of diffusers' `LatentConsistencyModelImg2ImgPipeline` (>= 0.25) with
`AutoencoderKL.encode` / `tiled_encode`, `DiagonalGaussianDistribution.sample` and
`LCMScheduler.set_timesteps(n, strength=...)` / `add_noise`.  diffusers is not installable offline,
so this is restated from its source and unpinned at the diffusers boundary (DESIGN.md §2), like the
rest of the oracle.  Key names follow the diffusers `AutoencoderKL` state dict (`encoder.*`,
`quant_conv.*`).  The init image, the posterior draw, the add_noise draw and the per-step noise are
inputs, so the CUDA path and the oracle consume identical randomness.
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from .pipeline import build_random_init, denormalize_to_u8
from .scheduler import OracleLCMScheduler, guidance_scale_embedding
from .unet import ResnetBlock2D
from .vae import VAEConfig, VAEMid, _blend_h, _blend_v


class Downsample2D(nn.Module):
    """`Downsample2D(use_conv=True, padding=0)`: F.pad(x, (0,1,0,1)) then conv3x3 stride 2, no padding."""

    def __init__(self, c):
        super().__init__()
        self.conv = nn.Conv2d(c, c, 3, stride=2, padding=0)

    def forward(self, x):
        return self.conv(F.pad(x, (0, 1, 0, 1), mode="constant", value=0))


class VAEDownBlock(nn.Module):
    """`DownEncoderBlock2D`: resnets (eps 1e-6, no temb), then the optional downsampler."""

    def __init__(self, cin, cout, n, groups, down):
        super().__init__()
        self.resnets = nn.ModuleList(
            [ResnetBlock2D(cin if i == 0 else cout, cout, None, groups, 1e-6) for i in range(n)])
        self.downsamplers = nn.ModuleList([Downsample2D(cout)]) if down else None

    def forward(self, x):
        for r in self.resnets:
            x = r(x)
        if self.downsamplers is not None:
            x = self.downsamplers[0](x)
        return x


class Encoder(nn.Module):
    """diffusers `Encoder(double_z=True)`: 2 * latent_channels output channels (mean | logvar)."""

    def __init__(self, cfg: VAEConfig):
        super().__init__()
        ch = cfg.block_out_channels
        g = cfg.norm_num_groups
        self.conv_in = nn.Conv2d(3, ch[0], 3, padding=1)
        self.down_blocks = nn.ModuleList()
        prev = ch[0]
        for i, c in enumerate(ch):
            self.down_blocks.append(VAEDownBlock(prev, c, cfg.layers_per_block, g, down=i != len(ch) - 1))
            prev = c
        self.mid_block = VAEMid(ch[-1], g)
        self.conv_norm_out = nn.GroupNorm(g, ch[-1], eps=1e-6)
        self.conv_out = nn.Conv2d(ch[-1], 2 * cfg.latent_channels, 3, padding=1)

    def forward(self, x):
        x = self.conv_in(x)
        for b in self.down_blocks:
            x = b(x)
        x = self.mid_block(x)
        return self.conv_out(F.silu(self.conv_norm_out(x)))


class OracleVAEEncoder(nn.Module):
    """`AutoencoderKL.encode` up to the posterior's moments: encoder + quant_conv (1x1, 2L -> 2L)."""

    def __init__(self, cfg: VAEConfig = VAEConfig()):
        super().__init__()
        self.cfg = cfg
        self.encoder = Encoder(cfg)
        self.quant_conv = nn.Conv2d(2 * cfg.latent_channels, 2 * cfg.latent_channels, 1)

    def encode(self, x):
        return self.quant_conv(self.encoder(x))

    def tiled_encode(self, x):
        """`AutoencoderKL.tiled_encode`: sample_size tiles at stride 0.75 tile, each encoded on its own,
        moments blended with the (already blended) upper / left neighbour, cropped, concatenated."""
        tile = self.cfg.sample_size
        tile_latent = tile // 8
        overlap = int(tile * (1 - 0.25))
        blend = int(tile_latent * 0.25)
        limit = tile_latent - blend
        rows = []
        for i in range(0, x.shape[2], overlap):
            rows.append([self.encode(x[:, :, i:i + tile, j:j + tile]) for j in range(0, x.shape[3], overlap)])
        out_rows = []
        for i, row in enumerate(rows):
            out_row = []
            for j, t in enumerate(row):
                if i > 0:
                    t = _blend_v(rows[i - 1][j], t, blend)
                if j > 0:
                    t = _blend_h(row[j - 1], t, blend)
                out_row.append(t[:, :, :limit, :limit])
            out_rows.append(torch.cat(out_row, dim=3))
        return torch.cat(out_rows, dim=2)

    def forward(self, x, tiling: bool = True):
        if tiling and (x.shape[-1] > self.cfg.sample_size or x.shape[-2] > self.cfg.sample_size):
            return self.tiled_encode(x)
        return self.encode(x)


def build_random_init_encoder(vae_cfg: VAEConfig = None, seed: int = 0) -> OracleVAEEncoder:
    """Random-init encoder weights (default PyTorch inits) from a seed of its own, so that the UNet and the
    decoder of `build_random_init(seed=seed)` are unchanged by it."""
    g = torch.random.get_rng_state()
    torch.manual_seed(seed + 7919)
    enc = OracleVAEEncoder(vae_cfg or VAEConfig()).eval()
    torch.random.set_rng_state(g)
    for p in enc.parameters():
        p.requires_grad_(False)
    return enc


def build_random_init_img2img(unet_cfg=None, vae_cfg: VAEConfig = None, seed: int = 0):
    unet, vae = build_random_init(unet_cfg, vae_cfg, seed)
    return unet, vae, build_random_init_encoder(vae_cfg, seed)


def preprocess(image_u8) -> torch.Tensor:
    """`VaeImageProcessor.preprocess` for an RGB u8 image of the exact size (no resize): NHWC u8 ->
    NCHW fp32 2 * (x / 255) - 1."""
    x = torch.as_tensor(np.asarray(image_u8)).to(torch.float32) / 255.0
    return (2.0 * x - 1.0).permute(0, 3, 1, 2).contiguous()


def sample_posterior(moments, eps, scaling_factor):
    """`DiagonalGaussianDistribution(moments).sample()` with the draw `eps`, times scaling_factor."""
    mean, logvar = torch.chunk(moments, 2, dim=1)
    logvar = torch.clamp(logvar, -30.0, 20.0)
    std = torch.exp(0.5 * logvar)
    return scaling_factor * (mean + std * eps)


class OracleLCMSchedulerImg2Img(OracleLCMScheduler):
    def set_timesteps(self, num_inference_steps: int, strength: float = 1.0):
        """`LCMScheduler.set_timesteps(n, strength=strength)`."""
        if not 0.0 < strength <= 1.0:
            raise ValueError(f"strength must be in (0, 1], got {strength}")
        k = self.num_train_timesteps // self.original_inference_steps
        origin = np.asarray(list(range(1, int(self.original_inference_steps * strength) + 1))) * k - 1
        if len(origin) // num_inference_steps < 1:
            raise ValueError(f"strength {strength}: {len(origin)} original timesteps < {num_inference_steps} steps")
        origin = origin[::-1].copy()
        idx = np.floor(np.linspace(0, len(origin), num=num_inference_steps, endpoint=False)).astype(np.int64)
        self.timesteps = torch.from_numpy(origin[idx]).to(torch.int64)
        self.num_inference_steps = num_inference_steps
        self._step_index = None
        return self.timesteps

    def add_noise(self, original, noise, t):
        a = self.alphas_cumprod[int(t)]
        return a ** 0.5 * original + (1 - a) ** 0.5 * noise


@torch.no_grad()
def run_pipeline_img2img(unet, vae, encoder: OracleVAEEncoder, prompt_embeds: torch.Tensor, image_u8,
                         eps_s: torch.Tensor, eps_n: torch.Tensor, step_noise: torch.Tensor,
                         num_inference_steps: int, strength: float, guidance_scale: float = 1.0,
                         tiling: bool = True, output_type: str = "u8", record: Optional[dict] = None):
    """`LatentConsistencyModelImg2ImgPipeline.__call__(prompt_embeds=..., image=..., strength=...)`:
    preprocess -> encode (+ quant_conv) -> posterior sample (eps_s) * scaling_factor -> add_noise (eps_n) at the
    first timestep of the strength schedule -> the LCM loop -> decode.  u8 NHWC images (or the final latents)."""
    sched = OracleLCMSchedulerImg2Img()
    timesteps = sched.set_timesteps(num_inference_steps, strength)
    B = prompt_embeds.shape[0]
    moments = encoder(preprocess(image_u8), tiling=tiling)
    x0 = sample_posterior(moments, eps_s, vae.cfg.scaling_factor)
    latents = sched.add_noise(x0, eps_n, timesteps[0])
    w_emb = None
    if unet.cfg.time_cond_proj_dim:
        w_emb = guidance_scale_embedding(torch.full((B,), guidance_scale - 1.0), unet.cfg.time_cond_proj_dim)
    if record is not None:
        record.update(timesteps=timesteps.clone(), moments=moments.clone(), init_latents=latents.clone(),
                      noise_pred=[], latents=[])
    for i, t in enumerate(timesteps):
        eps = unet(latents, t, prompt_embeds, w_emb)
        z = step_noise[i] if i < num_inference_steps - 1 else None
        latents, _ = sched.step(eps, int(t), latents, noise=z)
        if record is not None:
            record["noise_pred"].append(eps.clone())
            record["latents"].append(latents.clone())
    if output_type == "latent":
        return latents
    image = vae(latents / vae.cfg.scaling_factor, tiling=tiling)
    if record is not None:
        record["image_f32"] = image.clone()
    return denormalize_to_u8(image)
