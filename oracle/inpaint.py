"""Oracle inpainting (test infrastructure).

fp32 PyTorch restatement of diffusers' `StableDiffusionInpaintPipeline.__call__` with `LCMScheduler` swapped in (the
pipeline of diffusers' LCM-LoRA inpainting guide, and what the same pipeline does with an LCM-distilled UNet):
`retrieve_timesteps` + `get_timesteps` (the full schedule truncated by strength, `set_begin_index`), `mask_processor`
(grayscale, / 255, binarise at 0.5), `masked_image = image * (mask < 0.5)`, `prepare_latents` (image latents only for
a 4-channel UNet or strength < 1; pure noise at strength 1), `prepare_mask_latents` (nearest downsample, masked image
encoded), the 9-channel UNet input `cat([latents, mask, masked_image_latents])` or the 4-channel UNet's blend towards
the noised image latents, classifier-free guidance for UNets without `time_cond_proj_dim`.  diffusers is not
installable offline, so this is restated from its source and unpinned at the diffusers boundary (DESIGN.md §2).
Every random draw is an input, so the CUDA path and the oracle consume identical randomness.
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch
import torch.nn.functional as F

from .img2img import OracleLCMSchedulerImg2Img, OracleVAEEncoder, preprocess, sample_posterior
from .pipeline import denormalize_to_u8
from .scheduler import guidance_scale_embedding


class OracleLCMSchedulerInpaint(OracleLCMSchedulerImg2Img):
    def set_begin_index(self, begin_index: int):
        """`set_begin_index`: the first `step` runs at this index of the full schedule."""
        self._step_index = begin_index


def get_timesteps(sched: OracleLCMSchedulerInpaint, num_inference_steps: int, strength: float):
    """`StableDiffusionInpaintPipeline.get_timesteps` (scheduler.order = 1) -> (timesteps, steps that run)."""
    init_timestep = min(int(num_inference_steps * strength), num_inference_steps)
    t_start = max(num_inference_steps - init_timestep, 0)
    timesteps = sched.timesteps[t_start:]
    sched.set_begin_index(t_start)
    return timesteps, num_inference_steps - t_start


def truncated_schedule(num_inference_steps: int, strength: float):
    """`retrieve_timesteps` (set_timesteps(n)) + `get_timesteps`, with the pipeline's check -> (timesteps, t_start)."""
    sched = OracleLCMSchedulerInpaint()
    sched.set_timesteps(num_inference_steps)
    timesteps, n = get_timesteps(sched, num_inference_steps, strength)
    if n < 1:
        raise ValueError(f"strength {strength} leaves {n} of num_inference_steps={num_inference_steps} steps")
    return timesteps, num_inference_steps - n


def preprocess_mask(mask_u8) -> torch.Tensor:
    """`mask_processor.preprocess` of an "L" mask of the exact size (no resize): [B,H,W] u8 -> [B,1,H,W] fp32 in
    {0, 1}: / 255, then binarised (< 0.5 -> 0, else 1)."""
    m = torch.as_tensor(np.asarray(mask_u8)).to(torch.float32) / 255.0
    m = torch.where(m < 0.5, torch.zeros_like(m), torch.ones_like(m))
    return m[:, None].contiguous()


def prepare_mask_latents(mask, masked_image, encoder: OracleVAEEncoder, eps_m, scaling_factor, height, width,
                         do_cfg: bool, tiling: bool = True):
    """`prepare_mask_latents`: nearest downsample of the binarised mask to the latent size, the masked image's scaled
    posterior sample (draw eps_m); both doubled under classifier-free guidance."""
    mask = F.interpolate(mask, size=(height // 8, width // 8))
    masked_image_latents = sample_posterior(encoder(masked_image, tiling=tiling), eps_m, scaling_factor)
    if do_cfg:
        mask = torch.cat([mask] * 2)
        masked_image_latents = torch.cat([masked_image_latents] * 2)
    return mask, masked_image_latents


@torch.no_grad()
def run_pipeline_inpaint(unet, vae, encoder: OracleVAEEncoder, prompt_embeds: torch.Tensor, image_u8, mask_u8,
                         eps_s: Optional[torch.Tensor], eps_n: torch.Tensor, eps_m: torch.Tensor,
                         step_noise: torch.Tensor, num_inference_steps: int, strength: float = 1.0,
                         guidance_scale: float = 1.0, negative_prompt_embeds: Optional[torch.Tensor] = None,
                         tiling: bool = True, output_type: str = "u8", record: Optional[dict] = None):
    """`StableDiffusionInpaintPipeline.__call__(prompt_embeds=..., image=..., mask_image=..., strength=...)` with
    `LCMScheduler`.  eps_s: the image's posterior draw (unused, may be None, for a 9-channel UNet at strength 1);
    eps_n: the latents / add_noise draw; eps_m: the masked image's posterior draw; step_noise: one draw per non-final
    step of the truncated schedule.  -> u8 NHWC images (or the final latents)."""
    sched = OracleLCMSchedulerInpaint()
    sched.set_timesteps(num_inference_steps)
    timesteps, n = get_timesteps(sched, num_inference_steps, strength)
    if n < 1:
        raise ValueError(f"strength {strength} leaves no inference step")
    B = prompt_embeds.shape[0]
    H, W = np.asarray(image_u8).shape[1:3]
    sf = vae.cfg.scaling_factor
    nine = unet.cfg.in_channels == 9
    do_cfg = guidance_scale > 1.0 and not unet.cfg.time_cond_proj_dim
    init_image = preprocess(image_u8)
    mask_condition = preprocess_mask(mask_u8)
    masked_image = init_image * (mask_condition < 0.5)
    is_strength_max = strength == 1.0
    image_latents = None
    if not nine or not is_strength_max:
        image_latents = sample_posterior(encoder(init_image, tiling=tiling), eps_s, sf)
    noise = eps_n
    latents = noise * sched.init_noise_sigma if is_strength_max else sched.add_noise(image_latents, noise, timesteps[0])
    mask, masked_image_latents = prepare_mask_latents(mask_condition, masked_image, encoder, eps_m, sf, H, W, do_cfg,
                                                      tiling)
    ctx = prompt_embeds
    if do_cfg:
        neg = torch.zeros_like(prompt_embeds) if negative_prompt_embeds is None else negative_prompt_embeds
        ctx = torch.cat([neg, prompt_embeds], 0)
    w_emb = None
    if unet.cfg.time_cond_proj_dim:
        w_emb = guidance_scale_embedding(torch.full((B,), guidance_scale - 1.0), unet.cfg.time_cond_proj_dim)
    if record is not None:
        record.update(timesteps=timesteps.clone(), init_latents=latents.clone(), mask=mask[:B, 0].clone(),
                      masked_image_latents=masked_image_latents[:B].clone(), noise_pred=[], noise_pred_raw=[],
                      latents=[])
        if image_latents is not None:
            record["image_latents"] = image_latents.clone()
    for i, t in enumerate(timesteps):
        x = torch.cat([latents] * 2) if do_cfg else latents
        if nine:
            x = torch.cat([x, mask, masked_image_latents], dim=1)
        eps = unet(x, t, ctx, w_emb)
        if do_cfg:
            if record is not None:
                record["noise_pred_raw"].append(eps.clone())
            e_u, e_t = eps.chunk(2)
            eps = e_u + guidance_scale * (e_t - e_u)
        z = step_noise[i] if i < n - 1 else None
        latents, _ = sched.step(eps, int(t), latents, noise=z)
        if not nine:
            init_mask = mask.chunk(2)[0] if do_cfg else mask
            proper = image_latents
            if i < n - 1:
                proper = sched.add_noise(proper, noise, timesteps[i + 1])
            latents = (1 - init_mask) * proper + init_mask * latents
        if record is not None:
            record["noise_pred"].append(eps.clone())
            record["latents"].append(latents.clone())
    if output_type == "latent":
        return latents
    image = vae(latents / sf, tiling=tiling)
    if record is not None:
        record["image_f32"] = image.clone()
    return denormalize_to_u8(image)
