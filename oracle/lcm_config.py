"""Oracle `LCMScheduler.from_config(model scheduler config)` and SD2.x-class presets (test infrastructure).

The reference builds its scheduler from the model (`LCMScheduler.from_config(pipe.scheduler.config)`,
`backends/cuda_worker.py:88`, `:387`), so a model's `scheduler_config.json` decides the beta schedule, the
prediction type (`epsilon`, `v_prediction`, `sample`), the x0 clamp and the zero-terminal-SNR rescale.  This restates
those parts of diffusers' `LCMScheduler.__init__` / `step` (and `betas_for_alpha_bar`, `rescale_zero_terminal_snr`)
on top of the oracle schedulers in `scheduler.py`, `img2img.py` and `inpaint.py`, which stay as they are: their
defaults are SD1.5's constants, the default of every key here.

`configured(config)` runs the existing oracle loops (`run_pipeline_sdxl`, `run_pipeline_img2img`,
`run_pipeline_inpaint`, `truncated_schedule`) with this scheduler in place of the default one;
`run_pipeline_cfg` is the `StableDiffusionPipeline` loop with classifier-free guidance that SD2.x-class models run.
"""
from __future__ import annotations

import contextlib
import math
from typing import Optional

import torch

from .inpaint import OracleLCMSchedulerInpaint
from .pipeline import denormalize_to_u8
from .unet import UNetConfig

_INIT_KEYS = ("num_train_timesteps", "beta_start", "beta_end", "beta_schedule", "trained_betas",
              "original_inference_steps", "clip_sample", "clip_sample_range", "set_alpha_to_one", "steps_offset",
              "prediction_type", "thresholding", "dynamic_thresholding_ratio", "sample_max_value",
              "timestep_spacing", "timestep_scaling", "rescale_betas_zero_snr")


def betas_for_alpha_bar(num_diffusion_timesteps: int, max_beta: float = 0.999) -> torch.Tensor:
    def alpha_bar_fn(t):
        return math.cos((t + 0.008) / 1.008 * math.pi / 2) ** 2
    betas = []
    for i in range(num_diffusion_timesteps):
        t1 = i / num_diffusion_timesteps
        t2 = (i + 1) / num_diffusion_timesteps
        betas.append(min(1 - alpha_bar_fn(t2) / alpha_bar_fn(t1), max_beta))
    return torch.tensor(betas, dtype=torch.float32)


def rescale_zero_terminal_snr(betas: torch.Tensor) -> torch.Tensor:
    alphas = 1.0 - betas
    alphas_cumprod = torch.cumprod(alphas, dim=0)
    alphas_bar_sqrt = alphas_cumprod.sqrt()
    alphas_bar_sqrt_0 = alphas_bar_sqrt[0].clone()
    alphas_bar_sqrt_T = alphas_bar_sqrt[-1].clone()
    alphas_bar_sqrt -= alphas_bar_sqrt_T
    alphas_bar_sqrt *= alphas_bar_sqrt_0 / (alphas_bar_sqrt_0 - alphas_bar_sqrt_T)
    alphas_bar = alphas_bar_sqrt ** 2
    alphas = alphas_bar[1:] / alphas_bar[:-1]
    alphas = torch.cat([alphas_bar[0:1], alphas])
    return 1 - alphas


class OracleLCMSchedulerConfigured(OracleLCMSchedulerInpaint):
    """`LCMScheduler(**config)`: every `set_timesteps` / `add_noise` / `set_begin_index` of the oracle schedulers,
    with the config's alphas_cumprod, prediction type and clamp."""

    def __init__(self, num_train_timesteps: int = 1000, beta_start: float = 0.00085, beta_end: float = 0.012,
                 beta_schedule: str = "scaled_linear", trained_betas=None, original_inference_steps: int = 50,
                 clip_sample: bool = False, clip_sample_range: float = 1.0, set_alpha_to_one: bool = True,
                 prediction_type: str = "epsilon", timestep_scaling: float = 10.0,
                 rescale_betas_zero_snr: bool = False, **_unused):
        super().__init__(num_train_timesteps, beta_start, beta_end, original_inference_steps, timestep_scaling)
        if trained_betas is not None:
            betas = torch.tensor(trained_betas, dtype=torch.float32)
        elif beta_schedule == "linear":
            betas = torch.linspace(beta_start, beta_end, num_train_timesteps, dtype=torch.float32)
        elif beta_schedule == "scaled_linear":
            betas = torch.linspace(beta_start ** 0.5, beta_end ** 0.5, num_train_timesteps, dtype=torch.float32) ** 2
        elif beta_schedule == "squaredcos_cap_v2":
            betas = betas_for_alpha_bar(num_train_timesteps)
        else:
            raise NotImplementedError(beta_schedule)
        if rescale_betas_zero_snr:
            betas = rescale_zero_terminal_snr(betas)
        self.alphas_cumprod = torch.cumprod(1.0 - betas, dim=0)
        self.final_alpha_cumprod = torch.tensor(1.0) if set_alpha_to_one else self.alphas_cumprod[0]
        self.prediction_type = prediction_type
        self.clip_sample = clip_sample
        self.clip_sample_range = clip_sample_range

    @classmethod
    def from_config(cls, config: Optional[dict]) -> "OracleLCMSchedulerConfigured":
        return cls(**{k: v for k, v in (config or {}).items() if k in _INIT_KEYS})

    def step(self, model_output: torch.Tensor, timestep: int, sample: torch.Tensor,
             generator=None, noise: torch.Tensor | None = None):
        if self._step_index is None:
            self._step_index = int((self.timesteps == int(timestep)).nonzero()[0].item())
        i = self._step_index
        n = len(self.timesteps)
        prev_t = int(self.timesteps[i + 1]) if i + 1 < n else int(timestep)
        a_t = self.alphas_cumprod[int(timestep)]
        a_prev = self.alphas_cumprod[prev_t] if prev_t >= 0 else self.final_alpha_cumprod
        b_t = 1 - a_t
        b_prev = 1 - a_prev
        c_skip, c_out = self.boundary_scalings(int(timestep))
        if self.prediction_type == "epsilon":
            x0 = (sample - b_t.sqrt() * model_output) / a_t.sqrt()
        elif self.prediction_type == "sample":
            x0 = model_output
        elif self.prediction_type == "v_prediction":
            x0 = a_t.sqrt() * sample - b_t.sqrt() * model_output
        else:
            raise ValueError(self.prediction_type)
        if self.clip_sample:
            x0 = x0.clamp(-self.clip_sample_range, self.clip_sample_range)
        denoised = c_out * x0 + c_skip * sample
        if i != n - 1:
            if noise is None:
                noise = torch.randn(model_output.shape, generator=generator, dtype=denoised.dtype)
            prev = a_prev.sqrt() * denoised + b_prev.sqrt() * noise
        else:
            prev = denoised
        self._step_index += 1
        return prev, denoised


@contextlib.contextmanager
def configured(config: Optional[dict]):
    """Run the existing oracle loops with `LCMScheduler.from_config(config)`: they construct their scheduler by
    name, so the names are bound to this one for the duration."""
    from . import img2img, inpaint, pipeline

    def make():
        return OracleLCMSchedulerConfigured.from_config(config)
    saved = [(m, name, getattr(m, name)) for m, name in ((pipeline, "OracleLCMScheduler"),
                                                         (img2img, "OracleLCMSchedulerImg2Img"),
                                                         (inpaint, "OracleLCMSchedulerInpaint"))]
    try:
        for m, name, _ in saved:
            setattr(m, name, make)
        yield
    finally:
        for m, name, v in saved:
            setattr(m, name, v)


@torch.no_grad()
def run_pipeline_cfg(unet, vae, prompt_embeds: torch.Tensor, latents: torch.Tensor, step_noise: torch.Tensor,
                     num_inference_steps: int, guidance_scale: float, config: Optional[dict] = None,
                     negative_prompt_embeds: Optional[torch.Tensor] = None, tiling: bool = False,
                     output_type: str = "u8", record: Optional[dict] = None):
    """`StableDiffusionPipeline.__call__(prompt_embeds=..., guidance_scale=...)` with `LCMScheduler.from_config(config)`
    for a UNet without time_cond_proj (SD2.x): classifier-free guidance on a doubled batch [uncond, cond] when
    guidance_scale > 1 (zeros for the unconditional embeddings when no negative prompt is given, as the b200 engine
    does), `noise_pred = uncond + gs * (text - uncond)`, the configured step.  Runs where the models and inputs are
    (for the full-size UNet the tests run it on the device, inside `with torch.device("cuda")`, TF32 off)."""
    sched = OracleLCMSchedulerConfigured.from_config(config)
    timesteps = sched.set_timesteps(num_inference_steps)
    do_cfg = guidance_scale > 1.0 and not unet.cfg.time_cond_proj_dim
    ctx = prompt_embeds
    if do_cfg:
        neg = torch.zeros_like(prompt_embeds) if negative_prompt_embeds is None else negative_prompt_embeds
        ctx = torch.cat([neg, prompt_embeds], 0)
    latents = latents * sched.init_noise_sigma
    if record is not None:
        record.update(timesteps=timesteps.clone(), noise_pred=[], noise_pred_raw=[], latents=[])
    for i, t in enumerate(timesteps):
        x = torch.cat([latents] * 2, 0) if do_cfg else latents
        eps = unet(x, t.to(x.device), ctx)
        if record is not None:
            record["noise_pred_raw"].append(eps.clone())
        if do_cfg:
            e_u, e_t = eps.chunk(2)
            eps = e_u + guidance_scale * (e_t - e_u)
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
    return denormalize_to_u8(image.cpu())


def sd2_unet_config() -> UNetConfig:
    """stable-diffusion-2(-1)(-base) UNet: the SD1.5 4-level layout, `attention_head_dim` [5, 10, 20, 20] (= heads,
    64 wide at every level), linear projections, cross_attention_dim 1024, no time_cond_proj.  (`upcast_attention`
    is true in these configs; the oracle computes attention in fp32 throughout.)"""
    return UNetConfig(cross_attention_dim=1024, attention_head_dim=(5, 10, 20, 20), time_cond_proj_dim=None,
                      use_linear_projection=True)


def tiny_sd2_unet_config() -> UNetConfig:
    """SD2 topology (4 levels, linear projections, no time_cond_proj), small widths; head dim 32 everywhere."""
    return UNetConfig(block_out_channels=(64, 128, 256, 256), cross_attention_dim=96,
                      attention_head_dim=(2, 4, 8, 8), time_cond_proj_dim=None, use_linear_projection=True)


# stable-diffusion-2-1's scheduler/scheduler_config.json (a DDIMScheduler config; LCMScheduler.from_config keeps the
# keys it takes)
SD2_V_SCHEDULER_CONFIG = {
    "_class_name": "DDIMScheduler", "beta_end": 0.012, "beta_schedule": "scaled_linear", "beta_start": 0.00085,
    "clip_sample": False, "num_train_timesteps": 1000, "prediction_type": "v_prediction", "set_alpha_to_one": False,
    "skip_prk_steps": True, "steps_offset": 1, "trained_betas": None,
}
