"""Oracle samplers for guided models (test infrastructure): fp32 restatements of diffusers' `set_timesteps` /
`scale_model_input` / `step` of `EulerDiscreteScheduler` (s_churn = 0), `EulerAncestralDiscreteScheduler`,
`DDIMScheduler` (eta = 0) and `DPMSolverMultistepScheduler` (dpmsolver++, order 2, midpoint, lower_order_final,
final_sigmas_type "zero"; optionally Karras sigmas), each `from_config(model scheduler config)`.

Written from diffusers' semantics, independently of the product's `scheduler.py` (which restates the same classes
as per-step coefficients of one linear form): these step on tensors, in diffusers' expression order.  The step noise
of Euler ancestral is an input (one draw per step), like the LCM oracle's.

`run_pipeline_sampler` is the `StableDiffusionPipeline` / `StableDiffusionXLPipeline` loop with one of these:
latents * init_noise_sigma, scale_model_input on the doubled CFG batch, `noise_pred = uncond + gs (text - uncond)`.
"""
from __future__ import annotations

import math
from typing import Optional

import numpy as np
import torch

from .lcm_config import betas_for_alpha_bar, rescale_zero_terminal_snr
from .pipeline import denormalize_to_u8, sdxl_time_ids

NAMES = ("euler", "euler_a", "ddim", "dpmpp_2m", "dpmpp_2m_karras")

_BASE = dict(num_train_timesteps=1000, beta_start=0.0001, beta_end=0.02, beta_schedule="linear", trained_betas=None,
             prediction_type="epsilon", steps_offset=0, rescale_betas_zero_snr=False)
_DEFAULTS = {
    "euler": dict(_BASE, timestep_spacing="linspace"),
    "euler_a": dict(_BASE, timestep_spacing="linspace"),
    "ddim": dict(_BASE, timestep_spacing="leading", clip_sample=True, clip_sample_range=1.0, set_alpha_to_one=True),
    "dpmpp_2m": dict(_BASE, timestep_spacing="linspace"),
    "dpmpp_2m_karras": dict(_BASE, timestep_spacing="linspace"),
}


def _init_args(name: str, config: Optional[dict]) -> dict:
    """`from_config`: the class's keys from the file, its defaults otherwise; no file: SD1.5's betas."""
    a = dict(_DEFAULTS[name])
    if config is None:
        a.update(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")
    else:
        a.update({k: v for k, v in config.items() if k in a and v is not None})
    return a


def _alphas_cumprod(a: dict) -> torch.Tensor:
    n = a["num_train_timesteps"]
    if a["trained_betas"] is not None:
        betas = torch.tensor(a["trained_betas"], dtype=torch.float32)
    elif a["beta_schedule"] == "linear":
        betas = torch.linspace(a["beta_start"], a["beta_end"], n, dtype=torch.float32)
    elif a["beta_schedule"] == "scaled_linear":
        betas = torch.linspace(a["beta_start"] ** 0.5, a["beta_end"] ** 0.5, n, dtype=torch.float32) ** 2
    elif a["beta_schedule"] == "squaredcos_cap_v2":
        betas = betas_for_alpha_bar(n)
    else:
        raise NotImplementedError(a["beta_schedule"])
    if a["rescale_betas_zero_snr"]:
        betas = rescale_zero_terminal_snr(betas)
    alphas = 1.0 - betas
    return torch.cumprod(alphas, dim=0)


class OracleEuler:
    """EulerDiscreteScheduler (ancestral=False) / EulerAncestralDiscreteScheduler (ancestral=True)."""

    def __init__(self, config: Optional[dict] = None, ancestral: bool = False):
        self.cfg = _init_args("euler_a" if ancestral else "euler", config)
        self.ancestral = ancestral
        self.alphas_cumprod = _alphas_cumprod(self.cfg)
        if self.cfg["rescale_betas_zero_snr"]:
            self.alphas_cumprod[-1] = 2 ** -24

    def set_timesteps(self, num_inference_steps: int) -> torch.Tensor:
        N = self.cfg["num_train_timesteps"]
        sp = self.cfg["timestep_spacing"]
        if sp == "linspace":
            timesteps = np.linspace(0, N - 1, num_inference_steps, dtype=np.float32)[::-1].copy()
        elif sp == "leading":
            step_ratio = N // num_inference_steps
            timesteps = (np.arange(0, num_inference_steps) * step_ratio).round()[::-1].copy().astype(np.float32)
            timesteps += self.cfg["steps_offset"]
        elif sp == "trailing":
            step_ratio = N / num_inference_steps
            timesteps = (np.arange(N, 0, -step_ratio)).round().copy().astype(np.float32)
            timesteps -= 1
        else:
            raise ValueError(sp)
        sigmas = np.array(((1 - self.alphas_cumprod) / self.alphas_cumprod) ** 0.5)
        sigmas = np.interp(timesteps, np.arange(0, len(sigmas)), sigmas)
        sigmas = np.concatenate([sigmas, [0.0]]).astype(np.float32)
        self.sigmas = torch.from_numpy(sigmas)
        self.timesteps = torch.from_numpy(timesteps.astype(np.float32))
        self.step_index = 0
        return self.timesteps

    @property
    def init_noise_sigma(self):
        max_sigma = self.sigmas.max()
        if self.cfg["timestep_spacing"] in ["linspace", "trailing"]:
            return max_sigma
        return (max_sigma ** 2 + 1) ** 0.5

    def scale_model_input(self, sample: torch.Tensor) -> torch.Tensor:
        sigma = self.sigmas[self.step_index]
        return sample / ((sigma ** 2 + 1) ** 0.5)

    def step(self, model_output, sample, noise=None):
        sample = sample.to(torch.float32)
        sigma = self.sigmas[self.step_index]
        pt = self.cfg["prediction_type"]
        if pt == "epsilon":
            pred_original_sample = sample - sigma * model_output
        elif pt == "v_prediction":
            pred_original_sample = model_output * (-sigma / (sigma ** 2 + 1) ** 0.5) + (sample / (sigma ** 2 + 1))
        else:
            pred_original_sample = model_output
        if not self.ancestral:
            derivative = (sample - pred_original_sample) / sigma
            dt = self.sigmas[self.step_index + 1] - sigma
            prev_sample = sample + derivative * dt
        else:
            sigma_from = self.sigmas[self.step_index]
            sigma_to = self.sigmas[self.step_index + 1]
            sigma_up = (sigma_to ** 2 * (sigma_from ** 2 - sigma_to ** 2) / sigma_from ** 2) ** 0.5
            sigma_down = (sigma_to ** 2 - sigma_up ** 2) ** 0.5
            derivative = (sample - pred_original_sample) / sigma
            dt = sigma_down - sigma
            prev_sample = sample + derivative * dt
            prev_sample = prev_sample + noise * sigma_up
        self.step_index += 1
        return prev_sample, pred_original_sample


class OracleDDIM:
    """DDIMScheduler, eta = 0, use_clipped_model_output = False."""

    def __init__(self, config: Optional[dict] = None):
        self.cfg = _init_args("ddim", config)
        self.alphas_cumprod = _alphas_cumprod(self.cfg)
        self.final_alpha_cumprod = torch.tensor(1.0) if self.cfg["set_alpha_to_one"] else self.alphas_cumprod[0]
        self.init_noise_sigma = 1.0

    def set_timesteps(self, num_inference_steps: int) -> torch.Tensor:
        N = self.cfg["num_train_timesteps"]
        self.num_inference_steps = num_inference_steps
        sp = self.cfg["timestep_spacing"]
        if sp == "linspace":
            timesteps = np.linspace(0, N - 1, num_inference_steps).round()[::-1].copy().astype(np.int64)
        elif sp == "leading":
            step_ratio = N // num_inference_steps
            timesteps = (np.arange(0, num_inference_steps) * step_ratio).round()[::-1].copy().astype(np.int64)
            timesteps += self.cfg["steps_offset"]
        elif sp == "trailing":
            step_ratio = N / num_inference_steps
            timesteps = np.round(np.arange(N, 0, -step_ratio)).astype(np.int64)
            timesteps -= 1
        else:
            raise ValueError(sp)
        self.timesteps = torch.from_numpy(timesteps)
        return self.timesteps

    def scale_model_input(self, sample):
        return sample

    def step(self, model_output, timestep: int, sample, noise=None):
        prev_timestep = timestep - self.cfg["num_train_timesteps"] // self.num_inference_steps
        alpha_prod_t = self.alphas_cumprod[timestep]
        alpha_prod_t_prev = self.alphas_cumprod[prev_timestep] if prev_timestep >= 0 else self.final_alpha_cumprod
        beta_prod_t = 1 - alpha_prod_t
        pt = self.cfg["prediction_type"]
        if pt == "epsilon":
            pred_original_sample = (sample - beta_prod_t ** (0.5) * model_output) / alpha_prod_t ** (0.5)
            pred_epsilon = model_output
        elif pt == "sample":
            pred_original_sample = model_output
            pred_epsilon = (sample - alpha_prod_t ** (0.5) * pred_original_sample) / beta_prod_t ** (0.5)
        else:
            pred_original_sample = (alpha_prod_t ** 0.5) * sample - (beta_prod_t ** 0.5) * model_output
            pred_epsilon = (alpha_prod_t ** 0.5) * model_output + (beta_prod_t ** 0.5) * sample
        if self.cfg["clip_sample"]:
            r = self.cfg["clip_sample_range"]
            pred_original_sample = pred_original_sample.clamp(-r, r)
        std_dev_t = 0.0
        pred_sample_direction = (1 - alpha_prod_t_prev - std_dev_t ** 2) ** (0.5) * pred_epsilon
        prev_sample = alpha_prod_t_prev ** (0.5) * pred_original_sample + pred_sample_direction
        return prev_sample, pred_original_sample


class OracleDPMPP2M:
    """DPMSolverMultistepScheduler(algorithm_type="dpmsolver++", solver_order=2, solver_type="midpoint",
    lower_order_final=True, final_sigmas_type="zero", use_karras_sigmas=karras)."""

    def __init__(self, config: Optional[dict] = None, karras: bool = False):
        self.cfg = _init_args("dpmpp_2m_karras" if karras else "dpmpp_2m", config)
        self.karras = karras
        self.alphas_cumprod = _alphas_cumprod(self.cfg)
        if self.cfg["rescale_betas_zero_snr"]:
            self.alphas_cumprod[-1] = 2 ** -24
        self.init_noise_sigma = 1.0

    def set_timesteps(self, num_inference_steps: int) -> torch.Tensor:
        N = self.cfg["num_train_timesteps"]
        last_timestep = N                                   # lambda_min_clipped = -inf
        sp = self.cfg["timestep_spacing"]
        if sp == "linspace":
            timesteps = (np.linspace(0, last_timestep - 1, num_inference_steps + 1).round()[::-1][:-1]
                         .copy().astype(np.int64))
        elif sp == "leading":
            step_ratio = last_timestep // (num_inference_steps + 1)
            timesteps = ((np.arange(0, num_inference_steps + 1) * step_ratio).round()[::-1][:-1]
                         .copy().astype(np.int64))
            timesteps += self.cfg["steps_offset"]
        elif sp == "trailing":
            step_ratio = N / num_inference_steps
            timesteps = np.arange(last_timestep, 0, -step_ratio).round().copy().astype(np.int64)
            timesteps -= 1
        else:
            raise ValueError(sp)
        sigmas = np.array(((1 - self.alphas_cumprod) / self.alphas_cumprod) ** 0.5)
        log_sigmas = np.log(sigmas)
        if self.karras:
            sigmas = np.flip(sigmas).copy()
            sigma_min, sigma_max = sigmas[-1].item(), sigmas[0].item()
            rho = 7.0
            ramp = np.linspace(0, 1, num_inference_steps)
            min_inv_rho = sigma_min ** (1 / rho)
            max_inv_rho = sigma_max ** (1 / rho)
            sigmas = (max_inv_rho + ramp * (min_inv_rho - max_inv_rho)) ** rho
            timesteps = np.array([self._sigma_to_t(s, log_sigmas) for s in sigmas]).round()
        else:
            sigmas = np.interp(timesteps, np.arange(0, len(sigmas)), sigmas)
        sigmas = np.concatenate([sigmas, [0]]).astype(np.float32)
        self.sigmas = torch.from_numpy(sigmas)
        self.timesteps = torch.from_numpy(timesteps).to(dtype=torch.int64)
        self.model_outputs = [None, None]
        self.lower_order_nums = 0
        self.step_index = 0
        return self.timesteps

    @staticmethod
    def _sigma_to_t(sigma, log_sigmas):
        log_sigma = np.log(np.maximum(sigma, 1e-10))
        dists = log_sigma - log_sigmas[:, np.newaxis]
        low_idx = np.cumsum((dists >= 0), axis=0).argmax(axis=0).clip(max=log_sigmas.shape[0] - 2)
        high_idx = low_idx + 1
        low = log_sigmas[low_idx]
        high = log_sigmas[high_idx]
        w = (low - log_sigma) / (low - high)
        w = np.clip(w, 0, 1)
        t = (1 - w) * low_idx + w * high_idx
        return t.reshape(np.shape(sigma))

    @staticmethod
    def _alpha_sigma(sigma):
        alpha_t = 1 / ((sigma ** 2 + 1) ** 0.5)
        return alpha_t, sigma * alpha_t

    def scale_model_input(self, sample):
        return sample

    def step(self, model_output, sample, noise=None):
        n = len(self.timesteps)
        lower_order_final = self.step_index == n - 1            # final_sigmas_type "zero"
        alpha_t, sigma_t = self._alpha_sigma(self.sigmas[self.step_index])
        pt = self.cfg["prediction_type"]
        if pt == "epsilon":
            x0_pred = (sample - sigma_t * model_output) / alpha_t
        elif pt == "sample":
            x0_pred = model_output
        else:
            x0_pred = alpha_t * sample - sigma_t * model_output
        self.model_outputs = [self.model_outputs[1], x0_pred]
        sample = sample.to(torch.float32)
        if self.lower_order_nums < 1 or lower_order_final:
            a_t, s_t = self._alpha_sigma(self.sigmas[self.step_index + 1])
            a_s, s_s = self._alpha_sigma(self.sigmas[self.step_index])
            lambda_t = torch.log(a_t) - torch.log(s_t)
            lambda_s = torch.log(a_s) - torch.log(s_s)
            h = lambda_t - lambda_s
            prev_sample = (s_t / s_s) * sample - (a_t * (torch.exp(-h) - 1.0)) * x0_pred
        else:
            a_t, s_t = self._alpha_sigma(self.sigmas[self.step_index + 1])
            a_s0, s_s0 = self._alpha_sigma(self.sigmas[self.step_index])
            a_s1, s_s1 = self._alpha_sigma(self.sigmas[self.step_index - 1])
            lambda_t = torch.log(a_t) - torch.log(s_t)
            lambda_s0 = torch.log(a_s0) - torch.log(s_s0)
            lambda_s1 = torch.log(a_s1) - torch.log(s_s1)
            m0, m1 = self.model_outputs[-1], self.model_outputs[-2]
            h, h_0 = lambda_t - lambda_s0, lambda_s0 - lambda_s1
            r0 = h_0 / h
            D0, D1 = m0, (1.0 / r0) * (m0 - m1)
            prev_sample = ((s_t / s_s0) * sample - (a_t * (torch.exp(-h) - 1.0)) * D0
                           - 0.5 * (a_t * (torch.exp(-h) - 1.0)) * D1)
        if self.lower_order_nums < 2:
            self.lower_order_nums += 1
        self.step_index += 1
        return prev_sample, x0_pred


def make(name: str, config: Optional[dict] = None):
    if name in ("euler", "euler_a"):
        return OracleEuler(config, ancestral=name == "euler_a")
    if name == "ddim":
        return OracleDDIM(config)
    if name in ("dpmpp_2m", "dpmpp_2m_karras"):
        return OracleDPMPP2M(config, karras=name == "dpmpp_2m_karras")
    raise ValueError(name)


def step(sched, model_output, t, sample, noise=None):
    """One `scheduler.step` -> (prev_sample, pred_original_sample), whatever the class's argument list."""
    if isinstance(sched, OracleDDIM):
        return sched.step(model_output, int(t), sample)
    return sched.step(model_output, sample, noise)


def noise_draws(name: str, steps: int) -> int:
    return steps if name == "euler_a" else 0


@torch.no_grad()
def run_pipeline_sampler(unet, vae, prompt_embeds: torch.Tensor, latents: torch.Tensor, step_noise, sampler: str,
                         num_inference_steps: int, guidance_scale: float, config: Optional[dict] = None,
                         pooled_embeds: Optional[torch.Tensor] = None, height: Optional[int] = None,
                         width: Optional[int] = None, output_type: str = "u8", teacher=None,
                         record: Optional[dict] = None):
    """The text-to-image loop with `sampler`: classifier-free guidance on a doubled batch [uncond, cond] when
    guidance_scale > 1 (zeros for the unconditional embeddings, as the engine does without a negative prompt), SDXL
    text_time conditioning when pooled_embeds is given.  step_noise [steps, B, 4, h, w] (Euler ancestral only).
    teacher [steps, B, 4, h, w]: the latents the UNet sees at step i are taken from it (the scheduler state still
    advances on them), so per-step outputs can be compared on given inputs."""
    sched = make(sampler, config)
    timesteps = sched.set_timesteps(num_inference_steps)
    B = latents.shape[0]
    do_cfg = guidance_scale > 1.0 and not unet.cfg.time_cond_proj_dim
    ctx = prompt_embeds
    extra = {}
    if pooled_embeds is not None:
        pooled, tids = pooled_embeds, sdxl_time_ids(height, width, B).to(pooled_embeds.device)
        if do_cfg:
            pooled = torch.cat([torch.zeros_like(pooled_embeds), pooled_embeds], 0)
            tids = torch.cat([tids, tids], 0)
        extra = dict(text_embeds=pooled, time_ids=tids)
    if do_cfg:
        ctx = torch.cat([torch.zeros_like(prompt_embeds), prompt_embeds], 0)
    latents = latents * sched.init_noise_sigma
    if record is not None:
        record.update(timesteps=timesteps.clone(), init_latents=latents.clone(), noise_pred=[], noise_pred_raw=[],
                      latents=[], denoised=[])
    for i, t in enumerate(timesteps):
        if teacher is not None:
            latents = teacher[i].to(latents.device, latents.dtype)
        x = torch.cat([latents] * 2, 0) if do_cfg else latents
        x = sched.scale_model_input(x)
        eps = unet(x, t.to(x.device), ctx, None, **extra)
        if record is not None:
            record["noise_pred_raw"].append(eps.clone())
        if do_cfg:
            e_u, e_t = eps.chunk(2)
            eps = e_u + guidance_scale * (e_t - e_u)
        z = step_noise[i] if noise_draws(sampler, num_inference_steps) else None
        latents, x0 = step(sched, eps, t, latents, z)
        if record is not None:
            record["noise_pred"].append(eps.clone())
            record["latents"].append(latents.clone())
            record["denoised"].append(x0.clone())
    if output_type == "latent":
        return latents
    image = vae(latents / vae.cfg.scaling_factor, tiling=False)
    if record is not None:
        record["image_f32"] = image.clone()
    return denormalize_to_u8(image.cpu())
