"""Host side of the LCM scheduler (product code).

Integer timestep schedule and the fp32 coefficients of `LCMScheduler.step`, computed once per
(num_inference_steps) on the host exactly like diffusers does (fp32 torch scalars), then handed
to the fused device kernel `dl_lcm_step` — the reference's per-step host<->device sync
(indexing CPU `alphas_cumprod` with a CUDA scalar, SURVEY.md §3.2) disappears.

Reference: `pipe.scheduler = LCMScheduler.from_config(...)` (`backends/cuda_worker.py:88`),
`set_timesteps` / `step` call sites mirrored at `backends/rknnlcm.py:559-560, 596-598`.
"""
from __future__ import annotations

import math
from functools import lru_cache
from typing import List, Tuple

import numpy as np
import torch

NUM_TRAIN_TIMESTEPS = 1000
BETA_START, BETA_END = 0.00085, 0.012
ORIGINAL_INFERENCE_STEPS = 50
TIMESTEP_SCALING = 10.0
SIGMA_DATA = 0.5
INIT_NOISE_SIGMA = 1.0


@lru_cache(maxsize=1)
def alphas_cumprod() -> torch.Tensor:
    betas = torch.linspace(BETA_START ** 0.5, BETA_END ** 0.5, NUM_TRAIN_TIMESTEPS,
                           dtype=torch.float32) ** 2
    return torch.cumprod(1.0 - betas, dim=0)


def lcm_timesteps(num_inference_steps: int, strength: float = 1.0) -> List[int]:
    """`LCMScheduler.set_timesteps(n, strength=strength)`: image-to-image (strength < 1) draws the n steps from
    the first int(50 * strength) entries of the original 50-step schedule, counted from t = 19 upwards."""
    if not 1 <= num_inference_steps <= ORIGINAL_INFERENCE_STEPS:
        raise ValueError(f"num_inference_steps must be in [1, {ORIGINAL_INFERENCE_STEPS}], "
                         f"got {num_inference_steps}")
    if not 0.0 < strength <= 1.0:
        raise ValueError(f"strength must be in (0, 1], got {strength}")
    k = NUM_TRAIN_TIMESTEPS // ORIGINAL_INFERENCE_STEPS
    origin = (np.arange(1, int(ORIGINAL_INFERENCE_STEPS * strength) + 1) * k - 1)[::-1]
    if len(origin) // num_inference_steps < 1:
        raise ValueError(f"strength {strength} leaves {len(origin)} of the {ORIGINAL_INFERENCE_STEPS} original "
                         f"timesteps: fewer than num_inference_steps={num_inference_steps}")
    idx = np.floor(np.linspace(0, len(origin), num=num_inference_steps, endpoint=False)).astype(np.int64)
    return [int(t) for t in origin[idx]]


class LCMSchedule:
    """Timesteps + per-step coefficient tuples for `lib.lcm_step`.

    truncate=True (inpainting, `StableDiffusionInpaintPipeline.get_timesteps`): the full n-step schedule of
    `set_timesteps(n)`, of which only the tail from t_start = n - min(int(n * strength), n) runs
    (`set_begin_index(t_start)`).  Step i then uses the coefficients of full index t_start + i with
    prev_t = full[t_start + i + 1], i.e. those of the tail itself, and no noise is drawn at full index n - 1.
    Otherwise strength re-spaces the schedule (`set_timesteps(n, strength)`, image-to-image)."""

    def __init__(self, num_inference_steps: int, strength: float = 1.0, truncate: bool = False):
        self.num_inference_steps = num_inference_steps
        self.strength = strength
        self.begin_index = 0
        if truncate:
            if not 0.0 < strength <= 1.0:
                raise ValueError(f"strength must be in (0, 1], got {strength}")
            full = lcm_timesteps(num_inference_steps)
            init_timestep = min(int(num_inference_steps * strength), num_inference_steps)
            self.begin_index = max(num_inference_steps - init_timestep, 0)
            self.timesteps = full[self.begin_index:]
            if len(self.timesteps) < 1:
                raise ValueError(f"strength {strength} leaves no step of num_inference_steps={num_inference_steps} "
                                 f"(int(n * strength) = 0)")
        else:
            self.timesteps = lcm_timesteps(num_inference_steps, strength)
        ac = alphas_cumprod()
        self._coeffs: List[Tuple[float, ...]] = []
        n = len(self.timesteps)
        for i, t in enumerate(self.timesteps):
            prev_t = self.timesteps[i + 1] if i + 1 < n else t
            a_t, a_prev = ac[t], ac[prev_t]
            s = torch.as_tensor(t, dtype=torch.int64) * TIMESTEP_SCALING       # fp32 0-dim
            c_skip = SIGMA_DATA ** 2 / (s ** 2 + SIGMA_DATA ** 2)
            c_out = s / (s ** 2 + SIGMA_DATA ** 2) ** 0.5
            self._coeffs.append((a_t.sqrt().item(), (1 - a_t).sqrt().item(), c_skip.item(),
                                 c_out.item(), a_prev.sqrt().item(), (1 - a_prev).sqrt().item()))

    def add_noise_coeffs(self, t: int = None) -> Tuple[float, float]:
        """`LCMScheduler.add_noise` at t (default t0 = timesteps[0]): fp32 (sqrt(ac[t]), sqrt(1 - ac[t])) as `** 0.5`."""
        a = alphas_cumprod()[self.timesteps[0] if t is None else t]
        return (a ** 0.5).item(), ((1 - a) ** 0.5).item()

    def coeffs(self, i: int) -> Tuple[float, ...]:
        return self._coeffs[i]

    def has_noise(self, i: int) -> bool:
        return i != len(self.timesteps) - 1


def guidance_scale_embedding(w: torch.Tensor, embedding_dim: int = 256) -> torch.Tensor:
    """`get_guidance_scale_embedding` (`backends/rknnlcm.py:651-677`); w = guidance_scale - 1."""
    w = w.to(torch.float32) * 1000.0
    half = embedding_dim // 2
    e = math.log(10000.0) / (half - 1)
    f = torch.exp(torch.arange(half, dtype=torch.float32) * -e)
    emb = w[:, None] * f[None, :]
    emb = torch.cat([torch.sin(emb), torch.cos(emb)], dim=1)
    if embedding_dim % 2 == 1:
        emb = torch.nn.functional.pad(emb, (0, 1))
    return emb
