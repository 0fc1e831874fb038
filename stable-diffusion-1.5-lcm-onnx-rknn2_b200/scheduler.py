"""Host side of the LCM scheduler (product code).

Integer timestep schedule and the fp32 coefficients of `LCMScheduler.step`, computed once per
(num_inference_steps) on the host exactly like diffusers does (fp32 torch scalars), then handed
to the fused device kernel `dl_lcm_step` — the reference's per-step host<->device sync
(indexing CPU `alphas_cumprod` with a CUDA scalar, SURVEY.md §3.2) disappears.

Reference: `pipe.scheduler = LCMScheduler.from_config(...)` (`backends/cuda_worker.py:88`),
`set_timesteps` / `step` call sites mirrored at `backends/rknnlcm.py:559-560, 596-598`.

`SchedulerConfig` is that `from_config`: the model's `scheduler/scheduler_config.json` (beta schedule, prediction
type, clamp, zero-terminal-SNR rescale, ...) with `LCMScheduler`'s defaults for every key it leaves out.  Without the
file (and for single-file checkpoints) the defaults are SD1.5's constants below.
"""
from __future__ import annotations

import dataclasses
import json
import math
import os
from functools import lru_cache
from typing import List, Optional, Tuple

import numpy as np
import torch

NUM_TRAIN_TIMESTEPS = 1000
BETA_START, BETA_END = 0.00085, 0.012
ORIGINAL_INFERENCE_STEPS = 50
TIMESTEP_SCALING = 10.0
SIGMA_DATA = 0.5
INIT_NOISE_SIGMA = 1.0


BETA_SCHEDULES = ("linear", "scaled_linear", "squaredcos_cap_v2")
PREDICTION_TYPES = ("epsilon", "v_prediction", "sample")


@dataclasses.dataclass(frozen=True)
class SchedulerConfig:
    """The `LCMScheduler.__init__` arguments, defaults as diffusers has them (= SD1.5's constants above)."""
    num_train_timesteps: int = NUM_TRAIN_TIMESTEPS
    beta_start: float = BETA_START
    beta_end: float = BETA_END
    beta_schedule: str = "scaled_linear"
    trained_betas: Optional[Tuple[float, ...]] = None
    original_inference_steps: int = ORIGINAL_INFERENCE_STEPS
    clip_sample: bool = False
    clip_sample_range: float = 1.0
    # no effect under LCM: `step` reads final_alpha_cumprod only for prev_t < 0, and LCM's prev_t is a timestep of
    # the schedule (or t itself on the last step), never negative
    set_alpha_to_one: bool = True
    # no effect under LCM: `LCMScheduler.set_timesteps` builds its k * i - 1 grid without steps_offset
    steps_offset: int = 0
    prediction_type: str = "epsilon"
    thresholding: bool = False                      # refused when true (validate)
    dynamic_thresholding_ratio: float = 0.995       # read by thresholding only
    sample_max_value: float = 1.0                   # read by thresholding only
    # no effect under LCM: `LCMScheduler.set_timesteps` does not read timestep_spacing either
    timestep_spacing: str = "leading"
    timestep_scaling: float = TIMESTEP_SCALING
    rescale_betas_zero_snr: bool = False

    @classmethod
    def from_dict(cls, d: dict) -> "SchedulerConfig":
        """`LCMScheduler.from_config(d)`: keys `LCMScheduler.__init__` does not take (`_class_name`,
        `skip_prk_steps`, ...) are ignored, missing keys keep the defaults.  Refused values raise RuntimeError."""
        known = {f.name: f for f in dataclasses.fields(cls)}
        kw = {}
        for k, v in d.items():
            if k not in known:
                continue
            if k == "trained_betas":
                v = None if v is None else tuple(float(b) for b in v)
            elif v is not None and known[k].type in ("int", "float", "bool"):
                v = {"int": int, "float": float, "bool": bool}[known[k].type](v)
            elif v is None:
                continue
            kw[k] = v
        cfg = cls(**kw)
        cfg.validate()
        return cfg

    @classmethod
    def load(cls, model_dir: Optional[str]) -> "SchedulerConfig":
        """`<model_dir>/scheduler/scheduler_config.json`; the defaults when there is no such file (or no
        directory: single-file checkpoints carry no scheduler config)."""
        p = os.path.join(model_dir, "scheduler", "scheduler_config.json") if model_dir else None
        if p is None or not os.path.isfile(p):
            return cls()
        with open(p) as f:
            return cls.from_dict(json.load(f))

    def validate(self) -> None:
        def bad(key, why):
            raise RuntimeError(f"scheduler config: {key}={getattr(self, key)!r} {why}")
        if self.thresholding:
            bad("thresholding", "is not supported (dynamic thresholding of x0 is not implemented)")
        if self.beta_schedule not in BETA_SCHEDULES and self.trained_betas is None:
            bad("beta_schedule", f"is not supported (one of {', '.join(BETA_SCHEDULES)}, or trained_betas)")
        if self.prediction_type not in PREDICTION_TYPES:
            bad("prediction_type", f"is not supported (one of {', '.join(PREDICTION_TYPES)})")
        if self.rescale_betas_zero_snr and self.prediction_type == "epsilon":
            bad("rescale_betas_zero_snr", "cannot go with prediction_type='epsilon': the rescale makes "
                "alphas_cumprod[-1] = 0, and the epsilon x0 divides by its square root")
        if self.num_train_timesteps < 1:
            bad("num_train_timesteps", "must be positive")
        if not 1 <= self.original_inference_steps <= self.num_train_timesteps:
            bad("original_inference_steps", f"must be in [1, num_train_timesteps={self.num_train_timesteps}]")
        if self.trained_betas is not None and len(self.trained_betas) != self.num_train_timesteps:
            bad("num_train_timesteps", f"does not match the {len(self.trained_betas)} trained_betas")
        if self.clip_sample and not self.clip_sample_range >= 0.0:
            bad("clip_sample_range", "must be >= 0")


DEFAULT_CONFIG = SchedulerConfig()


def _betas_for_alpha_bar(n: int, max_beta: float = 0.999) -> torch.Tensor:
    """diffusers' `betas_for_alpha_bar` with the cosine alpha_bar (squaredcos_cap_v2): float64 host math, then fp32."""
    def alpha_bar(t):
        return math.cos((t + 0.008) / 1.008 * math.pi / 2) ** 2
    return torch.tensor([min(1 - alpha_bar((i + 1) / n) / alpha_bar(i / n), max_beta) for i in range(n)],
                        dtype=torch.float32)


def _rescale_zero_terminal_snr(betas: torch.Tensor) -> torch.Tensor:
    """diffusers' `rescale_zero_terminal_snr`: sqrt(alpha_bar) shifted so that its last entry is 0 and scaled so that
    its first is unchanged, squared, and turned back into betas (fp32 throughout)."""
    alphas_bar_sqrt = torch.cumprod(1.0 - betas, dim=0).sqrt()
    s0 = alphas_bar_sqrt[0].clone()
    sT = alphas_bar_sqrt[-1].clone()
    alphas_bar_sqrt -= sT
    alphas_bar_sqrt *= s0 / (s0 - sT)
    alphas_bar = alphas_bar_sqrt ** 2
    alphas = torch.cat([alphas_bar[0:1], alphas_bar[1:] / alphas_bar[:-1]])
    return 1 - alphas


@lru_cache(maxsize=8)
def alphas_cumprod(config: SchedulerConfig = DEFAULT_CONFIG) -> torch.Tensor:
    """fp32 alphas_cumprod of `LCMScheduler(**config)`, built as diffusers builds it."""
    c = config
    if c.trained_betas is not None:
        betas = torch.tensor(c.trained_betas, dtype=torch.float32)
    elif c.beta_schedule == "linear":
        betas = torch.linspace(c.beta_start, c.beta_end, c.num_train_timesteps, dtype=torch.float32)
    elif c.beta_schedule == "scaled_linear":
        betas = torch.linspace(c.beta_start ** 0.5, c.beta_end ** 0.5, c.num_train_timesteps,
                               dtype=torch.float32) ** 2
    elif c.beta_schedule == "squaredcos_cap_v2":
        betas = _betas_for_alpha_bar(c.num_train_timesteps)
    else:
        raise RuntimeError(f"scheduler config: beta_schedule={c.beta_schedule!r} is not supported")
    if c.rescale_betas_zero_snr:
        betas = _rescale_zero_terminal_snr(betas)
    return torch.cumprod(1.0 - betas, dim=0)


def lcm_timesteps(num_inference_steps: int, strength: float = 1.0,
                  config: SchedulerConfig = DEFAULT_CONFIG) -> List[int]:
    """`LCMScheduler.set_timesteps(n, strength=strength)`: image-to-image (strength < 1) draws the n steps from
    the first int(50 * strength) entries of the original 50-step schedule, counted from t = 19 upwards
    (50 = original_inference_steps, 19 = num_train_timesteps // 50 - 1 for the default config)."""
    orig = config.original_inference_steps
    if not 1 <= num_inference_steps <= orig:
        raise ValueError(f"num_inference_steps must be in [1, {orig}], got {num_inference_steps}")
    if not 0.0 < strength <= 1.0:
        raise ValueError(f"strength must be in (0, 1], got {strength}")
    k = config.num_train_timesteps // orig
    origin = (np.arange(1, int(orig * strength) + 1) * k - 1)[::-1]
    if len(origin) // num_inference_steps < 1:
        raise ValueError(f"strength {strength} leaves {len(origin)} of the {orig} original "
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

    def __init__(self, num_inference_steps: int, strength: float = 1.0, truncate: bool = False,
                 config: SchedulerConfig = DEFAULT_CONFIG):
        self.num_inference_steps = num_inference_steps
        self.strength = strength
        self.config = config
        # what the step kernel needs besides the coefficients: how x0 follows from the model output, and the clamp
        # of x0 (None: no clamp)
        self.prediction_type = config.prediction_type
        self.clip_range = float(config.clip_sample_range) if config.clip_sample else None
        self.begin_index = 0
        if truncate:
            if not 0.0 < strength <= 1.0:
                raise ValueError(f"strength must be in (0, 1], got {strength}")
            full = lcm_timesteps(num_inference_steps, config=config)
            init_timestep = min(int(num_inference_steps * strength), num_inference_steps)
            self.begin_index = max(num_inference_steps - init_timestep, 0)
            self.timesteps = full[self.begin_index:]
            if len(self.timesteps) < 1:
                raise ValueError(f"strength {strength} leaves no step of num_inference_steps={num_inference_steps} "
                                 f"(int(n * strength) = 0)")
        else:
            self.timesteps = lcm_timesteps(num_inference_steps, strength, config)
        ac = alphas_cumprod(config)
        self._coeffs: List[Tuple[float, ...]] = []
        n = len(self.timesteps)
        for i, t in enumerate(self.timesteps):
            prev_t = self.timesteps[i + 1] if i + 1 < n else t
            a_t, a_prev = ac[t], ac[prev_t]
            s = torch.as_tensor(t, dtype=torch.int64) * config.timestep_scaling  # fp32 0-dim
            c_skip = SIGMA_DATA ** 2 / (s ** 2 + SIGMA_DATA ** 2)
            c_out = s / (s ** 2 + SIGMA_DATA ** 2) ** 0.5
            self._coeffs.append((a_t.sqrt().item(), (1 - a_t).sqrt().item(), c_skip.item(),
                                 c_out.item(), a_prev.sqrt().item(), (1 - a_prev).sqrt().item()))

    def add_noise_coeffs(self, t: int = None) -> Tuple[float, float]:
        """`LCMScheduler.add_noise` at t (default t0 = timesteps[0]): fp32 (sqrt(ac[t]), sqrt(1 - ac[t])) as `** 0.5`."""
        a = alphas_cumprod(self.config)[self.timesteps[0] if t is None else t]
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
