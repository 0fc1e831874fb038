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
    # the config file as read (None: no file): the other samplers take their own keys and defaults from it
    raw: Optional[dict] = dataclasses.field(default=None, compare=False, repr=False)

    @classmethod
    def from_dict(cls, d: dict) -> "SchedulerConfig":
        """`LCMScheduler.from_config(d)`: keys `LCMScheduler.__init__` does not take (`_class_name`,
        `skip_prk_steps`, ...) are ignored, missing keys keep the defaults.  Refused values raise RuntimeError."""
        known = {f.name: f for f in dataclasses.fields(cls) if f.name != "raw"}
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
        cfg = cls(**kw, raw=dict(d))
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


# ---------------------------------------------------------------------------------------------------------------------
# Samplers for guided models (a request's `sampler`): Euler, Euler ancestral, DDIM (eta 0) and DPM++ 2M, each
# `<Class>.from_config(model's scheduler config)`.  Every step is one linear form (`lib.sampler_step`):
#   x0     = clamp(a_x x + a_e e)                     e: the (guided) model output
#   x_next = c_x x + c_e e + c_0 x0 + c_1 x0_prev + c_n z
# with the coefficients computed here, fp32 torch / float64 numpy where diffusers uses each.
# ---------------------------------------------------------------------------------------------------------------------
SAMPLERS = ("lcm", "euler", "euler_a", "ddim", "dpmpp_2m", "dpmpp_2m_karras")
TIMESTEP_SPACINGS = ("leading", "trailing", "linspace")

_COMMON_DEFAULTS = dict(num_train_timesteps=1000, beta_start=0.0001, beta_end=0.02, beta_schedule="linear",
                        trained_betas=None, prediction_type="epsilon", steps_offset=0, rescale_betas_zero_snr=False)
# `__init__` defaults of each diffusers class: a key the config file leaves out takes these, not LCMScheduler's
_CLASS_DEFAULTS = {
    "euler": dict(_COMMON_DEFAULTS, timestep_spacing="linspace", interpolation_type="linear", use_karras_sigmas=False,
                  use_exponential_sigmas=False, use_beta_sigmas=False, sigma_min=None, sigma_max=None,
                  timestep_type="discrete", final_sigmas_type="zero"),
    "euler_a": dict(_COMMON_DEFAULTS, timestep_spacing="linspace"),
    "ddim": dict(_COMMON_DEFAULTS, timestep_spacing="leading", clip_sample=True, clip_sample_range=1.0,
                 set_alpha_to_one=True, thresholding=False, dynamic_thresholding_ratio=0.995, sample_max_value=1.0),
    "dpmpp": dict(_COMMON_DEFAULTS, timestep_spacing="linspace", solver_order=2, algorithm_type="dpmsolver++",
                  solver_type="midpoint", lower_order_final=True, euler_at_final=False, use_karras_sigmas=False,
                  use_exponential_sigmas=False, use_beta_sigmas=False, use_lu_lambdas=False, final_sigmas_type="zero",
                  lambda_min_clipped=-math.inf, variance_type=None, thresholding=False,
                  dynamic_thresholding_ratio=0.995, sample_max_value=1.0),
}
# what the sampler name fixes, whatever the file says (`from_config(config, **these)`)
_FIXED = {
    "dpmpp_2m": dict(algorithm_type="dpmsolver++", solver_order=2, solver_type="midpoint", lower_order_final=True,
                     final_sigmas_type="zero", use_karras_sigmas=False),
    "dpmpp_2m_karras": dict(algorithm_type="dpmsolver++", solver_order=2, solver_type="midpoint",
                            lower_order_final=True, final_sigmas_type="zero", use_karras_sigmas=True),
}
# keys a class takes whose other values are not implemented here: refused unless they hold the class default
_NOT_BUILT = {
    "euler": ("interpolation_type", "use_karras_sigmas", "use_exponential_sigmas", "use_beta_sigmas", "sigma_min",
              "sigma_max", "timestep_type", "final_sigmas_type"),
    "euler_a": (),
    "ddim": ("thresholding",),
    "dpmpp": ("thresholding", "euler_at_final", "use_exponential_sigmas", "use_beta_sigmas", "use_lu_lambdas",
              "lambda_min_clipped", "variance_type"),
}
_SD15_BETAS = dict(num_train_timesteps=NUM_TRAIN_TIMESTEPS, beta_start=BETA_START, beta_end=BETA_END,
                   beta_schedule="scaled_linear", trained_betas=None)


def check_sampler(name) -> str:
    """A request's sampler name -> its canonical name ("lcm" for None); RuntimeError listing the accepted names."""
    s = "lcm" if name is None else name
    if s not in SAMPLERS:
        raise RuntimeError(f"unknown sampler {name!r}: one of {', '.join(SAMPLERS)}")
    return s


def sampler_noise_draws(sampler: str, steps: int) -> int:
    """Noise draws a text-to-image pass of `steps` steps consumes after the latents draw: one per non-final step
    under LCM, one per step under Euler ancestral (diffusers draws on the last step too), none otherwise."""
    s = check_sampler(sampler)
    return steps - 1 if s == "lcm" else steps if s == "euler_a" else 0


def sampler_config(sampler: str, config: SchedulerConfig = DEFAULT_CONFIG) -> dict:
    """`<Class>.from_config(config file)` for a non-LCM sampler: the file's keys the class takes, that class's defaults
    for the rest, and the settings the sampler name fixes.  Without a file: the betas, prediction type and
    zero-SNR rescale of `config` (SD1.5's constants for the default config) and the class defaults otherwise.
    Refused values raise RuntimeError naming the key."""
    s = check_sampler(sampler)
    if s == "lcm":
        raise RuntimeError("sampler_config: the LCM sampler is configured by SchedulerConfig itself")
    cls = "dpmpp" if s.startswith("dpmpp") else s
    d = dict(_CLASS_DEFAULTS[cls])
    if config.raw is None:
        d.update(num_train_timesteps=config.num_train_timesteps, beta_start=config.beta_start,
                 beta_end=config.beta_end, beta_schedule=config.beta_schedule, trained_betas=config.trained_betas,
                 prediction_type=config.prediction_type, rescale_betas_zero_snr=config.rescale_betas_zero_snr)
    else:
        for k, v in config.raw.items():
            if k in d and not (v is None and d[k] is not None):
                d[k] = v
    for k in _NOT_BUILT[cls]:
        if d[k] != _CLASS_DEFAULTS[cls][k]:
            raise RuntimeError(f"scheduler config: {k}={d[k]!r} is not supported by the {s} sampler")
    d.update(_FIXED.get(s, {}))

    def bad(key, why):
        raise RuntimeError(f"scheduler config: {key}={d[key]!r} {why} ({s} sampler)")
    if d["trained_betas"] is None and d["beta_schedule"] not in BETA_SCHEDULES:
        bad("beta_schedule", f"is not supported (one of {', '.join(BETA_SCHEDULES)}, or trained_betas)")
    if d["prediction_type"] not in PREDICTION_TYPES:
        bad("prediction_type", f"is not supported (one of {', '.join(PREDICTION_TYPES)})")
    if d["timestep_spacing"] not in TIMESTEP_SPACINGS:
        bad("timestep_spacing", f"is not supported (one of {', '.join(TIMESTEP_SPACINGS)})")
    if d["rescale_betas_zero_snr"] and d["prediction_type"] == "epsilon":
        bad("rescale_betas_zero_snr", "cannot go with prediction_type='epsilon'")
    if int(d["num_train_timesteps"]) < 1:
        bad("num_train_timesteps", "must be positive")
    if d["trained_betas"] is not None and len(d["trained_betas"]) != int(d["num_train_timesteps"]):
        bad("num_train_timesteps", f"does not match the {len(d['trained_betas'])} trained_betas")
    return d


def _sampler_alphas_cumprod(d: dict, zero_snr_floor: bool) -> torch.Tensor:
    """The class's fp32 alphas_cumprod (the LCM construction: same betas, same rescale); Euler, Euler ancestral and
    DPM++ then set alphas_cumprod[-1] = 2**-24 under zero-terminal SNR so that the last sigma is finite."""
    cfg = SchedulerConfig(num_train_timesteps=int(d["num_train_timesteps"]), beta_start=float(d["beta_start"]),
                          beta_end=float(d["beta_end"]), beta_schedule=d["beta_schedule"],
                          trained_betas=None if d["trained_betas"] is None else tuple(map(float, d["trained_betas"])),
                          rescale_betas_zero_snr=bool(d["rescale_betas_zero_snr"]))
    ac = alphas_cumprod(cfg).clone()
    if zero_snr_floor and cfg.rescale_betas_zero_snr:
        ac[-1] = 2 ** -24
    return ac


def _spaced(spacing: str, n_train: int, n: int, offset: int, dtype) -> np.ndarray:
    """`set_timesteps` grids of Euler (dtype float32) and DDIM (int64): `leading` (+ steps_offset), `trailing`,
    `linspace` (DDIM rounds it to integers, Euler keeps the float32 values)."""
    if spacing == "linspace":
        if dtype == np.float32:
            return np.linspace(0, n_train - 1, n, dtype=np.float32)[::-1].copy()
        return np.linspace(0, n_train - 1, n).round()[::-1].copy().astype(dtype)
    if spacing == "leading":
        return (np.arange(0, n) * (n_train // n)).round()[::-1].copy().astype(dtype) + offset
    return np.arange(n_train, 0, -n_train / n).round().astype(dtype) - 1


def _check_steps(n: int, limit: int, what: str) -> None:
    if not 1 <= n <= limit:
        raise ValueError(f"num_inference_steps must be in [1, {limit}] for the {what} sampler, got {n}")


class _SamplerSchedule:
    """What the denoise loop reads: `timesteps` (floats for Euler-family `linspace`, ints otherwise), `coeffs(i)` =
    (a_x, a_e, c_x, c_e, c_0, c_1, c_n) of the step kernel, `in_scale(i)` (scale_model_input), `has_noise(i)`,
    `n_draws`, `init_noise_sigma`, `prediction_type`, `clip_range` (None: no clamp of x0)."""
    name: str
    clip_range = None
    init_noise_sigma = 1.0

    def coeffs(self, i: int) -> Tuple[float, ...]:
        return self._coeffs[i]

    def in_scale(self, i: int) -> float:
        return 1.0

    def has_noise(self, i: int) -> bool:
        return False

    @property
    def n_draws(self) -> int:
        return sum(self.has_noise(i) for i in range(len(self.timesteps)))

    def uses_prev_x0(self, i: int) -> bool:
        return self._coeffs[i][5] != 0.0


def _x0_sigma_form(pred: str, sigma: torch.Tensor) -> Tuple[float, float]:
    """(a_x, a_e) of Euler's pred_original_sample at sigma (fp32): epsilon x - sigma e; v_prediction
    e * (-sigma / (sigma^2 + 1) ** 0.5) + x / (sigma^2 + 1); sample e."""
    if pred == "epsilon":
        return 1.0, (-sigma).item()
    if pred == "v_prediction":
        return (1.0 / (sigma ** 2 + 1)).item(), (-sigma / (sigma ** 2 + 1) ** 0.5).item()
    return 0.0, 1.0


class EulerSchedule(_SamplerSchedule):
    """`EulerDiscreteScheduler` (s_churn = 0): x_next = x + (x - x0) / sigma * (sigma_next - sigma), written as
    (1 + r) x - r x0 with r = (sigma_next - sigma) / sigma.  ancestral=True is `EulerAncestralDiscreteScheduler`:
    sigma_next becomes sigma_down and sigma_up * z is added, with a draw on every step (the last one's sigma_up is 0).
    Its `sample` prediction (which diffusers' class leaves unimplemented) uses x0 = e, as the Euler class does."""

    def __init__(self, num_inference_steps: int, config: SchedulerConfig = DEFAULT_CONFIG, ancestral: bool = False):
        self.name = "euler_a" if ancestral else "euler"
        d = sampler_config(self.name, config)
        self.config = d
        self.prediction_type = d["prediction_type"]
        n_train = int(d["num_train_timesteps"])
        _check_steps(num_inference_steps, n_train, self.name)
        self.num_inference_steps = num_inference_steps
        ac = _sampler_alphas_cumprod(d, zero_snr_floor=True)
        ts = _spaced(d["timestep_spacing"], n_train, num_inference_steps, int(d["steps_offset"]), np.float32)
        sig = (((1 - ac) / ac) ** 0.5).numpy()
        sig = np.interp(ts, np.arange(0, len(sig)), sig)
        self.sigmas = torch.from_numpy(np.concatenate([sig, [0.0]]).astype(np.float32))
        self.timesteps = [float(t) for t in ts.astype(np.float32)]
        smax = self.sigmas.max()
        self.init_noise_sigma = (smax if d["timestep_spacing"] in ("linspace", "trailing")
                                 else (smax ** 2 + 1) ** 0.5).item()
        self.ancestral = ancestral
        self._coeffs = []
        for i in range(len(self.timesteps)):
            s, s_next = self.sigmas[i], self.sigmas[i + 1]
            a_x, a_e = _x0_sigma_form(self.prediction_type, s)
            up = torch.zeros((), dtype=torch.float32)
            if ancestral:
                up = (s_next ** 2 * (s ** 2 - s_next ** 2) / s ** 2) ** 0.5
                s_next = (s_next ** 2 - up ** 2) ** 0.5
            r = (s_next - s) / s
            self._coeffs.append((a_x, a_e, (1 + r).item(), 0.0, (-r).item(), 0.0, up.item()))

    def in_scale(self, i: int) -> float:
        """`scale_model_input`: the UNet sees x / (sigma^2 + 1) ** 0.5."""
        return (1.0 / (self.sigmas[i] ** 2 + 1) ** 0.5).item()

    def has_noise(self, i: int) -> bool:
        return self.ancestral


class DDIMSchedule(_SamplerSchedule):
    """`DDIMScheduler` with eta = 0: x_next = sqrt(a_prev) x0 + sqrt(1 - a_prev) eps, with the previous timestep
    t - num_train_timesteps // n (`final_alpha_cumprod` below 0: 1 with set_alpha_to_one, else alphas_cumprod[0]).
    clip_sample clamps x0 only; eps stays the one computed from the raw model output (use_clipped_model_output
    False), so it is folded into c_x / c_e."""

    name = "ddim"

    def __init__(self, num_inference_steps: int, config: SchedulerConfig = DEFAULT_CONFIG):
        d = sampler_config("ddim", config)
        self.config = d
        self.prediction_type = d["prediction_type"]
        n_train = int(d["num_train_timesteps"])
        _check_steps(num_inference_steps, n_train, "ddim")
        self.num_inference_steps = num_inference_steps
        self.clip_range = float(d["clip_sample_range"]) if d["clip_sample"] else None
        ac = _sampler_alphas_cumprod(d, zero_snr_floor=False)
        final = torch.tensor(1.0) if d["set_alpha_to_one"] else ac[0]
        ts = _spaced(d["timestep_spacing"], n_train, num_inference_steps, int(d["steps_offset"]), np.int64)
        self.timesteps = [int(t) for t in ts]
        if max(self.timesteps) >= n_train:
            raise ValueError(f"steps_offset={d['steps_offset']} moves the last of {num_inference_steps} ddim timesteps "
                             f"past num_train_timesteps={n_train}")
        self._coeffs = []
        for t in self.timesteps:
            prev = t - n_train // num_inference_steps
            a, ap = ac[t], (ac[prev] if prev >= 0 else final)
            b = 1 - a
            dirn = (1 - ap) ** 0.5                            # (1 - a_prev - std_dev_t ** 2) ** 0.5, std_dev_t = 0
            if self.prediction_type == "epsilon":             # x0 = (x - b^.5 e) / a^.5; eps = e
                ax, ae, cx, ce = 1 / a ** 0.5, -(b ** 0.5) / a ** 0.5, 0.0, dirn
            elif self.prediction_type == "v_prediction":      # x0 = a^.5 x - b^.5 e; eps = a^.5 e + b^.5 x
                ax, ae, cx, ce = a ** 0.5, -(b ** 0.5), b ** 0.5 * dirn, a ** 0.5 * dirn
            else:                                             # x0 = e; eps = (x - a^.5 e) / b^.5
                ax, ae, cx, ce = 0.0, 1.0, dirn / b ** 0.5, -(a ** 0.5) * dirn / b ** 0.5
            self._coeffs.append(tuple(float(v) for v in (ax, ae, cx, ce, ap ** 0.5, 0.0, 0.0)))


class DPMSolverSchedule(_SamplerSchedule):
    """`DPMSolverMultistepScheduler(algorithm_type="dpmsolver++", solver_order=2, solver_type="midpoint",
    lower_order_final=True, final_sigmas_type="zero")`, karras: use_karras_sigmas=True.  With A = alpha_t (e^-h - 1):
    first order (step 0 and, sigma_next being 0, always the last step)  x_next = (s_t / s_s) x - A x0;
    second order  x_next = (s_t / s_s0) x - A (1 + 0.5 / r0) x0 + 0.5 A / r0 x0_prev,  r0 = h_0 / h.
    On the last step lambda_t is infinite and x_next = x0: the coefficients are (0, 1) there, set on the host."""

    def __init__(self, num_inference_steps: int, config: SchedulerConfig = DEFAULT_CONFIG, karras: bool = False):
        self.name = "dpmpp_2m_karras" if karras else "dpmpp_2m"
        d = sampler_config(self.name, config)
        self.config = d
        self.prediction_type = d["prediction_type"]
        n_train = int(d["num_train_timesteps"])
        n = num_inference_steps
        if not 1 <= n <= n_train - 1:
            raise ValueError(f"num_inference_steps must be in [1, {n_train - 1}] for the {self.name} sampler "
                             f"(its grid has num_inference_steps + 1 points), got {n}")
        self.num_inference_steps = n
        ac = _sampler_alphas_cumprod(d, zero_snr_floor=True)
        sp = d["timestep_spacing"]
        if sp == "linspace":
            ts = np.linspace(0, n_train - 1, n + 1).round()[::-1][:-1].copy().astype(np.int64)
        elif sp == "leading":
            ts = (np.arange(0, n + 1) * (n_train // (n + 1))).round()[::-1][:-1].copy().astype(np.int64)
            ts += int(d["steps_offset"])
        else:
            ts = np.arange(n_train, 0, -n_train / n).round().copy().astype(np.int64) - 1
        sig = (((1 - ac) / ac) ** 0.5).numpy()
        log_sig = np.log(sig)
        if karras:
            sig = _karras(np.flip(sig).copy(), n)
            ts = np.array([_sigma_to_t(s, log_sig) for s in sig]).round()
        else:
            sig = np.interp(ts, np.arange(0, len(sig)), sig)
        self.sigmas = torch.from_numpy(np.concatenate([sig, [0.0]]).astype(np.float32))
        self.timesteps = [int(t) for t in ts]
        self._coeffs = []
        for i in range(n):
            a_s = 1 / (self.sigmas[i] ** 2 + 1) ** 0.5           # _sigma_to_alpha_sigma_t
            s_s = self.sigmas[i] * a_s
            if self.prediction_type == "epsilon":
                ax, ae = (1 / a_s).item(), (-s_s / a_s).item()
            elif self.prediction_type == "v_prediction":
                ax, ae = a_s.item(), (-s_s).item()
            else:
                ax, ae = 0.0, 1.0
            if i == n - 1:                                      # sigma_next = 0: x_next = x0
                self._coeffs.append((ax, ae, 0.0, 0.0, 1.0, 0.0, 0.0))
                continue
            a_t = 1 / (self.sigmas[i + 1] ** 2 + 1) ** 0.5
            s_t = self.sigmas[i + 1] * a_t
            lam_t = torch.log(a_t) - torch.log(s_t)
            lam_s = torch.log(a_s) - torch.log(s_s)
            h = lam_t - lam_s
            A = a_t * (torch.exp(-h) - 1.0)
            if i == 0:
                c0, c1 = -A, torch.zeros(())
            else:
                a_p = 1 / (self.sigmas[i - 1] ** 2 + 1) ** 0.5
                lam_p = torch.log(a_p) - torch.log(self.sigmas[i - 1] * a_p)
                r0 = (lam_s - lam_p) / h
                c0, c1 = -A - 0.5 * A / r0, 0.5 * A / r0
            self._coeffs.append((ax, ae, (s_t / s_s).item(), 0.0, c0.item(), c1.item(), 0.0))


def _karras(in_sigmas: np.ndarray, n: int) -> np.ndarray:
    """`_convert_to_karras` (rho 7) between in_sigmas[-1] and in_sigmas[0], float64."""
    smin, smax = in_sigmas[-1].item(), in_sigmas[0].item()
    ramp = np.linspace(0, 1, n)
    lo, hi = smin ** (1 / 7.0), smax ** (1 / 7.0)
    return (hi + ramp * (lo - hi)) ** 7.0


def _sigma_to_t(sigma, log_sigmas: np.ndarray):
    """`_sigma_to_t`: the fractional timestep at which the interpolated log-sigma equals log(sigma)."""
    log_sigma = np.log(np.maximum(sigma, 1e-10))
    dists = log_sigma - log_sigmas[:, np.newaxis]
    low_idx = np.cumsum((dists >= 0), axis=0).argmax(axis=0).clip(max=log_sigmas.shape[0] - 2)
    high_idx = low_idx + 1
    low, high = log_sigmas[low_idx], log_sigmas[high_idx]
    w = np.clip((low - log_sigma) / (low - high), 0, 1)
    t = (1 - w) * low_idx + w * high_idx
    return t.reshape(np.shape(sigma))


def sampler_schedule(sampler: str, num_inference_steps: int, config: SchedulerConfig = DEFAULT_CONFIG):
    """The text-to-image schedule of a request's sampler: `LCMSchedule` for "lcm", else the class above."""
    s = check_sampler(sampler)
    if s == "lcm":
        return LCMSchedule(num_inference_steps, config=config)
    if s in ("euler", "euler_a"):
        return EulerSchedule(num_inference_steps, config, ancestral=s == "euler_a")
    if s == "ddim":
        return DDIMSchedule(num_inference_steps, config)
    return DPMSolverSchedule(num_inference_steps, config, karras=s == "dpmpp_2m_karras")


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
