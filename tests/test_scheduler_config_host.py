"""The model's scheduler config on the host (`LCMScheduler.from_config(scheduler/scheduler_config.json)`): defaults
and SD1.5's own config give today's coefficients bit for bit, every beta schedule / trained_betas / zero-SNR table
is the oracle's bit for bit, and configs the step cannot serve are refused naming the key (also by the worker,
before it touches a device)."""
import json
import os
from unittest.mock import patch

import pytest
import torch

from dreamlab_b200.scheduler import (DEFAULT_CONFIG, LCMSchedule, SchedulerConfig, alphas_cumprod, lcm_timesteps)
from oracle.lcm_config import SD2_V_SCHEDULER_CONFIG, OracleLCMSchedulerConfigured

# runwayml/stable-diffusion-v1-5 scheduler/scheduler_config.json
SD15_PNDM = {"_class_name": "PNDMScheduler", "_diffusers_version": "0.6.0", "beta_end": 0.012,
             "beta_schedule": "scaled_linear", "beta_start": 0.00085, "num_train_timesteps": 1000,
             "set_alpha_to_one": False, "skip_prk_steps": True, "steps_offset": 1, "trained_betas": None,
             "clip_sample": False}
# LCMScheduler's own defaults, written out (SimianLuo/LCM_Dreamshaper_v7 ships this class)
LCM_DEFAULT = {"_class_name": "LCMScheduler", "beta_end": 0.012, "beta_schedule": "scaled_linear",
               "beta_start": 0.00085, "clip_sample": False, "clip_sample_range": 1.0, "dynamic_thresholding_ratio": 0.995,
               "num_train_timesteps": 1000, "original_inference_steps": 50, "prediction_type": "epsilon",
               "rescale_betas_zero_snr": False, "sample_max_value": 1.0, "set_alpha_to_one": True, "steps_offset": 0,
               "thresholding": False, "timestep_scaling": 10.0, "timestep_spacing": "leading", "trained_betas": None}


def _schedules(config):
    """Every schedule kind a pass builds: text-to-image, image-to-image strengths, inpainting truncations."""
    out = []
    for n in (2, 4, 8):
        out.append(LCMSchedule(n, config=config) if config is not None else LCMSchedule(n))
        out.append(LCMSchedule(n, 0.5, config=config) if config is not None else LCMSchedule(n, 0.5))
        out.append(LCMSchedule(n, 0.75, truncate=True, config=config) if config is not None
                   else LCMSchedule(n, 0.75, truncate=True))
    out.append(LCMSchedule(1, config=config) if config is not None else LCMSchedule(1))
    return out


def _fingerprint(scheds):
    return [(s.timesteps, [s.coeffs(i) for i in range(len(s.timesteps))], s.add_noise_coeffs(),
             [s.add_noise_coeffs(t) for t in s.timesteps]) for s in scheds]


def _model_dir(tmp_path, config):
    d = tmp_path / "model"
    d.mkdir(exist_ok=True)
    if config is not None:
        (d / "scheduler").mkdir(exist_ok=True)
        (d / "scheduler" / "scheduler_config.json").write_text(json.dumps(config))
    return str(d)


@pytest.mark.parametrize("which", ["no_file", "lcm_default", "sd15_pndm", "no_dir"])
def test_default_configs_keep_todays_coefficients(tmp_path, which):
    cfg = {"no_file": None, "lcm_default": LCM_DEFAULT, "sd15_pndm": SD15_PNDM, "no_dir": None}[which]
    loaded = SchedulerConfig.load(None if which == "no_dir" else _model_dir(tmp_path, cfg))
    assert loaded.prediction_type == "epsilon" and not loaded.clip_sample
    today = _fingerprint(_schedules(None))
    assert _fingerprint(_schedules(loaded)) == today           # floats compared with ==: bit for bit
    assert torch.equal(alphas_cumprod(loaded), alphas_cumprod())
    assert all(s.prediction_type == "epsilon" and s.clip_range is None for s in _schedules(loaded))


def test_unknown_keys_ignored_and_missing_keys_default():
    c = SchedulerConfig.from_dict({"_class_name": "EulerDiscreteScheduler", "interpolation_type": "linear",
                                   "use_karras_sigmas": False, "prediction_type": "v_prediction"})
    assert c == SchedulerConfig(prediction_type="v_prediction")
    assert SchedulerConfig.from_dict({}) == DEFAULT_CONFIG


TABLES = {
    "scaled_linear": {},
    "linear": {"beta_schedule": "linear", "beta_start": 0.0001, "beta_end": 0.02},
    "squaredcos_cap_v2": {"beta_schedule": "squaredcos_cap_v2"},
    "trained_betas": {"trained_betas": [1e-4 + 2e-5 * i for i in range(1000)]},
    "zero_snr_scaled_linear": {"rescale_betas_zero_snr": True, "prediction_type": "v_prediction"},
    "zero_snr_linear": {"rescale_betas_zero_snr": True, "prediction_type": "v_prediction", "beta_schedule": "linear"},
    "zero_snr_cosine": {"rescale_betas_zero_snr": True, "prediction_type": "sample",
                        "beta_schedule": "squaredcos_cap_v2"},
    "short": {"num_train_timesteps": 500, "original_inference_steps": 25, "beta_end": 0.02},
}


@pytest.mark.parametrize("name", sorted(TABLES))
def test_alphas_cumprod_bit_exact_vs_oracle(name):
    d = TABLES[name]
    got = alphas_cumprod(SchedulerConfig.from_dict(d))
    want = OracleLCMSchedulerConfigured.from_config(d).alphas_cumprod
    assert got.dtype == torch.float32 and torch.equal(got, want)


@pytest.mark.parametrize("name", sorted(TABLES))
def test_schedule_coefficients_bit_exact_vs_oracle(name):
    """Timesteps and the step's (sqrt a_t, sqrt(1 - a_t), c_skip, c_out, sqrt a_prev, sqrt(1 - a_prev)) as the
    oracle's step computes them, for the config's table, original steps and timestep scaling."""
    d = {**TABLES[name], "timestep_scaling": 7.0}
    cfg = SchedulerConfig.from_dict(d)
    for n in (1, 4, 8):
        o = OracleLCMSchedulerConfigured.from_config(d)
        ts = o.set_timesteps(n).tolist()
        s = LCMSchedule(n, config=cfg)
        assert s.timesteps == ts == lcm_timesteps(n, config=cfg)
        for i, t in enumerate(ts):
            prev = ts[i + 1] if i + 1 < n else t
            a_t, a_p = o.alphas_cumprod[t], o.alphas_cumprod[prev]
            c_skip, c_out = o.boundary_scalings(t)
            want = (a_t.sqrt().item(), (1 - a_t).sqrt().item(), c_skip.item(), c_out.item(), a_p.sqrt().item(),
                    (1 - a_p).sqrt().item())
            assert s.coeffs(i) == want, (n, i)
            a = o.alphas_cumprod[t]
            assert s.add_noise_coeffs(t) == ((a ** 0.5).item(), ((1 - a) ** 0.5).item())


def test_zero_terminal_snr():
    base = alphas_cumprod()
    for sched in ("scaled_linear", "linear", "squaredcos_cap_v2"):
        d = {"rescale_betas_zero_snr": True, "prediction_type": "v_prediction", "beta_schedule": sched}
        ac = alphas_cumprod(SchedulerConfig.from_dict(d))
        plain = alphas_cumprod(SchedulerConfig.from_dict({"beta_schedule": sched}))
        assert ac[-1].item() == 0.0
        # ac[0] is unchanged up to the fp32 rounding of (s0 - sT) * (s0 / (s0 - sT)); exactly for scaled_linear
        assert abs(ac[0].item() - plain[0].item()) <= (0.0 if sched == "scaled_linear" else 1.2e-7)
        assert bool((ac[1:] < ac[:-1]).all())
    s = LCMSchedule(4, config=SchedulerConfig.from_dict({"rescale_betas_zero_snr": True,
                                                         "prediction_type": "v_prediction"}))
    assert s.timesteps[0] == 999 and s.coeffs(0)[:2] == (0.0, 1.0)       # v-prediction: x0 = -v at t = 999
    assert torch.equal(base, alphas_cumprod())


def test_prediction_type_and_clamp_travel_with_the_schedule():
    cfg = SchedulerConfig.from_dict({**SD2_V_SCHEDULER_CONFIG, "clip_sample": True, "clip_sample_range": 2})
    for s in (LCMSchedule(4, config=cfg), LCMSchedule(4, 0.5, config=cfg), LCMSchedule(4, 0.5, True, config=cfg)):
        assert s.prediction_type == "v_prediction" and s.clip_range == 2.0
    assert LCMSchedule(4, config=SchedulerConfig.from_dict(SD2_V_SCHEDULER_CONFIG)).clip_range is None


REFUSED = [
    ({"thresholding": True, "prediction_type": "v_prediction"}, "thresholding=True"),
    ({"beta_schedule": "sigmoid"}, "beta_schedule='sigmoid'"),
    ({"prediction_type": "flow"}, "prediction_type='flow'"),
    ({"rescale_betas_zero_snr": True}, "rescale_betas_zero_snr=True"),
    ({"rescale_betas_zero_snr": True, "prediction_type": "epsilon"}, "rescale_betas_zero_snr=True"),
    ({"trained_betas": [0.01] * 10}, "num_train_timesteps=1000"),
    ({"original_inference_steps": 2000}, "original_inference_steps=2000"),
]


@pytest.mark.parametrize("d,key", REFUSED)
def test_refused_configs_name_the_key(tmp_path, d, key):
    with pytest.raises(RuntimeError, match=key.replace("[", r"\[")):
        SchedulerConfig.from_dict(d)
    with pytest.raises(RuntimeError, match=key.replace("[", r"\[")):
        SchedulerConfig.load(_model_dir(tmp_path, d))


@pytest.mark.parametrize("d,key", REFUSED[:4])
def test_worker_refuses_at_construction(tmp_path, d, key):
    """The worker reads the config before it loads weights or asks for a device, so this holds without a GPU."""
    from backends.b200_worker import B200SDXLWorker, B200Worker
    root = _model_dir(tmp_path, d)
    with open(os.path.join(root, "model_index.json"), "w") as f:
        json.dump({"_class_name": "StableDiffusionPipeline"}, f)
    for cls in (B200Worker, B200SDXLWorker):
        with patch.dict(os.environ, {"MODEL_ROOT": str(tmp_path), "MODEL": "model"}):
            with pytest.raises(RuntimeError, match=key):
                cls(0)
