"""Host side of the guided-model samplers (CPU): the schedules of `scheduler.py` against known diffusers grids, against
the independent oracle restatement (`oracle/samplers.py`) coefficient for coefficient through the step kernel's linear
form, exactness on a point-mass data distribution, config handling, draw counts and refusals."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from dreamlab_b200 import scheduler as S
from dreamlab_b200.scheduler import SchedulerConfig

NAMES = ["euler", "euler_a", "ddim", "dpmpp_2m", "dpmpp_2m_karras"]
PREDS = ["epsilon", "v_prediction", "sample"]

# stable-diffusion-v1-5's scheduler/scheduler_config.json (PNDM; each sampler class keeps the keys it takes)
SD15 = {"_class_name": "PNDMScheduler", "beta_end": 0.012, "beta_schedule": "scaled_linear", "beta_start": 0.00085,
        "num_train_timesteps": 1000, "set_alpha_to_one": False, "skip_prk_steps": True, "steps_offset": 1,
        "trained_betas": None, "clip_sample": False}
# stable-diffusion-xl-base-1.0's
SDXL = {"_class_name": "EulerDiscreteScheduler", "beta_end": 0.012, "beta_schedule": "scaled_linear",
        "beta_start": 0.00085, "clip_sample": False, "interpolation_type": "linear", "num_train_timesteps": 1000,
        "prediction_type": "epsilon", "sample_max_value": 1.0, "set_alpha_to_one": False, "skip_prk_steps": True,
        "steps_offset": 1, "timestep_spacing": "leading", "trained_betas": None, "use_karras_sigmas": False}
V_ZERO_SNR = dict(SD15, prediction_type="v_prediction", rescale_betas_zero_snr=True, timestep_spacing="trailing")


def _cfg(d):
    return SchedulerConfig() if d is None else SchedulerConfig.from_dict(d)


def linear_step(sched, i, e, x, x0_prev=None, z=None):
    """The step kernel's linear form in fp32 torch (what `dl_sampler_step` computes)."""
    a_x, a_e, c_x, c_e, c_0, c_1, c_n = sched.coeffs(i)
    x0 = a_x * x + a_e * e
    if sched.clip_range is not None:
        x0 = x0.clamp(-sched.clip_range, sched.clip_range)
    out = c_x * x + c_e * e + c_0 * x0
    if x0_prev is not None and c_1 != 0.0:
        out = out + c_1 * x0_prev
    if z is not None and c_n != 0.0:
        out = out + c_n * z
    return out, x0


# ------------------------------------------------------------------------------------------------ known grids
def test_ddim_sd15_50_steps_leading_offset():
    s = S.DDIMSchedule(50, _cfg(SD15))
    assert s.timesteps == list(range(981, 0, -20))
    assert s.timesteps[0] == 981 and s.timesteps[1] == 961 and s.timesteps[-1] == 1
    assert s.clip_range is None and s.init_noise_sigma == 1.0       # SD15 states clip_sample false


def test_euler_sdxl_30_steps_leading_offset():
    s = S.EulerSchedule(30, _cfg(SDXL))
    assert s.timesteps[:3] == [958.0, 925.0, 892.0] and s.timesteps[-1] == 1.0 and len(s.timesteps) == 30
    smax = s.sigmas.max()
    assert s.init_noise_sigma == pytest.approx(float((smax ** 2 + 1) ** 0.5), rel=1e-7)   # leading: sqrt(max^2 + 1)


def test_euler_linspace_10_steps():
    s = S.EulerSchedule(10, SchedulerConfig())                      # no file: class default spacing linspace
    assert s.timesteps[0] == 999.0 and s.timesteps[-1] == 0.0
    assert S.EulerSchedule(7, SchedulerConfig()).timesteps[1] == 832.5   # fractional timesteps stay floats
    assert s.init_noise_sigma == pytest.approx(float(s.sigmas.max()), rel=1e-7)


def test_karras_sigmas_monotone_end_at_sigma_min_then_zero():
    s = S.DPMSolverSchedule(12, _cfg(SD15), karras=True)
    sig = s.sigmas.numpy()
    assert sig[-1] == 0.0 and np.all(np.diff(sig) < 0)
    ac = S.alphas_cumprod(SchedulerConfig.from_dict(SD15)).numpy()
    sigma_min = float(((1 - ac[0]) / ac[0]) ** 0.5)
    assert sig[-2] == pytest.approx(sigma_min, rel=1e-5)
    assert all(isinstance(t, int) for t in s.timesteps) and s.timesteps == sorted(s.timesteps, reverse=True)


def test_dpmpp_grid_drops_last_point():
    s = S.DPMSolverSchedule(10, SchedulerConfig())
    assert s.timesteps == [999, 899, 799, 699, 599, 500, 400, 300, 200, 100]


# ------------------------------------------------------------------------------------------------ vs oracle
def _oracle(name, d):
    from oracle.samplers import make
    o = make(name, d)
    return o


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("pred,base", [(p, b) for p in PREDS for b in ("sd15", "sdxl", "v_zero_snr", "none",
                                                                      "linspace", "trailing")
                                       if (p, b) != ("epsilon", "v_zero_snr")])     # refused (zero SNR + epsilon)
def test_product_matches_oracle_per_step(name, pred, base):
    """Random model outputs through the oracle's `step` and through the product's coefficients, on the same inputs
    at every step (teacher-forced on the oracle's trajectory): timesteps equal, init_noise_sigma, the UNet input scale,
    x0 and x_next agree to fp32 rounding."""
    from oracle.samplers import noise_draws, step
    d = {"sd15": SD15, "sdxl": SDXL, "v_zero_snr": V_ZERO_SNR, "none": None,
         "linspace": dict(SD15, timestep_spacing="linspace", clip_sample=True, clip_sample_range=1.5),
         "trailing": dict(SD15, timestep_spacing="trailing")}[base]
    if d is None and pred != "epsilon":
        d = {"prediction_type": pred}
    elif d is not None:
        d = dict(d, prediction_type=pred)
    n = 7
    sched = S.sampler_schedule(name, n, _cfg(d))
    o = _oracle(name, d)
    ts = o.set_timesteps(n)
    assert [float(t) for t in ts] == [float(t) for t in sched.timesteps]
    assert sched.init_noise_sigma == pytest.approx(float(o.init_noise_sigma), rel=1e-6)
    g = torch.Generator().manual_seed(3)
    shape = (2, 4, 8, 8)
    x = torch.randn(shape, generator=g) * float(o.init_noise_sigma)
    x0_prev = None
    assert sched.n_draws == noise_draws(name, n) == S.sampler_noise_draws(name, n)
    for i, t in enumerate(ts):
        e = torch.randn(shape, generator=g)
        z = torch.randn(shape, generator=g) if sched.has_noise(i) else None
        if hasattr(o, "sigmas"):
            want_in = o.scale_model_input(x)
            assert torch.allclose(x * sched.in_scale(i), want_in, rtol=2e-6, atol=0), i
        else:
            assert sched.in_scale(i) == 1.0
        ref_next, ref_x0 = step(o, e, t, x, z)
        got_next, got_x0 = linear_step(sched, i, e, x, x0_prev, z)
        scale = max(ref_next.abs().max().item(), x.abs().max().item())
        assert (got_x0 - ref_x0).abs().max().item() <= 2e-5 * max(ref_x0.abs().max().item(), 1.0), (i, "x0")
        assert (got_next - ref_next).abs().max().item() <= 2e-5 * scale, (i, "x_next")
        x0_prev = got_x0
        x = ref_next


# ------------------------------------------------------------------------------------------------ point mass
@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("pred", PREDS)
@pytest.mark.parametrize("n", [1, 2, 3, 5, 10, 25])
def test_point_mass_data_lands_exactly(name, pred, n):
    """Data distribution = a point mass at x*: the exact denoiser predicts x0 = x* from any x, i.e. the model output
    e = (x* - a_x x) / a_e.  Every sampler must then land on x* (DDIM with set_alpha_to_one: its last step reaches
    alphas_cumprod = 1)."""
    d = dict(SD15, prediction_type=pred, set_alpha_to_one=True)
    sched = S.sampler_schedule(name, n, _cfg(d))
    g = torch.Generator().manual_seed(n)
    x_star = torch.randn(1, 4, 8, 8, generator=g, dtype=torch.float64)
    x = torch.randn(1, 4, 8, 8, generator=g, dtype=torch.float64) * sched.init_noise_sigma
    x0_prev = None
    for i in range(n):
        a_x, a_e = sched.coeffs(i)[:2]
        e = (x_star - a_x * x) / a_e
        z = torch.randn(x.shape, generator=g, dtype=torch.float64) if sched.has_noise(i) else None
        x, x0 = linear_step(sched, i, e, x, x0_prev, z)
        assert torch.allclose(x0, x_star, rtol=0, atol=1e-5 * max(1.0, x.abs().max().item()))
        x0_prev = x0
    assert torch.allclose(x, x_star, rtol=0, atol=1e-5), (x - x_star).abs().max()


# ------------------------------------------------------------------------------------------------ config handling
def test_class_defaults_for_missing_keys():
    bare = SchedulerConfig.from_dict({"beta_schedule": "scaled_linear", "beta_start": 0.00085, "beta_end": 0.012})
    assert S.DDIMSchedule(4, bare).clip_range == 1.0                # DDIM's default clip_sample=True
    assert S.LCMSchedule(4, config=bare).clip_range is None         # LCM's default is False
    assert S.sampler_config("euler", bare)["timestep_spacing"] == "linspace"
    assert S.sampler_config("dpmpp_2m", bare)["timestep_spacing"] == "linspace"
    assert S.sampler_config("ddim", bare)["timestep_spacing"] == "leading"
    # a key the file leaves out takes the class default, also for the betas
    lin = S.sampler_config("euler", SchedulerConfig.from_dict({"prediction_type": "v_prediction"}))
    assert (lin["beta_schedule"], lin["beta_start"], lin["beta_end"]) == ("linear", 0.0001, 0.02)


def test_no_file_uses_sd15_betas_and_class_defaults():
    for name in NAMES:
        d = S.sampler_config(name, SchedulerConfig())
        assert (d["beta_schedule"], d["beta_start"], d["beta_end"]) == ("scaled_linear", 0.00085, 0.012)
        assert d["steps_offset"] == 0
    assert S.sampler_config("ddim", SchedulerConfig())["clip_sample"] is True
    ac = S._sampler_alphas_cumprod(S.sampler_config("ddim", SchedulerConfig()), False)
    assert torch.equal(ac, S.alphas_cumprod(SchedulerConfig()))


def test_sampler_name_fixes_dpmpp_settings():
    d = dict(SD15, _class_name="DPMSolverMultistepScheduler", solver_order=3, algorithm_type="dpmsolver",
             use_karras_sigmas=True)
    assert S.sampler_config("dpmpp_2m", _cfg(d))["solver_order"] == 2
    assert S.sampler_config("dpmpp_2m", _cfg(d))["use_karras_sigmas"] is False
    assert S.sampler_config("dpmpp_2m_karras", _cfg(d))["algorithm_type"] == "dpmsolver++"


@pytest.mark.parametrize("name,d,key", [
    ("euler", dict(SDXL, use_karras_sigmas=True), "use_karras_sigmas"),
    ("euler", dict(SDXL, interpolation_type="log_linear"), "interpolation_type"),
    ("euler_a", dict(SD15, timestep_spacing="weird"), "timestep_spacing"),
    ("dpmpp_2m", dict(SD15, euler_at_final=True), "euler_at_final"),
    ("dpmpp_2m", dict(SD15, variance_type="learned_range"), "variance_type"),
])
def test_refused_configs_name_the_key(name, d, key):
    with pytest.raises(RuntimeError, match=key):
        S.sampler_schedule(name, 4, _cfg(d))


@pytest.mark.parametrize("d,key", [(dict(SD15, thresholding=True), "thresholding"),
                                   (dict(SD15, beta_schedule="cosine"), "beta_schedule"),
                                   (dict(SD15, prediction_type="flow"), "prediction_type")])
def test_refused_at_load_name_the_key(d, key):
    with pytest.raises(RuntimeError, match=key):
        SchedulerConfig.from_dict(d)


def test_step_count_limits():
    for name in NAMES:
        with pytest.raises(ValueError):
            S.sampler_schedule(name, 0, SchedulerConfig())
        with pytest.raises(ValueError):
            S.sampler_schedule(name, 1001, SchedulerConfig())
    for name in ("euler", "euler_a"):
        assert len(S.sampler_schedule(name, 1000, SchedulerConfig()).timesteps) == 1000
    assert len(S.sampler_schedule("ddim", 1000, SchedulerConfig()).timesteps) == 1000
    with pytest.raises(ValueError):
        S.sampler_schedule("dpmpp_2m", 1000, SchedulerConfig())           # its grid has n + 1 points
    assert len(S.sampler_schedule("dpmpp_2m", 999, SchedulerConfig()).timesteps) == 999
    with pytest.raises(ValueError):
        S.sampler_schedule("lcm", 51, SchedulerConfig())                  # LCM keeps original_inference_steps


# ------------------------------------------------------------------------------------------------ draws, refusals
@pytest.mark.parametrize("n", [1, 4, 30])
def test_draw_counts(n):
    assert S.sampler_noise_draws("lcm", n) == n - 1
    assert S.sampler_noise_draws(None, n) == n - 1
    assert S.sampler_noise_draws("euler_a", n) == n
    for name in ("euler", "ddim", "dpmpp_2m", "dpmpp_2m_karras"):
        assert S.sampler_noise_draws(name, n) == 0
        assert S.sampler_schedule(name, n, SchedulerConfig()).n_draws == 0
    assert S.sampler_schedule("euler_a", n, SchedulerConfig()).n_draws == n


def test_unknown_sampler_refused_with_the_names():
    from backends.b200_worker import request_sampler
    with pytest.raises(RuntimeError, match="dpmpp_2m_karras"):
        S.check_sampler("heun")
    with pytest.raises(RuntimeError, match="euler_a"):
        request_sampler(SimpleNamespace(sampler="unipc"))
    assert request_sampler(SimpleNamespace()) == "lcm"
    assert request_sampler(SimpleNamespace(sampler=None)) == "lcm"
    assert request_sampler(SimpleNamespace(sampler="lcm", init_image=b"x")) == "lcm"


@pytest.mark.parametrize("field", ["init_image", "mask_image"])
def test_non_lcm_sampler_with_init_image_refused(field):
    from backends.b200_worker import request_sampler
    with pytest.raises(RuntimeError, match="LCM sampler only"):
        request_sampler(SimpleNamespace(sampler="ddim", **{field: b"png"}))


def test_pool_batch_key_keeps_lcm_keys_and_separates_samplers():
    from backends.base import GenSpec
    from backends.worker_pool import _batch_key

    def job(**kw):
        return SimpleNamespace(req=SimpleNamespace(size="512x512", num_inference_steps=4, guidance_scale=7.5, **kw))
    plain = _batch_key(job())
    assert _batch_key(job(sampler=None)) == plain and _batch_key(job(sampler="lcm")) == plain
    assert plain == ("512x512", 4, (None, 0))
    keys = {_batch_key(job(sampler=s)) for s in NAMES}
    assert len(keys) == len(NAMES) and plain not in keys
    assert _batch_key(job(sampler="ddim")) == plain + (("sampler", "ddim"),)
    assert _batch_key(job(sampler="ddim"), True) == plain + (("sampler", "ddim"), 7.5)
    assert GenSpec(prompt="p", size="512x512", steps=4, cfg=1.0).sampler is None


def test_pool_never_mixes_samplers_in_one_batch():
    import threading
    import time
    from test_worker_pool import make_config, make_registry
    from backends.worker_pool import GenerationJob, WorkerPool, reset_worker_pool

    class W:
        worker_id = 0

        def __init__(self):
            self.batches, self.lock = [], threading.Lock()

        def run_batch(self, jobs, with_latents=False):
            time.sleep(0.1)
            with self.lock:
                self.batches.append([getattr(j.req, "sampler", None) for j in jobs])
            return [(b"png", 1) for _ in jobs]

        def run_job(self, job):
            return self.run_batch([job])[0]
    w = W()
    reset_worker_pool()
    pool = WorkerPool(queue_max=64, mode_config=make_config(), registry=make_registry(),
                      worker_factory=lambda worker_id: w, num_workers=1, max_batch=16)
    try:
        def r(s):
            return SimpleNamespace(prompt="p", size="512x512", num_inference_steps=4, guidance_scale=1.0, seed=1,
                                   **({} if s == "absent" else {"sampler": s}))
        first = pool.submit_job(GenerationJob(req=r("absent")))
        time.sleep(0.03)
        order = ["absent", None, "lcm", "ddim", "ddim", "euler_a", "dpmpp_2m", "dpmpp_2m", "lcm"]
        futs = [pool.submit_job(GenerationJob(req=r(s))) for s in order]
        for f in [first] + futs:
            f.result(timeout=10)
    finally:
        pool.shutdown()
    assert w.batches[1:] == [[None, None, "lcm"], ["ddim", "ddim"], ["euler_a"], ["dpmpp_2m", "dpmpp_2m"], ["lcm"]]
