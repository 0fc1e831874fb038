"""The guided-model samplers on the device, random-init weights:
  * the step kernel: `dl_sampler_step` (guidance + step fused) against `dl_cfg_combine` + `dl_lcm_step_ex` on the same
    shape, both with the CFG halves as input: SDXL 1024^2 (latent [1, 128, 128, 4]) and SD1.5 512^2 at B = 16
    (latent [16, 64, 64, 4]).  CUDA events around `--kernel-reps` back-to-back launches (working set far below the
    126 MB of L2: the numbers are L2-resident launch-bound times), median of `--reps`;
  * the whole text-to-image pass per sampler against LCM at the same step count: the SDXL UNet and VAE at 1024^2, 30
    steps, classifier-free guidance 7.5, B = 1, one CUDA-graph replay each, alternated sampler by sampler within every
    round, a 512 MB write evicting L2 before each replay.  Median and minimum of `--reps` rounds.
The card's name, power limit and max SM clock are read in the same run.  Prints one JSON line.
  python tools/bench_samplers.py [--size 1024] [--steps 30] [--reps 5] [--kernel-reps 200] [--no-pass]"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.dont_write_bytecode = True

from tools.bench_img2img import card  # noqa: E402

SAMPLERS = ["lcm", "euler", "euler_a", "ddim", "dpmpp_2m", "dpmpp_2m_karras"]
# stable-diffusion-xl-base-1.0's scheduler/scheduler_config.json
SDXL_SCHEDULER_CONFIG = {"_class_name": "EulerDiscreteScheduler", "beta_end": 0.012, "beta_schedule": "scaled_linear",
                         "beta_start": 0.00085, "clip_sample": False, "interpolation_type": "linear",
                         "num_train_timesteps": 1000, "prediction_type": "epsilon", "sample_max_value": 1.0,
                         "set_alpha_to_one": False, "skip_prk_steps": True, "steps_offset": 1,
                         "timestep_spacing": "leading", "trained_betas": None, "use_karras_sigmas": False}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--gs", type=float, default=7.5)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--kernel-reps", type=int, default=200)
    ap.add_argument("--no-pass", action="store_true", help="kernel timings only")
    a = ap.parse_args()
    import torch
    from dreamlab_b200 import lib, synthetic as syn
    from dreamlab_b200.engine import LCMPipelineB200
    from dreamlab_b200.scheduler import LCMSchedule, SchedulerConfig, sampler_noise_draws, sampler_schedule
    lib.require_cuda()
    dev = torch.device("cuda:0")
    res = {"card": card()}

    def events(fn, reps):
        ms = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        ms.sort()
        return ms[len(ms) // 2], ms[0]

    # ---- the step kernel
    cfgd = SchedulerConfig.from_dict(SDXL_SCHEDULER_CONFIG)
    dpm = sampler_schedule("dpmpp_2m", a.steps, cfgd)
    lcm = LCMSchedule(4)
    kern = {}
    for name, shape in (("sdxl_1024_b1", (1, 128, 128, 4)), ("sd15_512_b16", (16, 64, 64, 4))):
        g = torch.Generator(device=dev).manual_seed(0)
        u, t, x, p = (torch.randn(*shape, device=dev, generator=g) for _ in range(4))
        xn, x0, eps = torch.empty_like(x), torch.empty_like(x), torch.empty_like(x)
        k = dpm.coeffs(1)                                   # a second-order step: every operand is read

        def fused():
            for _ in range(a.kernel_reps):
                lib.sampler_step(u, t, a.gs, x, p, None, xn, x0, k)

        def split():
            for _ in range(a.kernel_reps):
                lib.cfg_combine(u, t, a.gs, eps)
                lib.lcm_step_ex(eps, x, p, xn, x0, lcm.coeffs(0))
        for f in (fused, split):
            f()
        torch.cuda.synchronize()
        r = {}
        for _ in range(3):                                  # alternate the two
            for nm, f in (("sampler_step_us", fused), ("cfg_combine_plus_lcm_step_us", split)):
                med, _ = events(f, 5)
                r.setdefault(nm, []).append(1000.0 * med / a.kernel_reps)
        kern[name] = {nm: round(sorted(v)[len(v) // 2], 3) for nm, v in r.items()}
        kern[name]["elements"] = x.numel()
    res["kernel"] = kern
    if a.no_pass:
        print(json.dumps(res))
        return

    # ---- whole passes, SDXL at 1024^2
    ucfg, vcfg = syn.sdxl_unet_cfg(), syn.sdxl_vae_cfg()
    pipe = LCMPipelineB200(syn.random_state_dict(syn.unet_shapes(ucfg), 0), ucfg,
                           syn.random_state_dict(syn.vae_decoder_shapes(vcfg), 1), vcfg, "cuda:0",
                           scheduler_config=cfgd)
    S, n, B = a.size, a.steps, 1
    h = S // 8
    pdim = ucfg.projection_class_embeddings_input_dim - 6 * ucfg.addition_time_embed_dim
    g = torch.Generator().manual_seed(0)
    pe = torch.randn(B, 77, ucfg.cross_attention_dim, generator=g)
    pooled = torch.randn(B, pdim, generator=g)
    z = torch.randn(B, 4, h, h, generator=g)
    noise = torch.randn(n, B, 4, h, h, generator=g)
    flush = torch.empty(512 * 1024 * 1024, device=dev, dtype=torch.uint8)

    def run(s):
        nd = sampler_noise_draws(s, n)
        return pipe.generate(pe, z, noise[:nd] if nd else None, n, a.gs, pooled_embeds=pooled, use_graph=True,
                             sampler=s)
    for s in SAMPLERS:                                      # capture + warm-up
        run(s)
    torch.cuda.synchronize()
    times = {s: [] for s in SAMPLERS}
    for _ in range(a.reps):
        for s in SAMPLERS:
            flush.zero_()
            med, _ = events(lambda: run(s), 1)
            times[s].append(med)
    res["pass"] = {"shape": f"SDXL {S}x{S} B={B} steps={n} cfg={a.gs}",
                   **{s: {"median_ms": round(sorted(v)[len(v) // 2], 2), "min_ms": round(min(v), 2)}
                      for s, v in times.items()}}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
