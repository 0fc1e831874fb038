"""One SD2-architecture text-to-image pass at 768x768, random-init weights (UNet config of stable-diffusion-2-1:
head dim 64 at every level, linear projections, cross_attention_dim 1024; SD1.x VAE), `v_prediction` scheduler config,
classifier-free guidance 7.5 (doubled batch), 4 LCM steps, B = 1:
  * the whole pass (UNet x 4 x 2 CFG halves + scheduler steps + VAE decode), one CUDA-graph replay, CUDA events;
  * one UNet forward on the doubled batch (the per-step UNet time), one CUDA-graph replay, CUDA events;
  * the level-0 self-attention kernel: head dim 64, 5 heads, S = 96 * 96 = 9216, batch 2 (the CFG halves), from a
    fused QKV buffer as the engine lays it out, events around `--attn-reps` back-to-back launches, and its TFLOP/s
    against 4 * B * H * S^2 * d.
Every timed replay runs after a 512 MB write that evicts L2 (126 MB).  Medians (and minima) of `--reps`.
The card's name, power limit and max SM clock are read in the same run.  Prints one JSON line.
  python tools/bench_sd2.py [--size 768] [--steps 4] [--reps 10] [--attn-reps 50]"""
import argparse
import json
import math
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.dont_write_bytecode = True

from tools.bench_img2img import card  # noqa: E402

# stable-diffusion-2-1 unet/config.json, the keys the b200 worker reads (plus upcast_attention, which it accepts)
SD2_UNET_CONFIG = {"_class_name": "UNet2DConditionModel", "attention_head_dim": [5, 10, 20, 20],
                   "block_out_channels": [320, 640, 1280, 1280], "cross_attention_dim": 1024,
                   "down_block_types": ["CrossAttnDownBlock2D"] * 3 + ["DownBlock2D"], "in_channels": 4,
                   "layers_per_block": 2, "norm_eps": 1e-05, "norm_num_groups": 32, "out_channels": 4,
                   "upcast_attention": True, "use_linear_projection": True}
SD2_SCHEDULER_CONFIG = {"_class_name": "DDIMScheduler", "beta_end": 0.012, "beta_schedule": "scaled_linear",
                        "beta_start": 0.00085, "clip_sample": False, "num_train_timesteps": 1000,
                        "prediction_type": "v_prediction", "set_alpha_to_one": False, "skip_prk_steps": True,
                        "steps_offset": 1, "trained_betas": None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=768)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--gs", type=float, default=7.5)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--attn-reps", type=int, default=50)
    a = ap.parse_args()
    import torch
    from backends.b200_worker import unet_cfg_from_json
    from dreamlab_b200 import lib, synthetic as syn
    from dreamlab_b200.engine import LCMPipelineB200
    from dreamlab_b200.scheduler import SchedulerConfig
    lib.require_cuda()
    S, n, gs, B = a.size, a.steps, a.gs, 1
    h = S // 8
    ucfg, vcfg = unet_cfg_from_json(SD2_UNET_CONFIG), syn.sd_vae_cfg()
    pipe = LCMPipelineB200(syn.random_state_dict(syn.unet_shapes(ucfg), 0), ucfg,
                           syn.random_state_dict(syn.vae_decoder_shapes(vcfg), 1), vcfg, "cuda:0",
                           scheduler_config=SchedulerConfig.from_dict(SD2_SCHEDULER_CONFIG))
    dev = pipe.device
    flush = torch.empty(512 * 1024 * 1024, device=dev, dtype=torch.uint8)      # 512 MB > 126 MB of L2

    def graph_of(fn):
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            fn()
        torch.cuda.current_stream().wait_stream(s)
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr, stream=s):
            fn()
        return gr

    def timed(fn, reps, flush_first=True):
        ms = []
        for _ in range(reps):
            if flush_first:
                flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        ms.sort()
        return round(ms[len(ms) // 2], 3), round(ms[0], 3)

    res = {"card": card(), "size": S, "steps": n, "guidance_scale": gs, "batch": B,
           "prediction_type": pipe.scheduler_config.prediction_type}
    # the whole pass, one graph replay
    g = torch.Generator().manual_seed(0)
    pe = torch.randn(B, 77, 1024, generator=g)
    z = torch.randn(B, 4, h, h, generator=g)
    noise = torch.randn(n - 1, B, 4, h, h, generator=g)
    pipe.generate(pe, z, noise, n, gs, use_graph=True)
    torch.cuda.synchronize()
    res["pass_ms"], res["pass_ms_min"] = timed(lambda: pipe.generate(pe, z, noise, n, gs, use_graph=True), a.reps)

    # one UNet forward on the doubled CFG batch
    unet = pipe.unet
    sched = pipe.schedule(n)
    pe2 = torch.randn(2 * B, 77, 1024, generator=g).to(dev, pipe.dt)
    x = torch.randn(B, h, h, 4, generator=g).to(dev)
    kvs = unet.encode_context(pe2)
    tembs = unet.time_embeddings(sched.timesteps, 2 * B, None, None)
    gr = graph_of(lambda: unet.forward(x, tembs[0], kvs, repeat=2))
    res["unet_step_ms"], res["unet_step_ms_min"] = timed(gr.replay, a.reps)
    del gr

    # level-0 self-attention: head dim 64, 5 heads, S = (size / 8)^2, batch 2
    H, d, Sq, Ba = ucfg.attention_head_dim[0], 64, h * h, 2 * B
    hstride = (d + 1 + 15) // 16 * 16                 # the engine's head stride (weights.head_stride)
    hs = H * hstride
    qkv = (torch.randn(Ba * Sq, 3 * hs, device=dev) * 0.5).to(torch.bfloat16)
    qkv.view(Ba * Sq, 3, H, hstride)[..., d:] = 0
    qkv.view(Ba * Sq, 3, H, hstride)[:, 2, :, d] = 1  # V's ones column (the softmax row sum)
    out = torch.empty(Ba * Sq, H * d, device=dev, dtype=torch.bfloat16)

    def attn():
        for _ in range(a.attn_reps):
            lib.attention(qkv, qkv[:, hs:], qkv[:, 2 * hs:], out, batch=Ba, sq=Sq, skv=Sq, heads=H, d=d,
                          dh_stride=hstride, ldq=3 * hs, ldk=3 * hs, ldv=3 * hs, ldo=H * d, scale=1.0 / math.sqrt(d),
                          v_ones=True)
    attn()
    torch.cuda.synchronize()
    med, mn = timed(attn, a.reps, flush_first=False)
    per = med / a.attn_reps
    res.update(attn_shape=f"B={Ba} heads={H} d={d} S={Sq}", attn_ms=round(per, 4), attn_ms_min=round(mn / a.attn_reps, 4),
               attn_tflops=round(4.0 * Ba * H * Sq * Sq * d / per / 1e9, 1))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
