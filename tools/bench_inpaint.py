"""Inpainting against image-to-image and text-to-image at 512x512, 4 LCM steps, B = 1 and 16, random-init SD1.5-LCM
weights, for a 4-channel UNet (blend towards the noised image) and a 9-channel inpainting UNet (mask + masked image
latents as UNet input):
  * per-pass time: one CUDA-graph replay per batch, timed with CUDA events, the kinds alternated, median of --reps;
  * native kernel launches per replay (the captured graph's launch count).
Inpainting runs at strength 1.0 (its default: all 4 steps, like the other two kinds) and at 0.5 (the truncated
schedule: 2 steps; a 9-channel UNet then encodes the image and the masked image as one batch of 2B).  A 9-channel
UNet serves only inpainting.  The card's name and power limit are read in the same run.  Prints one JSON line.
  python tools/bench_inpaint.py [--size 512] [--steps 4] [--batches 1,16] [--reps 10]"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.dont_write_bytecode = True

from tools.bench_img2img import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--batches", default="1,16")
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    import torch
    from dreamlab_b200 import lib, synthetic as syn
    from dreamlab_b200.engine import LCMPipelineB200
    lib.require_cuda()
    S, n = a.size, a.steps
    h = S // 8
    vcfg = syn.sd_vae_cfg()
    vae_sd = syn.random_state_dict(syn.vae_decoder_shapes(vcfg), 1)
    vae_sd.update(syn.random_state_dict(syn.vae_encoder_shapes(vcfg), 3))
    res = {"card": card(), "size": S, "steps": n, "results": []}
    for cin in (4, 9):
        ucfg = syn.sd15_lcm_unet_cfg()
        ucfg.in_channels = cin
        pipe = LCMPipelineB200(syn.random_state_dict(syn.unet_shapes(ucfg), 0), ucfg, vae_sd, vcfg, "cuda:0")
        for B in (int(b) for b in a.batches.split(",")):
            g = torch.Generator().manual_seed(B)
            pe = torch.randn(B, 77, 768, generator=g)
            en, es, em = (torch.randn(B, 4, h, h, generator=g) for _ in range(3))
            noise = torch.randn(n - 1, B, 4, h, h, generator=g)
            img = torch.randint(0, 256, (B, S, S, 3), dtype=torch.uint8, generator=g)
            mask = torch.zeros(B, S, S, dtype=torch.uint8)
            mask[:, S // 4:3 * S // 4, S // 4:3 * S // 4] = 255

            def inpaint(strength):
                k = len(pipe.schedule(n, strength, inpaint=True).timesteps)
                return lambda: pipe.generate(pe, en, noise[:k - 1], n, 8.0, use_graph=True, init_images=img,
                                             mask_images=mask, strength=strength, posterior_noise=es,
                                             masked_posterior_noise=em)
            kinds = {"inpaint_s1.0": inpaint(1.0), "inpaint_s0.5": inpaint(0.5)}
            if cin == 4:
                kinds["txt2img"] = lambda: pipe.generate(pe, en, noise, n, 8.0, use_graph=True)
                kinds["img2img_s0.5"] = lambda: pipe.generate(pe, en, noise, n, 8.0, use_graph=True, init_images=img,
                                                              strength=0.5, posterior_noise=es)
            launches = {}
            for k, f in kinds.items():
                f()
                launches[k] = next(reversed(pipe._graphs.values())).launches     # the graph just replayed
            torch.cuda.synchronize()
            t = {k: [] for k in kinds}
            for _ in range(a.reps):
                for k, f in kinds.items():
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    f()
                    e1.record()
                    torch.cuda.synchronize()
                    t[k].append(e0.elapsed_time(e1))
            for k in kinds:
                ms = sorted(t[k])
                res["results"].append({"unet_in_channels": cin, "batch": B, "kind": k, "ms_median": round(ms[len(ms) // 2], 2),
                                       "ms_min": round(ms[0], 2), "images_per_s": round(B / ms[len(ms) // 2] * 1e3, 1),
                                       "launches": launches[k]})
        del pipe
        torch.cuda.empty_cache()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
