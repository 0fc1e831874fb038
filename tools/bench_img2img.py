"""Image-to-image at the C2 geometry (B = 16, 512x512, 4 LCM steps, strength 0.5), random-init SD1.5-LCM weights:
  * VAE encode per batch: CUDA-graph replay timed with CUDA events, L2 overwritten before every replay;
    achieved TFLOP/s against the encoder's algorithmic count (ENCODER_GFLOP_512, 2 * MAC from the shapes);
  * VAE decode per batch, the same way (a control);
  * images/s of the whole img2img pass and of text-to-image, alternated, each one CUDA-graph replay per batch;
  * the share of the three im2col_s2_pad01 launches in one eager encode with per-launch events.
The card's name and power limit are read in the same run.  Prints one JSON line at the end.
  python tools/bench_img2img.py [--batch 16] [--size 512] [--reps 10]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.dont_write_bytecode = True


def encoder_gflop(size: int, ch=(128, 256, 512, 512), lpb=2, latent=4) -> float:
    """Algorithmic GFLOP (2 * MAC) of AutoencoderKL.encode + quant_conv on one size x size image, from the shapes:
    convolutions, 1x1 shortcuts, the mid-block attention projections and its two S x S x C contractions.
    Norms, activations and softmax are not counted."""
    mac = 0
    hw = size * size
    mac += hw * ch[0] * 3 * 9                                      # conv_in
    prev = ch[0]
    for i, c in enumerate(ch):
        for j in range(lpb):
            cin = prev if j == 0 else c
            mac += hw * c * cin * 9 + hw * c * c * 9               # conv1, conv2
            if cin != c:
                mac += hw * c * cin                                 # conv_shortcut
        if i != len(ch) - 1:
            hw //= 4
            mac += hw * c * c * 9                                   # Downsample2D
        prev = c
    C = ch[-1]
    mac += 2 * hw * C * C * 9                                       # mid resnet 0
    mac += 4 * hw * C * C + 2 * hw * hw * C                         # q, k, v, out + QK^T, PV
    mac += 2 * hw * C * C * 9                                       # mid resnet 1
    mac += hw * 2 * latent * C * 9 + hw * 4 * latent * latent     # conv_out, quant_conv
    return 2.0 * mac / 1e9


ENCODER_GFLOP_512 = encoder_gflop(512)


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:                                            # noqa: BLE001
        return f"unknown ({e!r})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--strength", type=float, default=0.5)
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    import torch
    from dreamlab_b200 import lib, synthetic as syn
    from dreamlab_b200.engine import LCMPipelineB200
    lib.require_cuda()
    B, S, n = a.batch, a.size, a.steps
    h = S // 8
    ucfg, vcfg = syn.sd15_lcm_unet_cfg(), syn.sd_vae_cfg()
    vae_sd = syn.random_state_dict(syn.vae_decoder_shapes(vcfg), 1)
    vae_sd.update(syn.random_state_dict(syn.vae_encoder_shapes(vcfg), 3))
    pipe = LCMPipelineB200(syn.random_state_dict(syn.unet_shapes(ucfg), 0), ucfg, vae_sd, vcfg, "cuda:0")
    dev = pipe.device
    g = torch.Generator(device=dev).manual_seed(0)
    img = torch.randint(0, 256, (B, S, S, 3), device=dev, dtype=torch.uint8, generator=g)
    lat = torch.randn(B, h, h, 4, device=dev, generator=g)
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

    def time_graph(gr, reps):
        ms = []
        for _ in range(reps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            gr.replay()
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        ms.sort()
        return ms[len(ms) // 2], ms[0]

    enc_g = graph_of(lambda: pipe.vae_encoder.moments(img))
    dec_g = graph_of(lambda: pipe.vae.decode(lat))
    enc_ms, enc_min = time_graph(enc_g, a.reps)
    dec_ms, dec_min = time_graph(dec_g, a.reps)
    del enc_g, dec_g

    # whole passes: alternate img2img and text-to-image batches, one graph replay each
    pe = torch.randn(B, 77, 768)
    en = torch.randn(B, 4, h, h)
    es = torch.randn(B, 4, h, h)
    noise = torch.randn(n - 1, B, 4, h, h)
    init = img.cpu()
    run_i2i = lambda: pipe.generate(pe, en, noise, n, 8.0, use_graph=True, init_images=init,  # noqa: E731
                                    strength=a.strength, posterior_noise=es)
    run_t2i = lambda: pipe.generate(pe, en, noise, n, 8.0, use_graph=True)                     # noqa: E731
    for f in (run_i2i, run_t2i):
        f()
    torch.cuda.synchronize()
    t = {"img2img": [], "txt2img": []}
    for _ in range(a.reps):
        for k, f in (("img2img", run_i2i), ("txt2img", run_t2i)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f()
            e1.record()
            torch.cuda.synchronize()
            t[k].append(e0.elapsed_time(e1))
    med = {k: sorted(v)[len(v) // 2] for k, v in t.items()}

    # share of the stride-2 gathers in one eager, instrumented encode
    pipe.vae_encoder.moments(img)
    lib.profile_begin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    pipe.vae_encoder.moments(img)
    e1.record()
    prof = lib.profile_end()
    eager_ms = e0.elapsed_time(e1)
    s2 = prof.get("im2col_s2_pad01", {"ms": 0.0, "n": 0})
    res = {
        "card": card(), "batch": B, "size": S, "steps": n, "strength": a.strength,
        "encoder_gflop_per_image": round(ENCODER_GFLOP_512 * (S / 512) ** 2, 2),
        "encode_ms": round(enc_ms, 3), "encode_ms_min": round(enc_min, 3),
        "encode_tflops": round(ENCODER_GFLOP_512 * (S / 512) ** 2 * B / enc_ms, 1),
        "decode_ms": round(dec_ms, 3), "decode_ms_min": round(dec_min, 3),
        "img2img_batch_ms": round(med["img2img"], 2), "img2img_images_per_s": round(B / med["img2img"] * 1e3, 1),
        "txt2img_batch_ms": round(med["txt2img"], 2), "txt2img_images_per_s": round(B / med["txt2img"] * 1e3, 1),
        "eager_encode_ms_instrumented": round(eager_ms, 3), "im2col_s2_pad01_launches": s2["n"],
        "im2col_s2_pad01_ms": round(s2["ms"], 3),
        "im2col_s2_pad01_share_of_eager_encode": round(s2["ms"] / eager_ms, 4),
    }
    print(json.dumps(res))


if __name__ == "__main__":
    main()
