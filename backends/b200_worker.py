"""`b200` worker: the reference's `PipelineWorker` contract on the B200-native hot path.

Drop-in replacement for `DiffusersCudaWorker` (reference `backends/cuda_worker.py:20-304`):
same constructor (`B200Worker(worker_id)`), same env (`MODEL_ROOT`, `MODEL`, `CUDA_DEVICE`,
`CUDA_DTYPE`), same attributes (`worker_id`, `pipe`, `device`, `dtype`), same results
(`run_job -> (png, seed)`, `run_job_with_latents -> (png, seed, 512 B fp16 [1,4,8,8])`), same
errors (`RuntimeError("Invalid size '…', expected 'WIDTHxHEIGHT'")`, missing env ->
RuntimeError).  What changes is everything below `self.pipe(...)`: the LCM loop, UNet, scheduler
step and VAE decode run in `dreamlab_b200` (hand-written sm_100a kernels, no diffusers).

Extras the reference does not have (SURVEY.md §8f rank 1): `run_batch(jobs)` generates many
requests of the same geometry in ONE batched pass (per-request Philox streams preserved) and
`run_job_with_latents` returns the latent of the same pass instead of re-running the pipeline.
Requests carrying `init_image` (and `strength`, see `backends/base.py`) run image-to-image through
the same entry points (`LatentConsistencyModelImg2ImgPipeline` semantics, LCM UNets only); with a `mask_image`
as well they run inpainting (`StableDiffusionInpaintPipeline` semantics with `LCMScheduler`, 4- and 9-channel UNets).
"""
from __future__ import annotations

import io
import json
import collections
import os
import time
from typing import List, Sequence, Tuple

import torch

from .base import PipelineWorker


def parse_size(size) -> Tuple[int, int]:
    try:
        w_str, h_str = str(size).lower().split("x")
        return int(w_str), int(h_str)
    except Exception:
        raise RuntimeError(f"Invalid size '{size}', expected 'WIDTHxHEIGHT'")


def _device_for(worker_id: int) -> str:
    """One worker per GPU: worker k -> cuda:k, unless CUDA_DEVICE pins worker 0."""
    env = (os.environ.get("CUDA_DEVICE") or "").strip()
    if env and worker_id == 0:
        return env
    n = torch.cuda.device_count()
    return f"cuda:{worker_id % max(n, 1)}"


class _Cfg(dict):
    __getattr__ = dict.__getitem__


def _load_component(path: str):
    """diffusers-layout component dir -> (config dict, state dict)."""
    from safetensors.torch import load_file
    with open(os.path.join(path, "config.json")) as f:
        cfg = json.load(f)
    # plain names first, then the `variant="fp16"` names the reference's SDXL worker downloads
    # (`backends/cuda_worker.py:371-377`)
    for name in ("diffusion_pytorch_model.safetensors", "model.safetensors",
                 "diffusion_pytorch_model.fp16.safetensors", "model.fp16.safetensors"):
        p = os.path.join(path, name)
        if os.path.exists(p):
            return cfg, load_file(p)
    raise RuntimeError(f"no safetensors weights under {path}")


def unet_cfg_from_json(c: dict):
    from types import SimpleNamespace
    down = c.get("down_block_types", ["CrossAttnDownBlock2D"] * 3 + ["DownBlock2D"])
    heads = c.get("attention_head_dim", 8)
    heads = tuple(heads) if isinstance(heads, (list, tuple)) else heads
    tl = c.get("transformer_layers_per_block", 1)
    tl = tuple(tl) if isinstance(tl, (list, tuple)) else ((tl,) * len(down) if tl != 1 else ())
    aet = c.get("addition_embed_type")
    if aet not in (None, "text_time"):
        raise RuntimeError(f"b200 worker: addition_embed_type={aet!r} is not supported")
    return SimpleNamespace(
        in_channels=c.get("in_channels", 4), out_channels=c.get("out_channels", 4),
        block_out_channels=tuple(c.get("block_out_channels", (320, 640, 1280, 1280))),
        down_attn=tuple("CrossAttn" in t for t in down),
        layers_per_block=c.get("layers_per_block", 2),
        cross_attention_dim=c.get("cross_attention_dim", 768),
        attention_head_dim=heads, norm_num_groups=c.get("norm_num_groups", 32),
        norm_eps=c.get("norm_eps", 1e-5), time_cond_proj_dim=c.get("time_cond_proj_dim"),
        transformer_layers_per_block=tl, use_linear_projection=bool(c.get("use_linear_projection", False)),
        addition_embed_type=aet, addition_time_embed_dim=c.get("addition_time_embed_dim", 256),
        projection_class_embeddings_input_dim=c.get("projection_class_embeddings_input_dim", 2816))


def vae_cfg_from_json(c: dict):
    from types import SimpleNamespace
    return SimpleNamespace(
        latent_channels=c.get("latent_channels", 4), out_channels=c.get("out_channels", 3),
        block_out_channels=tuple(c.get("block_out_channels", (128, 256, 512, 512))),
        layers_per_block=c.get("layers_per_block", 2), norm_num_groups=c.get("norm_num_groups", 32),
        scaling_factor=c.get("scaling_factor", 0.18215), sample_size=c.get("sample_size", 512))


class B200Worker(PipelineWorker):
    _tag = "b200"
    _env_what = "BACKEND=cuda"

    def __init__(self, worker_id: int):
        self.worker_id = worker_id
        model_root = (os.environ.get("MODEL_ROOT") or "").strip()
        model_name = (os.environ.get("MODEL") or "").strip()
        if not model_root:
            raise RuntimeError(f"MODEL_ROOT is required for {self._env_what}")
        if not model_name:
            raise RuntimeError(f"MODEL is required for {self._env_what}")
        path = os.path.join(model_root, model_name)
        # a diffusers-layout directory (`from_pretrained`, reference `backends/cuda_worker.py:70-77`) or a
        # single-file checkpoint in the original layout (`from_single_file`, `:79-85`; every model of the
        # reference's modes.yaml.example is one)
        single = os.path.isfile(path) and path.lower().endswith(".safetensors")
        if not single and not (os.path.isdir(path) and os.path.exists(os.path.join(path, "model_index.json"))):
            raise RuntimeError(f"b200 worker needs a diffusers-layout model directory or a single-file "
                               f".safetensors checkpoint, got: {path}")
        if not torch.cuda.is_available():
            raise RuntimeError("b200 worker needs a CUDA device (sm_100a); there is no CPU fallback")

        from dreamlab_b200.engine import LCMPipelineB200
        from dreamlab_b200 import lib
        lib.load()

        self.device = _device_for(worker_id)
        # CUDA_DTYPE keeps its meaning for the *noise stream*: the reference draws latents and
        # step noise in this dtype (fp16 default, `backends/cuda_worker.py:55-61`).  fp16 / bf16
        # compute in bf16 (fp32 accumulate) on the tensor cores; fp32 runs the fp32 precision mode.
        dtype_str = os.environ.get("CUDA_DTYPE", "fp16").lower().strip()
        self.dtype = {"bf16": torch.bfloat16, "fp32": torch.float32}.get(dtype_str, torch.float16)
        torch.cuda.set_device(self.device)

        self._single = None
        if single:
            from dreamlab_b200.single_file import load_single_file
            self._single = load_single_file(path)
            self._model_index = self._single["model_index"]
            ucfg_json, unet_sd = self._single["unet"]
            vcfg_json, vae_sd = self._single["vae"]
        else:
            with open(os.path.join(path, "model_index.json")) as f:
                self._model_index = json.load(f)
            ucfg_json, unet_sd = _load_component(os.path.join(path, "unet"))
            vcfg_json, vae_sd = _load_component(os.path.join(path, "vae"))
        # vae_tiling: the reference switches `pipe.vae.enable_tiling()` on unconditionally
        # (`backends/cuda_worker.py:91`, `:390`)
        # CUDA_DTYPE=fp32 selects the fp32 precision mode (CUDA-core kernels, parity bar 1e-4);
        # fp16 / bf16 both run the bf16 tcgen05 path
        self.pipe = LCMPipelineB200(unet_sd, unet_cfg_from_json(ucfg_json), vae_sd,
                                    vae_cfg_from_json(vcfg_json), self.device, vae_tiling=True,
                                    precision="fp32" if dtype_str == "fp32" else "bf16")
        self._text = self._make_text_encoder(path)
        self._single = None                               # the converted state dicts are packed: drop the copies
        # the attributes the reference's worker tests look for on `pipe` (`tests/test_sdxl_worker.py:127-130`)
        towers = getattr(self._text, "models", None) or (getattr(self._text, "model", None),)
        self.pipe.text_encoder = towers[0] if towers else None
        if len(towers) > 1:
            self.pipe.text_encoder_2 = towers[1]
        elif self.pipe.is_sdxl:
            self.pipe.text_encoder_2 = None
        self._load_styles({k: tuple(v.shape) for k, v in unet_sd.items()})
        print(f"[{self._tag}] worker {worker_id} loaded: {model_name} on {self.device} "
              f"(noise dtype={dtype_str}, compute {self.pipe.precision}, styles={sorted(self._style_loaded)})")

    # ------------------------------------------------------------------ styles
    def _load_styles(self, unet_shapes):
        """Preload every registry style whose cross-attention dim matches the model (reference
        `backends/cuda_worker.py:123-147`); a style that fails to load is skipped, not fatal."""
        from backends import styles
        from dreamlab_b200.lora import StyleManager
        from safetensors.torch import load_file
        self._style_loaded = {}
        self._style_api = "merged"
        self._styles = StyleManager(self.pipe.unet, unet_shapes)
        self._registry = dict(styles.STYLE_REGISTRY) or styles.load_registry()
        cad = self.pipe.unet.cfg.cross_attention_dim
        for sid, sd in self._registry.items():
            if sd.required_cross_attention_dim is not None and int(sd.required_cross_attention_dim) != int(cad):
                print(f"[{self._tag}] skip style '{sid}': incompatible cross_attention_dim "
                      f"(model={cad} style={sd.required_cross_attention_dim})")
                self._style_loaded[sd.adapter_name] = False
                continue
            try:
                ad = self._styles.load(sd.adapter_name, load_file(sd.lora_path))
                self._style_loaded[sd.adapter_name] = True
                print(f"[{self._tag}] loaded style LoRA: {sid} -> {sd.lora_path} (adapter={sd.adapter_name}, "
                      f"{ad.num_tensors} packed tensors, {len(ad.skipped)} entries skipped)")
            except Exception as e:                         # noqa: BLE001 - same policy as the reference
                self._style_loaded[sd.adapter_name] = False
                print(f"[{self._tag}] FAILED to load style LoRA {sid}: {e!r}")

    def _apply_style(self, style_id, level) -> None:
        """Exclusive style selection (reference `backends/cuda_worker.py:165-196`)."""
        from backends.styles import clamp_level
        if not style_id or int(level) <= 0:
            self._styles.disable()
            return
        sd = self._registry.get(style_id)
        if not sd or not self._style_loaded.get(sd.adapter_name, False):
            self._styles.disable()
            return
        weight = float(sd.levels[clamp_level(level, len(sd.levels)) - 1])
        self._styles.set_adapter(sd.adapter_name, weight)

    @staticmethod
    def _style_of(req):
        sl = getattr(req, "style_lora", None)
        style = getattr(sl, "style", None) if sl else None
        level = int(getattr(sl, "level", 0) or 0) if sl else 0
        return (style, level) if style and level > 0 else (None, 0)

    def _make_text_encoder(self, path):
        return _TextEncoder(path, self.device, self.pipe.unet.cfg.cross_attention_dim, single=self._single)

    # one CUDA-graph replay per request batch (captured per (batch, size, steps) on first use; LRU
    # of LCMPipelineB200.max_graphs geometries): at small batches the eager path is bound by
    # launch latency, not by the GPU.  B200_CUDA_GRAPH=0 runs eagerly.
    _use_graph = os.environ.get("B200_CUDA_GRAPH", "1").lower() not in ("0", "false", "no", "off")

    @property
    def batch_same_guidance(self) -> bool:
        """A UNet without the LCM guidance embedding (time_cond_proj_dim None: vanilla SD1.5 checkpoints such
        as the reference's dreamshaper / realisticvision modes) runs classifier-free guidance on a doubled batch
        when guidance_scale > 1: one scale per batch, so the pool must group requests by it."""
        return not self.pipe.unet.cfg.time_cond_proj_dim

    def _negative(self, n: int):
        """Unconditional half under CFG: `StableDiffusionPipeline.encode_prompt` encodes the EMPTY prompt
        (zeros are an SDXL-only convention, `force_zeros_for_empty_prompt`)."""
        return self._text.encode([""] * n)

    def _generate(self, prompts, lat, noise, steps, gs, height, width, decode=True, init=None):
        """init (image-to-image): (u8 images [B,H,W,3], posterior draw [B,4,h,w], strength); lat is then the
        add_noise draw.  Inpainting appends (u8 masks [B,H,W], the masked image's posterior draw)."""
        pe = self._text.encode(prompts)
        neg = self._negative(len(prompts)) if self.pipe.cfg_scale_for(gs) is not None else None
        i2i = {}
        if init is not None:
            i2i = dict(init_images=init[0], posterior_noise=init[1], strength=init[2])
            if len(init) > 3:
                i2i.update(mask_images=init[3], masked_posterior_noise=init[4])
        return self.pipe.generate(pe, lat, noise, steps, gs, return_latents=True, use_graph=self._use_graph,
                                  negative_prompt_embeds=neg, decode=decode, **i2i)

    def _check_img2img(self) -> None:
        """Refuse image-to-image where this engine does not implement diffusers' semantics."""
        if not self.pipe.unet.cfg.time_cond_proj_dim:
            raise RuntimeError("image-to-image needs an LCM UNet (time_cond_proj_dim): the LCM img2img pipeline has "
                               "no classifier-free guidance branch, and CFG img2img is not implemented")
        self.pipe.require_encoder()

    def _check_inpaint(self) -> None:
        """Refuse inpainting where this engine does not implement diffusers' semantics."""
        self.pipe.require_encoder()

    def _inpaint_plan(self, steps: int, strength: float):
        """-> (steps of the truncated schedule, whether the image's posterior draw is consumed: diffusers encodes the
        image only for a 4-channel UNet or strength < 1).  ValueError when the strength leaves no step."""
        from dreamlab_b200.scheduler import LCMSchedule
        k = len(LCMSchedule(steps, strength, truncate=True).timesteps)
        return k, getattr(self.pipe.unet.cfg, "in_channels", 4) != 9 or strength < 1.0

    @staticmethod
    def _mask_image(obj, width: int, height: int):
        """A request's mask_image (image bytes PIL opens, converted to "L", or an HxW uint8 array of L values) ->
        contiguous uint8 [height, width].  No resizing: any other size is refused."""
        import numpy as np
        if isinstance(obj, (bytes, bytearray, memoryview)):
            from PIL import Image
            with Image.open(io.BytesIO(bytes(obj))) as im:
                arr = np.asarray(im.convert("L"))
        else:
            arr = np.asarray(obj)
            if arr.dtype != np.uint8 or arr.ndim != 2:
                raise RuntimeError(f"mask_image: image bytes or an HxW uint8 array expected, got "
                                   f"{arr.dtype} {list(arr.shape)}")
        if arr.shape != (height, width):
            raise RuntimeError(f"mask_image is {arr.shape[1]}x{arr.shape[0]}, the request's size is "
                               f"{width}x{height} (masks are not resized)")
        return np.ascontiguousarray(arr)

    @staticmethod
    def _init_image(obj, width: int, height: int):
        """A request's init_image (image bytes PIL opens, or an HxWx3 uint8 array) -> contiguous RGB uint8
        [height, width, 3].  No resizing: any other size is refused."""
        import numpy as np
        if isinstance(obj, (bytes, bytearray, memoryview)):
            from PIL import Image
            with Image.open(io.BytesIO(bytes(obj))) as im:
                arr = np.asarray(im.convert("RGB"))
        else:
            arr = np.asarray(obj)
            if arr.dtype != np.uint8 or arr.ndim != 3 or arr.shape[2] != 3:
                raise RuntimeError(f"init_image: image bytes or an HxWx3 uint8 array expected, got "
                                   f"{arr.dtype} {list(arr.shape)}")
        if arr.shape[:2] != (height, width):
            raise RuntimeError(f"init_image is {arr.shape[1]}x{arr.shape[0]}, the request's size is "
                               f"{width}x{height} (init images are not resized)")
        return np.ascontiguousarray(arr)

    # ------------------------------------------------------------------ jobs
    def _parse(self, req):
        width, height = parse_size(req.size)
        if width % 8 or height % 8 or width <= 0 or height <= 0:
            raise RuntimeError(f"Invalid size '{req.size}', expected 'WIDTHxHEIGHT'")
        # every UNet level halves the latent (stride-2 conv, padding 1): this engine implements the exact-halving
        # case only; diffusers' ceil-mode downsample + `upsample_size` path for other sizes is not built
        m = 8 << (len(self.pipe.unet.cfg.block_out_channels) - 1)
        if width % m or height % m:
            raise RuntimeError(f"Invalid size '{req.size}': the b200 worker needs WIDTH and HEIGHT to be multiples "
                               f"of {m} for this model (e.g. {max(m, width // m * m)}x{max(m, height // m * m)})")
        seed = int(req.seed) if getattr(req, "seed", None) is not None else \
            int(torch.randint(0, 100_000_000, (1,)).item())
        return width, height, seed

    def _draw(self, seed: int, h8: int, w8: int, steps: int, raw: bool = False, posterior: bool = False,
              masked: bool = False):
        """The reference's per-request Philox stream (`backends/cuda_worker.py:212-213`,
        SURVEY.md App. A.5): latents first, then one draw per non-final step.
        posterior (image-to-image): the posterior sample's draw comes first and is returned third; the
        "latents" draw is then the add_noise noise (diffusers' prepare_latents order).
        masked (inpainting): the masked image's posterior draw follows the latents draw (prepare_mask_latents runs
        after prepare_latents) and is returned fourth; steps is then the truncated schedule's length."""
        gen = torch.Generator(device=self.device)
        gen.manual_seed(seed)
        shape = (1, 4, h8, w8)
        eps_s = torch.randn(shape, generator=gen, device=self.device, dtype=torch.float32) if posterior else None
        lat = torch.randn(shape, generator=gen, device=self.device, dtype=torch.float32)
        eps_m = torch.randn(shape, generator=gen, device=self.device, dtype=torch.float32) if masked else None
        noise = [torch.randn(shape, generator=gen, device=self.device, dtype=torch.float32)
                 for _ in range(steps - 1)]
        if not raw:
            lat = lat.to(self.dtype).float()
            noise = [z.to(self.dtype).float() for z in noise]
            eps_s = eps_s.to(self.dtype).float() if posterior else None
            eps_m = eps_m.to(self.dtype).float() if masked else None
        if masked:
            return lat, noise, eps_s, eps_m
        return (lat, noise, eps_s) if posterior else (lat, noise)

    supports_deferred = True      # run_batch(..., deferred=True) -> thunks (see WorkerPool)

    @torch.no_grad()
    def run_batch(self, jobs: Sequence, with_latents: bool = False, deferred: bool = False,
                  raw: bool = False, latents_only: bool = False) -> List:
        """All jobs must share size / steps / style; guidance may differ per job.
        deferred=True returns one zero-argument callable per job that PNG-encodes its image when
        called: the pool runs them on encoder threads while this worker's thread already drives
        the next batch on the GPU (PIL's ~20 ms per 512^2 image would otherwise cap a worker at
        ~50 img/s, SURVEY.md §8f rank 1)."""
        timing = _BATCH_TIMING is not None
        with torch.cuda.device(self.device):
            if timing:
                t_in = time.perf_counter()
                ev0 = torch.cuda.Event(enable_timing=True)
                ev0.record()
            parsed = [self._parse(j.req) for j in jobs]
            width, height = parsed[0][0], parsed[0][1]
            steps = int(jobs[0].req.num_inference_steps)
            for (w, h, _), j in zip(parsed, jobs):
                if (w, h) != (width, height) or int(j.req.num_inference_steps) != steps:
                    raise RuntimeError("run_batch: jobs must share size and num_inference_steps")
            inits = [getattr(j.req, "init_image", None) for j in jobs]
            masks = [getattr(j.req, "mask_image", None) for j in jobs]
            inpaint = any(m is not None for m in masks)
            init = None
            k, posterior = steps, False           # steps that run; whether the image's posterior draw is consumed
            if inpaint or any(x is not None for x in inits):
                if len({(x is not None, m is not None) for x, m in zip(inits, masks)}) != 1:
                    raise RuntimeError("run_batch: inpainting, image-to-image and text-to-image jobs cannot share a "
                                       "batch")
                if inits[0] is None:
                    raise RuntimeError("mask_image without init_image: inpainting repaints part of a given picture")
                default = 1.0 if inpaint else 0.8
                strengths = {default if getattr(j.req, "strength", None) is None else float(j.req.strength)
                             for j in jobs}
                if len(strengths) != 1:
                    raise RuntimeError("run_batch: image-to-image and inpainting jobs must share strength")
                strength = next(iter(strengths))
                if inpaint:
                    self._check_inpaint()
                else:
                    self._check_img2img()
                # host work on this thread: PNG / JPEG decoding of the init images (and masks)
                import numpy as np
                imgs = torch.from_numpy(np.stack([self._init_image(x, width, height) for x in inits]))
                init = [imgs, None, strength]
                posterior = True
                if inpaint:
                    init += [torch.from_numpy(np.stack([self._mask_image(m, width, height) for m in masks])), None]
                    k, posterior = self._inpaint_plan(steps, strength)
            # per-request Philox streams; the round trip through the noise dtype (CUDA_DTYPE) is applied once to
            # the assembled batch instead of per tensor (same values, ~8 fewer launches per request)
            draws = [self._draw(seed, height // 8, width // 8, k, raw=True, posterior=posterior, masked=inpaint)
                     for _, _, seed in parsed]
            if posterior:
                init[1] = torch.cat([d[2] for d in draws], 0).to(self.dtype).float()
            if inpaint:
                init[4] = torch.cat([d[3] for d in draws], 0).to(self.dtype).float()
            lat = torch.cat([d[0] for d in draws], 0).to(self.dtype).float()
            noise = (torch.stack([torch.cat([d[1][i] for d in draws], 0) for i in range(k - 1)]).to(self.dtype).float()
                     if k > 1 else None)
            gs = torch.tensor([float(j.req.guidance_scale) for j in jobs])
            styles = {self._style_of(j.req) for j in jobs}
            if len(styles) != 1:
                raise RuntimeError("run_batch: jobs must share style and level")
            self._apply_style(*next(iter(styles)))
            try:
                img, final = self._generate([str(j.req.prompt) for j in jobs], lat, noise, steps, gs,
                                            height, width, decode=not latents_only,
                                            **({"init": tuple(init)} if init is not None else {}))
            finally:
                self._apply_style(None, 0)          # reset: no state bleed into the next job
            from dreamlab_b200 import lib
            if latents_only:
                # denoised latents, fp32 NCHW like the reference's `output_type="latent"` pass
                # (`backends/cuda_worker.py:273-283`): no VAE decode, no PNG
                lat_out = final.permute(0, 3, 1, 2).contiguous().cpu().numpy()
                return [(lat_out[i], parsed[i][2]) for i in range(len(jobs))]
            pooled = None
            if with_latents:
                pooled = torch.empty(len(jobs), 4, 8, 8, device=self.device, dtype=torch.float16)
                lib.latent_pool8(final, pooled)
                pooled = pooled.cpu().numpy()
            png_size = 0
            gpu_png = not raw and _png_mode() == "gpu"
            if gpu_png:
                # the finished PNG files come off the device (csrc/png.cu): no zlib on the host
                png_dev, png_size = lib.png_stored(img.contiguous())
                host, done = _to_host_async(png_dev)
            else:
                host, done = _to_host_async(img)
            if timing:
                # debug aid (B200_BATCH_TIMING=1): host time to enqueue the batch, device time from its first to its
                # last command, and when both happened — enough to tell an idle GPU from a slow one
                ev1 = torch.cuda.Event(enable_timing=True)
                ev1.record()
                _BATCH_TIMING.append((self.worker_id, len(jobs), t_in, time.perf_counter(), ev0, ev1))
            self._admit(done)

        def finish(i):
            done.synchronize()                      # this batch's GPU work and its copy to `host` have finished
            seed = parsed[i][2]
            arr = host.numpy()
            if raw:
                return (arr[i], seed, pooled[i:i + 1].tobytes(order="C")) if with_latents else (arr[i], seed)
            png = arr[i, :png_size].tobytes() if gpu_png else _encode_png(arr[i])
            return (png, seed, pooled[i:i + 1].tobytes(order="C")) if with_latents else (png, seed)

        if deferred:
            return [_Deferred(finish, i, done) for i in range(len(jobs))]
        if len(jobs) == 1:
            return [finish(0)]
        return list(_encoders().map(finish, range(len(jobs))))      # PIL releases the GIL in zlib

    def _admit(self, done) -> None:
        """Bound how far this thread runs ahead of the GPU: with `deferred=True` run_batch returns as soon as a
        batch is enqueued, and the host work of batch k+1 (request parsing, token ids, draws, launches) overlaps
        batch k on the device.  At most B200_BATCHES_IN_FLIGHT (default 2) batches are outstanding — their pinned
        result buffers are what would pile up otherwise."""
        q = self.__dict__.setdefault("_in_flight", collections.deque())
        q.append(done)
        limit = max(1, int(os.environ.get("B200_BATCHES_IN_FLIGHT", "2")))
        while len(q) > limit:
            q.popleft().synchronize()

    def drain(self) -> None:
        """Wait for every batch this worker has enqueued (the pool calls it before it drops a worker)."""
        q = self.__dict__.get("_in_flight")
        while q:
            q.popleft().synchronize()

    def run_job(self, job) -> Tuple[bytes, int]:
        return self.run_batch([job])[0]

    def run_job_with_latents(self, job) -> Tuple[bytes, int, bytes]:
        return self.run_batch([job], with_latents=True)[0]

    def run_job_latents(self, job):
        """Extension for callers that score candidates in latent space (SURVEY.md §8f rank 4, the Yume dream
        loop `yume/dream_worker.py:203-306` renders a 64x64 1-step candidate only to hash / score it): the
        denoise loop alone -> (fp32 latents [4, H/8, W/8], seed); the VAE decode and the PNG are skipped.
        `run_batch(jobs, latents_only=True)` does the same for many candidates in one pass."""
        return self.run_batch([job], latents_only=True)[0]

    def run_job_array(self, job):
        """Extension for callers that score pixels instead of shipping a file (the Yume dream
        loop renders 64x64 1-step candidates through `run_job` and immediately decodes the PNG
        again, `yume/dream_worker.py:294-299`): -> (uint8 HxWx3 array, seed), no PNG round trip."""
        return self.run_batch([job], raw=True)[0]


class B200SDXLWorker(B200Worker):
    """Drop-in for `DiffusersSDXLCudaWorker` (reference `backends/cuda_worker.py:307-614`): same
    constructor / env / attributes / results / errors; SDXL-class UNet (text_time conditioning,
    two text encoders -> [B,77,2048] + pooled [B,1280]), LCMScheduler, classifier-free guidance
    when guidance_scale > 1 (all jobs of one batch must then share the scale), SDXL VAE."""
    _tag = "b200-sdxl"
    _env_what = "SDXL CUDA worker"

    def _check_img2img(self) -> None:
        raise RuntimeError("image-to-image is not implemented for SDXL: StableDiffusionXLImg2ImgPipeline truncates "
                           "the full schedule (get_timesteps), which is different semantics from the LCM img2img "
                           "pipeline built here")

    def _check_inpaint(self) -> None:
        raise RuntimeError("inpainting is not implemented for SDXL: StableDiffusionXLInpaintPipeline is not built, "
                           "only the SD1.5-class inpainting pipeline")

    def _make_text_encoder(self, path):
        ucfg = self.pipe.unet.cfg
        if not self.pipe.is_sdxl:
            raise RuntimeError("B200SDXLWorker needs an SDXL-class UNet (addition_embed_type=text_time)")
        pooled = ucfg.projection_class_embeddings_input_dim - 6 * ucfg.addition_time_embed_dim
        return _SDXLTextEncoder(path, self.device, ucfg.cross_attention_dim, pooled, single=self._single)

    def _generate(self, prompts, lat, noise, steps, gs, height, width, decode=True):
        pe, pooled = self._text.encode(prompts)
        neg = negp = None
        # `force_zeros_for_empty_prompt` (model_index.json; True for SDXL-base): zeros for the unconditional
        # half, which is the engine's default; otherwise the empty prompt is encoded like any other
        if self.pipe.cfg_scale_for(gs) is not None and not self._model_index.get("force_zeros_for_empty_prompt", True):
            neg, negp = self._text.encode([""] * len(prompts))
        return self.pipe.generate(pe, lat, noise, steps, gs, return_latents=True, pooled_embeds=pooled,
                                  use_graph=self._use_graph, negative_prompt_embeds=neg,
                                  negative_pooled_embeds=negp, decode=decode)


_ENCODERS = None


def _encoders():
    """Process-wide PNG encoder threads (shared by all workers and the pool)."""
    global _ENCODERS
    if _ENCODERS is None:
        from concurrent.futures import ThreadPoolExecutor
        n = int(os.environ.get("B200_PNG_THREADS", "0")) or min(16, os.cpu_count() or 4)
        _ENCODERS = ThreadPoolExecutor(max_workers=n, thread_name_prefix="png")
    return _ENCODERS


# B200_BATCH_TIMING=1: run_batch appends (worker, batch size, t_enter, t_enqueued, first event, last event)
_BATCH_TIMING = [] if os.environ.get("B200_BATCH_TIMING", "0") not in ("0", "", "false") else None


def batch_timing_summary():
    """-> per-worker medians of the B200_BATCH_TIMING records (call after the work has finished)."""
    import statistics
    out = {}
    for wid in sorted({r[0] for r in _BATCH_TIMING or []}):
        rows = [r for r in _BATCH_TIMING if r[0] == wid]
        gpu = [r[4].elapsed_time(r[5]) for r in rows]
        host = [(r[3] - r[2]) * 1e3 for r in rows]
        period = [(b[2] - a[2]) * 1e3 for a, b in zip(rows, rows[1:])]
        out[wid] = {"batches": len(rows), "device_ms_median": statistics.median(gpu),
                    "device_ms_max": max(gpu), "host_enqueue_ms_median": statistics.median(host),
                    "host_enqueue_ms_max": max(host),
                    "period_ms_median": statistics.median(period) if period else None}
    return out


class _Deferred:
    """One request's result, still on its way: `()` -> the result tuple (blocks until the batch's GPU work is done,
    then encodes / slices this request's bytes); `wait()` only blocks — the pool parks ONE waiter per batch on it and
    fans the per-request calls out to the encoder threads afterwards, instead of blocking a thread per request."""
    __slots__ = ("_finish", "_i", "_done")

    def __init__(self, finish, i, done):
        self._finish, self._i, self._done = finish, i, done

    def wait(self):
        self._done.synchronize()

    def __call__(self):
        return self._finish(self._i)


def _to_host_async(t: torch.Tensor):
    """Device tensor -> (pinned host tensor, CUDA event): the copy is only ENQUEUED behind the work that produces
    `t`; whoever reads the host tensor waits on the event first (the PNG thunks do, on the encoder threads), so the
    worker's thread is free to enqueue the next batch while this one is still on the GPU.  Pinned staging: torch's
    caching host allocator recycles the blocks, and a pageable `.cpu()` of a 12.6 MB batch runs at a fraction of the
    link rate.  The thunks keep the pinned tensor alive until the last one that reads it is done."""
    host = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    host.copy_(t, non_blocking=True)
    ev = torch.cuda.Event()
    ev.record(torch.cuda.current_stream(t.device))
    return host, ev


def _png_mode() -> str:
    """B200_PNG: "pil" (default) = the reference's exact call `img.save(buf, format="PNG")`
    (`backends/cuda_worker.py:234-239`) on encoder threads; "gpu" = PNG files assembled on the device by
    `dl_png_stored` (stored deflate blocks, CRC-32 / Adler-32 in CUDA): same pixels in any PNG reader,
    deterministic bytes, ~1 ms instead of 70-100 ms of host zlib per 512x512 image — the host encoder caps an
    8-GPU box at a few hundred images/s."""
    v = os.environ.get("B200_PNG", "pil").strip().lower()
    if v not in ("pil", "gpu"):
        raise RuntimeError(f"B200_PNG must be 'pil' or 'gpu', got {v!r}")
    return v


def _png_level():
    """B200_PNG_COMPRESS_LEVEL (0-9): zlib level of the PNG encoder.  Unset = PIL's default (6), i.e.
    exactly the reference's `img.save(buf, format="PNG")` (`backends/cuda_worker.py:234-239`).  The pixels
    are the same at every level; level 1 encodes a 512x512 image in ~45 ms instead of 70-100 ms per core,
    which matters once one GPU produces > 130 images/s."""
    v = os.environ.get("B200_PNG_COMPRESS_LEVEL", "").strip()
    if not v:
        return None
    lvl = int(v)
    if not 0 <= lvl <= 9:
        raise RuntimeError(f"B200_PNG_COMPRESS_LEVEL must be 0..9, got {v!r}")
    return lvl


def _encode_png(arr) -> bytes:
    from PIL import Image
    buf = io.BytesIO()
    lvl = _png_level()
    if lvl is None:
        Image.fromarray(arr).save(buf, format="PNG")
    else:
        Image.fromarray(arr).save(buf, format="PNG", compress_level=lvl)
    return buf.getvalue()


def _load_clip(te_dir: str, device: str):
    """`text_encoder/` of a diffusers model dir -> on-device CLIP tower (dreamlab_b200.clip)."""
    from safetensors.torch import load_file
    from dreamlab_b200.clip import CLIPTextB200, clip_cfg_from_json
    with open(os.path.join(te_dir, "config.json")) as f:
        cfg = clip_cfg_from_json(json.load(f))
    for name in ("model.safetensors", "model.fp16.safetensors"):
        p = os.path.join(te_dir, name)
        if os.path.exists(p):
            return CLIPTextB200(load_file(p), cfg, device)
    raise RuntimeError(f"no safetensors weights under {te_dir}")


def _clip_from(component, device: str):
    """(config dict, transformers-named state dict) of a converted single-file text tower -> CLIPTextB200."""
    from dreamlab_b200.clip import CLIPTextB200, clip_cfg_from_json
    cfg, sd = component
    return CLIPTextB200(sd, clip_cfg_from_json(cfg), device)


def _side_tokenizer(checkpoint_path: str, name: str):
    """A single-file checkpoint carries no tokenizer files (diffusers fetches them from the hub): look for
    `<name>/vocab.json` next to the file, or under B200_TOKENIZER_ROOT.  None -> hashed stand-in tokens."""
    for root in (os.path.dirname(checkpoint_path), os.environ.get("B200_TOKENIZER_ROOT", "")):
        tk = os.path.join(root, name) if root else ""
        if tk and os.path.exists(os.path.join(tk, "vocab.json")):
            from transformers import CLIPTokenizer
            return CLIPTokenizer.from_pretrained(tk)
    print(f"[b200] no {name}/vocab.json next to {checkpoint_path} (or under B200_TOKENIZER_ROOT): prompts are "
          f"tokenised by a hashing stand-in")
    return None


def _hash_tokens(prompts: List[str], eos: int = 49407, bos: int = 49406) -> torch.Tensor:
    """Deterministic stand-in token ids when the model dir ships no tokenizer files (offline
    fixtures): good for synthetic load, meaningless for real prompts."""
    import numpy as np
    ids = np.full((len(prompts), 77), eos, dtype=np.int64)
    ids[:, 0] = bos
    j = np.arange(75, dtype=np.int64)
    for i, p in enumerate(prompts):
        b = np.frombuffer(p.encode("utf-8")[:75], dtype=np.uint8).astype(np.int64)
        ids[i, 1:1 + b.size] = (b * 193 + j[:b.size] * 7919) % bos
    return torch.from_numpy(ids)


def _seeded_embeds(prompts: List[str], dims, device):
    out = [[] for _ in dims]
    for p in prompts:
        g = torch.Generator().manual_seed(int.from_bytes(p.encode("utf-8")[:7] or b"\0", "little"))
        for o, shape in zip(out, dims):
            o.append(torch.randn(1, *shape, generator=g))
    return [torch.cat(o, 0).to(device) for o in out]


class _TextEncoder:
    """Prompt -> [B,77,D] embeddings: the step *before* the hot path (SURVEY.md §8f rank 2), on
    the device through `dreamlab_b200.clip.CLIPTextB200` when the model dir ships `text_encoder/`
    (tokenisation is the stock `transformers` CLIPTokenizer, pure host code).  Without a text
    tower (offline fixtures): seeded N(0,1) embeddings keyed by the prompt."""

    def __init__(self, model_dir: str, device: str, dim: int, single=None):
        self.device, self.dim = device, dim
        self.model = None
        self.tokenizer = None
        if single is not None:
            if single.get("text_encoder"):
                self.model = _clip_from(single["text_encoder"], device)
            self.tokenizer = _side_tokenizer(model_dir, "tokenizer")
            return
        te = os.path.join(model_dir, "text_encoder")
        if os.path.exists(os.path.join(te, "config.json")):
            self.model = _load_clip(te, device)
            tk = os.path.join(model_dir, "tokenizer")
            if os.path.exists(os.path.join(tk, "vocab.json")):
                from transformers import CLIPTokenizer
                self.tokenizer = CLIPTokenizer.from_pretrained(tk)

    @torch.no_grad()
    def encode(self, prompts: List[str]) -> torch.Tensor:
        if self.model is None:
            return _seeded_embeds(prompts, [(77, self.dim)], self.device)[0]
        if self.tokenizer is not None:
            ids = self.tokenizer(prompts, padding="max_length", max_length=77, truncation=True,
                                 return_tensors="pt").input_ids
        else:
            ids = _hash_tokens(prompts)
        return self.model.forward_graphed(ids)["last_hidden_state"].float()


class _SDXLTextEncoder:
    """Prompt -> ([B,77,D] embeddings, [B,P] pooled) for SDXL: penultimate hidden states of
    `text_encoder` (CLIP-L, 768) and `text_encoder_2` (OpenCLIP-bigG, 1280) concatenated, pooled =
    `text_encoder_2`'s projected embedding (SURVEY.md App. A.2); both towers run on the device
    (`dreamlab_b200.clip`).  Without them in the model dir (offline fixtures): seeded N(0,1)
    embeddings keyed by the prompt."""

    def __init__(self, model_dir: str, device: str, dim: int, pooled_dim: int, single=None):
        self.device, self.dim, self.pooled_dim = device, dim, pooled_dim
        self.models = None
        self.tokenizers = (None, None)
        if single is not None:
            if single.get("text_encoder") and single.get("text_encoder_2"):
                self.models = (_clip_from(single["text_encoder"], device), _clip_from(single["text_encoder_2"], device))
            self.tokenizers = (_side_tokenizer(model_dir, "tokenizer"), _side_tokenizer(model_dir, "tokenizer_2"))
            return
        te1, te2 = os.path.join(model_dir, "text_encoder"), os.path.join(model_dir, "text_encoder_2")
        if os.path.exists(os.path.join(te1, "config.json")) and os.path.exists(os.path.join(te2, "config.json")):
            self.models = (_load_clip(te1, device), _load_clip(te2, device))
            toks = []
            for t in ("tokenizer", "tokenizer_2"):
                tk = os.path.join(model_dir, t)
                if os.path.exists(os.path.join(tk, "vocab.json")):
                    from transformers import CLIPTokenizer
                    toks.append(CLIPTokenizer.from_pretrained(tk))
                else:
                    toks.append(None)
            self.tokenizers = tuple(toks)

    @torch.no_grad()
    def encode(self, prompts: List[str]):
        if self.models is None:
            return tuple(_seeded_embeds(prompts, [(77, self.dim), (self.pooled_dim,)], self.device))
        hs, pooled = [], None
        for tok, m in zip(self.tokenizers, self.models):
            if tok is not None:
                ids = tok(prompts, padding="max_length", max_length=77, truncation=True,
                          return_tensors="pt").input_ids
            else:
                ids = _hash_tokens(prompts, eos=m.cfg.vocab_size - 1, bos=m.cfg.vocab_size - 2)
            out = m.forward_graphed(ids, want_hidden=-2)
            hs.append(out["hidden"].float())
            pooled = out.get("text_embeds", out["pooler_output"]).float()   # the last tower's pooled embedding
        return torch.cat(hs, -1), pooled
