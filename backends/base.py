"""Worker interface — the drop-in boundary (restates reference `backends/base.py:8-58`).

`PipelineWorker` is what `WorkerPool` drives (`job.execute(worker)` -> `worker.run_job(job)`,
reference `backends/worker_pool.py:84-88`).  A request object is duck-typed: workers read
`req.prompt`, `req.size` ("WIDTHxHEIGHT"), `req.num_inference_steps`, `req.guidance_scale`,
`req.seed` (optional) and `getattr(req, "style_lora", None)`.

Image-to-image (`LatentConsistencyModelImg2ImgPipeline` semantics) is requested with two more optional
fields, also read with `getattr`: `init_image` — image bytes PIL can open (PNG, JPEG, ...) or an HxWx3
uint8 array (what `run_job_array` returns), RGB and exactly `size` (no resizing) — and `strength` in
(0, 1] (default 0.8): how far the init image is noised before the LCM steps redraw it.

Inpainting (`StableDiffusionInpaintPipeline` semantics with `LCMScheduler`) adds `mask_image` to `init_image`, also
read with `getattr`: image bytes PIL can open (converted to "L") or an HxW uint8 array of L values, exactly `size`.
Pixels with L >= 128 are repainted, the others kept.  `strength` then defaults to 1.0 and truncates the full step
schedule (int(steps * strength) of its last steps run).  A model whose UNet has 9 input channels (an inpainting UNet)
serves only such requests.

Only names, fields and return conventions are shared with the reference — they ARE the
interface; everything a caller can observe is pinned by `tests/test_worker_pool.py` and
`tests/test_worker_factory.py`.
"""
from __future__ import annotations

import os
from concurrent.futures import Future
from dataclasses import dataclass, field
from typing import Any, Optional, Protocol, Tuple, runtime_checkable

LATENT_THUMB_SHAPE = (1, 4, 8, 8)            # run_job_with_latents: fp16 little-endian, 512 bytes
LATENT_THUMB_BYTES = 2 * 4 * 8 * 8


@runtime_checkable
class PipelineWorker(Protocol):
    """One worker = one device, driven serially by one pool thread."""

    worker_id: int

    def run_job(self, spec) -> Tuple[bytes, int]:
        """-> (PNG bytes, the seed that was used — drawn when the request carried none)."""

    def run_job_with_latents(self, spec) -> Tuple[bytes, int, bytes]:
        """-> (PNG bytes, seed, latent thumbnail): the final latent average-pooled to
        `LATENT_THUMB_SHAPE` (NCHW), serialised as little-endian float16 (`LATENT_THUMB_BYTES`)."""


@dataclass(frozen=True)
class StyleLora:
    """Style selection carried by a request: `style` names a registry entry, `level` indexes its
    strength presets (0 switches the style off)."""
    style: Optional[str] = None
    level: int = 0


@dataclass
class GenSpec:
    """Flat request record (the REST layer's GenerateRequest carries the same information as
    `num_inference_steps` / `guidance_scale`)."""
    prompt: str
    size: str
    steps: int
    cfg: float
    seed: Optional[int] = None
    style_lora: StyleLora = field(default_factory=StyleLora)
    init_image: Any = None                   # image-to-image: image bytes or HxWx3 uint8 array
    strength: Optional[float] = None         # image-to-image strength (None: 0.8; inpainting: 1.0)
    mask_image: Any = None                   # inpainting: image bytes or HxW uint8 array, with init_image


@dataclass
class Job:
    """What the legacy service queues: the request, the future its HTTP handler awaits, and the
    enqueue time (queue-latency metric)."""
    req: Any
    fut: Future
    submitted_at: float


@dataclass(frozen=True)
class ModelPaths:
    """Sub-paths of a component-per-directory model root (the layout the reference's RKNN worker loads from,
    reference `backends/base.py`).  Not used by the b200 path, which reads a diffusers directory; kept so that
    `from backends.base import ModelPaths` keeps working when this package replaces the reference's."""
    root: str

    @property
    def scheduler_config(self) -> str:
        return os.path.join(self.root, "scheduler", "scheduler_config.json")

    @property
    def text_encoder(self) -> str:
        return os.path.join(self.root, "text_encoder")

    @property
    def unet(self) -> str:
        return os.path.join(self.root, "unet")

    @property
    def vae_decoder(self) -> str:
        return os.path.join(self.root, "vae_decoder")
