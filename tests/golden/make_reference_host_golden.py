"""Pins the oracle's host pieces to the REFERENCE ITSELF.

The reference's hot path delegates its arithmetic to `diffusers` (absent offline), but four host
pieces of the path are stated in the reference tree in plain NumPy and need nothing but numpy /
torch / PIL to run:

  * `RKNN2LatentConsistencyPipeline.get_guidance_scale_embedding`  backends/rknnlcm.py:651-677
  * `RKNN2LatentConsistencyPipeline.postprocess`                   backends/rknnlcm.py:212-264
  * `RKNN2LatentConsistencyPipeline.prepare_latents`               backends/rknnlcm.py:423-447
  * `_downsample_to_8x8_nchw` (the 8x8 latent pooling contract)    backends/rknn_worker.py:223-248

The module itself cannot be imported (it imports `diffusers` and `rknnlite` at load), so the
function sources are cut out of the file with `ast` and executed UNMODIFIED in a namespace that
holds numpy / torch / PIL.  `python tests/golden/make_reference_host_golden.py <reference checkout>`
writes the committed fixture `reference_host_pieces.npz` that tests/test_reference_pin.py compares
against.  Nothing of the reference's source is copied into the repo.
"""
from __future__ import annotations

import ast
import logging
import os
import sys
import textwrap
from types import SimpleNamespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
FIXTURE = os.path.join(HERE, "reference_host_pieces.npz")


def _cut(path: str, names) -> dict:
    """{name: source text of the function `name`} for (possibly nested-in-class) defs in `path`."""
    src = open(path).read()
    tree = ast.parse(src)
    lines = src.splitlines()
    out = {}
    for node in ast.walk(tree):
        if isinstance(node, ast.FunctionDef) and node.name in names and node.name not in out:
            start = min([node.lineno] + [d.lineno for d in node.decorator_list]) - 1
            out[node.name] = textwrap.dedent("\n".join(lines[start:node.end_lineno]))
    missing = set(names) - set(out)
    if missing:
        raise RuntimeError(f"{path}: functions not found: {sorted(missing)}")
    return out


def extract(reference_root: str) -> SimpleNamespace:
    """The reference's own functions, executed from its own source text."""
    from typing import List, Optional, Union
    from PIL import Image
    ns = {"np": np, "torch": torch, "Image": Image, "Optional": Optional, "List": List, "Union": Union,
          "logger": logging.getLogger("reference.rknnlcm")}
    cut = _cut(os.path.join(reference_root, "backends", "rknnlcm.py"),
               ["get_guidance_scale_embedding", "postprocess", "prepare_latents"])
    cut.update(_cut(os.path.join(reference_root, "backends", "rknn_worker.py"), ["_downsample_to_8x8_nchw"]))
    for name, text in cut.items():
        exec(compile(text, f"<reference:{name}>", "exec"), ns)
    # the two methods that take `self` read only these attributes (rknnlcm.py:209, :445)
    self_ = SimpleNamespace(vae_scale_factor=8, scheduler=SimpleNamespace(init_noise_sigma=1.0))
    post = ns["postprocess"]
    post = post.__func__ if isinstance(post, staticmethod) else post
    return SimpleNamespace(
        guidance_scale_embedding=lambda w, dim, dtype=np.float32: ns["get_guidance_scale_embedding"](self_, w, dim, dtype),
        postprocess=lambda image: post(image, output_type="np", do_denormalize=[True] * image.shape[0]),
        postprocess_pil=lambda image: post(image, output_type="pil", do_denormalize=[True] * image.shape[0]),
        prepare_latents=lambda b, c, h, w, dtype, gen: ns["prepare_latents"](self_, b, c, h, w, dtype, gen),
        downsample_8x8=ns["_downsample_to_8x8_nchw"])


GUIDANCE = [1.0, 1.5, 2.0, 4.0, 7.5, 8.0, 12.0, 0.0]        # guidance_scale values; w = gs - 1 (rknnlcm.py:574)
LATENT_SEEDS = [0, 42, 12345678]


def inputs():
    g = np.random.RandomState(20261018)
    image = (g.randn(2, 3, 48, 40) * 0.9).astype(np.float32)            # decoder output range incl. clipping
    # exact ties of the *255 rounding and the clip edges
    image[0, 0, 0, :8] = np.array([-1.0, 1.0, -1.5, 1.5, 0.0, 2 * (0.5 / 255) - 1, 2 * (1.5 / 255) - 1,
                                   2 * (2.5 / 255) - 1], dtype=np.float32)
    lat = g.randn(1, 4, 64, 64).astype(np.float32)
    lat96 = g.randn(1, 4, 96, 96).astype(np.float32)
    return image, lat, lat96


def generate(reference_root: str) -> dict:
    ref = extract(reference_root)
    image, lat, lat96 = inputs()
    out = {"image_in": image, "lat64": lat, "lat96": lat96}
    w = np.asarray(GUIDANCE, dtype=np.float32) - 1.0
    out["w"] = w
    out["w_emb_256"] = ref.guidance_scale_embedding(w, 256)
    out["w_emb_255"] = ref.guidance_scale_embedding(w, 255)             # odd dim: zero pad branch
    out["post_np"] = ref.postprocess(image)                             # float NHWC in [0,1]
    out["post_u8"] = np.stack([np.asarray(im) for im in ref.postprocess_pil(image)])
    for s in LATENT_SEEDS:
        out[f"latents_torch_{s}"] = ref.prepare_latents(1, 4, 512, 512, np.float32, torch.Generator().manual_seed(s))
        out[f"latents_np_{s}"] = ref.prepare_latents(1, 4, 512, 512, np.float32, np.random.RandomState(s))
    out["pool8_64"] = ref.downsample_8x8(lat)
    out["pool8_96"] = ref.downsample_8x8(lat96)
    return out


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: python tests/golden/make_reference_host_golden.py <checkout of the reference repository>")
    np.savez_compressed(FIXTURE, **generate(sys.argv[1]))
    print("wrote", FIXTURE, os.path.getsize(FIXTURE), "bytes")
