"""The oracle's (and the product's) host pieces pinned to the REFERENCE ITSELF.

`tests/golden/make_reference_host_golden.py` cuts four plain-NumPy functions out of the reference
tree with `ast` and executes their source unmodified (guidance-scale embedding, postprocess,
prepare_latents: `backends/rknnlcm.py:651-677, 212-264, 423-447`; 8x8 latent pooling:
`backends/rknn_worker.py:223-248`).  Their outputs on seeded inputs are the committed fixture
`tests/golden/reference_host_pieces.npz`.  Here:
  * CPU: `oracle/` + the product's host scheduler code are compared against the fixture;
  * GPU (-m gpu): the CUDA kernels that implement the same pieces (u8 image tail — fused conv
    epilogue and the crop kernel —, 8x8 pooling) are compared against it through the C-ABI.
Bars: bit-exact for u8 / integer work and the latent draw; fp32 results within the rounding of the
reference's float64 evaluation (the tolerance is derived next to each assert).
"""
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import make_reference_host_golden as mk  # noqa: E402

FIX = np.load(mk.FIXTURE)


def _emb_tol(w, dim):
    # the reference evaluates sin / cos of a = (1000 w) f_i in float64 (NumPy 2 promotes its np.float64
    # `np.log(10000.0) / (half - 1)`); the fp32 evaluation rounds w*1000 (2^-24), the exponent i*e <= 9.2 of
    # f_i = exp(-i*e) (absolute 9.2 * 2^-24 -> relative on f_i), exp itself (2 ulp) and the product (2^-24):
    # |delta a| <= 16 * 2^-24 * |a|, and |d sin|, |d cos| <= |delta a|; plus 1 ulp of the result
    half = dim // 2
    f = np.exp(np.arange(half) * -(np.log(10000.0) / (half - 1)))
    a = np.abs(w.astype(np.float64))[:, None] * 1000.0 * f[None, :]
    t = 16.0 * 2.0 ** -24 * np.maximum(a, 1.0) + 2.0 ** -23
    t = np.concatenate([t, t], axis=1)
    return np.pad(t, [(0, 0), (0, dim - 2 * half)], constant_values=1e-30)


@pytest.mark.parametrize("which", ["oracle", "product"])
@pytest.mark.parametrize("dim", [256, 255])
def test_guidance_scale_embedding_matches_reference(which, dim):
    if which == "oracle":
        from oracle.scheduler import guidance_scale_embedding
    else:
        from dreamlab_b200.scheduler import guidance_scale_embedding
    w = torch.from_numpy(FIX["w"])
    ours = guidance_scale_embedding(w, dim).numpy().astype(np.float64)
    ref = FIX[f"w_emb_{dim}"]
    assert ours.shape == ref.shape
    err = np.abs(ours - ref)
    assert (err <= _emb_tol(FIX["w"], dim)).all(), float((err / _emb_tol(FIX["w"], dim)).max())
    # guidance_scale = 1 (w = 0): exactly 128 zeros then 128 ones (SURVEY.md App. A.6)
    i = list(mk.GUIDANCE).index(1.0)
    half = dim // 2
    assert np.array_equal(ours[i, :half], np.zeros(half)) and np.array_equal(ours[i, half:2 * half], np.ones(half))


def test_oracle_postprocess_bit_exact_vs_reference():
    from oracle.pipeline import denormalize_to_u8
    img = torch.from_numpy(FIX["image_in"])
    assert np.array_equal(denormalize_to_u8(img), FIX["post_u8"])
    # the float NHWC intermediate as well
    x = (img / 2 + 0.5).clamp(0, 1).permute(0, 2, 3, 1).numpy()
    assert np.array_equal(x, FIX["post_np"])


def test_oracle_latent_draw_bit_exact_vs_reference():
    """`synthetic_inputs` (the oracle's and the product's, same function body) draws the initial latents
    exactly as the reference's prepare_latents does from a torch.Generator: randn(1,4,h/8,w/8) * 1.0."""
    from oracle.pipeline import synthetic_inputs as oracle_inputs
    from dreamlab_b200.synthetic import synthetic_inputs as product_inputs
    for s in mk.LATENT_SEEDS:
        ref = FIX[f"latents_torch_{s}"]
        for fn in (oracle_inputs, product_inputs):
            _, lat, _ = fn(1, 512, 512, 4, seed_base=s)
            assert lat.shape == ref.shape
            assert np.array_equal(lat.numpy().astype(np.float64), ref)
        # the RandomState branch differs from the torch branch (different generator), same contract
        assert FIX[f"latents_np_{s}"].shape == ref.shape


def test_oracle_latent_pooling_vs_reference():
    from oracle.pipeline import pooled_latent_bytes
    for k in ("64", "96"):
        lat = torch.from_numpy(FIX[f"lat{k}"])
        ours = np.frombuffer(pooled_latent_bytes(lat), dtype=np.float16).reshape(1, 4, 8, 8)
        ref = FIX[f"pool8_{k}"].astype(np.float16)
        # both are fp32 block means cast to fp16; the summation order differs, so allow the last fp16 bit
        assert len(ours.tobytes()) == 512
        d = np.abs(ours.astype(np.float32) - ref.astype(np.float32))
        assert (d <= np.spacing(np.abs(ref)).astype(np.float32)).all()
        assert (ours == ref).mean() > 0.98


# ------------------------------------------------------------------------------------------------
# CUDA kernels against the reference's outputs
# ------------------------------------------------------------------------------------------------
def _lib():
    import dreamlab_b200.lib as lib
    lib.load()
    return lib


@pytest.mark.gpu
def test_cuda_image_crop_u8_bit_exact_vs_reference():
    """`dl_image_crop_u8` (tiled-decode tail).  The kernel rounds the decoder output to bf16 first (the
    decoder's activation dtype), so it is fed bf16-representable values and must then equal the reference's
    `postprocess` of those very values byte for byte."""
    lib = _lib()
    img = torch.from_numpy(FIX["image_in"]).to(torch.bfloat16).float()
    from oracle.pipeline import denormalize_to_u8         # pinned to the reference bit-exactly above
    ref = denormalize_to_u8(img)
    src = img.permute(0, 2, 3, 1).contiguous().cuda()
    n, h, w, c = src.shape
    out = torch.zeros(n, h, w, c, device="cuda", dtype=torch.uint8)
    lib.image_crop_u8(src, h, w, out)
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy(), ref)


@pytest.mark.gpu
def test_cuda_conv_u8_image_epilogue_bit_exact_vs_reference():
    """The fused VaeImageProcessor tail of the last conv (`DL_EPI_U8_IMAGE`): a 3x3 conv whose centre tap
    copies channels 0..2 reproduces its (bf16) input exactly in the fp32 accumulator, so the u8 it
    stores must equal the reference's postprocess of that input."""
    lib = _lib()
    img = torch.from_numpy(FIX["image_in"]).to(torch.bfloat16)                 # [2,3,48,40]
    from oracle.pipeline import denormalize_to_u8
    ref = denormalize_to_u8(img.float())
    n, _, h, w = img.shape
    x = torch.zeros(n, h, w, 64, device="cuda", dtype=torch.bfloat16)
    x[..., :3] = img.permute(0, 2, 3, 1).cuda()
    wgt = torch.zeros(3, 9, 64, device="cuda", dtype=torch.bfloat16)
    for j in range(3):
        wgt[j, 4, j] = 1.0
    out = torch.zeros(n, h, w, 3, device="cuda", dtype=torch.uint8)
    lib.igemm(x, wgt.view(3, 9 * 64), out, nimg=n, h=h, w=w, taps=9, n=3, mode=lib.EPI_U8_IMAGE, ldo=3)
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy(), ref)


@pytest.mark.gpu
def test_cuda_latent_pool8_vs_reference():
    lib = _lib()
    for k in ("64", "96"):
        lat = torch.from_numpy(FIX[f"lat{k}"])
        nhwc = lat.permute(0, 2, 3, 1).contiguous().cuda()
        out = torch.empty(1, 4, 8, 8, device="cuda", dtype=torch.float16)
        lib.latent_pool8(nhwc, out)
        torch.cuda.synchronize()
        ours = out.cpu().numpy()
        ref = FIX[f"pool8_{k}"].astype(np.float16)
        d = np.abs(ours.astype(np.float32) - ref.astype(np.float32))
        assert (d <= np.spacing(np.abs(ref)).astype(np.float32)).all()
        assert (ours == ref).mean() > 0.98
        assert len(ours.tobytes()) == 512


@pytest.mark.gpu
def test_cuda_latent_pool8_adaptive_bins_for_sizes_not_divisible_by_8():
    """`adaptive_avg_pool2d(lat, (8, 8))` of the reference's CUDA worker (`backends/cuda_worker.py:299`)
    for latent extents that are not multiples of 8 (e.g. 600x600 -> 75x75 latents)."""
    lib = _lib()
    g = torch.Generator().manual_seed(5)
    for (h, w) in [(75, 75), (90, 160), (12, 20)]:
        lat = torch.randn(2, 4, h, w, generator=g)
        out = torch.empty(2, 4, 8, 8, device="cuda", dtype=torch.float16)
        lib.latent_pool8(lat.permute(0, 2, 3, 1).contiguous().cuda(), out)
        torch.cuda.synchronize()
        ref = torch.nn.functional.adaptive_avg_pool2d(lat, (8, 8))
        assert (out.cpu().float() - ref).abs().max().item() < 2e-3
