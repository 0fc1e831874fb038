"""Per-kernel parity of the hand-written sm_100a kernels (through the C-ABI) against plain
PyTorch fp32 references of the same op on the same bf16-rounded inputs."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda"
# the torch references below (F.conv2d, matmul, SDPA in fp32) must be real fp32: no TF32 in cuDNN / cuBLAS
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False


def L():
    import dreamlab_b200.lib as lib
    lib.load()
    return lib


def bf(x):
    return x.to(torch.bfloat16)


def rel_err(a, b):
    a, b = a.float(), b.float()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-6)).item()


def rand(*shape, seed=0, scale=1.0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(DEV)


# ------------------------------------------------------------------ igemm: linear
@pytest.mark.parametrize("M,K,N,bn", [
    (256, 320, 320, 0), (128, 64, 32, 32), (154, 768, 640, 0), (4096, 320, 960, 160),
    (1000, 1280, 1280, 256), (300, 5120, 1280, 64), (512, 640, 1920, 0), (128, 128, 96, 96),
    (8192, 320, 2560, 0),
])
def test_igemm_linear(M, K, N, bn):
    lib = L()
    x = bf(rand(M, K, seed=1))
    w = bf(rand(N, K, seed=2, scale=K ** -0.5))
    bias = rand(N, seed=3)
    out = torch.empty(M, N, device=DEV, dtype=torch.bfloat16)
    lib.igemm(x, w, out, nimg=1, h=1, w=M, taps=1, n=N, bias=bias, bn=bn)
    ref = x.float() @ w.float().t() + bias
    torch.cuda.synchronize()
    e = rel_err(out, ref)
    assert e < 1e-2, f"rel err {e}"


def test_igemm_linear_epilogues():
    lib = L()
    M, K, N = 640, 320, 640
    x = bf(rand(M, K, seed=1))
    w = bf(rand(N, K, seed=2, scale=K ** -0.5))
    bias = rand(N, seed=3)
    res = bf(rand(M, N, seed=4))
    # rowadd: 5 "images" of 128 rows each
    rowadd = rand(5, N, seed=5)
    out = torch.empty(M, N, device=DEV, dtype=torch.bfloat16)
    lib.igemm(x.view(5, 1, 128, K), w, out, nimg=5, h=1, w=128, taps=1, n=N, bias=bias,
              rowadd=rowadd, residual=res)
    ref = (x.float() @ w.float().t()) + bias + rowadd.repeat_interleave(128, 0) + res.float()
    torch.cuda.synchronize()
    assert rel_err(out, ref) < 1e-2
    # residual into a 160-wide N tile (partial last 64-column identity chunk), odd M, alpha
    for bn in (160, 96, 256):
        o2 = torch.empty(M, N, device=DEV, dtype=torch.bfloat16)
        lib.igemm(x[:600], w, o2[:600], nimg=1, h=1, w=600, taps=1, n=N, residual=res[:600], bn=bn)
        torch.cuda.synchronize()
        assert rel_err(o2[:600], x[:600].float() @ w.float().t() + res[:600].float()) < 1e-2, bn
    o3 = torch.empty(M, N, device=DEV, dtype=torch.bfloat16)
    lib.igemm(x, w, o3, nimg=1, h=1, w=M, taps=1, n=N, bias=bias, alpha=0.5)
    torch.cuda.synchronize()
    assert rel_err(o3, 0.5 * (x.float() @ w.float().t()) + bias) < 1e-2
    # fp32 output, N = 4 (UNet conv_out shape class)
    w4 = bf(rand(4, K, seed=6, scale=K ** -0.5))
    o4 = torch.zeros(M, 4, device=DEV, dtype=torch.float32)
    lib.igemm(x, w4, o4, nimg=1, h=1, w=M, taps=1, n=4, bias=bias[:4].contiguous(), mode=lib.EPI_F32)
    ref4 = x.float() @ w4.float().t() + bias[:4]
    torch.cuda.synchronize()
    assert rel_err(o4, ref4) < 2e-3
    # GEGLU: interleaved (value, gate) rows
    inner = 1280
    wg = bf(rand(2 * inner, K, seed=7, scale=K ** -0.5))
    bg = rand(2 * inner, seed=8)
    wi = torch.stack([wg[:inner], wg[inner:]], 1).reshape(2 * inner, K).contiguous()
    bi = torch.stack([bg[:inner], bg[inner:]], 1).reshape(-1).contiguous()
    og = torch.empty(M, inner, device=DEV, dtype=torch.bfloat16)
    lib.igemm(x, wi, og, nimg=1, h=1, w=M, taps=1, n=2 * inner, bias=bi, mode=lib.EPI_GEGLU)
    proj = x.float() @ wg.float().t() + bg
    refg = proj[:, :inner] * F.gelu(proj[:, inner:])
    torch.cuda.synchronize()
    assert rel_err(og, refg) < 1e-2


# ------------------------------------------------------------------ igemm: conv3x3
@pytest.mark.parametrize("B,H,W,C0,C1,N", [
    (2, 16, 16, 64, 0, 64), (1, 64, 64, 320, 0, 320), (3, 8, 8, 1280, 1280, 1280),
    (2, 32, 32, 640, 320, 640), (1, 24, 24, 128, 0, 128), (1, 96, 96, 64, 0, 128),
    (1, 128, 128, 256, 0, 128), (2, 12, 12, 64, 0, 64),
    (2, 256, 256, 64, 0, 128), (1, 593, 128, 64, 0, 128), (1, 600, 128, 64, 64, 64),   # two M sub-tiles per CTA tile
])
def test_igemm_conv3x3(B, H, W, C0, C1, N):
    lib = L()
    C = C0 + C1
    x0 = bf(rand(B, H, W, C0, seed=1))
    x1 = bf(rand(B, H, W, C1, seed=2)) if C1 else None
    wt = bf(rand(N, C, 3, 3, seed=3, scale=(9 * C) ** -0.5))          # torch OIHW
    bias = rand(N, seed=4)
    w_pack = wt.permute(0, 2, 3, 1).reshape(N, 9 * C).contiguous()    # [N, tap, C]
    out = torch.empty(B, H, W, N, device=DEV, dtype=torch.bfloat16)
    lib.igemm(x0, w_pack, out, nimg=B, h=H, w=W, taps=9, n=N, a1=x1, bias=bias)
    xin = x0 if x1 is None else torch.cat([x0, x1], -1)
    ref = F.conv2d(xin.float().permute(0, 3, 1, 2), wt.float(), bias, padding=1).permute(0, 2, 3, 1)
    torch.cuda.synchronize()
    e = rel_err(out, ref)
    assert e < 1e-2, f"rel err {e}"


def test_igemm_conv3x3_residual_rowadd_partial_tiles():
    lib = L()
    B, H, W, C, N = 3, 24, 24, 128, 320          # 24x24: clipped tiles in x and y; N=320 -> BN 160
    x = bf(rand(B, H, W, C, seed=1))
    wt = bf(rand(N, C, 3, 3, seed=3, scale=(9 * C) ** -0.5))
    bias, rowadd = rand(N, seed=4), rand(B, N, seed=5)
    res = bf(rand(B, H, W, N, seed=6))
    w_pack = wt.permute(0, 2, 3, 1).reshape(N, 9 * C).contiguous()
    out = torch.full((B, H, W, N), 7.0, device=DEV, dtype=torch.bfloat16)
    lib.igemm(x, w_pack, out, nimg=B, h=H, w=W, taps=9, n=N, bias=bias, rowadd=rowadd, residual=res)
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), wt.float(), bias, padding=1).permute(0, 2, 3, 1)
    ref = ref + rowadd[:, None, None, :] + res.float()
    torch.cuda.synchronize()
    e = rel_err(out, ref)
    assert e < 1e-2, f"rel err {e}"


@pytest.mark.parametrize("B,H,W,C", [(2, 16, 16, 64), (1, 64, 64, 256), (3, 8, 8, 1280), (1, 24, 40, 128)])
def test_igemm_upsample_fold(B, H, W, C):
    """nearest-2x + conv3x3 as four 2x2-tap phase convs (weights pre-summed in fp32)."""
    lib = L()
    from dreamlab_b200.weights import pack_upsample_conv3x3
    x = bf(rand(B, H, W, C, seed=1))
    wt = rand(C, C, 3, 3, seed=2, scale=(9 * C) ** -0.5)
    bias = rand(C, seed=3)
    wp = pack_upsample_conv3x3(wt, DEV)
    out = torch.zeros(B, 2 * H, 2 * W, C, device=DEV, dtype=torch.bfloat16)
    strides = (2 * C, 4 * W * C, 4 * H * W * C)
    for ph in range(4):
        lib.igemm(x, wp[ph], out[:, ph >> 1:, ph & 1:, :], nimg=B, h=H, w=W, taps=4, n=C, bias=bias,
                  tap_phase=ph, ldo=C, out_strides=strides)
    up = F.interpolate(x.float().permute(0, 3, 1, 2), scale_factor=2.0, mode="nearest")
    ref = F.conv2d(up, wt.bfloat16().float(), bias, padding=1).permute(0, 2, 3, 1)
    torch.cuda.synchronize()
    e = rel_err(out, ref)
    assert e < 1.5e-2, f"rel err {e}"


def test_igemm_u8_image_tail():
    lib = L()
    B, H, W, C = 1, 64, 64, 128
    x = bf(rand(B, H, W, C, seed=1))
    wt = bf(rand(3, C, 3, 3, seed=2, scale=3 * (9 * C) ** -0.5))
    bias = rand(3, seed=3, scale=0.1)
    w_pack = wt.permute(0, 2, 3, 1).reshape(3, 9 * C).contiguous()
    out = torch.zeros(B, H, W, 3, device=DEV, dtype=torch.uint8)
    lib.igemm(x, w_pack, out, nimg=B, h=H, w=W, taps=9, n=3, bias=bias, mode=lib.EPI_U8_IMAGE, ldo=3)
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), wt.float(), bias, padding=1).permute(0, 2, 3, 1)
    ref = ((ref.bfloat16().float() / 2 + 0.5).clamp(0, 1) * 255).round()
    torch.cuda.synchronize()
    diff = (out.float() - ref).abs()
    assert diff.max().item() <= 2 and (diff > 0).float().mean().item() < 0.05


# ------------------------------------------------------------------ norms
@pytest.mark.parametrize("B,HW,C0,C1,silu", [
    (2, 4096, 320, 0, True), (2, 1024, 640, 320, True), (3, 64, 1280, 1280, True),
    (1, 65536, 128, 0, True), (2, 256, 1280, 640, False), (1, 4096, 512, 0, False),
    (2, 300, 256, 0, True), (16, 64, 1280, 1280, True), (4, 1024, 640, 320, True), (3, 1024, 320, 0, False),
    (2, 256, 1280, 640, True), (2, 16, 64, 0, True), (1, 4, 256, 128, True),
])
def test_groupnorm(B, HW, C0, C1, silu):
    lib = L()
    C = C0 + C1
    x0 = bf(rand(B, HW, C0, seed=1) * 2 + 0.5)
    x1 = bf(rand(B, HW, C1, seed=2) - 1.0) if C1 else None
    gamma, beta = rand(C, seed=3) * 0.2 + 1, rand(C, seed=4) * 0.2
    out = torch.empty(B, HW, C, device=DEV, dtype=torch.bfloat16)
    ws = torch.empty(lib.groupnorm_workspace_bytes(B), device=DEV, dtype=torch.uint8)
    lib.groupnorm(x0, out, gamma, beta, ws, nimg=B, hw=HW, eps=1e-5, silu=silu, x1=x1)
    xin = x0 if x1 is None else torch.cat([x0, x1], -1)
    ref = F.group_norm(xin.float().transpose(1, 2), 32, gamma, beta, 1e-5).transpose(1, 2)
    if silu:
        ref = F.silu(ref)
    torch.cuda.synchronize()
    assert (out.float() - ref).abs().max().item() < 3e-2


@pytest.mark.parametrize("rows,C", [(4096, 320), (1000, 640), (77, 1280), (5, 64)])
def test_layernorm(rows, C):
    lib = L()
    x = bf(rand(rows, C, seed=1) * 3 + 1)
    gamma, beta = rand(C, seed=2) * 0.2 + 1, rand(C, seed=3) * 0.2
    out = torch.empty_like(x)
    lib.layernorm(x, out, gamma, beta, 1e-5)
    ref = F.layer_norm(x.float(), (C,), gamma, beta, 1e-5)
    torch.cuda.synchronize()
    assert (out.float() - ref).abs().max().item() < 3e-2


# ------------------------------------------------------------------ attention
def _attn_case(lib, B, Sq, Skv, heads, d, impl, seed=0, v_ones=False, qscale=1.0):
    d16 = (d + 15) // 16 * 16
    hs = (d + 1 + 15) // 16 * 16 if v_ones else d16      # zero-padded per-head stride
    q = torch.zeros(B * Sq, heads * hs, device=DEV, dtype=torch.bfloat16)
    k = torch.zeros(B * Skv, heads * hs, device=DEV, dtype=torch.bfloat16)
    v = torch.zeros(B * Skv, heads * hs, device=DEV, dtype=torch.bfloat16)
    qr, kr, vr = (bf(rand(B, n, heads, d, seed=seed + i)) for i, n in enumerate((Sq, Skv, Skv)))
    qr = bf(qr.float() * qscale)          # > 1: peaked rows, the running max moves and O is rescaled
    q.view(B, Sq, heads, hs)[..., :d] = qr
    k.view(B, Skv, heads, hs)[..., :d] = kr
    v.view(B, Skv, heads, hs)[..., :d] = vr
    if v_ones:
        v.view(B, Skv, heads, hs)[..., d] = 1.0
    out = torch.zeros(B * Sq, heads * d, device=DEV, dtype=torch.bfloat16)
    lib.attention(q, k, v, out, batch=B, sq=Sq, skv=Skv, heads=heads, d=d, dh_stride=hs,
                  ldq=heads * hs, ldk=heads * hs, ldv=heads * hs, ldo=heads * d,
                  scale=1 / math.sqrt(d), impl=impl, v_ones=v_ones)
    ref = F.scaled_dot_product_attention(qr.float().transpose(1, 2), kr.float().transpose(1, 2),
                                         vr.float().transpose(1, 2)).transpose(1, 2)
    torch.cuda.synchronize()
    return rel_err(out.view(B, Sq, heads, d), ref)


@pytest.mark.parametrize("B,Sq,Skv,heads,d", [
    (1, 256, 256, 8, 160), (2, 64, 77, 8, 160), (1, 1024, 1024, 2, 80), (1, 300, 77, 8, 40),
    (1, 1024, 1024, 4, 40),
])
def test_attention_simt(B, Sq, Skv, heads, d):
    assert _attn_case(L(), B, Sq, Skv, heads, d, 1) < 2e-2


@pytest.mark.parametrize("B,Sq,Skv,heads,d", [
    (1, 128, 128, 1, 64), (1, 256, 256, 2, 64), (1, 128, 128, 1, 40), (1, 4096, 4096, 2, 40),
    (2, 1024, 1024, 8, 80), (2, 256, 256, 8, 160), (2, 64, 64, 8, 160), (2, 1024, 77, 8, 80),
    (1, 4096, 77, 8, 40), (3, 64, 77, 8, 160), (1, 2304, 2304, 2, 80), (1, 576, 576, 2, 160),
])
def test_attention_tc(B, Sq, Skv, heads, d):
    e = _attn_case(L(), B, Sq, Skv, heads, d, 0)
    assert e < 2e-2, f"rel err {e}"
    e1 = _attn_case(L(), B, Sq, Skv, heads, d, 0, v_ones=True)     # denominator on the tensor core
    assert e1 < 2e-2, f"rel err (v_ones) {e1}"


@pytest.mark.parametrize("B,Sq,Skv,heads,d", [
    (1, 4096, 77, 8, 40), (2, 1024, 77, 8, 80), (2, 256, 77, 8, 160), (1, 300, 77, 3, 40), (2, 512, 100, 4, 64),
    (1, 384, 128, 2, 40), (16, 4096, 77, 8, 40), (1, 2304, 77, 8, 80), (1, 9216, 77, 2, 40), (3, 256, 5, 2, 40),
])
def test_attention_x_short_keys(B, Sq, Skv, heads, d):
    """attention_x.cu (cross-attention: one key tile, a CTA walks a range of query tiles of one (image, head)):
    77 text tokens with the 80-key tile, other short key lists with the 128-key tile, query counts that are not
    a multiple of 128, one to three 64-column chunks per head (d = 40 / 80 / 160)."""
    e = _attn_case(L(), B, Sq, Skv, heads, d, 0, v_ones=True)
    assert e < 2e-2, f"rel err {e}"
    e2 = _attn_case(L(), B, Sq, Skv, heads, d, 0, v_ones=True, qscale=6.0, seed=11)
    assert e2 < 2e-2, f"rel err (peaked rows) {e2}"


@pytest.mark.parametrize("B,Sq,Skv,heads,d", [
    (1, 512, 512, 2, 40), (2, 1024, 1024, 3, 40), (1, 300, 600, 2, 40), (1, 4096, 4096, 1, 40),
    (1, 768, 1000, 2, 56), (1, 512, 640, 2, 48), (2, 9216, 9216, 1, 40),
])
@pytest.mark.parametrize("inputs", ["random", "peaked"])
def test_attention_pp_two_query_tiles(B, Sq, Skv, heads, d, inputs):
    """attention_pp.cu (one softmax thread per row, P in its own TMEM columns) on the default path: ragged key
    tiles, query counts that are not a multiple of 256, both K-step variants; random and peaked rows (the running
    max moves and O is rescaled).  The variants of the DL_ATTN_PP_POLY / DL_ATTN_PP_NQ knobs are checked in
    test_attention_edges_gpu.py::test_attention_knob_variants."""
    if inputs == "random":
        e = _attn_case(L(), B, Sq, Skv, heads, d, 0, v_ones=True)
    else:
        e = _attn_case(L(), B, Sq, Skv, heads, d, 0, v_ones=True, qscale=6.0, seed=7)
    assert e < 2e-2, f"rel err ({inputs}) {e}"


@pytest.mark.parametrize("B,Sq,Skv,d", [
    (2, 1024, 1024, 512), (1, 4096, 4096, 512), (1, 256, 448, 256), (3, 128, 64, 128), (1, 512, 2048, 384),
])
@pytest.mark.parametrize("qscale", [1.0, 5.0])
def test_attention_wide_vae_head(B, Sq, Skv, d, qscale):
    """attention_wide.cu (one head, head dim up to 512, the output columns split over two CTAs per query tile)
    against an fp32 softmax(QK^T / sqrt(d)) V of the same bf16 inputs; q and k are read out of one fused [.., 2d]
    projection buffer as the VAE mid block passes them; peaked rows exercise the running-max rescale of O."""
    lib = L()
    g = torch.Generator(device="cuda").manual_seed(B * 1000 + Sq + d)
    qk = (torch.randn(B * max(Sq, Skv), 2 * d, device="cuda", generator=g) * qscale).to(torch.bfloat16)
    v = torch.randn(B * Skv, d, device="cuda", generator=g).to(torch.bfloat16)
    q = qk[:B * Sq, :d]
    k = qk[:B * Skv, d:]
    out = torch.full((B * Sq, d), float("nan"), device="cuda", dtype=torch.bfloat16)
    scale = 1.0 / math.sqrt(d)
    lib.attention_wide(q, k, v, out, batch=B, sq=Sq, skv=Skv, d=d, ldq=2 * d, ldk=2 * d, ldv=d, ldo=d, scale=scale)
    torch.cuda.synchronize()
    qf = q.float().reshape(B, Sq, d)
    kf = k.float().reshape(B, Skv, d)
    vf = v.float().reshape(B, Skv, d)
    ref = torch.softmax(qf @ kf.transpose(1, 2) * scale, dim=-1) @ vf
    got = out.float().reshape(B, Sq, d)
    assert torch.isfinite(got).all()
    e = ((got - ref).norm() / ref.norm()).item()
    assert e < 2e-2, f"rel err {e}"


# ------------------------------------------------------------------ elementwise / scheduler
def test_upsample_im2col_pack():
    lib = L()
    B, H, W, C = 2, 8, 16, 64
    x = bf(rand(B, H, W, C, seed=1))
    up = torch.empty(B, 2 * H, 2 * W, C, device=DEV, dtype=torch.bfloat16)
    lib.upsample2x(x, up, nimg=B, h=H, w=W)
    ref = F.interpolate(x.float().permute(0, 3, 1, 2), scale_factor=2.0, mode="nearest").permute(0, 2, 3, 1)
    torch.cuda.synchronize()
    assert torch.equal(up.float(), ref)
    cols = torch.empty(B * (H // 2) * (W // 2), 9 * C, device=DEV, dtype=torch.bfloat16)
    lib.im2col_s2(x, cols, nimg=B, h=H, w=W)
    un = F.unfold(x.float().permute(0, 3, 1, 2), 3, padding=1, stride=2)       # [B, C*9, L]
    un = un.view(B, C, 9, -1).permute(0, 3, 2, 1).reshape(-1, 9 * C)
    torch.cuda.synchronize()
    assert torch.equal(cols.float(), un)
    lat = rand(B, 8, 8, 4, seed=2)
    packed = torch.empty(B, 8, 8, 64, device=DEV, dtype=torch.bfloat16)
    lib.pack_latent(lat, packed, cin=4, scale=2.0)
    torch.cuda.synchronize()
    assert torch.equal(packed[..., :4], (lat * 2.0).bfloat16()) and packed[..., 4:].abs().sum() == 0
    a = rand(B, 4, 8, 8, seed=3)
    o = torch.empty(B, 8, 8, 4, device=DEV)
    lib.nchw_to_nhwc_f32(a, o)
    back = torch.empty_like(a)
    lib.nhwc_to_nchw_f32(o, back)
    torch.cuda.synchronize()
    assert torch.equal(o, a.permute(0, 2, 3, 1).contiguous()) and torch.equal(back, a)


def test_lcm_step_bit_exact_vs_oracle():
    """Scheduler update is bit-exact against the oracle's fp32 arithmetic (SURVEY §8c)."""
    lib = L()
    from oracle.scheduler import OracleLCMScheduler
    from dreamlab_b200.scheduler import LCMSchedule
    for n in (1, 2, 4, 8):
        osch = OracleLCMScheduler()
        ts = osch.set_timesteps(n)
        sch = LCMSchedule(n)
        assert sch.timesteps == ts.tolist()
        x = torch.randn(2, 4, 64, 64, generator=torch.Generator().manual_seed(5))
        for i, t in enumerate(ts):
            eps = torch.randn(2, 4, 64, 64, generator=torch.Generator().manual_seed(10 + i))
            z = torch.randn(2, 4, 64, 64, generator=torch.Generator().manual_seed(20 + i)) if i < n - 1 else None
            ref_prev, ref_den = osch.step(eps, int(t), x, noise=z)
            xn = torch.empty(2, 4, 64, 64, device=DEV)
            dn = torch.empty_like(xn)
            lib.lcm_step(eps.to(DEV), x.to(DEV), None if z is None else z.to(DEV), xn, dn, sch.coeffs(i))
            torch.cuda.synchronize()
            assert torch.equal(xn.cpu(), ref_prev), f"prev_sample mismatch n={n} i={i}"
            assert torch.equal(dn.cpu(), ref_den), f"denoised mismatch n={n} i={i}"
            x = ref_prev


def test_time_embedding_pieces():
    lib = L()
    from oracle.unet import timestep_embedding
    t = torch.tensor([999.0, 759.0, 499.0, 259.0], device=DEV)
    out = torch.empty(4, 320, device=DEV)
    lib.timestep_sinusoid(t, out)
    ref = timestep_embedding(t.cpu(), 320)
    torch.cuda.synchronize()
    assert (out.cpu() - ref).abs().max().item() < 2e-3      # sin/cos of ~1e3 rad in fp32
    x = rand(20, 320, seed=1)
    w = bf(rand(1280, 320, seed=2, scale=320 ** -0.5))
    b = rand(1280, seed=3)
    add = rand(20, 1280, seed=4)
    o = torch.empty(20, 1280, device=DEV)
    lib.small_linear(x, w, o, bias=b, add=add, silu_in=True, silu_out=True)
    ref = F.silu(F.silu(x) @ w.float().t() + b + add)
    torch.cuda.synchronize()
    assert (o - ref).abs().max().item() < 1e-3


def test_latent_pool8():
    lib = L()
    from oracle.pipeline import pooled_latent_bytes
    lat = torch.randn(1, 4, 64, 64, generator=torch.Generator().manual_seed(3))
    nhwc = lat.permute(0, 2, 3, 1).contiguous().to(DEV)
    out = torch.empty(1, 4, 8, 8, device=DEV, dtype=torch.float16)
    lib.latent_pool8(nhwc, out)
    torch.cuda.synchronize()
    ref = torch.frombuffer(bytearray(pooled_latent_bytes(lat)), dtype=torch.float16).view(1, 4, 8, 8)
    assert (out.cpu().float() - ref.float()).abs().max().item() < 1e-3
    assert len(out.cpu().numpy().tobytes()) == 512


@pytest.mark.parametrize("B,H,W,C,N,res", [(2, 32, 32, 128, 128, True), (1, 64, 48, 64, 256, False),
                                           (3, 16, 16, 256, 512, True), (2, 24, 48, 128, 128, False)])
def test_igemm_groupnorm_partials(B, H, W, C, N, res):
    """The conv epilogue's GroupNorm records of its own bf16 output (sum, sumsq per M tile and
    group) -> dl_groupnorm_finalize -> (mean, M2) equal to statistics taken from the output
    tensor itself, with and without the fused residual."""
    lib = L()
    G = 32
    cpg = N // G
    x = bf(rand(B, H, W, C, seed=1))
    wt = bf(rand(N, 9 * C, seed=3, scale=(9 * C) ** -0.5))
    bias = rand(N, seed=4)
    r = bf(rand(B, H, W, N, seed=5)) if res else None
    out = torch.empty(B, H, W, N, device=DEV, dtype=torch.bfloat16)
    slots = lib.igemm_tiles_per_image(H, W)
    assert slots > 0
    part = torch.full((B, slots, G, 2), float("nan"), device=DEV)
    lib.igemm(x, wt, out, nimg=B, h=H, w=W, taps=9, n=N, bias=bias, residual=r, gn_partial=part, gn_cpg=cpg)
    stats = torch.empty(B, G, 2, device=DEV)
    lib.groupnorm_finalize(part, stats, H * W * cpg)
    torch.cuda.synchronize()
    assert not torch.isnan(part).any()                       # every (slot, group) was written
    o = out.float().view(B, H * W, G, cpg).permute(0, 2, 1, 3).reshape(B, G, -1).double()
    mean = o.mean(-1)
    m2 = ((o - mean[..., None]) ** 2).sum(-1)
    assert torch.allclose(stats[..., 0].double(), mean, atol=1e-5, rtol=1e-5)
    assert torch.allclose(stats[..., 1].double(), m2, rtol=1e-4, atol=1e-3)
    # and the one-pass norm built on them matches the fused two-phase kernel
    gw, gb = rand(N, seed=6), rand(N, seed=7)
    a = torch.empty_like(out)
    lib.groupnorm_apply(out, a, gw, gb, stats.unsqueeze(0), nimg=B, hw=H * W, groups=G, eps=1e-6, silu=True)
    ws = torch.empty(lib.groupnorm_workspace_bytes(B, G), device=DEV, dtype=torch.uint8)
    b = torch.empty_like(out)
    lib.groupnorm(out, b, gw, gb, ws, nimg=B, hw=H * W, groups=G, eps=1e-6, silu=True)
    torch.cuda.synchronize()
    assert (a.float() - b.float()).abs().max().item() <= 0.0625


@pytest.mark.parametrize("B,H,W,C0,C1,res", [(2, 32, 32, 320, 0, True), (3, 16, 16, 1280, 640, False),
                                              (2, 64, 64, 320, 320, True), (1, 48, 48, 640, 0, False),
                                              (2, 24, 32, 640, 320, True)])
def test_igemm_groupnorm_channel_records(B, H, W, C0, C1, res):
    """Per-CHANNEL GroupNorm records (gn_cpg = 1: the UNet's 10 / 20 / 40 / 60 channels per group do not line up
    with the epilogue's 32-column chunks): the records of one producer, or of the two producers of a
    skip-concat [x0 | x1] whose groups straddle the two sources, -> dl_groupnorm_finalize_channels ->
    (mean, M2) equal to statistics of the tensors themselves; the one-pass norm on them matches the two-phase
    kernel."""
    lib = L()
    G = 32
    outs, parts = [], []
    for k, N in enumerate([C0, C1]):
        if N == 0:
            outs.append(None); parts.append(None)
            continue
        Cin = 64
        x = bf(rand(B, H, W, Cin, seed=1 + k))
        wt = bf(rand(N, 9 * Cin, seed=3 + k, scale=(9 * Cin) ** -0.5))
        bias = rand(N, seed=4 + k)
        r = bf(rand(B, H, W, N, seed=5 + k)) if res else None
        out = torch.empty(B, H, W, N, device=DEV, dtype=torch.bfloat16)
        slots = lib.igemm_tiles_per_image(H, W)
        assert slots > 0
        part = torch.full((B, slots, N, 2), float("nan"), device=DEV)
        lib.igemm(x, wt, out, nimg=B, h=H, w=W, taps=9, n=N, bias=bias, residual=r, gn_partial=part, gn_cpg=1)
        outs.append(out); parts.append(part)
    C = C0 + C1
    cpg = C // G
    stats = torch.empty(B, G, 2, device=DEV)
    lib.groupnorm_finalize_channels(parts[0], parts[1], stats, G, H * W * cpg)
    torch.cuda.synchronize()
    assert not any(torch.isnan(p_).any() for p_ in parts if p_ is not None)     # every (slot, channel) written
    cat = torch.cat([o for o in outs if o is not None], -1).float()
    o = cat.view(B, H * W, G, cpg).permute(0, 2, 1, 3).reshape(B, G, -1).double()
    mean = o.mean(-1)
    m2 = ((o - mean[..., None]) ** 2).sum(-1)
    assert torch.allclose(stats[..., 0].double(), mean, atol=1e-5, rtol=1e-5)
    assert torch.allclose(stats[..., 1].double(), m2, rtol=1e-4, atol=1e-3)
    gw, gb = rand(C, seed=6), rand(C, seed=7)
    a = torch.empty(B, H, W, C, device=DEV, dtype=torch.bfloat16)
    lib.groupnorm_apply(outs[0], a, gw, gb, stats.unsqueeze(0), nimg=B, hw=H * W, groups=G, eps=1e-5, silu=True,
                        x1=outs[1])
    ws = torch.empty(lib.groupnorm_workspace_bytes(B, G), device=DEV, dtype=torch.uint8)
    b = torch.empty_like(a)
    lib.groupnorm(outs[0], b, gw, gb, ws, nimg=B, hw=H * W, groups=G, eps=1e-5, silu=True, x1=outs[1])
    torch.cuda.synchronize()
    assert (a.float() - b.float()).abs().max().item() <= 0.0625


def test_linear_groupnorm_channel_records_token_rows():
    """The same records from a token-row GEMM (Transformer2DModel.proj_out + residual): M = B*S rows, one slot
    per 128 rows of an image."""
    lib = L()
    B, S, K, N, G = 3, 1024, 640, 640, 32
    x = bf(rand(B * S, K, seed=1))
    wt = bf(rand(N, K, seed=2, scale=K ** -0.5))
    r = bf(rand(B * S, N, seed=3))
    out = torch.empty(B * S, N, device=DEV, dtype=torch.bfloat16)
    part = torch.full((B, S // 128, N, 2), float("nan"), device=DEV)
    lib.igemm(x, wt, out, nimg=1, h=1, w=B * S, taps=1, n=N, bias=rand(N, seed=4), residual=r, ldr=N, ldo=N,
              gn_partial=part, gn_cpg=1, gn_rows_per_img=S)
    stats = torch.empty(B, G, 2, device=DEV)
    lib.groupnorm_finalize_channels(part, None, stats, G, S * (N // G))
    torch.cuda.synchronize()
    assert not torch.isnan(part).any()
    o = out.float().view(B, S, G, N // G).permute(0, 2, 1, 3).reshape(B, G, -1).double()
    mean = o.mean(-1)
    assert torch.allclose(stats[..., 0].double(), mean, atol=1e-5, rtol=1e-5)
    assert torch.allclose(stats[..., 1].double(), ((o - mean[..., None]) ** 2).sum(-1), rtol=1e-4, atol=1e-3)


def test_igemm_dual_subtile_residual_and_u8():
    """Narrow-N layers big enough for the two-sub-tile mode (two 128-pixel tiles share a weight
    tile): fused residual + GroupNorm partials, and the u8 image tail (N = 3), odd tile count."""
    lib = L()
    B, H, W, C, N = 1, 593, 128, 64, 128
    x = bf(rand(B, H, W, C, seed=1))
    wt = bf(rand(N, C, 3, 3, seed=3, scale=(9 * C) ** -0.5))
    bias = rand(N, seed=4)
    res = bf(rand(B, H, W, N, seed=6))
    w_pack = wt.permute(0, 2, 3, 1).reshape(N, 9 * C).contiguous()
    out = torch.empty(B, H, W, N, device=DEV, dtype=torch.bfloat16)
    slots = lib.igemm_tiles_per_image(H, W)
    part = torch.full((B, slots, 32, 2), float("nan"), device=DEV)
    lib.igemm(x, w_pack, out, nimg=B, h=H, w=W, taps=9, n=N, bias=bias, residual=res, gn_partial=part, gn_cpg=4)
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), wt.float(), bias, padding=1).permute(0, 2, 3, 1) + res.float()
    torch.cuda.synchronize()
    assert rel_err(out, ref) < 1e-2
    assert not torch.isnan(part).any()
    tot = part.double().sum(1)                                  # [B, 32, 2]
    o = out.float().view(B, H * W, 32, 4).double()
    assert torch.allclose(tot[..., 0], o.sum((1, 3)), rtol=1e-4, atol=1e-2)
    assert torch.allclose(tot[..., 1], (o * o).sum((1, 3)), rtol=1e-4, atol=1e-2)
    w3 = bf(rand(3, C, 3, 3, seed=8, scale=(9 * C) ** -0.5))
    img = torch.empty(B, H, W, 3, device=DEV, dtype=torch.uint8)
    lib.igemm(x, w3.permute(0, 2, 3, 1).reshape(3, 9 * C).contiguous(), img, nimg=B, h=H, w=W, taps=9, n=3,
              bias=rand(3, seed=9), mode=lib.EPI_U8_IMAGE, ldo=3)
    r3 = F.conv2d(x.float().permute(0, 3, 1, 2), w3.float(), rand(3, seed=9), padding=1).permute(0, 2, 3, 1)
    r8 = (r3.bfloat16().float() * 0.5 + 0.5).clamp(0, 1) * 255
    torch.cuda.synchronize()
    assert (img.float() - r8).abs().max().item() <= 1.5


@pytest.mark.parametrize("rows,cols", [(64, 4096), (33, 256), (16, 192), (8, 4100), (5, 1023)])
def test_softmax_rows(rows, cols):
    """fp32 scores -> bf16 probabilities (VAE mid-block attention): register-resident variant
    (cols <= 4096, multiple of 4) and the generic one."""
    lib = L()
    s = rand(rows, cols, seed=1, scale=4.0)
    out = torch.empty(rows, cols, device=DEV, dtype=torch.bfloat16)
    lib.softmax_rows(s, out)
    ref = torch.softmax(s.float(), dim=-1)
    torch.cuda.synchronize()
    assert (out.float() - ref).abs().max().item() <= 4e-3 * ref.max().item() + 1e-6
    assert torch.allclose(out.float().sum(-1), torch.ones(rows, device=DEV), atol=2e-2)


@pytest.mark.parametrize("M,C,N,mode", [(4096, 320, 1152, 0), (1024, 640, 768, 0), (512, 1280, 2560, 1), (300, 320, 384, 0),
                                        (65536, 320, 2560, 1)])
def test_layernorm_folded_into_gemms(M, C, N, mode):
    """LayerNorm without a LayerNorm pass (dl_igemm_desc.row_stats_out / ln_*): GEMM 1 (+ residual) leaves per-row
    (sum, sumsq) records of its bf16 output h; GEMM 2 multiplies h by gamma-scaled weights and applies mean / rstd /
    beta in its epilogue.  Reference: LayerNorm(h) in fp32 -> Linear (-> GEGLU); also against the unfused kernels."""
    lib = L()
    from dreamlab_b200.weights import fold_layernorm, interleave_geglu
    x = bf(rand(M, C, seed=1))
    w1 = bf(rand(C, C, seed=2, scale=C ** -0.5))
    res = bf(rand(M, C, seed=3) + 0.7)                       # a row mean well away from zero
    h = torch.empty(M, C, device=DEV, dtype=torch.bfloat16)
    rs = lib.igemm(x, w1, h, nimg=1, h=1, w=M, taps=1, n=C, bias=rand(C, seed=4), residual=res, ldr=C, ldo=C,
                   row_stats=True)
    torch.cuda.synchronize()
    tot = rs.double().sum(1)                                 # [M, 2]
    assert torch.allclose(tot[:, 0], h.double().sum(1), rtol=1e-5, atol=1e-3)
    assert torch.allclose(tot[:, 1], (h.double() ** 2).sum(1), rtol=1e-5, atol=1e-3)
    gamma, beta = rand(C, seed=5) * 0.3 + 1.0, rand(C, seed=6) * 0.3
    w2 = rand(N, C, seed=7, scale=C ** -0.5)
    b2 = rand(N, seed=8)
    if mode == 1:
        w2p, b2p = interleave_geglu(w2), interleave_geglu(b2)
    else:
        w2p, b2p = w2, b2
    wf, cs, bfold = fold_layernorm(w2p, b2p, gamma, beta, DEV)
    cols = N // 2 if mode == 1 else N
    out = torch.empty(M, cols, device=DEV, dtype=torch.bfloat16)
    lib.igemm(h, wf, out, nimg=1, h=1, w=M, taps=1, n=N, bias=bfold, mode=mode, ldo=cols, ln=(rs, cs, 1e-5))
    # reference in fp32 from the same bf16 h
    ln = F.layer_norm(h.float(), (C,), gamma, beta, 1e-5)
    y = ln @ w2.t() + b2
    if mode == 1:
        y = y[:, :N // 2] * F.gelu(y[:, N // 2:])
    # the unfused product path: LayerNorm kernel (bf16 out) -> GEMM
    n1 = torch.empty_like(h)
    lib.layernorm(h, n1, gamma, beta, 1e-5)
    out2 = torch.empty_like(out)
    lib.igemm(n1, bf(w2p), out2, nimg=1, h=1, w=M, taps=1, n=N, bias=b2p, mode=mode, ldo=cols)
    torch.cuda.synchronize()
    e_fold, e_plain = rel_err(out, y), rel_err(out2, y)
    assert e_fold < 1e-2, e_fold
    assert e_fold <= 1.5 * e_plain + 1e-3, (e_fold, e_plain)      # no worse than the pass it replaces
