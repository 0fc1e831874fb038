"""Per-kernel parity of the fp32 precision mode (csrc/fp32_path.cu, `CUDA_DTYPE=fp32`) against float64
references of the same op on the same fp32 inputs.

The fp32 mode is the yardstick the bf16 path is judged by (test_fp32_mode_gpu.py), so its kernels are held to
fp32 arithmetic: relative error (max|out - ref| / max|ref|) at most 1e-5 for the GEMM, attention and norm
kernels, and bit-exact results where the op involves no arithmetic (im2col) or a single rounding step.
Each test names the entry point it reaches through the dtype-dispatching binding (`dl_igemm_f32`, ...).
Sentinel NaNs in padding columns and past the output's last column show that nothing outside the described
operands is read or written."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda"
# the float64 references below do not use TF32, but the switches are off so that no fp32 helper does either
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False

NAN = float("nan")
BAR = 1e-5          # relative error bar of the fp32 kernels against float64


def L():
    import dreamlab_b200.lib as lib
    lib.load()
    return lib


def rel_err(a, b):
    a, b = a.double(), b.double()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


def rand(*shape, seed=0, scale=1.0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(DEV)


def check(what, err, bar=BAR):
    print(f"{what}: rel err {err:.3e} (bar {bar:.0e})")
    assert err <= bar, f"{what}: rel err {err:.3e} > {bar:.0e}"


def conv3x3_ref(x_nhwc, wt, bias=None):
    """float64 conv3x3 stride 1 pad 1, NHWC in and out."""
    b = None if bias is None else bias.double()
    return F.conv2d(x_nhwc.double().permute(0, 3, 1, 2), wt.double(), b, padding=1).permute(0, 2, 3, 1)


def pack3x3(wt):
    """torch OIHW -> [O, tap*C + c] (the igemm weight layout)."""
    return wt.permute(0, 2, 3, 1).reshape(wt.shape[0], -1).contiguous()


# ------------------------------------------------------------------ dl_igemm_f32: linear
@pytest.mark.parametrize("M,K,N", [(100, 80, 3), (333, 64, 4), (130, 48, 77), (64, 16, 64), (257, 320, 200)])
@pytest.mark.parametrize("mode", [0, 2])        # DL_EPI_BF16 and DL_EPI_F32 both store fp32 in this mode
def test_igemm_f32_linear(M, K, N, mode):
    """dl_igemm_f32 as a Linear with M and N off the 64 x 64 tile, N as small as the conv_out widths; the
    columns of the output rows past N stay untouched."""
    lib = L()
    x = rand(M, K, seed=1)
    w = rand(N, K, seed=2, scale=K ** -0.5)
    bias = rand(N, seed=3)
    buf = torch.full((M, N + 5), NAN, device=DEV)
    lib.igemm(x, w, buf[:, :N], nimg=1, h=1, w=M, taps=1, n=N, bias=bias, mode=mode)
    ref = x.double() @ w.double().t() + bias.double()
    torch.cuda.synchronize()
    check(f"linear M={M} K={K} N={N}", rel_err(buf[:, :N], ref))
    assert torch.isnan(buf[:, N:]).all(), "wrote past column n"


# ------------------------------------------------------------------ dl_igemm_f32: conv3x3
@pytest.mark.parametrize("B,H,W,C0,C1,N", [
    (2, 9, 13, 48, 32, 40), (1, 16, 16, 16, 0, 64), (1, 5, 70, 32, 16, 3), (3, 1, 1, 64, 64, 96), (1, 33, 3, 16, 48, 65),
])
def test_igemm_f32_conv3x3(B, H, W, C0, C1, N):
    """dl_igemm_f32 conv3x3 over a two-source channel concat [x0 | x1] (c0, c1 multiples of 16 but not of 64),
    image sides that cut the 64-pixel tiles anywhere, 1 x 1 images (only the centre tap is inside)."""
    lib = L()
    C = C0 + C1
    x0 = rand(B, H, W, C0, seed=1)
    x1 = rand(B, H, W, C1, seed=2) if C1 else None
    wt = rand(N, C, 3, 3, seed=3, scale=(9 * C) ** -0.5)
    bias = rand(N, seed=4)
    out = torch.full((B, H, W, N), NAN, device=DEV)
    lib.igemm(x0, pack3x3(wt), out, nimg=B, h=H, w=W, taps=9, n=N, a1=x1, bias=bias)
    xin = x0 if x1 is None else torch.cat([x0, x1], -1)
    ref = conv3x3_ref(xin, wt, bias)
    torch.cuda.synchronize()
    check(f"conv3x3 {B}x{H}x{W} C={C0}+{C1} N={N}", rel_err(out, ref))


@pytest.mark.parametrize("B,H,W,C,N", [(2, 5, 7, 32, 48), (1, 8, 8, 16, 16), (1, 1, 9, 48, 3)])
def test_igemm_f32_upsample_fold(B, H, W, C, N):
    """nearest-2x upsample + conv3x3 as four 4-tap phase convs (dl_igemm_f32 taps = 4, tap_phase 0..3), each
    stored through the strided phase view of the 2H x 2W output (out_strides), against the float64 conv of
    the upsampled image with the unfolded weights."""
    lib = L()
    from dreamlab_b200.weights import pack_dtype, pack_upsample_conv3x3
    x = rand(B, H, W, C, seed=1)
    wt = rand(N, C, 3, 3, seed=2, scale=(9 * C) ** -0.5)
    bias = rand(N, seed=3)
    with pack_dtype(torch.float32):
        wp = pack_upsample_conv3x3(wt, DEV)
    assert wp.dtype == torch.float32
    out = torch.full((B, 2 * H, 2 * W, N), NAN, device=DEV)
    strides = (2 * N, 4 * W * N, 4 * H * W * N)
    for ph in range(4):
        lib.igemm(x, wp[ph], out[:, ph >> 1:, ph & 1:, :], nimg=B, h=H, w=W, taps=4, n=N, bias=bias,
                  tap_phase=ph, ldo=N, out_strides=strides)
    up = F.interpolate(x.double().permute(0, 3, 1, 2), scale_factor=2.0, mode="nearest").permute(0, 2, 3, 1)
    ref = conv3x3_ref(up, wt, bias)
    torch.cuda.synchronize()
    check(f"upsample fold {B}x{H}x{W} C={C} N={N}", rel_err(out, ref))


@pytest.mark.parametrize("r0,h", [(0, 4), (4, 6), (10, 6), (3, 5)])
def test_igemm_f32_halo_strip(r0, h):
    """A halo-padded row strip (in_rows = h + 2, in_row0 = 1): the rows above and below the strip come from the
    neighbouring rows of the full image (zeros past its edges); the strip's output equals rows [r0, r0 + h) of
    the dense conv of the full image."""
    lib = L()
    B, H, W, C, N = 2, 16, 12, 32, 48
    x = rand(B, H, W, C, seed=1)
    wt = rand(N, C, 3, 3, seed=2, scale=(9 * C) ** -0.5)
    bias = rand(N, seed=3)
    strip = torch.zeros(B, h + 2, W, C, device=DEV)
    lo, hi = max(r0 - 1, 0), min(r0 + h + 1, H)
    strip[:, lo - (r0 - 1):hi - (r0 - 1)] = x[:, lo:hi]
    out = torch.full((B, h, W, N), NAN, device=DEV)
    lib.igemm(strip, pack3x3(wt), out, nimg=B, h=h, w=W, taps=9, n=N, bias=bias, in_rows=h + 2, in_row0=1)
    ref = conv3x3_ref(x, wt, bias)[:, r0:r0 + h]
    torch.cuda.synchronize()
    check(f"halo strip rows [{r0}, {r0 + h})", rel_err(out, ref))


def test_igemm_f32_conv_epilogue_rowadd_residual_alpha():
    """dl_igemm_f32 epilogue: acc * alpha + bias + rowadd + residual, with rowadd the strided slice of a wider
    per-image time-embedding row (ld_rowadd > n), as the ResNet blocks pass it."""
    lib = L()
    B, H, W, C, N, T = 3, 7, 9, 32, 40, 200
    x = rand(B, H, W, C, seed=1)
    wt = rand(N, C, 3, 3, seed=2, scale=(9 * C) ** -0.5)
    bias = rand(N, seed=3)
    temb = rand(B, T, seed=4)
    rowadd = temb[:, 37:37 + N]
    assert rowadd.stride(0) == T
    res = rand(B, H, W, N, seed=5)
    alpha = 0.37
    out = torch.full((B, H, W, N), NAN, device=DEV)
    lib.igemm(x, pack3x3(wt), out, nimg=B, h=H, w=W, taps=9, n=N, bias=bias, rowadd=rowadd, residual=res,
              alpha=alpha)
    ref = alpha * conv3x3_ref(x, wt) + bias.double() + rowadd.double()[:, None, None, :] + res.double()
    torch.cuda.synchronize()
    check("conv epilogue", rel_err(out, ref))


def test_igemm_f32_strided_operands_geglu():
    """dl_igemm_f32 Linear with the activation read at a pixel stride > c0 and the weight at a row stride > K
    (the gaps hold NaN, so any read of them shows), in DL_EPI_F32 and in GEGLU with interleaved (value, gate)
    columns and the exact erf GELU."""
    lib = L()
    M, K, inner = 150, 96, 40
    xbuf = torch.full((M, K + 32), NAN, device=DEV)
    xbuf[:, :K] = rand(M, K, seed=1)
    x = xbuf[:, :K]
    wv, wg = rand(inner, K, seed=2, scale=K ** -0.5), rand(inner, K, seed=3, scale=K ** -0.5)
    bv, bg = rand(inner, seed=4), rand(inner, seed=5)
    wi = torch.stack([wv, wg], 1).reshape(2 * inner, K)
    wbuf = torch.full((2 * inner, K + 16), NAN, device=DEV)
    wbuf[:, :K] = wi
    w = wbuf[:, :K]
    bi = torch.stack([bv, bg], 1).reshape(-1).contiguous()
    # fp32 output of the interleaved projection itself
    o1 = torch.full((M, 2 * inner + 3), NAN, device=DEV)
    lib.igemm(x, w, o1[:, :2 * inner], nimg=1, h=1, w=M, taps=1, n=2 * inner, bias=bi, mode=lib.EPI_F32)
    ref1 = x.double() @ wi.double().t() + bi.double()
    # GEGLU
    o2 = torch.full((M, inner + 3), NAN, device=DEV)
    lib.igemm(x, w, o2[:, :inner], nimg=1, h=1, w=M, taps=1, n=2 * inner, bias=bi, mode=lib.EPI_GEGLU)
    v = x.double() @ wv.double().t() + bv.double()
    g = x.double() @ wg.double().t() + bg.double()
    ref2 = v * (0.5 * g * (1.0 + torch.erf(g / math.sqrt(2.0))))
    torch.cuda.synchronize()
    check("strided operands, fp32 out", rel_err(o1[:, :2 * inner], ref1))
    check("strided operands, GEGLU", rel_err(o2[:, :inner], ref2))
    assert torch.isnan(o1[:, 2 * inner:]).all() and torch.isnan(o2[:, inner:]).all(), "wrote past the output"


def test_igemm_f32_u8_image_tail():
    """DL_EPI_U8_IMAGE in the fp32 mode: clamp(x / 2 + 0.5, 0, 1) * 255, round to nearest, with no bf16 rounding
    of x in between.  Bit-exact with the float64 result except next to a .5 tie, where the GEMM's own fp32
    error (the 1e-5 bar, in units of 255 / 2 per unit of x) may round the other way, by one."""
    lib = L()
    B, H, W, C = 2, 19, 23, 32
    x = rand(B, H, W, C, seed=1)
    wt = rand(3, C, 3, 3, seed=2, scale=1.3 * (9 * C) ** -0.5)          # outputs past +-1: both clamps
    bias = rand(3, seed=3, scale=0.1)
    out = torch.zeros(B, H, W, 3, device=DEV, dtype=torch.uint8)
    lib.igemm(x, pack3x3(wt), out, nimg=B, h=H, w=W, taps=9, n=3, bias=bias, mode=lib.EPI_U8_IMAGE, ldo=3)
    ref = conv3x3_ref(x, wt, bias)
    f = (ref * 0.5 + 0.5).clamp(0, 1) * 255.0
    tol = 127.5 * BAR * ref.abs().max().item()
    torch.cuda.synchronize()
    assert (ref.abs() > 1).any() and (f > 0).any() and (f < 255).any()
    diff = (out.double() - f.round()).abs()
    near_tie = (f - f.floor() - 0.5).abs() <= tol
    print(f"u8 tail: {(diff > 0).sum().item()} of {diff.numel()} differ (near-tie tolerance {tol:.1e})")
    assert diff.max().item() <= 1
    assert near_tie[diff > 0].all(), "u8 value off away from a rounding tie"


@pytest.mark.parametrize("field", ["gn_partial", "row_stats", "ln", "peer_outs"])
def test_igemm_f32_refuses_fused_statistics_and_peer_stores(field):
    """dl_igemm_f32 has no fused GroupNorm / row statistics, no folded LayerNorm and no peer stores: a descriptor
    asking for one is refused on the host (nothing is launched, the output keeps its contents) instead of
    leaving the caller's statistics buffer unwritten."""
    lib = L()
    M, K, N = 128, 64, 64
    x = rand(M, K, seed=1)
    w = rand(N, K, seed=2, scale=K ** -0.5)
    out = torch.full((M, N), NAN, device=DEV)
    kw = {
        "gn_partial": dict(gn_partial=torch.zeros(1, 1, N, 2, device=DEV), gn_cpg=1, gn_rows_per_img=M),
        "row_stats": dict(row_stats=True),
        "ln": dict(ln=(torch.zeros(M, 2, 2, device=DEV), torch.zeros(N, device=DEV), 1e-5)),
        "peer_outs": dict(peer_outs=[out.data_ptr()]),
    }[field]
    with pytest.raises(RuntimeError, match="fp32 mode has no"):
        lib.igemm(x, w, out, nimg=1, h=1, w=M, taps=1, n=N, **kw)
    torch.cuda.synchronize()
    assert torch.isnan(out).all()
    # the same descriptor without the field runs
    lib.igemm(x, w, out, nimg=1, h=1, w=M, taps=1, n=N)
    torch.cuda.synchronize()
    check("plain linear after the refusal", rel_err(out, x.double() @ w.double().t()))


# ------------------------------------------------------------------ dl_attention_f32
def _attn_f32(B, sq, skv, heads, d, seed=0, qscale=1.0, causal=False):
    """Heads at a per-head stride dh_stride = d + 8 whose pad columns hold NaN; the output rows are 3 columns
    wider than heads * d (NaN too).  float64 reference; causal = keys <= query, by an explicit mask."""
    lib = L()
    hs = d + 8
    q = torch.full((B * sq, heads * hs), NAN, device=DEV)
    k = torch.full((B * skv, heads * hs), NAN, device=DEV)
    v = torch.full((B * skv, heads * hs), NAN, device=DEV)
    qr = rand(B, sq, heads, d, seed=seed) * qscale
    kr, vr = rand(B, skv, heads, d, seed=seed + 1), rand(B, skv, heads, d, seed=seed + 2)
    q.view(B, sq, heads, hs)[..., :d] = qr
    k.view(B, skv, heads, hs)[..., :d] = kr
    v.view(B, skv, heads, hs)[..., :d] = vr
    ldo = heads * d + 3
    out = torch.full((B * sq, ldo), NAN, device=DEV)
    scale = 1 / math.sqrt(d)
    lib.attention(q, k, v, out, batch=B, sq=sq, skv=skv, heads=heads, d=d, dh_stride=hs, ldq=heads * hs,
                  ldk=heads * hs, ldv=heads * hs, ldo=ldo, scale=scale,
                  impl=lib.ATTN_SIMT_CAUSAL if causal else lib.ATTN_SIMT)
    qd, kd, vd = (t.double().transpose(1, 2) for t in (qr, kr, vr))           # [B, heads, S, d]
    s = (qd @ kd.transpose(-1, -2)) * scale
    if causal:
        mask = torch.ones(sq, skv, dtype=torch.bool, device=DEV).triu(1)     # key j > query i
        s = s.masked_fill(mask, float("-inf"))
    ref = (torch.softmax(s, -1) @ vd).transpose(1, 2)                         # [B, sq, heads, d]
    torch.cuda.synchronize()
    assert torch.isnan(out[:, heads * d:]).all(), "wrote past heads * d"
    return rel_err(out[:, :heads * d].reshape(B, sq, heads, d), ref)


@pytest.mark.parametrize("skv", [1, 33, 77, 1000])
@pytest.mark.parametrize("d", [40, 64, 80, 160, 512])
@pytest.mark.parametrize("qscale", [1.0, 6.0])
def test_attention_f32(d, skv, qscale):
    """dl_attention_f32: head dims of the UNet (40 / 80 / 160), CLIP (64) and the VAE mid block (512); key
    counts of one, a partial 32-key step, the 77 text tokens, and many steps; 37 queries (not a multiple of
    the 8 per CTA); two heads; peaked rows (q x 6) move the running max and rescale the accumulator."""
    check(f"attention d={d} skv={skv} q x{qscale:g}", _attn_f32(2, 37, skv, 2, d, seed=d + skv, qscale=qscale))


@pytest.mark.parametrize("B,S,heads,d", [(2, 77, 3, 64), (1, 100, 2, 40), (1, 40, 1, 512)])
def test_attention_f32_causal(B, S, heads, d):
    """DL_ATTN_SIMT_CAUSAL in the fp32 mode (the fp32 CLIP text tower) against an explicitly masked softmax."""
    check(f"causal attention S={S} d={d}", _attn_f32(B, S, S, heads, d, seed=5, causal=True))
    check(f"causal attention S={S} d={d} q x6", _attn_f32(B, S, S, heads, d, seed=6, qscale=6.0, causal=True))


# ------------------------------------------------------------------ dl_groupnorm_f32 / dl_layernorm_f32
@pytest.mark.parametrize("B,HW,C0,C1,G", [(2, 64, 320, 640, 32), (1, 300, 48, 16, 4), (3, 17, 128, 0, 32)])
@pytest.mark.parametrize("silu", [False, True])
@pytest.mark.parametrize("eps", [1e-5, 1e-6])
def test_groupnorm_f32(B, HW, C0, C1, G, silu, eps):
    """dl_groupnorm_f32 over [x0 | x1] with groups that straddle the two sources (C = 320 + 640, 30 channels per
    group: group 10 holds channels 300..329), on inputs with a large common offset (x * 2 + 50), where a
    one-pass E[x^2] - E[x]^2 variance would lose its digits."""
    lib = L()
    C = C0 + C1
    x0 = rand(B, HW, C0, seed=1) * 2 + 50
    x1 = rand(B, HW, C1, seed=2) * 2 + 50 if C1 else None
    gamma, beta = rand(C, seed=3) * 0.2 + 1, rand(C, seed=4) * 0.2
    out = torch.full((B, HW, C), NAN, device=DEV)
    lib.groupnorm(x0, out, gamma, beta, None, nimg=B, hw=HW, groups=G, eps=eps, silu=silu, x1=x1)
    xin = x0 if x1 is None else torch.cat([x0, x1], -1)
    ref = F.group_norm(xin.double().transpose(1, 2), G, gamma.double(), beta.double(), eps).transpose(1, 2)
    if silu:
        ref = F.silu(ref)
    torch.cuda.synchronize()
    check(f"groupnorm C={C0}+{C1} G={G} silu={silu} eps={eps:g}", rel_err(out, ref))


@pytest.mark.parametrize("rows,C", [(1003, 77), (5, 200), (77, 1280), (9, 33)])
def test_layernorm_f32(rows, C):
    """dl_layernorm_f32 with C not a multiple of the 32 lanes and row counts not a multiple of the 8 rows per CTA;
    the input has a common offset as well."""
    lib = L()
    x = rand(rows, C, seed=1) * 3 + 20
    gamma, beta = rand(C, seed=2) * 0.2 + 1, rand(C, seed=3) * 0.2
    buf = torch.full((rows + 1, C), NAN, device=DEV)
    out = buf[:rows]
    lib.layernorm(x, out, gamma, beta, 1e-5)
    ref = F.layer_norm(x.double(), (C,), gamma.double(), beta.double(), 1e-5)
    torch.cuda.synchronize()
    check(f"layernorm rows={rows} C={C}", rel_err(out, ref))
    assert torch.isnan(buf[rows:]).all(), "wrote past the last row"


# ------------------------------------------------------------------ dl_softmax_rows_f32
@pytest.mark.parametrize("cols", [1, 5, 4100])
def test_softmax_rows_f32(cols):
    """dl_softmax_rows_f32 with one column, a handful, and more than 16 per thread; scores x 30 (rows dominated
    by one entry, most exponentials underflow)."""
    lib = L()
    rows = 37
    s = rand(rows, cols, seed=1, scale=30.0)
    out = torch.full((rows, cols), NAN, device=DEV)
    lib.softmax_rows(s, out)
    ref = torch.softmax(s.double(), dim=-1)
    torch.cuda.synchronize()
    check(f"softmax_rows cols={cols}", rel_err(out, ref))
    assert (out.double().sum(-1) - 1).abs().max().item() < 1e-5


# ------------------------------------------------------------------ dl_small_linear_f32
@pytest.mark.parametrize("k", [77, 320])
@pytest.mark.parametrize("silu_in", [False, True])
@pytest.mark.parametrize("silu_out", [False, True])
@pytest.mark.parametrize("with_add", [False, True])
def test_small_linear_f32(k, silu_in, silu_out, with_add):
    """dl_small_linear_f32 with more rows than the bf16 kernel's 64 and k off the 32 lanes, every combination
    of the input / output SiLU and the per-row add."""
    lib = L()
    m, n = 80, 96
    x = rand(m, k, seed=1)
    w = rand(n, k, seed=2, scale=k ** -0.5)
    b = rand(n, seed=3)
    add = rand(m, n, seed=4) if with_add else None
    out = torch.full((m, n), NAN, device=DEV)
    lib.small_linear(x, w, out, bias=b, add=add, silu_in=silu_in, silu_out=silu_out)
    xd = F.silu(x.double()) if silu_in else x.double()
    ref = xd @ w.double().t() + b.double() + (add.double() if with_add else 0.0)
    if silu_out:
        ref = F.silu(ref)
    torch.cuda.synchronize()
    check(f"small_linear k={k} silu_in={silu_in} silu_out={silu_out} add={with_add}", rel_err(out, ref))


# ------------------------------------------------------------------ dl_pack_latent_f32 / dl_im2col_s2_f32
@pytest.mark.parametrize("cpad", [8, 16])
@pytest.mark.parametrize("fold", ["none", "mat", "mat_vec"])
def test_pack_latent_f32(cpad, fold):
    """dl_pack_latent_f32: fp32 [npix, cin] * scale, optionally through the folded post_quant_conv (mat, vec),
    zero-padded to cpad > cin channels."""
    lib = L()
    B, H, W, cin, scale = 2, 9, 7, 4, 1.0 / 0.18215
    x = rand(B, H, W, cin, seed=1)
    mat = rand(cin, cin, seed=2) if fold != "none" else None
    vec = rand(cin, seed=3) if fold == "mat_vec" else None
    out = torch.full((B, H, W, cpad), NAN, device=DEV)
    lib.pack_latent(x, out, cin=cin, scale=scale, mat=mat, vec=vec)
    torch.cuda.synchronize()
    assert torch.equal(out[..., cin:], torch.zeros_like(out[..., cin:]))
    if mat is None:
        assert torch.equal(out[..., :cin], x * scale)        # one fp32 rounding, the same as torch's
        return
    ref = (x.double() * scale) @ mat.double().t() + (vec.double() if vec is not None else 0.0)
    check(f"pack_latent fold={fold}", rel_err(out[..., :cin], ref))


@pytest.mark.parametrize("B,H,W,C", [(2, 8, 16, 4), (1, 6, 10, 36), (3, 2, 2, 64)])
def test_im2col_s2_f32(B, H, W, C):
    """dl_im2col_s2_f32 (conv3x3 stride 2 pad 1 columns, K index = tap * C + c) bit-exact with F.unfold."""
    lib = L()
    x = rand(B, H, W, C, seed=1)
    cols = torch.full((B * (H // 2) * (W // 2), 9 * C), NAN, device=DEV)
    lib.im2col_s2(x, cols, nimg=B, h=H, w=W)
    un = F.unfold(x.permute(0, 3, 1, 2), 3, padding=1, stride=2)          # [B, C*9, L]
    un = un.view(B, C, 9, -1).permute(0, 3, 2, 1).reshape(-1, 9 * C)
    torch.cuda.synchronize()
    assert torch.equal(cols, un)
