"""Per-kernel parity of the bf16-path entry points that the pipelines reach but no other kernel test calls, and
of the igemm operand layouts the engine uses beyond those of test_kernels_gpu.py.

Where a kernel claims a rounding sequence (CFG combine, tile blend, tap sum, token embedding) the test is
bit-exact with the same sequence in torch fp32; elsewhere it compares with a plain fp32 / float64 reference of
the same op on the same bf16-rounded inputs, at the bar of the kernel's arithmetic."""
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


def bf16_ulp(ref):
    """One bf16 unit in the last place at |ref| (8 significant bits; subnormal spacing below 2^-126)."""
    e = torch.floor(torch.log2(ref.double().abs().clamp_min(2.0 ** -126)))
    return torch.exp2(e - 7)


# ------------------------------------------------------------------ cfg_combine
@pytest.mark.parametrize("gs", [1.0, 7.5, 0.0])
def test_cfg_combine_bit_exact(gs):
    """dl_cfg_combine is the oracle's `e_u + gs * (e_t - e_u)` (oracle/pipeline.py) in fp32, three roundings and
    no contraction, bit for bit; the larger tensor has more float4s than the grid (num_sms * 16 CTAs of 256
    threads), so the grid-stride loop runs more than once."""
    lib = L()
    cap = lib.load().dl_device_sm_count() * 16 * 256
    for n in (2 * 4 * 64 * 64, 4 * (cap + cap // 3 + 5)):
        g = torch.Generator().manual_seed(n)
        e_u = torch.randn(n, generator=g)
        e_t = e_u + torch.randn(n, generator=g) * 0.3
        ref = e_u + gs * (e_t - e_u)
        out = torch.full((n,), float("nan"), device=DEV)
        lib.cfg_combine(e_u.to(DEV), e_t.to(DEV), gs, out)
        torch.cuda.synchronize()
        got = out.cpu()
        assert torch.equal(got, ref), (f"gs={gs} n={n}: {(got != ref).sum().item()} elements differ, max "
                                       f"{(got - ref).abs().max().item():.3e}")


# ------------------------------------------------------------------ tile_blend
def _nchw(t):
    return t.permute(0, 3, 1, 2)


@pytest.mark.parametrize("ha,hb,blend", [(48, 48, 16), (48, 20, 16), (12, 40, 16), (16, 16, 16), (5, 3, 8)])
def test_tile_blend_bit_exact(ha, hb, blend):
    """dl_tile_blend against oracle.vae._blend_v / _blend_h (diffusers' blend_v / blend_h) on the same fp32 NHWC
    tiles, bit for bit: full tiles and the ragged bottom / right tiles whose blend extent is the min(...) that
    tiled_decode passes."""
    lib = L()
    from oracle.vae import _blend_h, _blend_v
    B, W, C = 2, 24, 3
    for vertical in (True, False):
        if vertical:
            a, b = rand(B, ha, W, C, seed=1), rand(B, hb, W, C, seed=2)
            ext = min(ha, hb, blend)
        else:
            a, b = rand(B, W, ha, C, seed=1), rand(B, W, hb, C, seed=2)
            ext = min(ha, hb, blend)
        ref = b.cpu().clone()
        (_blend_v if vertical else _blend_h)(_nchw(a.cpu()), _nchw(ref), blend)
        lib.tile_blend(a, b, ext, vertical=vertical)
        torch.cuda.synchronize()
        got = b.cpu()
        assert torch.equal(got, ref), (f"vertical={vertical} extent={ext}: {(got != ref).sum().item()} differ, max "
                                       f"{(got - ref).abs().max().item():.3e}")


def test_tile_blend_sequence_of_tiled_decode():
    """The sequence tiled_decode runs on one tile: blended with the (already blended) tile above, then with the
    tile to its left, the right-most tile being ragged in width and the bottom one in height."""
    lib = L()
    from oracle.vae import _blend_h, _blend_v
    B, C, blend = 1, 3, 16
    up = rand(B, 48, 30, C, seed=1)            # above: same width as the tile
    left = rand(B, 20, 48, C, seed=2)          # left: same height as the tile
    tile = rand(B, 20, 30, C, seed=3)
    ref = tile.cpu().clone()
    _blend_v(_nchw(up.cpu()), _nchw(ref), blend)
    _blend_h(_nchw(left.cpu()), _nchw(ref), blend)
    lib.tile_blend(up, tile, min(up.shape[1], tile.shape[1], blend), vertical=True)
    lib.tile_blend(left, tile, min(left.shape[2], tile.shape[2], blend), vertical=False)
    torch.cuda.synchronize()
    assert torch.equal(tile.cpu(), ref)


# ------------------------------------------------------------------ conv_tapsum
def _tapsum_ref(y, bias, nout):
    """bias first, then taps 0..8 in order, out-of-image taps contributing nothing (fp32, one add per tap)."""
    B, H, W, _ = y.shape
    acc = bias.view(1, 1, 1, nout).expand(B, H, W, nout).clone()
    for t in range(9):
        dy, dx = t // 3 - 1, t % 3 - 1
        part = torch.zeros(B, H, W, nout, device=y.device)
        ys, yd = slice(max(dy, 0), H + min(dy, 0)), slice(max(-dy, 0), H - max(dy, 0))
        xs, xd = slice(max(dx, 0), W + min(dx, 0)), slice(max(-dx, 0), W - max(dx, 0))
        part[:, yd, xd] = y[:, ys, xs, t * nout:(t + 1) * nout]
        acc = acc + part          # + 0.0 where the tap is outside: exact
    return acc


def _image_tail(x):
    """VaeImageProcessor tail of the decoder's bf16 output: round(clamp(x / 2 + 0.5, 0, 1) * 255), ties to even."""
    xb = x.bfloat16().float()
    return ((xb * 0.5 + 0.5).clamp(0, 1) * 255.0).round()


@pytest.mark.parametrize("nout", [1, 2, 3, 4])
@pytest.mark.parametrize("B,H,W", [(2, 7, 5), (1, 1, 9), (2, 6, 1), (1, 1, 1)])
@pytest.mark.parametrize("pad", [3, 32])
def test_conv_tapsum_bit_exact(nout, B, H, W, pad):
    """dl_conv_tapsum on tap-major partial products y [.., ldy] (ldy = 9 * nout + pad > 9 * nout; the engine
    uses 32 for nout = 3), fp32 and u8 outputs, images one pixel high or wide: bit-exact with the same sum."""
    lib = L()
    ldy = 9 * nout + pad
    y = rand(B, H, W, ldy, seed=nout + H, scale=0.4)
    y[..., 9 * nout:] = float("nan")                    # the row padding is never read
    bias = rand(nout, seed=7, scale=0.2)
    ref = _tapsum_ref(y, bias, nout)
    o32 = torch.full((B, H, W, nout), float("nan"), device=DEV)
    lib.conv_tapsum(y, bias, o32)
    o8 = torch.zeros(B, H, W, nout, device=DEV, dtype=torch.uint8)
    lib.conv_tapsum(y, bias, o8)
    torch.cuda.synchronize()
    assert torch.equal(o32, ref), f"max diff {(o32 - ref).abs().max().item():.3e}"
    assert torch.equal(o8.float(), _image_tail(ref))


@pytest.mark.parametrize("B,H,W", [(2, 24, 40), (1, 1, 17), (1, 33, 1)])
def test_conv_tapsum_engine_path(B, H, W):
    """The VAE conv_out as the engine runs it: one 1x1 igemm with the tap-major regrouped weights (27 rows padded
    to 32) in DL_EPI_F32, then dl_conv_tapsum; against F.conv2d on the same bf16 input and weights."""
    lib = L()
    C = 128
    x = bf(rand(B, H, W, C, seed=1))
    wt = bf(rand(3, C, 3, 3, seed=2, scale=1.5 * (9 * C) ** -0.5))
    bias = rand(3, seed=3, scale=0.1)
    w_pack = wt.permute(0, 2, 3, 1).reshape(3, 9 * C)                         # [3, tap*C + c]
    w27 = w_pack.view(3, 9, C).permute(1, 0, 2).reshape(27, C)
    w32 = torch.cat([w27, w27.new_zeros(5, C)], 0).contiguous()
    y = torch.empty(B, H, W, 32, device=DEV)
    lib.igemm(x, w32, y, nimg=B, h=H, w=W, taps=1, n=32, mode=lib.EPI_F32, ldo=32)
    o32 = torch.empty(B, H, W, 3, device=DEV)
    lib.conv_tapsum(y, bias, o32)
    o8 = torch.empty(B, H, W, 3, device=DEV, dtype=torch.uint8)
    lib.conv_tapsum(y, bias, o8)
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), wt.float(), bias, padding=1).permute(0, 2, 3, 1)
    torch.cuda.synchronize()
    assert rel_err(o32, ref) < 1e-2
    # one fp32-rounding difference can move the bf16 rounding of the decoder output by one bf16 step: <= 1 LSB
    assert (o8.float() - _image_tail(ref)).abs().max().item() <= 1


# ------------------------------------------------------------------ act_bf16 / embed_tokens
@pytest.mark.parametrize("mode", [0, 1])
def test_act_bf16(mode):
    """dl_act_bf16 mode 0 = quick_gelu x * sigmoid(1.702 x), mode 1 = exact erf GELU, against torch's fp32 ops on
    the same bf16 inputs, within one bf16 ulp; |x| up to 100, where exp(1.702 |x|) overflows fp32."""
    lib = L()
    g = torch.Generator().manual_seed(3)
    x = torch.cat([torch.linspace(-100, 100, 4001), torch.randn(8192, generator=g) * 4,
                   torch.tensor([0.0, -0.0, 1e-30, -1e-30, 88.0, -88.0, 52.0, -52.0])])
    x = bf(x[: x.numel() // 8 * 8].to(DEV))
    out = torch.empty_like(x)
    lib.act_bf16(x, out, mode)
    xf = x.float()
    ref = xf * torch.sigmoid(1.702 * xf) if mode == 0 else F.gelu(xf)
    torch.cuda.synchronize()
    assert torch.isfinite(out.float()).all()
    diff = (out.double() - ref.double()).abs()
    ulp = bf16_ulp(ref)
    worst = (diff / ulp).max().item()
    print(f"act_bf16 mode {mode}: max |out - ref| = {worst:.2f} bf16 ulp")
    assert worst <= 1.0, f"{worst:.2f} ulp at x = {xf[(diff / ulp).argmax()].item()}"


def test_embed_tokens_bit_exact():
    """dl_embed_tokens for a batch of three prompts (n = 3 * seq: position r % seq) with token ids outside
    [0, V) clamped to the table: bit-exact with bf16(tok[id].float() + pos[r % seq].float())."""
    lib = L()
    V, seq, D = 1000, 77, 96
    tok = bf(rand(V, D, seed=1))
    pos = bf(rand(seq, D, seed=2, scale=0.5))
    g = torch.Generator().manual_seed(4)
    ids = torch.randint(0, V, (3 * seq,), generator=g)
    ids[[0, 5, 80, 200]] = torch.tensor([-1, V, V + 123, -(2 ** 40)])
    ids[[1, 78]] = torch.tensor([V - 1, 0])
    ids = ids.to(DEV)
    out = torch.empty(3 * seq, D, device=DEV, dtype=torch.bfloat16)
    lib.embed_tokens(ids, tok, pos, out, seq)
    r = torch.arange(3 * seq, device=DEV)
    ref = (tok[ids.clamp(0, V - 1)].float() + pos[r % seq].float()).bfloat16()
    torch.cuda.synchronize()
    assert torch.equal(out, ref)


# ------------------------------------------------------------------ pack_latent / im2col_s2_halo
@pytest.mark.parametrize("with_vec", [False, True])
def test_pack_latent_post_quant_conv(with_vec):
    """dl_pack_latent with the folded VAE post_quant_conv (mat, vec) and `/ scaling_factor`, bf16 out, zero pad to
    64 channels: within one bf16 ulp of the float64 result."""
    lib = L()
    B, H, W, cin, cpad, scale = 2, 16, 24, 4, 64, 1.0 / 0.18215
    x = rand(B, H, W, cin, seed=1)
    mat = rand(cin, cin, seed=2)                      # not symmetric: a transposed read shows
    vec = rand(cin, seed=3) if with_vec else None
    out = torch.full((B, H, W, cpad), float("nan"), device=DEV, dtype=torch.bfloat16)
    lib.pack_latent(x, out, cin=cin, scale=scale, mat=mat, vec=vec)
    ref = (x.double() * scale) @ mat.double().t() + (vec.double() if vec is not None else 0.0)
    torch.cuda.synchronize()
    assert torch.equal(out[..., cin:].float(), torch.zeros(B, H, W, cpad - cin, device=DEV))
    worst = ((out[..., :cin].double() - ref).abs() / bf16_ulp(ref)).max().item()
    assert worst <= 1.0, f"{worst:.2f} bf16 ulp"


@pytest.mark.parametrize("r0,h", [(0, 4), (4, 6), (10, 6)])
def test_im2col_s2_halo(r0, h):
    """dl_im2col_s2_halo on the downsample input of a patch-parallel strip: rows [r0, r0 + h) of a full image
    plus one halo row above and below taken from the neighbouring rows (zero outside the image),
    in_rows = h + 2, in_row0 = 1: bit-exact with the matching output rows of dl_im2col_s2 on the full image.
    And the top strip without a halo row (in_row0 = 0): rows above the buffer read as zero."""
    lib = L()
    B, H, W, C = 2, 16, 12, 64
    x = bf(rand(B, H, W, C, seed=1))
    full = torch.empty(B, H // 2, W // 2, 9 * C, device=DEV, dtype=torch.bfloat16)
    lib.im2col_s2(x, full.view(-1, 9 * C), nimg=B, h=H, w=W)
    strip = torch.zeros(B, h + 2, W, C, device=DEV, dtype=torch.bfloat16)
    lo, hi = max(r0 - 1, 0), min(r0 + h + 1, H)
    strip[:, lo - (r0 - 1):hi - (r0 - 1)] = x[:, lo:hi]
    cols = torch.empty(B, h // 2, W // 2, 9 * C, device=DEV, dtype=torch.bfloat16)
    lib.im2col_s2_halo(strip, cols.view(-1, 9 * C), nimg=B, in_rows=h + 2, in_row0=1, h=h, w=W)
    torch.cuda.synchronize()
    assert torch.equal(cols, full[:, r0 // 2:(r0 + h) // 2])
    if r0 == 0:
        top = x[:, :h + 1].contiguous()
        cols0 = torch.empty_like(cols)
        lib.im2col_s2_halo(top, cols0.view(-1, 9 * C), nimg=B, in_rows=h + 1, in_row0=0, h=h, w=W)
        torch.cuda.synchronize()
        assert torch.equal(cols0, full[:, :h // 2])


# ------------------------------------------------------------------ attention: the CUDA-core kernel at d = 512
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


@pytest.mark.parametrize("S", [144, 841])
@pytest.mark.parametrize("qscale", [1.0, 6.0])
def test_attention_simt_vae_mid_block(S, qscale):
    """ATTN_SIMT with one head of d = 512 at the token counts of ragged tiled-decode tiles (12 x 12, 29 x 29):
    the mid-block attention path for tiles the wide flash kernel and the GEMM form cannot take."""
    e = _attn_case(L(), 1, S, S, 1, 512, 1, seed=S, qscale=qscale)
    assert e < 2e-2, f"rel err {e}"


# ------------------------------------------------------------------ the unfused VAE mid-block attention GEMMs
@pytest.mark.parametrize("S,B", [(576, 2), (1600, 1)])
def test_vae_mid_attention_gemm_sequence(S, B):
    """VAEDecoderB200._mid_attention's GEMM form (S % 128 != 0, S % 64 == 0; 24^2 and 40^2 latents) at C = 512:
    V^T with the activation as the weight operand, Q K^T reading q and k out of one [S, 2C] buffer (c0 = C,
    a0_stride = ldw = 2C) into fp32 scores scaled by alpha = 1/sqrt(C), the bf16 row softmax, and P V^T into
    the image's rows of the output.  Each intermediate against fp32 torch on the kernel's own inputs, and the
    output against fp32 attention from the start."""
    lib = L()
    C = 512
    hn = bf(rand(B * S, C, seed=1))
    v_w = bf(rand(C, C, seed=2, scale=C ** -0.5))
    qk = bf(rand(B * S, 2 * C, seed=3))
    scores = torch.empty(S, S, device=DEV)
    probs = torch.empty(S, S, device=DEV, dtype=torch.bfloat16)
    vt = torch.empty(C, S, device=DEV, dtype=torch.bfloat16)
    o = torch.empty(B * S, C, device=DEV, dtype=torch.bfloat16)
    for b in range(B):
        rows = slice(b * S, (b + 1) * S)
        lib.igemm(v_w, hn[rows], vt, nimg=1, h=1, w=C, taps=1, n=S, a0_stride=C, ldo=S)
        q, k = qk[rows, :C], qk[rows, C:]
        lib.igemm(q, k, scores, nimg=1, h=1, w=S, taps=1, n=S, c0=C, a0_stride=2 * C,
                  mode=lib.EPI_F32, alpha=1.0 / math.sqrt(C), ldo=S)
        lib.softmax_rows(scores, probs)
        lib.igemm(probs, vt, o[rows], nimg=1, h=1, w=S, taps=1, n=C, a0_stride=S, ldo=C)
        vt_ref = v_w.float() @ hn[rows].float().t()
        s_ref = (q.float() @ k.float().t()) / math.sqrt(C)
        p_ref = torch.softmax(scores, -1)
        o_ref = probs.float() @ vt.float().t()
        full_ref = torch.softmax(s_ref, -1) @ vt_ref.t()
        torch.cuda.synchronize()
        e_vt, e_s = rel_err(vt, vt_ref), rel_err(scores, s_ref)
        e_p = (probs.float() - p_ref).abs().max().item() / p_ref.max().item()
        e_o, e_full = rel_err(o[rows], o_ref), rel_err(o[rows], full_ref)
        print(f"S={S} image {b}: V^T {e_vt:.2e}, scores {e_s:.2e}, probs {e_p:.2e}, PV {e_o:.2e}, all {e_full:.2e}")
        assert e_vt < 1e-2, e_vt
        assert e_s < 1e-4, e_s            # exact bf16 products, fp32 sums over K = 512, one scale
        assert e_p < 4e-3, e_p
        assert e_o < 1e-2, e_o
        assert e_full < 2e-2, e_full


# ------------------------------------------------------------------ igemm bf16 operand variants
def test_igemm_conv3x3_rowadd_strided_time_embedding():
    """The ResNet time-embedding add as the engine passes it: rowadd = temb[:, off:off + cout], a strided view of
    the fused per-image projection (ld_rowadd = its full width), on a conv3x3 with partial tiles in x and y."""
    lib = L()
    B, H, W, C, N, T, off = 3, 24, 20, 128, 320, 2240, 640
    x = bf(rand(B, H, W, C, seed=1))
    wt = bf(rand(N, C, 3, 3, seed=2, scale=(9 * C) ** -0.5))
    bias = rand(N, seed=3)
    temb = rand(B, T, seed=4)
    rowadd = temb[:, off:off + N]
    assert rowadd.stride(0) == T
    w_pack = wt.permute(0, 2, 3, 1).reshape(N, 9 * C).contiguous()
    out = torch.empty(B, H, W, N, device=DEV, dtype=torch.bfloat16)
    lib.igemm(x, w_pack, out, nimg=B, h=H, w=W, taps=9, n=N, bias=bias, rowadd=rowadd)
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), wt.float(), bias, padding=1).permute(0, 2, 3, 1)
    ref = ref + rowadd[:, None, None, :]
    torch.cuda.synchronize()
    e = rel_err(out, ref)
    assert e < 1e-2, f"rel err {e}"


@pytest.mark.parametrize("M,C0,C1,N", [(300, 640, 320, 320), (1024, 128, 64, 64), (77, 64, 1280, 640)])
def test_igemm_two_source_linear(M, C0, C1, N):
    """taps = 1 over two sources (the ResNet 1x1 shortcut on a skip-concat): a0 and a1 each read at their own
    pixel stride (a1 a column slice of a wider buffer), against cat([x0, x1]) @ W^T."""
    lib = L()
    x0 = bf(rand(M, C0, seed=1))
    x1buf = bf(rand(M, C1 + 64, seed=2))
    x1 = x1buf[:, :C1]
    w = bf(rand(N, C0 + C1, seed=3, scale=(C0 + C1) ** -0.5))
    bias = rand(N, seed=4)
    out = torch.empty(M, N, device=DEV, dtype=torch.bfloat16)
    lib.igemm(x0, w, out, nimg=1, h=1, w=M, taps=1, n=N, a1=x1, bias=bias, a0_stride=C0, a1_stride=C1 + 64)
    ref = torch.cat([x0, x1], -1).float() @ w.float().t() + bias
    torch.cuda.synchronize()
    e = rel_err(out, ref)
    assert e < 1e-2, f"rel err {e}"
