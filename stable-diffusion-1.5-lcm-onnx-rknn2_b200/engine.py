"""Host orchestration of the hot path: LCM denoise loop (UNet + scheduler step) + VAE decode.

Every arithmetic op is a launch of a hand-written sm_100a kernel through the C-ABI (`lib.py`);
torch only owns device memory, streams and the CUDA graph.  Activations are NHWC bf16,
latents / time embeddings / noise_pred fp32.

What this replaces in the reference: the body of `self.pipe(...)` at
`backends/cuda_worker.py:221-229` (loop restated in-tree at `backends/rknnlcm.py:586-618`).
Structural differences from the diffusers pipeline, all result-preserving:
  * cross-attention K/V projections of the prompt are hoisted out of the step loop (the text
    is constant across steps), time embeddings for all steps are computed before the loop;
  * skip-concat, GroupNorm+SiLU, bias/temb/residual adds, GEGLU and the image denormalise
    are fused into the producing kernels; no host sync inside the loop.
"""
from __future__ import annotations

import math
from typing import List, Optional

import torch

from . import lib
from .scheduler import (DEFAULT_CONFIG, LCMSchedule, SchedulerConfig, check_sampler, guidance_scale_embedding,
                        sampler_schedule)
from .weights import Packed, has_vae_encoder, pack_taesd_decoder, pack_unet, pack_vae_decoder, pack_vae_encoder

BF16 = torch.bfloat16


_gnx_ws = {}


class Padded:
    """A row strip with one halo row above and below: t is bf16 [B, h+2, W, C]; rows 1..h are
    the strip, rows 0 / h+1 the neighbours' boundary rows (zeros at the image border)."""
    __slots__ = ("t",)

    def __init__(self, t):
        self.t = t


class _Ctx:
    """Per-forward scratch: device, batch, the GroupNorm workspace and (patch-parallel runs)
    the strip communicator.  comm=None is the single-GPU path."""

    def __init__(self, device, batch, comm=None, gn_fuse=0, dt=BF16, ln_fold=False):
        self.device = device
        self.batch = batch
        self.comm = comm
        # LayerNorm folded into the neighbouring GEMMs (transformer_block); bf16 one-GPU path only
        self.ln_fold = bool(ln_fold) and comm is None and dt == BF16
        self.dt = dt          # activation dtype: bf16 (tcgen05 path) or fp32 (precision mode, CUDA cores)
        if dt != BF16:
            gn_fuse = 0
        # > 0: convs emit GroupNorm partial statistics of their output for norms with this many
        # groups (VAE decoder: 4/8/16 channels per group line up with the epilogue's 32-column
        # chunks); the consumer norm then reads its input once instead of twice
        self.gn_fuse = gn_fuse if comm is None else 0
        self.gn_ws = torch.empty(lib.groupnorm_workspace_bytes(batch, 32), device=device,
                                 dtype=torch.uint8)
        if comm is not None:
            # zero-initialised once per (device, batch): the stats kernel leaves its counters zero
            import threading
            key = (str(device), batch, threading.get_ident())    # virtual ranks (threads) never share it
            if key not in _gnx_ws:
                _gnx_ws[key] = torch.zeros(lib.groupnorm_split_workspace_bytes(batch, 64), device=device,
                                           dtype=torch.uint8)
            self.gnx_ws = _gnx_ws[key]

    def empty(self, *shape, dtype=None):
        return torch.empty(*shape, device=self.device, dtype=dtype or self.dt)

    def pad_rows(self, x):
        """Strip [B,h,W,C] -> Padded copy with exchanged halo rows."""
        B, H, W, C = x.shape
        t = self.empty(B, H + 2, W, C)
        t[:, 1:H + 1].copy_(x)
        self.comm.halo_exchange(t)
        return Padded(t)


# ------------------------------------------------------------------------------------------------
# building blocks
# ------------------------------------------------------------------------------------------------
def _gn_request(ctx, B, n_out, slots, phases=1):
    """(partial-statistics buffer, channels per record) for an igemm whose output feeds a GroupNorm, or
    (None, 0).  Channels per group 4 / 8 / 16 / 32 (VAE decoder) line up with the epilogue's 32-column
    chunks: per-group records [B, slots, groups, 2].  Anything else (UNet: 10 / 20 / 40): per-CHANNEL records
    [B, slots, n_out, 2] (cpg 1), reduced per group by `groupnorm_finalize_channels`."""
    g = ctx.gn_fuse
    if not g or n_out % g or n_out % 32 or slots <= 0:
        return None, 0
    if (n_out // g) in (4, 8, 16, 32):
        return ctx.empty(B, slots * phases, g, 2, dtype=torch.float32), n_out // g
    return ctx.empty(B, slots * phases, n_out, 2, dtype=torch.float32), 1


def _carry_gn(src, dst):
    """Views are new tensor objects: hand the producer's GroupNorm records on."""
    if hasattr(src, "_gn"):
        dst._gn, dst._gn_cpg = src._gn, src._gn_cpg
    return dst


def conv3x3(ctx, x, w, b, n_out, *, x1=None, rowadd=None, residual=None, mode=lib.EPI_BF16,
            out=None, ldo=None, feeds_norm=False):
    """x: dense [B,H,W,C] (zero padding all round) or a Padded strip (halo rows supplied)."""
    halo = isinstance(x, Padded)
    if halo:
        x = x.t
    B, H, W, _ = x.shape
    if halo:
        H -= 2
    if out is None:
        out = ctx.empty(B, H, W, n_out, dtype=torch.float32 if mode == lib.EPI_F32 else None)
    part, cpg = None, 0
    if feeds_norm and ctx.gn_fuse and mode == lib.EPI_BF16 and not halo:
        part, cpg = _gn_request(ctx, B, n_out, lib.igemm_tiles_per_image(H, W))
    lib.igemm(x, w, out, nimg=B, h=H, w=W, taps=9, n=n_out, a1=x1, bias=b, rowadd=rowadd,
              residual=residual, mode=mode, ldo=ldo, in_rows=H + 2 if halo else 0,
              in_row0=1 if halo else 0, gn_partial=part, gn_cpg=cpg)
    if part is not None:
        out._gn, out._gn_cpg = part, cpg
    return out


def linear(ctx, x, w, b, n_out, *, x1=None, residual=None, mode=lib.EPI_BF16, out_cols=None,
           alpha=1.0, out=None, norm_rows_per_img=0, row_stats=False, ln=None):
    """x: [..., K] bf16 rows (any leading shape); returns [..., n_out] (or n_out/2 for GEGLU).
    norm_rows_per_img > 0: the output (token rows of images of that many pixels) feeds a GroupNorm.
    row_stats: the output feeds a LayerNorm that is folded into its consumer — the epilogue leaves per-row
    (sum, sumsq) records in `out._rs`.  ln=(records, colsum, eps): this GEMM consumes LayerNorm(x) (w is the
    gamma-scaled weight, b the folded bias)."""
    lead = x.shape[:-1]
    M = x.numel() // x.shape[-1]
    cols = out_cols if out_cols is not None else (n_out // 2 if mode == lib.EPI_GEGLU else n_out)
    if out is None:
        out = ctx.empty(*lead, cols, dtype=torch.float32 if mode == lib.EPI_F32 else None)
    part, cpg = None, 0
    if norm_rows_per_img and norm_rows_per_img % 128 == 0 and mode == lib.EPI_BF16 and M % norm_rows_per_img == 0:
        part, cpg = _gn_request(ctx, M // norm_rows_per_img, n_out, norm_rows_per_img // 128)
    rs = lib.igemm(x, w, out, nimg=1, h=1, w=M, taps=1, n=n_out, a1=x1, bias=b, residual=residual,
                   mode=mode, alpha=alpha, a0_stride=x.stride(-2), a1_stride=None if x1 is None else x1.stride(-2),
                   ldo=cols, ldr=None if residual is None else residual.shape[-1], gn_partial=part,
                   gn_cpg=cpg, gn_rows_per_img=norm_rows_per_img if part is not None else 0,
                   row_stats=row_stats, ln=ln)
    if part is not None:
        out._gn, out._gn_cpg = part, cpg
    if rs is not None:
        out._rs = rs
    return out


def groupnorm(ctx, x, gw, gb, *, eps, silu, x1=None, groups=32, halo=False):
    """halo=True (feeds a conv3x3): under a strip communicator the result is a Padded strip."""
    B, H, W, C0 = x.shape
    C = C0 + (x1.shape[-1] if x1 is not None else 0)
    part = getattr(x, "_gn", None)
    if ctx.comm is None and part is not None and x1 is None and x._gn_cpg > 1 and part.shape[2] == groups:
        # the producing conv left (sum, sumsq) per M tile: one tiny reduction, then ONE pass over x
        stats = ctx.empty(1, B, groups, 2, dtype=torch.float32)
        lib.groupnorm_finalize(part, stats, H * W * (C // groups))
        out = ctx.empty(B, H, W, C)
        lib.groupnorm_apply(x, out, gw, gb, stats, nimg=B, hw=H * W, groups=groups, eps=eps, silu=silu)
        return out
    part1 = getattr(x1, "_gn", None) if x1 is not None else None
    if (ctx.comm is None and part is not None and x._gn_cpg == 1 and
            (x1 is None or (part1 is not None and x1._gn_cpg == 1))):
        # per-channel records of the producer(s) (the skip-concat partner included): finalize per group,
        # then ONE pass over [x | x1] — no statistics pass, no grid barrier
        stats = ctx.empty(1, B, groups, 2, dtype=torch.float32)
        lib.groupnorm_finalize_channels(part, part1, stats, groups, H * W * (C // groups))
        out = ctx.empty(B, H, W, C)
        lib.groupnorm_apply(x, out, gw, gb, stats, nimg=B, hw=H * W, groups=groups, eps=eps, silu=silu, x1=x1)
        return out
    if ctx.comm is None:
        out = ctx.empty(B, H, W, C)
        lib.groupnorm(x, out, gw, gb, ctx.gn_ws, nimg=B, hw=H * W, groups=groups, eps=eps, silu=silu, x1=x1)
        return out
    # row strips: local (mean, M2) -> all-gather over the patch group -> merge + normalise
    stats = ctx.empty(B, groups, 2, dtype=torch.float32)
    lib.groupnorm_stats(x, stats, ctx.gnx_ws, nimg=B, hw=H * W, groups=groups, x1=x1)
    stats_all = ctx.comm.all_gather(stats)
    if not halo:
        out = ctx.empty(B, H, W, C)
        lib.groupnorm_apply(x, out, gw, gb, stats_all, nimg=B, hw=H * W, groups=groups, eps=eps,
                            silu=silu, x1=x1)
        return out
    t = ctx.empty(B, H + 2, W, C)
    lib.groupnorm_apply(x, t[:, 1:], gw, gb, stats_all, nimg=B, hw=H * W, groups=groups, eps=eps,
                        silu=silu, x1=x1, out_img_stride=(H + 2) * W * C)
    ctx.comm.halo_exchange(t)
    return Padded(t)


def resnet(ctx, x, p: Packed, *, temb=None, x1=None, eps=1e-5, groups=32):
    """ResnetBlock2D on x (or on the channel concat [x | x1])."""
    cout = p["cout"]
    h = groupnorm(ctx, x, p["norm1_w"], p["norm1_b"], eps=eps, silu=True, x1=x1, groups=groups, halo=True)
    rowadd = None
    if temb is not None:
        rowadd = temb[:, p["temb_off"]:p["temb_off"] + cout]     # view: ld = temb_total
    h = conv3x3(ctx, h, p["conv1_w"], p["conv1_b"], cout, rowadd=rowadd, feeds_norm=True)
    h = groupnorm(ctx, h, p["norm2_w"], p["norm2_b"], eps=eps, silu=True, groups=groups, halo=True)
    if p["sc_w"] is not None:
        sc = linear(ctx, x, p["sc_w"], p["sc_b"], cout, x1=x1)
    else:
        assert x1 is None
        sc = x
    return conv3x3(ctx, h, p["conv2_w"], p["conv2_b"], cout, residual=sc, feeds_norm=True)


def transformer_block(ctx, h, q: Packed, kv, *, B, S, C, heads, d, hstride, last=True):
    """One BasicTransformerBlock on token rows h [B*S, C]; kv = hoisted cross-attn K/V.
    With `ctx.ln_fold` (one GPU, bf16, no style LoRA on the weights) the three LayerNorms are never
    materialised: every GEMM that produces a LayerNorm input leaves per-row (sum, sumsq) records in its
    epilogue (`h._rs`) and the consuming projection applies mean / rstd / gamma / beta in its own epilogue
    (weights pre-multiplied by gamma at load, `weights.fold_layernorm`).  last=False: the block's output
    feeds the next block's LayerNorm, so the final GEMM emits records too."""
    hs = heads * hstride
    scale = 1.0 / math.sqrt(d)
    fold = ctx.ln_fold and ctx.comm is None and q["qkv_wf"] is not None and hasattr(h, "_rs")
    # --- self attention
    a = ctx.empty(B * S, C)
    if ctx.comm is None:
        if fold:
            qkv = linear(ctx, h, q["qkv_wf"], q["qkv_bf"], 3 * hs, ln=(h._rs, q["qkv_cs"], 1e-5))
        else:
            n1 = ctx.empty(B * S, C)
            lib.layernorm(h, n1, q["ln1_w"], q["ln1_b"])
            qkv = linear(ctx, n1, q["qkv_w"], q["qkv_b"], 3 * hs)
        lib.attention(qkv, qkv[:, hs:], qkv[:, 2 * hs:], a, batch=B, sq=S, skv=S, heads=heads, d=d,
                      dh_stride=hstride, ldq=3 * hs, ldk=3 * hs, ldv=3 * hs, ldo=C, scale=scale, v_ones=True)
    else:
        n1 = ctx.empty(B * S, C)
        lib.layernorm(h, n1, q["ln1_w"], q["ln1_b"])
        # row strips: queries stay local, keys/values of every strip are all-gathered
        # (SURVEY.md §8e exchange X2); key order = rank order = image row order
        qs = linear(ctx, n1, q["qkv_w"][:hs], None, hs)
        if hasattr(ctx.comm, "gather_linear") and S % 128 == 0 and ctx.dt == BF16:
            # gather fused into the K/V projection: its epilogue TMA-stores every tile into the
            # peers' K/V buffers as well (NVLink writes overlap the GEMM), a flag barrier follows
            def kv_proj(out_view, peer_ptrs):
                lib.igemm(n1, q["qkv_w"][hs:], out_view, nimg=B, h=1, w=S, taps=1, n=2 * hs, bias=q["qkv_b"][hs:],
                          ldo=2 * hs, out_strides=(2 * hs, S * 2 * hs, out_view.stride(0)), peer_outs=peer_ptrs)
            kvf = ctx.comm.gather_linear(kv_proj, B, S, 2 * hs)
        else:
            kvl = linear(ctx, n1, q["qkv_w"][hs:], q["qkv_b"][hs:], 2 * hs)
            kvf = ctx.comm.gather_rows(kvl.view(B, S, 2 * hs))            # [B, R*S, 2hs]
        skv_all = kvf.shape[1]
        kvf = kvf.view(B * skv_all, 2 * hs)
        lib.attention(qs, kvf, kvf[:, hs:], a, batch=B, sq=S, skv=skv_all, heads=heads, d=d,
                      dh_stride=hstride, ldq=hs, ldk=2 * hs, ldv=2 * hs, ldo=C, scale=scale, v_ones=True)
    h = linear(ctx, a, q["o1_w"], q["o1_b"], C, residual=h, row_stats=fold)
    # --- cross attention (K/V precomputed once per request)
    if fold:
        qq = linear(ctx, h, q["q2_wf"], q["q2_bf"], hs, ln=(h._rs, q["q2_cs"], 1e-5))
    else:
        n2 = ctx.empty(B * S, C)
        lib.layernorm(h, n2, q["ln2_w"], q["ln2_b"])
        qq = linear(ctx, n2, q["q2_w"], None, hs)
    skv = kv.shape[0] // B
    a2 = ctx.empty(B * S, C)
    lib.attention(qq, kv, kv[:, hs:], a2, batch=B, sq=S, skv=skv, heads=heads, d=d, dh_stride=hstride,
                  ldq=hs, ldk=2 * hs, ldv=2 * hs, ldo=C, scale=scale, v_ones=True)
    h = linear(ctx, a2, q["o2_w"], q["o2_b"], C, residual=h, row_stats=fold)
    # --- GEGLU feed-forward
    if fold:
        g = linear(ctx, h, q["ff1_wf"], q["ff1_bf"], 8 * C, mode=lib.EPI_GEGLU, ln=(h._rs, q["ff1_cs"], 1e-5))
    else:
        n3 = ctx.empty(B * S, C)
        lib.layernorm(h, n3, q["ln3_w"], q["ln3_b"])
        g = linear(ctx, n3, q["ff1_w"], q["ff1_b"], 8 * C, mode=lib.EPI_GEGLU)
    return linear(ctx, g, q["ff2_w"], q["ff2_b"], C, residual=h, row_stats=fold and not last)


def transformer(ctx, x, p: Packed, kvs, *, groups=32):
    """Transformer2DModel.  kvs: one hoisted cross-attn K/V [B*77, 2*heads*hstride] per block."""
    B, H, W, C = x.shape
    S = H * W
    hn = groupnorm(ctx, x, p["norm_w"], p["norm_b"], eps=1e-6, silu=False, groups=groups)
    h = linear(ctx, hn.view(B * S, C), p["proj_in_w"], p["proj_in_b"], C,
               row_stats=ctx.ln_fold and ctx.comm is None and ctx.dt == BF16)
    nb = len(p["blocks"])
    for i, (q, kv) in enumerate(zip(p["blocks"], kvs)):
        h = transformer_block(ctx, h, q, kv, B=B, S=S, C=C, heads=p["heads"], d=p["d"],
                              hstride=p["hstride"], last=i == nb - 1)
    out = linear(ctx, h, p["proj_out_w"], p["proj_out_b"], C, residual=x.view(B * S, C), norm_rows_per_img=S)
    return _carry_gn(out, out.view(B, H, W, C))


def downsample(ctx, x, p: Packed):
    B, H, W, C = x.shape
    cols = ctx.empty(B * (H // 2) * (W // 2), 9 * C)
    if ctx.comm is None:
        lib.im2col_s2(x, cols, nimg=B, h=H, w=W)
    else:
        xp = ctx.pad_rows(x)
        lib.im2col_s2_halo(xp.t, cols, nimg=B, in_rows=H + 2, in_row0=1, h=H, w=W)
    out = linear(ctx, cols, p["w"], p["b"], C, norm_rows_per_img=(H // 2) * (W // 2))
    return _carry_gn(out, out.view(B, H // 2, W // 2, C))


def upsample(ctx, x, p: Packed):
    """Upsample2D = nearest-2x + conv3x3, folded: four 2x2-tap convs on the low-res input, one
    per output phase, each TMA-storing into its strided quarter of the output."""
    B, H, W, C = x.shape
    out = ctx.empty(B, 2 * H, 2 * W, C)
    strides = (2 * C, 4 * W * C, 4 * H * W * C)            # x, row, image strides of a phase view
    src, halo = x, {}
    if ctx.comm is not None:
        src, halo = ctx.pad_rows(x).t, dict(in_rows=H + 2, in_row0=1)
    T = lib.igemm_tiles_per_image(H, W) if ctx.gn_fuse else 0
    part, cpg = _gn_request(ctx, B, C, T, phases=4)
    for ph in range(4):
        a, b = ph >> 1, ph & 1
        view = out[:, a:, b:, :]                            # base pointer of phase (a, b)
        lib.igemm(src, p["w"][ph], view, nimg=B, h=H, w=W, taps=4, n=C, bias=p["b"], tap_phase=ph,
                  ldo=C, out_strides=strides, gn_partial=part, gn_cpg=cpg, gn_slot0=ph * T, **halo)
    if part is not None:
        out._gn, out._gn_cpg = part, cpg
    return out


# ------------------------------------------------------------------------------------------------
# UNet
# ------------------------------------------------------------------------------------------------
def _dt_of(precision: str):
    if precision not in ("bf16", "fp32"):
        raise RuntimeError(f"precision must be 'bf16' or 'fp32', got {precision!r}")
    return BF16 if precision == "bf16" else torch.float32


class UNetB200:
    def __init__(self, state_dict, cfg, device="cuda:0", precision="bf16"):
        lib.require_cuda()
        lib.load()
        self.device = torch.device(device)
        self.cfg = cfg
        self.dt = _dt_of(precision)
        from .weights import pack_dtype
        with pack_dtype(self.dt):
            self.P = pack_unet(state_dict, cfg, self.device)
        self.groups = getattr(cfg, "norm_num_groups", 32)
        import os
        self.fuse_gn_stats = os.environ.get("DL_UNET_GN_FUSE", "1") not in ("0", "false")
        # DL_UNET_LN_FOLD=0 keeps the standalone LayerNorm kernel (A/B).  Style LoRAs update the packed
        # projection weights in place (lora.py): `StyleManager` switches the fold off for such a UNet
        self.fold_ln = os.environ.get("DL_UNET_LN_FOLD", "1") not in ("0", "false")

    @torch.no_grad()
    def encode_context(self, prompt_embeds: torch.Tensor) -> List[List[torch.Tensor]]:
        """Hoisted cross-attention K/V: per Transformer2DModel, one tensor per block.
        prompt_embeds [B,77,D]."""
        B, T, D = prompt_embeds.shape
        ctx = _Ctx(self.device, B, dt=self.dt)
        pe = prompt_embeds.to(self.device, self.dt).contiguous().view(B * T, D)
        return [[linear(ctx, pe, q["kv2_w"], q["kv2_b"], 2 * t["heads"] * t["hstride"])
                 for q in t["blocks"]] for t in self.P["transformers"]]

    @torch.no_grad()
    def addition_embedding(self, text_embeds: torch.Tensor, time_ids: torch.Tensor) -> torch.Tensor:
        """SDXL `text_time` embedding (constant over the steps): fp32 [B, 4*ch0].
        text_embeds [B, P] pooled text, time_ids [B, 6]."""
        P = self.P
        B = text_embeds.shape[0]
        td = self.cfg.addition_time_embed_dim
        ids = time_ids.to(self.device, torch.float32).reshape(-1).contiguous()
        sin = torch.empty(ids.numel(), td, device=self.device, dtype=torch.float32)
        lib.timestep_sinusoid(ids, sin)
        add = torch.cat([text_embeds.to(self.device, torch.float32), sin.view(B, -1)], dim=1).contiguous()
        e1 = torch.empty(B, P["add1_w"].shape[0], device=self.device, dtype=torch.float32)
        lib.small_linear(add, P["add1_w"], e1, bias=P["add1_b"], silu_out=True)
        out = torch.empty_like(e1)
        lib.small_linear(e1, P["add2_w"], out, bias=P["add2_b"])
        return out

    @torch.no_grad()
    def time_embeddings(self, timesteps: List[int], batch: int, w_emb: Optional[torch.Tensor],
                        aug_emb: Optional[torch.Tensor] = None):
        """Per step: all ResnetBlock2D time projections, fp32 [B, temb_total].
        aug_emb: SDXL addition embedding, added to the time embedding (`emb = emb + aug_emb`)."""
        P = self.P
        ch0 = self.cfg.block_out_channels[0]
        out = []
        for t in timesteps:
            tt = torch.full((batch,), float(t), device=self.device, dtype=torch.float32)
            sin = torch.empty(batch, ch0, device=self.device, dtype=torch.float32)
            lib.timestep_sinusoid(tt, sin)
            if P["cond_w"] is not None and w_emb is not None:
                x = torch.empty_like(sin)
                lib.small_linear(w_emb, P["cond_w"], x, add=sin)
            else:
                x = sin
            e1 = torch.empty(batch, ch0 * 4, device=self.device, dtype=torch.float32)
            lib.small_linear(x, P["t1_w"], e1, bias=P["t1_b"], silu_out=True)
            emb = torch.empty_like(e1)
            # `emb` is only ever consumed as SiLU(emb) (ResnetBlock2D.time_emb_proj): apply it once
            # here instead of once per output column of the 20160-wide projection
            lib.small_linear(e1, P["t2_w"], emb, bias=P["t2_b"], add=aug_emb, silu_out=True)
            temb = torch.empty(batch, P["temb_total"], device=self.device, dtype=torch.float32)
            lib.small_linear(emb, P["temb_w"], temb, bias=P["temb_b"])
            out.append(temb)
        return out

    @torch.no_grad()
    def forward(self, latents_nhwc: torch.Tensor, temb: torch.Tensor, kvs: List[List[torch.Tensor]],
                eps_out: Optional[torch.Tensor] = None, repeat: int = 1, comm=None, inpaint_cond=None,
                in_scale: float = 1.0) -> torch.Tensor:
        """latents_nhwc fp32 [b,h,w,4] -> noise_pred fp32 [b*repeat,h,w,4].  repeat=2 is the
        classifier-free-guidance doubled batch `cat([latents]*2)`: the same latents are packed
        twice, temb / kvs carry the [uncond, cond] halves.

        inpaint_cond (a 9-channel inpainting UNet, and only there): (latent mask fp32 [b,h,w], masked_image_latents
        fp32 NHWC [b,h,w,4]); the UNet input is cat([latents, mask, masked_image_latents]) per image, doubled
        together with the latents under guidance.

        in_scale: the samplers' `scale_model_input` (Euler: 1 / sqrt(sigma^2 + 1)), applied as the latents are packed.

        comm (patch parallel, SURVEY.md §8e): this rank computes rows
        [rank*h/R, (rank+1)*h/R) of every image and returns that strip [b*repeat, h/R, w, 4];
        latents_nhwc is still the full latent (it is tiny and every rank holds it)."""
        P = self.P
        b0, H, W, Cin = latents_nhwc.shape
        B = b0 * repeat
        if comm is not None and self.dt != BF16:
            raise RuntimeError("patch parallel runs on the bf16 path only (the split GroupNorm kernels have no "
                               "fp32 variant); the fp32 precision mode is a one-GPU parity mode")
        if comm is not None and inpaint_cond is not None:
            raise RuntimeError("patch parallel does not implement the inpainting conditioning (9-channel conv_in)")
        cin_model = getattr(self.cfg, "in_channels", 4)
        if cin_model == 9 and inpaint_cond is None:
            raise RuntimeError("this UNet has in_channels=9 (an inpainting UNet): it needs the mask and the masked "
                               "image latents; text-to-image and image-to-image are not defined for it")
        if cin_model != 9 and inpaint_cond is not None:
            raise RuntimeError(f"inpaint_cond is the input of a 9-channel UNet, this one has in_channels={cin_model}")
        g = self.groups
        # GroupNorm statistics from the producers' epilogues (per-channel records): every GroupNorm of the
        # UNet becomes finalize + ONE pass; DL_UNET_GN_FUSE=0 keeps the cooperative two-phase kernel (A/B)
        ctx = _Ctx(self.device, B, comm, gn_fuse=g if self.fuse_gn_stats else 0, dt=self.dt, ln_fold=self.fold_ln)
        ch = self.cfg.block_out_channels
        kv_it = iter(kvs)
        if comm is None:
            xin = ctx.empty(B, H, W, 64)
            if inpaint_cond is not None:
                lib.pack_latent_inpaint(latents_nhwc, inpaint_cond[0], inpaint_cond[1], xin, repeat=repeat)
            else:
                for r in range(repeat):
                    lib.pack_latent(latents_nhwc, xin[r * b0:(r + 1) * b0], cin=Cin, scale=in_scale)
        else:
            n_lv = len(ch)
            if H % (comm.world << (n_lv - 1)):
                raise RuntimeError(f"patch parallel: {H} latent rows do not split into {comm.world} strips "
                                   f"of a multiple of {1 << (n_lv - 1)} rows")
            hl = H // comm.world
            r0 = comm.rank * hl
            lo, hi = max(r0 - 1, 0), min(r0 + hl + 1, H)      # strip + halo rows inside the image
            xp = torch.zeros(B, hl + 2, W, 64, device=self.device, dtype=self.dt)
            for r in range(repeat):
                for i in range(b0):
                    lib.pack_latent(latents_nhwc[i, lo:hi], xp[r * b0 + i, lo - (r0 - 1):hi - (r0 - 1)], cin=Cin,
                                    scale=in_scale)
            xin = Padded(xp)
            H = hl
        h = conv3x3(ctx, xin, P["conv_in_w"], P["conv_in_b"], ch[0], feeds_norm=True)
        skips = [h]
        for blk in P["down"]:
            for j, r in enumerate(blk["resnets"]):
                h = resnet(ctx, h, r, temb=temb, groups=g)
                if blk["attns"]:
                    h = transformer(ctx, h, blk["attns"][j], next(kv_it), groups=g)
                skips.append(h)
            if blk["down"] is not None:
                h = downsample(ctx, h, blk["down"])
                skips.append(h)
        h = resnet(ctx, h, P["mid"]["resnets"][0], temb=temb, groups=g)
        h = transformer(ctx, h, P["mid"]["attns"][0], next(kv_it), groups=g)
        h = resnet(ctx, h, P["mid"]["resnets"][1], temb=temb, groups=g)
        for blk in P["up"]:
            for j, r in enumerate(blk["resnets"]):
                h = resnet(ctx, h, r, temb=temb, x1=skips.pop(), groups=g)
                if blk["attns"]:
                    h = transformer(ctx, h, blk["attns"][j], next(kv_it), groups=g)
            if blk["up"] is not None:
                h = upsample(ctx, h, blk["up"])
        hn = groupnorm(ctx, h, P["norm_out_w"], P["norm_out_b"], eps=1e-5, silu=True, groups=g, halo=True)
        cout = getattr(self.cfg, "out_channels", Cin)
        if eps_out is None:
            eps_out = torch.empty(B, H, W, cout, device=self.device, dtype=torch.float32)
        conv3x3(ctx, hn, P["conv_out_w"], P["conv_out_b"], cout, mode=lib.EPI_F32, out=eps_out, ldo=cout)
        return eps_out


# ------------------------------------------------------------------------------------------------
# VAE mid-block attention (shared by the encoder and the decoder)
# ------------------------------------------------------------------------------------------------
def _vae_flash_ok(flash, sq, skv, C):
    return flash and sq % 128 == 0 and skv % 64 == 0 and C % 128 == 0 and C <= 512


def vae_mid_attention(ctx, x, a: Packed, *, groups: int, flash: bool):
    """AutoencoderKL mid-block attention (encoder and decoder): heads=1, d=C (512).  Token counts the wide flash
    kernel tiles (multiples of 128: every full decode) go through it; otherwise QK^T and PV through the tcgen05 GEMM with fp32 scores per image, or the CUDA-core
    flash kernel for ragged tiles."""
    B, H, W, C = x.shape
    S = H * W
    hn = groupnorm(ctx, x, a["norm_w"], a["norm_b"], eps=1e-6, silu=False, groups=groups)
    hn2 = hn.view(B * S, C)
    if ctx.comm is not None:
        return _vae_mid_attention_strips(ctx, x, hn2, a, flash)
    qk = linear(ctx, hn2, a["qk_w"], a["qk_b"], 2 * C)                 # [B*S, 2C]
    o = ctx.empty(B * S, C)
    if _vae_flash_ok(flash, S, S, C):
        # b_v is folded into the out-proj bias (softmax rows sum to 1), as in the other branches
        v = linear(ctx, hn2, a["v_w"], None, C)
        lib.attention_wide(qk, qk[:, C:], v, o, batch=B, sq=S, skv=S, d=C, ldq=2 * C, ldk=2 * C, ldv=C, ldo=C,
                           scale=1.0 / math.sqrt(C))
        out = linear(ctx, o, a["o_w"], a["o_b"], C, residual=x.view(B * S, C), norm_rows_per_img=S)
        return _carry_gn(out, out.view(B, H, W, C))
    if S % 64 or ctx.dt != BF16:
        # fp32 precision mode, and ragged tiles of a tiled decode (token count not a multiple of the 64-deep GEMM K
        # chunk, e.g. a 29 x 29 corner tile): the CUDA-core flash kernel takes any length.
        # b_v is folded into the out-proj bias exactly as below (softmax rows sum to 1).
        v = linear(ctx, hn2, a["v_w"], None, C)
        lib.attention(qk, qk[:, C:], v, o, batch=B, sq=S, skv=S, heads=1, d=C, dh_stride=C,
                      ldq=2 * C, ldk=2 * C, ldv=C, ldo=C, scale=1.0 / math.sqrt(C), impl=lib.ATTN_SIMT)
        out = linear(ctx, o, a["o_w"], a["o_b"], C, residual=x.view(B * S, C))
        return out.view(B, H, W, C)
    scores = ctx.empty(S, S, dtype=torch.float32)
    probs = ctx.empty(S, S)
    vt = ctx.empty(C, S)
    for b in range(B):
        rows = slice(b * S, (b + 1) * S)
        # V^T[c, s] = sum_k Wv[c,k] X[s,k]  (bias folded into the out-proj bias)
        lib.igemm(a["v_w"], hn2[rows], vt, nimg=1, h=1, w=C, taps=1, n=S, a0_stride=C, ldo=S)
        q, k = qk[rows, :C], qk[rows, C:]
        lib.igemm(q, k, scores, nimg=1, h=1, w=S, taps=1, n=S, c0=C, a0_stride=2 * C,
                  mode=lib.EPI_F32, alpha=1.0 / math.sqrt(C), ldo=S)
        lib.softmax_rows(scores, probs)
        lib.igemm(probs, vt, o[rows], nimg=1, h=1, w=S, taps=1, n=C, a0_stride=S, ldo=C)
    out = linear(ctx, o, a["o_w"], a["o_b"], C, residual=x.view(B * S, C), norm_rows_per_img=S)
    return _carry_gn(out, out.view(B, H, W, C))


def _vae_mid_attention_strips(ctx, x, hn2, a: Packed, flash: bool):
    """Row strips (SURVEY.md §8e, VAE row): the queries of this rank's S tokens attend to the
    keys / values of all R*S tokens.  ONE exchange: the normalised tokens are all-gathered
    (rank order = image row order) and every rank projects K and V^T from them itself — the
    two projections are 2*R*S*C^2 MACs, far cheaper than a second and third gather."""
    B, H, W, C = x.shape
    S = H * W
    comm = ctx.comm
    hn_all = comm.gather_rows(hn2.view(B, S, C))                        # [B, R*S, C]
    Sa = hn_all.shape[1]
    hn_all = hn_all.reshape(B * Sa, C)
    scale = 1.0 / math.sqrt(C)
    q = linear(ctx, hn2, a["qk_w"][:C], a["qk_b"][:C], C)               # [B*S, C]
    k = linear(ctx, hn_all, a["qk_w"][C:], a["qk_b"][C:], C)            # [B*Sa, C]
    o = ctx.empty(B * S, C)
    if _vae_flash_ok(flash, S, Sa, C):
        v = linear(ctx, hn_all, a["v_w"], None, C)
        lib.attention_wide(q, k, v, o, batch=B, sq=S, skv=Sa, d=C, ldq=C, ldk=C, ldv=C, ldo=C, scale=scale)
    elif Sa % 64:                     # ragged key count: the CUDA-core flash kernel takes any length
        v = linear(ctx, hn_all, a["v_w"], None, C)
        lib.attention(q, k, v, o, batch=B, sq=S, skv=Sa, heads=1, d=C, dh_stride=C,
                      ldq=C, ldk=C, ldv=C, ldo=C, scale=scale, impl=lib.ATTN_SIMT)
    else:
        scores = ctx.empty(S, Sa, dtype=torch.float32)
        probs = ctx.empty(S, Sa)
        vt = ctx.empty(C, Sa)
        for b in range(B):
            rows, keys = slice(b * S, (b + 1) * S), slice(b * Sa, (b + 1) * Sa)
            lib.igemm(a["v_w"], hn_all[keys], vt, nimg=1, h=1, w=C, taps=1, n=Sa, a0_stride=C, ldo=Sa)
            lib.igemm(q[rows], k[keys], scores, nimg=1, h=1, w=S, taps=1, n=Sa, c0=C, a0_stride=C,
                      mode=lib.EPI_F32, alpha=scale, ldo=Sa)
            lib.softmax_rows(scores, probs)
            lib.igemm(probs, vt, o[rows], nimg=1, h=1, w=S, taps=1, n=C, a0_stride=Sa, ldo=C)
    out = linear(ctx, o, a["o_w"], a["o_b"], C, residual=x.view(B * S, C))
    return out.view(B, H, W, C)


# ------------------------------------------------------------------------------------------------
# VAE decoder
# ------------------------------------------------------------------------------------------------
class VAEDecoderB200:
    def __init__(self, state_dict, cfg, device="cuda:0", precision="bf16"):
        lib.require_cuda()
        lib.load()
        self.device = torch.device(device)
        self.cfg = cfg
        self.dt = _dt_of(precision)
        from .weights import pack_dtype
        with pack_dtype(self.dt):
            self.P = pack_vae_decoder(state_dict, cfg, self.device)
        self.groups = cfg.norm_num_groups
        import os
        self.fuse_gn_stats = os.environ.get("DL_VAE_GN_FUSE", "1") not in ("0", "false")
        self.conv_out_tapsum = (os.environ.get("DL_VAE_CONV_OUT_TAPSUM", "1") not in ("0", "false")
                                and self.dt == BF16 and self.P["conv_out_w"].shape[0] == 3)
        # flash attention for the mid block (csrc/attention_wide.cu); DL_VAE_FLASH=0 keeps the unfused GEMM form
        self.flash_attention = os.environ.get("DL_VAE_FLASH", "1") not in ("0", "false") and self.dt == BF16
        if self.conv_out_tapsum:
            # conv_out weights regrouped tap-major for the 1x1-GEMM + tap-sum form: row t*3 + oc = w[oc, tap t, :]
            cl = self.P["conv_out_w"].shape[1] // 9
            w27 = self.P["conv_out_w"].view(3, 9, cl).permute(1, 0, 2).reshape(27, cl)
            self.P["conv_out_w27"] = torch.cat([w27, w27.new_zeros(5, cl)], 0).contiguous()

    @torch.no_grad()
    def decode(self, latents_nhwc: torch.Tensor, out_u8: Optional[torch.Tensor] = None,
               tiling: bool = False) -> torch.Tensor:
        """latents fp32 NHWC [B,h,w,4] (un-scaled, as the scheduler leaves them) -> u8 [B,8h,8w,3].
        tiling: `vae.enable_tiling()` semantics (reference `backends/cuda_worker.py:91`): latents
        larger than sample_size/8 in either dim are decoded tile by tile and blended."""
        t = self.cfg.sample_size // 8
        if tiling and (latents_nhwc.shape[1] > t or latents_nhwc.shape[2] > t):
            return self.tiled_decode(latents_nhwc, out_u8)
        return self._decode(latents_nhwc, out_u8)

    @torch.no_grad()
    def tiled_decode(self, latents_nhwc: torch.Tensor, out_u8: Optional[torch.Tensor] = None) -> torch.Tensor:
        """diffusers `AutoencoderKL.tiled_decode` (SURVEY.md App. A.4): tiles of sample_size/8
        latents at stride 0.75 tile, each decoded on its own (own GroupNorm statistics and
        attention), blended over sample_size/4 pixels with the already blended upper / left
        neighbour, cropped to 0.75 sample_size and written into the canvas."""
        B, H, W, _ = latents_nhwc.shape
        tl = self.cfg.sample_size // 8
        stride = int(tl * (1 - 0.25))
        blend = int(self.cfg.sample_size * 0.25)
        limit = self.cfg.sample_size - blend
        if out_u8 is None:
            out_u8 = torch.empty(B, 8 * H, 8 * W, 3, device=self.device, dtype=torch.uint8)
        prev_row = []
        oy = 0
        for i in range(0, H, stride):
            row = []
            ox = 0
            for jn, j in enumerate(range(0, W, stride)):
                tile = self._decode(latents_nhwc[:, i:i + tl, j:j + tl].contiguous(), f32_out=True)
                if i > 0:
                    up = prev_row[jn]
                    lib.tile_blend(up, tile, min(up.shape[1], tile.shape[1], blend), vertical=True)
                if jn > 0:
                    left = row[jn - 1]
                    lib.tile_blend(left, tile, min(left.shape[2], tile.shape[2], blend), vertical=False)
                row.append(tile)
                ch, cw = min(limit, tile.shape[1]), min(limit, tile.shape[2])
                lib.image_crop_u8(tile, ch, cw, out_u8[:, oy:, ox:])
                ox += cw
            prev_row = row
            oy += min(limit, row[0].shape[1])
        return out_u8

    @torch.no_grad()
    def decode_strips(self, latents_nhwc: torch.Tensor, comm, f32_out: bool = False) -> torch.Tensor:
        """One image decoded by all ranks of `comm` (a patch_parallel.StripComm), SURVEY.md §8e
        "VAE decode in C5": rank r owns latent rows [r*H/R, (r+1)*H/R) and therefore 8x as many
        pixel rows at the output.  Same kernels as the one-GPU decode; exchanges: one halo row to
        each neighbour in front of every 3x3 conv (the upsample convs included), the per-(image,
        group) GroupNorm records, the mid-block attention tokens (`_mid_attention_strips`), and at
        the end the pixel rows (3 bytes / pixel).  latents: the FULL fp32 NHWC latent, identical on
        every rank (as `PatchParallelDenoiser.denoise` leaves it).  -> the full u8 (or fp32)
        image [B,8H,8W,3] on every rank."""
        B, H, W, _ = latents_nhwc.shape
        R = comm.world
        if self.dt != BF16:
            raise RuntimeError("strip decode runs on the bf16 path only (the split GroupNorm kernels have no "
                               "fp32 variant); the fp32 precision mode is a one-GPU parity mode")
        if H % R:
            raise RuntimeError(f"strip decode: {H} latent rows do not split into {R} strips")
        hl = H // R
        mine = latents_nhwc[:, comm.rank * hl:(comm.rank + 1) * hl].contiguous()
        strip = self._decode(mine, f32_out=f32_out, comm=comm)                # [B, 8*hl, 8W, 3]
        return comm.gather_rows(strip)

    @torch.no_grad()
    def _decode(self, latents_nhwc: torch.Tensor, out_u8: Optional[torch.Tensor] = None,
                f32_out: bool = False, comm=None) -> torch.Tensor:
        """One untiled decode.  Fuses `/ scaling_factor`, post_quant_conv and (u8 output) the
        VaeImageProcessor denormalise; f32_out returns the decoder output fp32 [B,8h,8w,3].
        comm: latents_nhwc is this rank's row strip (see `decode_strips`), so is the result."""
        P = self.P
        B, H, W, Cin = latents_nhwc.shape
        g = self.groups
        ctx = _Ctx(self.device, B, comm=comm, gn_fuse=g if self.fuse_gn_stats else 0, dt=self.dt)
        ch = self.cfg.block_out_channels
        z = ctx.empty(B, H, W, 64)
        lib.pack_latent(latents_nhwc, z, cin=Cin, scale=1.0 / self.cfg.scaling_factor,
                        mat=P["pq_w"], vec=P["pq_b"])
        # `/ scaling_factor` is computed as a multiply by the fp32 reciprocal
        if comm is not None:
            z = ctx.pad_rows(z)
        h = conv3x3(ctx, z, P["conv_in_w"], P["conv_in_b"], ch[-1], feeds_norm=True)
        h = resnet(ctx, h, P["mid_res"][0], eps=1e-6, groups=g)
        h = vae_mid_attention(ctx, h, P["mid_attn"], groups=g, flash=self.flash_attention)
        h = resnet(ctx, h, P["mid_res"][1], eps=1e-6, groups=g)
        for blk in P["up"]:
            for r in blk["resnets"]:
                h = resnet(ctx, h, r, eps=1e-6, groups=g)
            if blk["up"] is not None:
                h = upsample(ctx, h, blk["up"])
        hn = groupnorm(ctx, h, P["norm_out_w"], P["norm_out_b"], eps=1e-6, silu=True, groups=g,
                       halo=comm is not None)
        Bo, Ho, Wo, Cl = h.shape
        if comm is None and self.dt == BF16 and self.conv_out_tapsum:
            # conv_out (C -> 3) as ONE 1x1 GEMM over the input (27 tap-major partial products per pixel, input
            # read once) + a tap-sum kernel with the image tail, instead of a 3x3 implicit GEMM with a 16-wide
            # N tile that re-reads the 1 GB input nine times at 2 % of the tensor peak
            y = ctx.empty(Bo, Ho, Wo, 32, dtype=torch.float32)
            lib.igemm(hn, P["conv_out_w27"], y, nimg=Bo, h=Ho, w=Wo, taps=1, n=32, mode=lib.EPI_F32, ldo=32)
            img = (torch.empty(Bo, Ho, Wo, 3, device=self.device, dtype=torch.float32) if f32_out else
                   (out_u8 if out_u8 is not None else torch.empty(Bo, Ho, Wo, 3, device=self.device, dtype=torch.uint8)))
            lib.conv_tapsum(y, P["conv_out_b"], img)
            return img
        if f32_out:
            img = torch.empty(Bo, Ho, Wo, 3, device=self.device, dtype=torch.float32)
            conv3x3(ctx, hn, P["conv_out_w"], P["conv_out_b"], 3, mode=lib.EPI_F32, out=img, ldo=3)
            return img
        if out_u8 is None:
            out_u8 = torch.empty(Bo, Ho, Wo, 3, device=self.device, dtype=torch.uint8)
        conv3x3(ctx, hn, P["conv_out_w"], P["conv_out_b"], 3, mode=lib.EPI_U8_IMAGE, out=out_u8, ldo=3)
        return out_u8


class TAESDDecoderB200:
    """The tiny autoencoder's decoder (diffusers `AutoencoderTiny`, `madebyollin/taesd` / `taesdxl`): 64-channel
    conv3x3 layers only, no GroupNorm, no attention.  `dl_taesd_latent_in` computes `tanh(x / 3) * 3` into the
    first conv's operand; every conv followed by a ReLU stores through the igemm's DL_EPI_BF16_RELU epilogue, a
    Block's last conv with its skip added on the tensor core first (relu(conv + b + x)); the upsamples are the
    four-phase folded convs of the KL decoder without bias; the output map `x * 2 - 1` is folded into the final
    conv's weights (`weights.taesd_conv_out_fold`), so the u8 tail is the KL decoder's.  Always untiled: its working
    set is 64 channels (~32 MB per 512x512 image in bf16); diffusers' `AutoencoderTiny._tiled_decode` is not
    restated.  Same interface as `VAEDecoderB200` (`decode`, `_decode`)."""

    def __init__(self, state_dict, cfg, device="cuda:0", precision="bf16"):
        lib.require_cuda()
        lib.load()
        self.device = torch.device(device)
        self.cfg = cfg
        self.dt = _dt_of(precision)
        ch = tuple(cfg.decoder_block_out_channels)
        if (cfg.latent_channels != 4 or cfg.out_channels != 3 or cfg.act_fn != "relu" or cfg.upsample_fn != "nearest"
                or cfg.upsampling_scaling_factor != 2 or cfg.scaling_factor != 1.0 or len(set(ch)) != 1
                or ch[0] % 64 or len(ch) != len(cfg.num_decoder_blocks)):
            raise RuntimeError(f"AutoencoderTiny decoder: only latent_channels=4, out_channels=3, act_fn=relu, nearest "
                               f"2x upsampling, scaling_factor=1.0 and one width (a multiple of 64) for every level are "
                               f"built, got {vars(cfg) if hasattr(cfg, '__dict__') else cfg}")
        self.ch = ch[0]
        from .weights import pack_dtype
        with pack_dtype(self.dt):
            self.P = pack_taesd_decoder(state_dict, cfg, self.device)
        # final conv (64 -> 3): a 3x3 implicit GEMM with the u8 epilogue (False), or one 1x1 GEMM with 27 tap-major
        # partial products per pixel + the tap-sum kernel with the u8 tail (True, bf16 only).  At 64 input channels
        # the first is faster (B = 16 at 512x512 on a B200 at 1000 W: 4.48 against 4.93 ms per decode);
        # tools/bench_taesd.py times both
        self.conv_out_tapsum = False

    @torch.no_grad()
    def decode(self, latents_nhwc: torch.Tensor, out_u8: Optional[torch.Tensor] = None,
               tiling: bool = False) -> torch.Tensor:
        """latents fp32 NHWC [B,h,w,4] -> u8 [B,8h,8w,3].  tiling is accepted for the `VAEDecoderB200` interface and
        ignored: this decoder always decodes untiled."""
        return self._decode(latents_nhwc, out_u8)

    @torch.no_grad()
    def _decode(self, latents_nhwc: torch.Tensor, out_u8: Optional[torch.Tensor] = None,
                f32_out: bool = False) -> torch.Tensor:
        """One decode; f32_out returns the decoder output (x * 2 - 1 applied) fp32 [B,8h,8w,3]."""
        P, C = self.P, self.ch
        B, H, W, _ = latents_nhwc.shape
        ctx = _Ctx(self.device, B, dt=self.dt)
        relu = lib.EPI_BF16_RELU
        z = ctx.empty(B, H, W, 64)
        lib.taesd_latent_in(latents_nhwc.contiguous(), z)
        h = conv3x3(ctx, z, P["conv_in_w"], P["conv_in_b"], C, mode=relu)
        for lev in P["levels"]:
            for blk in lev["blocks"]:
                a = conv3x3(ctx, h, blk["w0"], blk["b0"], C, mode=relu)
                a = conv3x3(ctx, a, blk["w1"], blk["b1"], C, mode=relu)
                h = conv3x3(ctx, a, blk["w2"], blk["b2"], C, residual=h, mode=relu)
            if lev["up"] is not None:
                h = upsample(ctx, h, lev["up"])
        Bo, Ho, Wo, _ = h.shape
        if self.conv_out_tapsum and self.dt == BF16:
            y = ctx.empty(Bo, Ho, Wo, 32, dtype=torch.float32)
            lib.igemm(h, P["conv_out_w27"], y, nimg=Bo, h=Ho, w=Wo, taps=1, n=32, mode=lib.EPI_F32, ldo=32)
            img = (torch.empty(Bo, Ho, Wo, 3, device=self.device, dtype=torch.float32) if f32_out else
                   (out_u8 if out_u8 is not None else torch.empty(Bo, Ho, Wo, 3, device=self.device, dtype=torch.uint8)))
            lib.conv_tapsum(y, P["conv_out_b"], img)
            return img
        if f32_out:
            img = torch.empty(Bo, Ho, Wo, 3, device=self.device, dtype=torch.float32)
            conv3x3(ctx, h, P["conv_out_w"], P["conv_out_b"], 3, mode=lib.EPI_F32, out=img, ldo=3)
            return img
        if out_u8 is None:
            out_u8 = torch.empty(Bo, Ho, Wo, 3, device=self.device, dtype=torch.uint8)
        conv3x3(ctx, h, P["conv_out_w"], P["conv_out_b"], 3, mode=lib.EPI_U8_IMAGE, out=out_u8, ldo=3)
        return out_u8


# ------------------------------------------------------------------------------------------------
# VAE encoder (image-to-image)
# ------------------------------------------------------------------------------------------------
class VAEEncoderB200:
    """`AutoencoderKL.encode` up to the posterior's moments: encoder + quant_conv, untiled or tiled
    (`enable_tiling()`).  The u8 image goes straight into conv_in's im2col operand (`dl_pack_image_im2col`),
    conv_in runs as a 1x1 GEMM with K = 64, Downsample2D(padding=0) through `dl_im2col_s2_pad01`, quant_conv
    in fp32 in the latent-packing kernel.  Moments are fp32 NHWC [B, H/8, W/8, 2 * latent_channels]."""

    def __init__(self, state_dict, cfg, device="cuda:0", precision="bf16"):
        lib.require_cuda()
        lib.load()
        self.device = torch.device(device)
        self.cfg = cfg
        self.dt = _dt_of(precision)
        if cfg.latent_channels != 4:
            raise RuntimeError(f"VAE encoder: latent_channels={cfg.latent_channels}, only 4 is implemented")
        from .weights import pack_dtype
        with pack_dtype(self.dt):
            self.P = pack_vae_encoder(state_dict, cfg, self.device)
        self.groups = cfg.norm_num_groups
        import os
        self.fuse_gn_stats = os.environ.get("DL_VAE_GN_FUSE", "1") not in ("0", "false")
        self.flash_attention = os.environ.get("DL_VAE_FLASH", "1") not in ("0", "false") and self.dt == BF16

    @torch.no_grad()
    def moments(self, img_u8: torch.Tensor, tiling: bool = False, comm=None, mask=None,
                keep_unmasked: bool = False) -> torch.Tensor:
        """img_u8: u8 NHWC [B,H,W,3] on the device (H, W multiples of 8).  tiling: images larger than
        sample_size in either dim are encoded tile by tile and blended (`tiled_encode`).
        mask (inpainting): u8 [B,H,W]; the masked images (pixels with m >= 128 at 0.0) are encoded instead, or,
        with keep_unmasked, after the unmasked ones in one batch of 2B: moments [2B, ...] = [image; masked image]."""
        if comm is not None:
            raise RuntimeError("VAE encoder: strip-parallel encode is not implemented")
        t = self.cfg.sample_size
        if tiling and (img_u8.shape[1] > t or img_u8.shape[2] > t):
            return self.tiled_moments(img_u8, mask, keep_unmasked)
        return self._encode(img_u8, mask, keep_unmasked)

    @torch.no_grad()
    def tiled_moments(self, img_u8: torch.Tensor, mask=None, keep_unmasked: bool = False) -> torch.Tensor:
        """diffusers `AutoencoderKL.tiled_encode`: tiles of sample_size pixels at stride 0.75 tile, each encoded
        on its own (own GroupNorm statistics and attention, zero padding at the tile border), moments blended
        over sample_size/32 latents with the already blended upper / left neighbour, cropped to 0.75 of a tile
        and written into the result."""
        B, H, W, _ = img_u8.shape
        t = self.cfg.sample_size
        stride = int(t * (1 - 0.25))
        tl = t // 8
        blend = int(tl * 0.25)
        limit = tl - blend
        nb = 2 * B if mask is not None and keep_unmasked else B
        out = torch.empty(nb, H // 8, W // 8, 2 * self.cfg.latent_channels, device=self.device, dtype=torch.float32)
        prev_row = []
        oy = 0
        for i in range(0, H, stride):
            row = []
            ox = 0
            for jn, j in enumerate(range(0, W, stride)):
                tile = self._encode(img_u8[:, i:i + t, j:j + t],          # views: read in place
                                    None if mask is None else mask[:, i:i + t, j:j + t], keep_unmasked)
                if i > 0:
                    up = prev_row[jn]
                    lib.tile_blend(up, tile, min(up.shape[1], tile.shape[1], blend), vertical=True)
                if jn > 0:
                    left = row[jn - 1]
                    lib.tile_blend(left, tile, min(left.shape[2], tile.shape[2], blend), vertical=False)
                row.append(tile)
                ch, cw = min(limit, tile.shape[1]), min(limit, tile.shape[2])
                out[:, oy:oy + ch, ox:ox + cw].copy_(tile[:, :ch, :cw])
                ox += cw
            prev_row = row
            oy += min(limit, row[0].shape[1])
        return out

    def _downsample(self, ctx, x, p: Packed):
        """Downsample2D(padding=0): F.pad(x, (0,1,0,1)) + conv3x3 stride 2, as im2col + GEMM."""
        B, H, W, C = x.shape
        cols = ctx.empty(B * (H // 2) * (W // 2), 9 * C)
        lib.im2col_s2_pad01(x, cols, nimg=B, h=H, w=W)
        out = linear(ctx, cols, p["w"], p["b"], C, norm_rows_per_img=(H // 2) * (W // 2))
        return _carry_gn(out, out.view(B, H // 2, W // 2, C))

    @torch.no_grad()
    def _encode(self, img_u8: torch.Tensor, mask=None, keep_unmasked: bool = False) -> torch.Tensor:
        """One untiled encode (img_u8 and mask may be windows of a larger canvas)."""
        P = self.P
        B0, H, W, _ = img_u8.shape
        if H % 8 or W % 8:
            raise RuntimeError(f"VAE encoder: image {W}x{H} is not a multiple of 8")
        B = 2 * B0 if mask is not None and keep_unmasked else B0
        g = self.groups
        ctx = _Ctx(self.device, B, gn_fuse=g if self.fuse_gn_stats else 0, dt=self.dt)
        ch = self.cfg.block_out_channels
        cols = ctx.empty(B * H * W, 64)
        if mask is None or keep_unmasked:
            lib.pack_image_im2col(img_u8, cols[:B0 * H * W])
        if mask is not None:
            lib.pack_image_im2col(img_u8, cols[(B - B0) * H * W:], mask=mask)
        h = linear(ctx, cols, P["conv_in_w"], P["conv_in_b"], ch[0], norm_rows_per_img=H * W)
        h = _carry_gn(h, h.view(B, H, W, ch[0]))
        for blk in P["down"]:
            for r in blk["resnets"]:
                h = resnet(ctx, h, r, eps=1e-6, groups=g)
            if blk["down"] is not None:
                h = self._downsample(ctx, h, blk["down"])
        h = resnet(ctx, h, P["mid_res"][0], eps=1e-6, groups=g)
        h = vae_mid_attention(ctx, h, P["mid_attn"], groups=g, flash=self.flash_attention)
        h = resnet(ctx, h, P["mid_res"][1], eps=1e-6, groups=g)
        hn = groupnorm(ctx, h, P["norm_out_w"], P["norm_out_b"], eps=1e-6, silu=True, groups=g)
        Bo, Ho, Wo, _ = h.shape
        m = P["q_w"].shape[0]
        raw = torch.empty(Bo, Ho, Wo, m, device=self.device, dtype=torch.float32)
        conv3x3(ctx, hn, P["conv_out_w"], P["conv_out_b"], m, mode=lib.EPI_F32, out=raw, ldo=m)
        mom = torch.empty_like(raw)
        lib.pack_latent(raw, mom, cin=m, mat=P["q_w"], vec=P["q_b"])         # quant_conv, fp32
        return mom


# ------------------------------------------------------------------------------------------------
# pipeline: denoise loop + decode
# ------------------------------------------------------------------------------------------------
# Warm-up + capture of ALL pipelines of the process are serialised: the WorkerPool runs one worker thread
# per GPU in one process and every worker captures lazily on first use of a geometry.  The capture itself
# uses capture_error_mode="thread_local", so CUDA calls of the OTHER worker threads (caching-allocator
# cudaMalloc, event queries) neither fail with "operation not permitted when stream is capturing" nor
# invalidate this capture.
import threading as _threading

CAPTURE_LOCK = _threading.Lock()


def _pinned(x: torch.Tensor) -> torch.Tensor:
    """Host tensors -> page-locked staging (torch's caching host allocator; it keeps the block until the async copy
    that reads it has run); device tensors pass through."""
    return x.pin_memory() if x.device.type == "cpu" and not x.is_pinned() else x


class _StaticGraph:
    """One captured CUDA graph of the whole hot path for a fixed (B, h, w, steps[, gs][, strength][, inpaint]).
    strength set: image-to-image; the init images and the posterior draw are static inputs too, and `lat`
    holds the add_noise draw.  inpaint: the masks and the masked image's posterior draw are static inputs as well,
    and `noise` holds one draw per non-final step of the truncated schedule.  sampler (text-to-image only): `noise`
    holds the draws the sampler consumes (none for the deterministic ones; a one-entry placeholder then)."""

    def __init__(self, pipe: "LCMPipelineB200", B, h, w, steps, cfg_scale=None, decode=True, strength=None,
                 inpaint=False, sampler="lcm"):
        dev = pipe.device
        ucfg = pipe.unet.cfg
        D = ucfg.cross_attention_dim
        Bc = 2 * B if cfg_scale is not None else B          # CFG: [uncond, cond] context rows
        self.pe = torch.zeros(Bc, 77, D, device=dev, dtype=pipe.dt)
        cd = ucfg.time_cond_proj_dim
        self.w_emb = torch.zeros(B, cd, device=dev, dtype=torch.float32) if cd else None
        self.add = None
        if pipe.unet.P["add1_w"] is not None:
            pdim = ucfg.projection_class_embeddings_input_dim - 6 * ucfg.addition_time_embed_dim
            self.add = (torch.zeros(Bc, pdim, device=dev, dtype=torch.float32),
                        torch.zeros(Bc, 6, device=dev, dtype=torch.float32))
        self.lat = torch.zeros(B, 4, h, w, device=dev, dtype=torch.float32)
        if sampler != "lcm":
            nd = pipe.schedule(steps, sampler=sampler).n_draws
        else:
            nd = (len(pipe.schedule(steps, strength, inpaint).timesteps) if inpaint else steps) - 1
        self.noise = torch.zeros(max(nd, 1), B, 4, h, w, device=dev, dtype=torch.float32)
        self.steps = steps
        self.init_u8 = self.eps_s = self.mask_u8 = self.eps_m = None
        if strength is not None:
            self.init_u8 = torch.zeros(B, 8 * h, 8 * w, 3, device=dev, dtype=torch.uint8)
            self.eps_s = torch.zeros(B, 4, h, w, device=dev, dtype=torch.float32)
        if inpaint:
            self.mask_u8 = torch.zeros(B, 8 * h, 8 * w, device=dev, dtype=torch.uint8)
            self.eps_m = torch.zeros(B, 4, h, w, device=dev, dtype=torch.float32)
        args = (self.pe, self.w_emb, self.lat, self.noise, steps)
        kw = dict(add=self.add, cfg_scale=cfg_scale, decode=decode, init_u8=self.init_u8, eps_s=self.eps_s,
                  strength=strength, mask_u8=self.mask_u8, eps_m=self.eps_m, sampler=sampler)
        with CAPTURE_LOCK:
            # warm-up on a side stream (lazy per-device init: smem attributes, module load)
            s = torch.cuda.Stream(device=dev)
            s.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(s):
                pipe.run_static(*args, **kw)
            torch.cuda.current_stream(dev).wait_stream(s)
            torch.cuda.synchronize(dev)
            self.graph = torch.cuda.CUDAGraph()
            n0 = lib.launch_count
            # an explicit capture stream on THIS device: torch.cuda.graph's default capture stream is one
            # class-wide stream created on whichever device captured first, so a second worker (another GPU,
            # same process) would capture on the wrong device
            # one memory pool for all graphs of a pipeline: they replay one at a time on the worker's thread, so
            # their intermediates may share addresses (a dozen private pools at SDXL 1024^2 is a lot of HBM)
            with torch.cuda.graph(self.graph, pool=pipe._graph_pool(), stream=s, capture_error_mode="thread_local"):
                self.img, self.final = pipe.run_static(*args, **kw)
            self.launches = lib.launch_count - n0        # native kernel launches per replay


class LCMPipelineB200:
    """The hot path as one object: `generate()` = n x (UNet + scheduler step) + VAE decode.

    SD1.5-LCM (guidance through the w-embedding, no CFG) and SDXL-class UNets (text_time
    micro-conditioning; classifier-free guidance on a doubled batch when guidance_scale > 1 and
    the UNet has no time_cond_proj — `StableDiffusionXLPipeline.__call__` behind reference
    `backends/cuda_worker.py:532`) share this loop."""

    def __init__(self, unet_sd, unet_cfg, vae_sd, vae_cfg, device="cuda:0", vae_tiling: bool = False,
                 precision: str = "bf16", vae_kind: str = "kl", scheduler_config: SchedulerConfig = DEFAULT_CONFIG):
        """vae_tiling: `pipe.vae.enable_tiling()` (the reference workers always switch it on,
        `backends/cuda_worker.py:91`): requests larger than the VAE's sample_size decode tiled.
        vae_kind: "kl" (`AutoencoderKL`) or "taesd" (`AutoencoderTiny`, decoder only, always untiled).
        scheduler_config: `LCMScheduler.from_config(model's scheduler config)` (`SchedulerConfig.load`); it is fixed
        for the pipeline, so its coefficients are baked into the captured graphs like the timesteps are."""
        if vae_kind not in ("kl", "taesd"):
            raise RuntimeError(f"vae_kind must be 'kl' or 'taesd', got {vae_kind!r}")
        scheduler_config.validate()
        self.scheduler_config = scheduler_config
        self.device = torch.device(device)
        self.precision = precision
        self.dt = _dt_of(precision)
        self.vae_kind = vae_kind
        self.unet = UNetB200(unet_sd, unet_cfg, device, precision)
        if vae_kind == "taesd":
            self.vae = TAESDDecoderB200(vae_sd, vae_cfg, device, precision)
            self.vae_encoder = None
        else:
            self.vae = VAEDecoderB200(vae_sd, vae_cfg, device, precision)
            # image-to-image needs the encoder half of the VAE; a VAE shipped without it still serves text-to-image
            self.vae_encoder = (VAEEncoderB200(vae_sd, vae_cfg, device, precision) if has_vae_encoder(vae_sd)
                                else None)
        self.vae_tiling = vae_tiling
        self._graphs = {}

    @property
    def is_sdxl(self) -> bool:
        return self.unet.P["add1_w"] is not None

    def _w_emb(self, B, guidance_scale):
        cd = self.unet.cfg.time_cond_proj_dim
        if not cd:
            return None
        gs = torch.as_tensor(guidance_scale, dtype=torch.float32).reshape(-1).expand(B)
        return guidance_scale_embedding(gs - 1.0, cd)           # host, fp32 [B, cd]

    def cfg_scale_for(self, guidance_scale) -> Optional[float]:
        """The CFG weight, or None when the pass is not classifier-free guided
        (`do_classifier_free_guidance = guidance_scale > 1 and time_cond_proj_dim is None`)."""
        if self.unet.cfg.time_cond_proj_dim:
            return None
        gs = torch.as_tensor(guidance_scale, dtype=torch.float32).reshape(-1)
        if gs.numel() > 1 and not bool((gs == gs[0]).all()):
            raise RuntimeError("classifier-free guidance needs one guidance_scale per batch")
        g = float(gs[0])
        return g if g > 1.0 else None

    @torch.no_grad()
    def run_static(self, pe_bf16, w_emb, lat_nchw, noise_nchw, steps: int, record: dict = None,
                   add=None, cfg_scale: Optional[float] = None, teacher=None, decode: bool = True,
                   init_u8=None, eps_s=None, strength: Optional[float] = None, mask_u8=None, eps_m=None,
                   sampler: str = "lcm"):
        """Everything on device, no host sync, graph-capturable.  Returns (u8 images, latents).
        pe_bf16 / add carry 2B rows ([uncond, cond]) when cfg_scale is set.
        init_u8 (image-to-image): u8 NHWC init images; the pass becomes encode -> posterior sample with eps_s ->
        add_noise at the first timestep of the strength schedule with lat_nchw as the noise -> denoise -> decode.
        mask_u8 (inpainting, with init_u8): u8 [B,H,W] masks; see `inpaint_latents`, eps_m is the masked image's
        posterior draw, the schedule is the truncated one and noise_nchw holds its non-final steps' draws."""
        B = lat_nchw.shape[0]
        Bu = 2 * B if cfg_scale is not None else B
        sched = self.schedule(steps, strength if init_u8 is not None else None, mask_u8 is not None, sampler)
        kvs = self.unet.encode_context(pe_bf16)
        aug = self.unet.addition_embedding(*add) if add is not None else None
        tembs = self.unet.time_embeddings(sched.timesteps, Bu, w_emb, aug)
        start = inpaint = None
        if mask_u8 is not None:
            start, inpaint = self.inpaint_latents(init_u8, mask_u8, eps_s, eps_m, lat_nchw, sched, record)
        elif init_u8 is not None:
            start = self.init_latents(init_u8, eps_s, lat_nchw, sched, record)
        lat = self.denoise(lat_nchw, noise_nchw, sched, kvs, tembs, record, cfg_scale=cfg_scale, teacher=teacher,
                           start_nhwc=start, inpaint=inpaint)
        if not decode:                   # latent-only callers (candidate scoring): no VAE pass at all
            return None, lat
        return self.vae.decode(lat, tiling=self.vae_tiling), lat

    def init_latents(self, init_u8, eps_s, eps_n, sched: LCMSchedule, record: dict = None) -> torch.Tensor:
        """`LatentConsistencyModelImg2ImgPipeline.prepare_latents`: moments of the init images, posterior sample
        mean + std * eps_s, times scaling_factor, then `add_noise` with eps_n at t0 = sched.timesteps[0], in one
        kernel.  -> fp32 NHWC latents [B, h, w, 4]."""
        enc = self.require_encoder()
        mom = enc.moments(init_u8, tiling=self.vae_tiling)
        B, h, w, _ = mom.shape
        x = torch.empty(B, h, w, 4, device=self.device, dtype=torch.float32)
        sa, sb = sched.add_noise_coeffs()
        lib.vae_sample_latents(mom, eps_s, eps_n, x, scaling_factor=self.vae.cfg.scaling_factor, sqrt_alpha=sa,
                               sqrt_one_minus_alpha=sb)
        if record is not None:
            record["moments"] = mom.permute(0, 3, 1, 2).clone()
            record["init_latents"] = x.permute(0, 3, 1, 2).clone()
        return x

    def inpaint_latents(self, init_u8, mask_u8, eps_s, eps_m, noise_nchw, sched: LCMSchedule, record: dict = None):
        """`StableDiffusionInpaintPipeline.prepare_latents` + `prepare_mask_latents`.  image_latents =
        scaling_factor * posterior sample (eps_s) of the image, only where diffusers computes it (a 4-channel UNet, or
        strength < 1); masked_image_latents likewise of the masked image (eps_m), for a 9-channel UNet only (a
        4-channel UNet never reads it).  Both encodes run as one batch.  The starting latents are the noise draw
        itself at strength 1, else add_noise(image_latents, noise, timesteps[0]).
        -> (starting latents fp32 NHWC [B,h,w,4], dict(cond=(mask, masked) for a 9-channel UNet or None,
        blend=(image_latents, noise NHWC, mask) for a 4-channel UNet or None)); mask is the fp32 latent mask [B,h,w]."""
        enc = self.require_encoder()
        nine = getattr(self.unet.cfg, "in_channels", 4) == 9
        need_img = not nine or sched.strength < 1.0
        B, H, W, _ = init_u8.shape
        h, w = H // 8, W // 8
        f32 = dict(device=self.device, dtype=torch.float32)
        sf = self.vae.cfg.scaling_factor
        mom = enc.moments(init_u8, tiling=self.vae_tiling, mask=mask_u8 if nine else None, keep_unmasked=need_img)
        mask = torch.empty(B, h, w, **f32)
        lib.inpaint_latent_mask(mask_u8, mask)
        noise = torch.empty(B, h, w, 4, **f32)
        lib.nchw_to_nhwc_f32(noise_nchw, noise)
        image = masked = None
        if need_img:          # (sqrt_alpha, sqrt_one_minus_alpha) = (1, 0): the scaled posterior sample itself
            image = torch.empty(B, h, w, 4, **f32)
            lib.vae_sample_latents(mom[:B], eps_s, eps_s, image, scaling_factor=sf, sqrt_alpha=1.0,
                                   sqrt_one_minus_alpha=0.0)
        if nine:
            masked = torch.empty(B, h, w, 4, **f32)
            lib.vae_sample_latents(mom[mom.shape[0] - B:], eps_m, eps_m, masked, scaling_factor=sf, sqrt_alpha=1.0,
                                   sqrt_one_minus_alpha=0.0)
        if sched.strength >= 1.0:            # is_strength_max: latents = noise * init_noise_sigma (1.0)
            start = noise
        else:
            start = torch.empty(B, h, w, 4, **f32)
            sa, sb = sched.add_noise_coeffs()
            lib.vae_sample_latents(mom[:B], eps_s, noise_nchw, start, scaling_factor=sf, sqrt_alpha=sa,
                                   sqrt_one_minus_alpha=sb)
        if record is not None:
            record["moments"] = mom.permute(0, 3, 1, 2).clone()
            record["mask"] = mask.clone()
            record["init_latents"] = start.permute(0, 3, 1, 2).clone()
            if image is not None:
                record["image_latents"] = image.permute(0, 3, 1, 2).clone()
            if masked is not None:
                record["masked_image_latents"] = masked.permute(0, 3, 1, 2).clone()
        return start, dict(cond=(mask, masked) if nine else None, blend=None if nine else (image, noise, mask))

    def schedule(self, steps: int, strength: Optional[float] = None, inpaint: bool = False, sampler: str = "lcm"):
        """The pass's schedule: text-to-image (strength None), image-to-image (re-spaced by strength) or
        inpainting (the full schedule truncated by strength).  sampler: "lcm" (`LCMSchedule`), or one of the
        guided-model samplers of `scheduler.SAMPLERS` (text-to-image only)."""
        cfg = self.scheduler_config
        if check_sampler(sampler) != "lcm":
            if strength is not None or inpaint:
                raise RuntimeError(f"sampler {sampler!r}: image-to-image and inpainting run the LCM sampler only")
            return sampler_schedule(sampler, steps, cfg)
        if inpaint:
            return LCMSchedule(steps, strength, truncate=True, config=cfg)
        return LCMSchedule(steps, config=cfg) if strength is None else LCMSchedule(steps, strength, config=cfg)

    def require_encoder(self) -> VAEEncoderB200:
        if self.vae_kind == "taesd":
            raise RuntimeError("image-to-image and inpainting need a VAE encoder, and this model's VAE is the tiny "
                               "autoencoder (AutoencoderTiny): its encoder is not built, only its decoder")
        if self.vae_encoder is None:
            raise RuntimeError("image-to-image and inpainting need the VAE encoder, and this model's VAE has no "
                               "encoder weights (encoder.* / quant_conv.*)")
        return self.vae_encoder

    max_graphs = 12       # captured geometries kept per pipeline
    # batch sizes a CUDA graph is captured for: a request batch is padded up to the next one (micro-batching
    # produces every B in 1..16; one graph per exact B would thrash the LRU and re-capture constantly)
    batch_buckets = (1, 2, 4, 8, 16)

    def _graph_pool(self):
        if getattr(self, "_pool", None) is None:
            self._pool = torch.cuda.graph_pool_handle()
        return self._pool

    def graph_for(self, B, h, w, steps, cfg_scale=None, decode=True, strength=None, inpaint=False,
                  sampler="lcm") -> _StaticGraph:
        key = (B, h, w, steps, cfg_scale, decode)
        if sampler != "lcm":                                     # the LCM keys stay as they were
            key += ("sampler", sampler)
        if inpaint:                                              # inpainting: its own graph per strength
            key += ("inpaint", strength)
        elif strength is not None:                               # image-to-image: its own graph per strength
            key += ("img2img", strength)
        g = self._graphs.pop(key, None)
        if g is None:
            while len(self._graphs) >= self.max_graphs:          # least recently used goes first
                self._graphs.pop(next(iter(self._graphs)))
            with torch.cuda.device(self.device):
                g = _StaticGraph(self, B, h, w, steps, cfg_scale, decode, strength, inpaint, sampler)
        self._graphs[key] = g                                     # dict order = recency
        return g

    @torch.no_grad()
    def denoise(self, latents_nchw, step_noise_nchw, sched, kvs, tembs, record: dict = None,
                cfg_scale: Optional[float] = None, teacher=None, start_nhwc=None, inpaint=None):
        """latents fp32 NCHW [B,4,h,w]; step_noise [steps-1,B,4,h,w] (steps = len(sched.timesteps)).  Returns final
        latents NHWC.
        start_nhwc (image-to-image, inpainting): the initial latents, already NHWC; latents_nchw then only gives the
        shape.  inpaint: the second result of `inpaint_latents` — the 9-channel UNet input, or the 4-channel UNet's
        blend fused into the scheduler step.
        teacher (parity tests): fp32 NCHW [steps,B,4,h,w] — the latents fed to the UNet at step i
        come from this tensor (an oracle trajectory) instead of from the previous step, so every
        step's noise_pred is compared on identical inputs (teacher forcing).
        A guided-model sampler's schedule (not `LCMSchedule`) runs `_denoise_sampler`."""
        if not isinstance(sched, LCMSchedule):
            return self._denoise_sampler(latents_nchw, step_noise_nchw, sched, kvs, tembs, record, cfg_scale, teacher)
        B, C, H, W = latents_nchw.shape
        if start_nhwc is not None:
            x = start_nhwc
        else:
            x = torch.empty(B, H, W, C, device=self.device, dtype=torch.float32)
            lib.nchw_to_nhwc_f32(latents_nchw, x)
        n = len(sched.timesteps)
        noise = None
        if n > 1:
            noise = torch.empty(n - 1, B, H, W, C, device=self.device, dtype=torch.float32)
            lib.nchw_to_nhwc_f32(step_noise_nchw[:n - 1].reshape((n - 1) * B, C, H, W),
                                 noise.view((n - 1) * B, H, W, C))
        den = torch.empty_like(x)
        tx = None
        if teacher is not None:
            tx = torch.empty(n, B, H, W, C, device=self.device, dtype=torch.float32)
            lib.nchw_to_nhwc_f32(teacher.to(self.device, torch.float32).reshape(n * B, C, H, W).contiguous(),
                                 tx.view(n * B, H, W, C))
        cond = inpaint["cond"] if inpaint is not None else None
        blend = inpaint["blend"] if inpaint is not None else None
        for i in range(n):
            if tx is not None:
                x = tx[i]
            if cfg_scale is None:
                eps = self.unet.forward(x, tembs[i], kvs, inpaint_cond=cond)
            else:
                eps2 = self.unet.forward(x, tembs[i], kvs, repeat=2, inpaint_cond=cond)
                eps = torch.empty_like(x)
                lib.cfg_combine(eps2[:B], eps2[B:], cfg_scale, eps)
                if record is not None:      # the UNet output before guidance: [uncond; text]
                    record.setdefault("noise_pred_raw", []).append(eps2.permute(0, 3, 1, 2).clone())
            x_next = torch.empty_like(x)
            z = noise[i] if sched.has_noise(i) else None
            if blend is not None:
                # latents = (1 - m) * add_noise(image_latents, noise, timesteps[i + 1]) + m * latents; image_latents
                # itself after the last step
                last = i == n - 1
                lib.lcm_step_inpaint_ex(eps, x, z, blend[0], None if last else blend[1], blend[2], x_next, den,
                                        sched.coeffs(i), (1.0, 0.0) if last else
                                        sched.add_noise_coeffs(sched.timesteps[i + 1]), last,
                                        sched.prediction_type, sched.clip_range)
            else:
                lib.lcm_step_ex(eps, x, z, x_next, den, sched.coeffs(i), sched.prediction_type, sched.clip_range)
            if record is not None:
                record.setdefault("noise_pred", []).append(eps.permute(0, 3, 1, 2).clone())
                record.setdefault("latents", []).append(x_next.permute(0, 3, 1, 2).clone())
            x = x_next
        return x

    def _denoise_sampler(self, latents_nchw, step_noise_nchw, sched, kvs, tembs, record, cfg_scale, teacher):
        """Text-to-image with a guided-model sampler: latents * init_noise_sigma, then per step the UNet on
        x * in_scale(i) and one `lib.sampler_step` (guidance fused).  step_noise holds sched.n_draws draws.  The
        x0 of the previous step (DPM++'s second-order term) stays in one of two device buffers."""
        B, C, H, W = latents_nchw.shape
        n = len(sched.timesteps)
        f32 = dict(device=self.device, dtype=torch.float32)
        x = torch.empty(B, H, W, C, **f32)
        lib.nchw_to_nhwc_f32(latents_nchw, x)
        if sched.init_noise_sigma != 1.0:
            # latents * init_noise_sigma as the step's x0 with a_x = sigma (a_e = 0 leaves e out of the product)
            x_init = torch.empty_like(x)
            lib.sampler_step(x, None, 1.0, x, None, None, torch.empty_like(x), x_init,
                             (sched.init_noise_sigma, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0))
            x = x_init
        noise = None
        if sched.n_draws:
            noise = torch.empty(sched.n_draws, B, H, W, C, **f32)
            lib.nchw_to_nhwc_f32(step_noise_nchw[:sched.n_draws].reshape(sched.n_draws * B, C, H, W),
                                 noise.view(sched.n_draws * B, H, W, C))
        den = (torch.empty_like(x), torch.empty_like(x))
        tx = None
        if teacher is not None:
            tx = torch.empty(n, B, H, W, C, **f32)
            lib.nchw_to_nhwc_f32(teacher.to(self.device, torch.float32).reshape(n * B, C, H, W).contiguous(),
                                 tx.view(n * B, H, W, C))
        k = 0                                                   # draws consumed so far
        for i in range(n):
            if tx is not None:
                x = tx[i]
            s = sched.in_scale(i)
            if cfg_scale is None:
                out = self.unet.forward(x, tembs[i], kvs, in_scale=s)
                u, t = out, None
            else:
                out = self.unet.forward(x, tembs[i], kvs, repeat=2, in_scale=s)
                u, t = out[:B], out[B:]
            z = None
            if sched.has_noise(i):
                z, k = noise[k], k + 1
            x_next = torch.empty_like(x)
            lib.sampler_step(u, t, 1.0 if cfg_scale is None else cfg_scale, x,
                             den[(i + 1) % 2] if sched.uses_prev_x0(i) else None, z, x_next, den[i % 2],
                             sched.coeffs(i), sched.clip_range)
            if record is not None:
                if t is None:
                    record.setdefault("noise_pred", []).append(out.permute(0, 3, 1, 2).clone())
                else:
                    guided = torch.empty_like(x)
                    lib.cfg_combine(u, t, cfg_scale, guided)
                    record.setdefault("noise_pred", []).append(guided.permute(0, 3, 1, 2).clone())
                    record.setdefault("noise_pred_raw", []).append(out.permute(0, 3, 1, 2).clone())
                record.setdefault("latents", []).append(x_next.permute(0, 3, 1, 2).clone())
                record.setdefault("denoised", []).append(den[i % 2].permute(0, 3, 1, 2).clone())
            x = x_next
        return x

    def _conditioning(self, prompt_embeds, pooled_embeds, time_ids, negative_prompt_embeds,
                      negative_pooled_embeds, cfg_scale, height, width):
        """-> (context rows, (pooled, time_ids) or None), doubled [uncond, cond] under CFG.
        With no negative prompt the unconditional half is zeros (`force_zeros_for_empty_prompt`,
        SDXL-base pipeline config)."""
        B = prompt_embeds.shape[0]
        pe = prompt_embeds
        add = None
        if self.is_sdxl:
            if pooled_embeds is None:
                raise RuntimeError("SDXL-class UNet needs pooled_embeds (text_time conditioning)")
            if time_ids is None:
                time_ids = torch.tensor([[height, width, 0, 0, height, width]],
                                        dtype=torch.float32).repeat(B, 1)
            add = (pooled_embeds.float(), time_ids.float())
        if cfg_scale is not None:
            neg = torch.zeros_like(pe) if negative_prompt_embeds is None else negative_prompt_embeds
            pe = torch.cat([neg.to(pe.device, pe.dtype), pe], 0)
            if add is not None:
                negp = (torch.zeros_like(add[0]) if negative_pooled_embeds is None
                        else negative_pooled_embeds.to(add[0].device).float())
                add = (torch.cat([negp, add[0]], 0), torch.cat([add[1], add[1]], 0))
        return pe, add

    @torch.no_grad()
    def generate(self, prompt_embeds, latents_nchw, step_noise_nchw, num_inference_steps: int,
                 guidance_scale=1.0, record: dict = None, return_latents: bool = False,
                 use_graph: bool = False, pooled_embeds=None, time_ids=None,
                 negative_prompt_embeds=None, negative_pooled_embeds=None, teacher_latents=None,
                 decode: bool = True, init_images=None, strength: Optional[float] = None, posterior_noise=None,
                 mask_images=None, masked_posterior_noise=None, sampler: str = "lcm"):
        """Public entry: host or device tensors in -> u8 images [B,H,W,3] on device (and the
        final latents NHWC fp32 if asked).  With use_graph the whole pass is one CUDA-graph
        replay; the returned tensors are the graph's static outputs (consume before next call).

        Image-to-image (`LatentConsistencyModelImg2ImgPipeline`): init_images u8 [B,H,W,3] (H = 8h, W = 8w),
        strength in (0, 1] (default 0.8), posterior_noise fp32 [B,4,h,w] (the posterior sample's draw);
        latents_nchw is then the add_noise draw.  Needs an LCM UNet (time_cond_proj_dim) and VAE encoder
        weights.

        Inpainting (`StableDiffusionInpaintPipeline` with `LCMScheduler`): init_images as above plus mask_images u8
        [B,H,W] (L values; m >= 128 is repainted), strength in (0, 1] (default 1.0) truncating the full schedule.
        latents_nchw is the latents / add_noise draw, posterior_noise the image's posterior draw (needed by a 4-channel
        UNet, and by a 9-channel one at strength < 1), masked_posterior_noise the masked image's (9-channel UNets);
        step_noise_nchw holds len(truncated schedule) - 1 draws.  A 9-channel (inpainting) UNet serves nothing else;
        classifier-free guidance applies as for text-to-image.

        sampler: "lcm" (`LCMScheduler`, the default), or "euler", "euler_a", "ddim", "dpmpp_2m", "dpmpp_2m_karras"
        (text-to-image only; `scheduler.sampler_schedule`).  step_noise_nchw then holds the draws the sampler consumes:
        num_inference_steps for "euler_a", none for the others (None is accepted)."""
        B, _, h, w = latents_nchw.shape
        steps = int(num_inference_steps)
        nine = getattr(self.unet.cfg, "in_channels", 4) == 9
        inpaint = mask_images is not None
        sampler = check_sampler(sampler)
        if sampler != "lcm" and (init_images is not None or inpaint):
            raise RuntimeError(f"sampler {sampler!r}: image-to-image and inpainting run the LCM sampler only")
        k = steps                                         # steps that run (inpainting: the truncated schedule's)
        if nine and not inpaint:
            raise RuntimeError("this model's UNet has in_channels=9 (an inpainting UNet): it serves inpainting only "
                               "(init_images + mask_images); text-to-image and image-to-image are not defined for it")
        if inpaint:
            if init_images is None:
                raise RuntimeError("mask_images without init_images: inpainting repaints part of a given picture")
            strength = 1.0 if strength is None else float(strength)
            self.require_encoder()
            if tuple(init_images.shape) != (B, 8 * h, 8 * w, 3) or init_images.dtype != torch.uint8:
                raise RuntimeError(f"init_images: u8 [{B}, {8 * h}, {8 * w}, 3] expected, got "
                                   f"{init_images.dtype} {list(init_images.shape)}")
            if tuple(mask_images.shape) != (B, 8 * h, 8 * w) or mask_images.dtype != torch.uint8:
                raise RuntimeError(f"mask_images: u8 [{B}, {8 * h}, {8 * w}] expected, got "
                                   f"{mask_images.dtype} {list(mask_images.shape)}")
            k = len(self.schedule(steps, strength, inpaint=True).timesteps)     # ValueError when no step remains
            if (not nine or strength < 1.0) and (posterior_noise is None or
                                                 tuple(posterior_noise.shape) != (B, 4, h, w)):
                raise RuntimeError(f"inpainting needs posterior_noise [{B}, 4, {h}, {w}] (the image's posterior draw)")
            if nine and (masked_posterior_noise is None or tuple(masked_posterior_noise.shape) != (B, 4, h, w)):
                raise RuntimeError(f"inpainting with a 9-channel UNet needs masked_posterior_noise [{B}, 4, {h}, {w}]")
        elif init_images is not None:
            strength = 0.8 if strength is None else float(strength)
            if not self.unet.cfg.time_cond_proj_dim:
                raise RuntimeError("image-to-image is implemented for LCM UNets (time_cond_proj_dim) only: the LCM "
                                   "img2img pipeline has no classifier-free guidance branch")
            self.require_encoder()
            if tuple(init_images.shape) != (B, 8 * h, 8 * w, 3) or init_images.dtype != torch.uint8:
                raise RuntimeError(f"init_images: u8 [{B}, {8 * h}, {8 * w}, 3] expected, got "
                                   f"{init_images.dtype} {list(init_images.shape)}")
            if posterior_noise is None or tuple(posterior_noise.shape) != (B, 4, h, w):
                raise RuntimeError(f"image-to-image needs posterior_noise [{B}, 4, {h}, {w}]")
            self.schedule(steps, strength)                # ValueError for a strength the schedule cannot serve
        else:
            strength = None
        # step noise draws the pass consumes
        nd = k - 1 if sampler == "lcm" else self.schedule(steps, sampler=sampler).n_draws
        if nd > 0 and (step_noise_nchw is None or step_noise_nchw.shape[0] < nd):
            raise RuntimeError(f"step_noise_nchw: {nd} draws [{nd}, {B}, 4, {h}, {w}] expected")
        if use_graph and record is None and teacher_latents is None:
            Bp = next((b for b in self.batch_buckets if b >= B), B)
            if Bp != B:
                # pad to the bucket by repeating the last request (images are independent: per-image GroupNorm,
                # per-image attention), run the bucket's graph, return the first B results
                def pad(t, dim=0):
                    if t is None or not torch.is_tensor(t) or t.dim() == 0:
                        return t
                    idx = [slice(None)] * t.dim()
                    idx[dim] = slice(t.shape[dim] - 1, t.shape[dim])
                    return torch.cat([t] + [t[tuple(idx)]] * (Bp - B), dim)
                gs = torch.as_tensor(guidance_scale, dtype=torch.float32).reshape(-1)
                out = self.generate(pad(prompt_embeds), pad(latents_nchw),
                                    pad(step_noise_nchw, 1) if nd > 0 else step_noise_nchw, steps,
                                    pad(gs) if gs.numel() > 1 else guidance_scale, return_latents=True, use_graph=True,
                                    pooled_embeds=pad(pooled_embeds), time_ids=pad(time_ids),
                                    negative_prompt_embeds=pad(negative_prompt_embeds),
                                    negative_pooled_embeds=pad(negative_pooled_embeds), decode=decode,
                                    init_images=pad(init_images), strength=strength,
                                    posterior_noise=pad(posterior_noise), mask_images=pad(mask_images),
                                    masked_posterior_noise=pad(masked_posterior_noise), sampler=sampler)
                img, lat = out
                img = img[:B] if img is not None else None
                return (img, lat[:B]) if return_latents else img
        w_emb = self._w_emb(B, guidance_scale)
        cfg_scale = self.cfg_scale_for(guidance_scale)
        pe_all, add = self._conditioning(prompt_embeds, pooled_embeds, time_ids, negative_prompt_embeds,
                                         negative_pooled_embeds, cfg_scale, 8 * h, 8 * w)
        with torch.cuda.device(self.device):
            if use_graph and record is None and teacher_latents is None:
                g = self.graph_for(B, h, w, steps, cfg_scale, decode, strength, inpaint, sampler)
                # host inputs go through pinned staging: a copy from PAGEABLE host memory first waits for the stream to
                # drain (CUDA's documented behaviour), i.e. for the previous batch — the thread could then not enqueue
                # this batch behind it
                g.pe.copy_(_pinned(pe_all), non_blocking=True)
                if w_emb is not None:
                    g.w_emb.copy_(_pinned(w_emb), non_blocking=True)
                if add is not None:
                    g.add[0].copy_(_pinned(add[0]), non_blocking=True)
                    g.add[1].copy_(_pinned(add[1]), non_blocking=True)
                g.lat.copy_(_pinned(latents_nchw), non_blocking=True)
                if nd > 0:
                    g.noise.copy_(_pinned(step_noise_nchw[:nd]), non_blocking=True)
                if strength is not None:
                    g.init_u8.copy_(_pinned(init_images), non_blocking=True)
                    if posterior_noise is not None:
                        g.eps_s.copy_(_pinned(posterior_noise), non_blocking=True)
                if inpaint:
                    g.mask_u8.copy_(_pinned(mask_images), non_blocking=True)
                    if masked_posterior_noise is not None:
                        g.eps_m.copy_(_pinned(masked_posterior_noise), non_blocking=True)
                g.graph.replay()
                img, lat = g.img, g.final
            else:
                pe = pe_all.to(self.device, self.dt).contiguous()
                we = w_emb.to(self.device) if w_emb is not None else None
                if add is not None:
                    add = (add[0].to(self.device), add[1].to(self.device))
                lat0 = latents_nchw.to(self.device, torch.float32).contiguous()
                nz = (step_noise_nchw.to(self.device, torch.float32).contiguous()
                      if nd > 0 else None)
                init = eps = mask = eps_m = None
                if strength is not None:
                    init = init_images.to(self.device).contiguous()
                    if posterior_noise is not None:
                        eps = posterior_noise.to(self.device, torch.float32).contiguous()
                if inpaint:
                    mask = mask_images.to(self.device).contiguous()
                    if masked_posterior_noise is not None:
                        eps_m = masked_posterior_noise.to(self.device, torch.float32).contiguous()
                img, lat = self.run_static(pe, we, lat0, nz, steps, record, add=add, cfg_scale=cfg_scale,
                                           teacher=teacher_latents, decode=decode, init_u8=init, eps_s=eps,
                                           strength=strength, mask_u8=mask, eps_m=eps_m, sampler=sampler)
        return (img, lat) if return_latents else img
