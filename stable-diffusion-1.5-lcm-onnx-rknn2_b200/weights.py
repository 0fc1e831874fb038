"""Weight packing: diffusers-keyed state dicts -> device tensors in the layouts the kernels want.

Keys follow the diffusers `UNet2DConditionModel` / `AutoencoderKL` state dicts (the reference
loads them with `StableDiffusionPipeline.from_pretrained/from_single_file`,
`backends/cuda_worker.py:70-85`), so a real checkpoint's tensors drop in unchanged.

Layouts
  conv3x3  [O,I,3,3] -> bf16 [O, 9*I]   K index = (ky*3+kx)*I + i   (OHWI, K-major)
  conv1x1 / Linear   -> bf16 [O, I]
  attention q/k/v    -> fused, per-head rows zero-padded from d to d16 = ceil16(d) so the
                        tcgen05 K-steps over the pad contribute exact zeros
  GEGLU proj         -> rows interleaved (value_j, gate_j) for the fused epilogue
  norms, biases      -> fp32
"""
from __future__ import annotations

import threading
from typing import Dict

import torch


def ceil16(d: int) -> int:
    return (d + 15) // 16 * 16


_tls = threading.local()


class pack_dtype:
    """Context: dtype of the packed GEMM operands (bf16 for the kernels; fp32 when packing LoRA
    deltas, `lora.py`).  Thread-local: pool workers load concurrently."""

    def __init__(self, dtype):
        self.dtype = dtype

    def __enter__(self):
        self.prev = getattr(_tls, "dtype", torch.bfloat16)
        _tls.dtype = self.dtype

    def __exit__(self, *exc):
        _tls.dtype = self.prev
        return False


def _bf(t, device):
    return t.to(device=device, dtype=getattr(_tls, "dtype", torch.bfloat16)).contiguous()


def _f32(t, device):
    return t.to(device=device, dtype=torch.float32).contiguous()


def pack_conv3x3(w: torch.Tensor, device, pad_in_to: int = 0) -> torch.Tensor:
    o, i = w.shape[0], w.shape[1]
    w = w.float().permute(0, 2, 3, 1)                      # [O,3,3,I]
    if pad_in_to and pad_in_to > i:
        w = torch.nn.functional.pad(w, (0, pad_in_to - i))
    return _bf(w.reshape(o, -1), device)


def pack_upsample_conv3x3(w: torch.Tensor, device) -> torch.Tensor:
    """Nearest-2x upsample followed by conv3x3 == four 2x2 convs on the low-res input, one per
    output phase (a, b) = (row parity, column parity), with the 3x3 taps that land on the same
    low-res pixel pre-summed (in fp32): 2.25x fewer MACs and no upsampled tensor in HBM.
    Returns bf16 [4, O, 4*I]: phase 2a+b, K index = (ty*2+tx)*I + i."""
    o, i = w.shape[0], w.shape[1]
    w = w.float()
    groups = {0: ([0], [1, 2]), 1: ([0, 1], [2])}       # parity -> (taps of low-res -1+p, of +p)
    out = torch.zeros(4, o, 2, 2, i, device=w.device)
    for a in (0, 1):
        for b in (0, 1):
            for ty in (0, 1):
                for tx in (0, 1):
                    acc = torch.zeros(o, i, device=w.device)
                    for ky in groups[a][ty]:
                        for kx in groups[b][tx]:
                            acc += w[:, :, ky, kx]
                    out[2 * a + b, :, ty, tx] = acc
    return _bf(out.reshape(4, o, 4 * i), device)


def pack_conv1x1(w: torch.Tensor, device) -> torch.Tensor:
    return _bf(w.reshape(w.shape[0], -1), device)


def head_stride(d: int) -> int:
    """Per-head column stride of the packed Q/K/V: room for d values, zero padding up to a
    multiple of 16 (tcgen05 K-steps) and one extra column that holds 1.0 in V (the PV MMA then
    accumulates the softmax denominator for free)."""
    return ceil16(d + 1)


def pad_heads(w: torch.Tensor, heads: int) -> torch.Tensor:
    """[heads*d, K] -> [heads*stride, K] with zero rows after each head's d rows."""
    c, k = w.shape
    d = c // heads
    hs = head_stride(d)
    out = w.new_zeros(heads, hs, k)
    out[:, :d] = w.view(heads, d, k)
    return out.reshape(heads * hs, k)


def ones_bias(heads: int, d: int, sections: int, v_section: int) -> torch.Tensor:
    """fp32 bias for a fused projection of `sections` head-padded blocks: 1.0 in column d of
    every head of the V block (its weight rows are zero), 0 elsewhere."""
    hs = head_stride(d)
    b = torch.zeros(sections, heads, hs)
    b[v_section, :, d] = 1.0
    return b.reshape(-1)


def interleave_geglu(w: torch.Tensor) -> torch.Tensor:
    """[2*inner, ...] (values then gates) -> rows (v0,g0,v1,g1,...)."""
    inner = w.shape[0] // 2
    return torch.stack([w[:inner], w[inner:]], dim=1).reshape(w.shape)


def fold_layernorm(w: torch.Tensor, bias, gamma: torch.Tensor, beta: torch.Tensor, device):
    """LayerNorm folded into the Linear that consumes it (SURVEY.md K8, `dl_igemm_desc.ln_*`):
        LN(x) W^T + b = rstd (x W'^T - mean colsum(W')) + (b + W beta),   W'[j,k] = W[j,k] gamma[k].
    w: packed fp32 [N, K] (head padding / GEGLU interleave already applied), bias fp32 [N] or None.
    -> (W' in the packing dtype, colsum(W') fp32 of the ROUNDED W' the tensor core multiplies, folded bias
    fp32), or (None, None, None) outside the bf16 tensor-core path."""
    if getattr(_tls, "dtype", torch.bfloat16) != torch.bfloat16:
        return None, None, None
    w = w.float()
    wf = _bf(w * gamma.float()[None, :].to(w.device), device)
    colsum = wf.float().sum(1)
    b = w.to(torch.bfloat16).float() @ beta.float().to(w.device)
    if bias is not None:
        b = b + bias.float().to(w.device)
    return wf, _f32(colsum, device), _f32(b, device)


class Packed(dict):
    """dict with attribute access; values are device tensors or nested Packed."""
    __getattr__ = dict.__getitem__


def pack_resnet(sd: Dict[str, torch.Tensor], prefix: str, device) -> Packed:
    p = Packed()
    p["norm1_w"], p["norm1_b"] = _f32(sd[prefix + "norm1.weight"], device), _f32(sd[prefix + "norm1.bias"], device)
    p["norm2_w"], p["norm2_b"] = _f32(sd[prefix + "norm2.weight"], device), _f32(sd[prefix + "norm2.bias"], device)
    p["conv1_w"], p["conv1_b"] = pack_conv3x3(sd[prefix + "conv1.weight"], device), _f32(sd[prefix + "conv1.bias"], device)
    p["conv2_w"], p["conv2_b"] = pack_conv3x3(sd[prefix + "conv2.weight"], device), _f32(sd[prefix + "conv2.bias"], device)
    p["cin"] = sd[prefix + "conv1.weight"].shape[1]
    p["cout"] = sd[prefix + "conv1.weight"].shape[0]
    if prefix + "conv_shortcut.weight" in sd:
        p["sc_w"] = pack_conv1x1(sd[prefix + "conv_shortcut.weight"], device)
        p["sc_b"] = _f32(sd[prefix + "conv_shortcut.bias"], device)
    else:
        p["sc_w"] = None
    p["has_temb"] = prefix + "time_emb_proj.weight" in sd
    return p


def pack_transformer(sd, prefix: str, heads: int, device, depth: int = 1) -> Packed:
    """Transformer2DModel with `depth` BasicTransformerBlocks.  proj_in/proj_out are 1x1 convs
    (SD1.5) or Linears (SDXL, use_linear_projection): the same [C, C] matrix on NHWC rows."""
    p = Packed()
    p["norm_w"], p["norm_b"] = _f32(sd[prefix + "norm.weight"], device), _f32(sd[prefix + "norm.bias"], device)
    p["proj_in_w"], p["proj_in_b"] = pack_conv1x1(sd[prefix + "proj_in.weight"], device), _f32(sd[prefix + "proj_in.bias"], device)
    p["proj_out_w"], p["proj_out_b"] = pack_conv1x1(sd[prefix + "proj_out.weight"], device), _f32(sd[prefix + "proj_out.bias"], device)
    c = sd[prefix + "transformer_blocks.0.attn1.to_q.weight"].shape[0]
    p["c"], p["heads"], p["d"] = c, heads, c // heads
    p["hstride"] = head_stride(c // heads)
    p["blocks"] = []
    for l in range(depth):
        b = prefix + f"transformer_blocks.{l}."
        q = Packed()
        for i in (1, 2, 3):
            q[f"ln{i}_w"], q[f"ln{i}_b"] = _f32(sd[b + f"norm{i}.weight"], device), _f32(sd[b + f"norm{i}.bias"], device)
        qkv = torch.cat([pad_heads(sd[b + f"attn1.to_{n}.weight"].float(), heads) for n in "qkv"], 0)
        q["qkv_w"] = _bf(qkv, device)
        q["qkv_b"] = _f32(ones_bias(heads, c // heads, 3, 2), device)
        q["qkv_wf"], q["qkv_cs"], q["qkv_bf"] = fold_layernorm(qkv, ones_bias(heads, c // heads, 3, 2),
                                                               sd[b + "norm1.weight"], sd[b + "norm1.bias"], device)
        q["o1_w"], q["o1_b"] = _bf(sd[b + "attn1.to_out.0.weight"], device), _f32(sd[b + "attn1.to_out.0.bias"], device)
        q["q2_w"] = _bf(pad_heads(sd[b + "attn2.to_q.weight"].float(), heads), device)
        q["q2_wf"], q["q2_cs"], q["q2_bf"] = fold_layernorm(pad_heads(sd[b + "attn2.to_q.weight"].float(), heads), None,
                                                            sd[b + "norm2.weight"], sd[b + "norm2.bias"], device)
        kv = torch.cat([pad_heads(sd[b + f"attn2.to_{n}.weight"].float(), heads) for n in "kv"], 0)
        q["kv2_w"] = _bf(kv, device)
        q["kv2_b"] = _f32(ones_bias(heads, c // heads, 2, 1), device)
        q["o2_w"], q["o2_b"] = _bf(sd[b + "attn2.to_out.0.weight"], device), _f32(sd[b + "attn2.to_out.0.bias"], device)
        q["ff1_w"] = _bf(interleave_geglu(sd[b + "ff.net.0.proj.weight"].float()), device)
        q["ff1_b"] = _f32(interleave_geglu(sd[b + "ff.net.0.proj.bias"].float()), device)
        q["ff1_wf"], q["ff1_cs"], q["ff1_bf"] = fold_layernorm(interleave_geglu(sd[b + "ff.net.0.proj.weight"].float()),
                                                               interleave_geglu(sd[b + "ff.net.0.proj.bias"].float()),
                                                               sd[b + "norm3.weight"], sd[b + "norm3.bias"], device)
        q["ff2_w"], q["ff2_b"] = _bf(sd[b + "ff.net.2.weight"], device), _f32(sd[b + "ff.net.2.bias"], device)
        p["blocks"].append(q)
    return p


def _heads_at(cfg, i):
    a = cfg.attention_head_dim
    return a if isinstance(a, int) else a[i]


def _depth_at(cfg, i):
    t = getattr(cfg, "transformer_layers_per_block", None)
    return t[i] if t else 1


def pack_unet(sd: Dict[str, torch.Tensor], cfg, device) -> Packed:
    """cfg: anything with block_out_channels, down_attn, layers_per_block, attention_head_dim,
    time_cond_proj_dim (oracle.unet.UNetConfig or a dict-like parsed from unet/config.json)."""
    ch = cfg.block_out_channels
    n_lv = len(ch)
    P = Packed()
    P["cfg"] = cfg
    P["conv_in_w"] = pack_conv3x3(sd["conv_in.weight"], device, pad_in_to=64)
    P["conv_in_b"] = _f32(sd["conv_in.bias"], device)
    P["t1_w"], P["t1_b"] = _bf(sd["time_embedding.linear_1.weight"], device), _f32(sd["time_embedding.linear_1.bias"], device)
    P["t2_w"], P["t2_b"] = _bf(sd["time_embedding.linear_2.weight"], device), _f32(sd["time_embedding.linear_2.bias"], device)
    P["cond_w"] = (_bf(sd["time_embedding.cond_proj.weight"], device)
                   if "time_embedding.cond_proj.weight" in sd else None)
    if "add_embedding.linear_1.weight" in sd:        # SDXL text_time micro-conditioning MLP
        P["add1_w"], P["add1_b"] = _bf(sd["add_embedding.linear_1.weight"], device), _f32(sd["add_embedding.linear_1.bias"], device)
        P["add2_w"], P["add2_b"] = _bf(sd["add_embedding.linear_2.weight"], device), _f32(sd["add_embedding.linear_2.bias"], device)
    else:
        P["add1_w"] = None
    resnets = []          # in execution order, for the fused time_emb_proj matrix

    def res(prefix):
        r = pack_resnet(sd, prefix, device)
        r["temb_off"] = sum(x["cout"] for x in resnets)
        r["prefix"] = prefix
        resnets.append(r)
        return r

    P["down"] = []
    for i in range(len(ch)):
        blk = Packed(resnets=[], attns=[], down=None)
        for j in range(cfg.layers_per_block):
            blk["resnets"].append(res(f"down_blocks.{i}.resnets.{j}."))
            if cfg.down_attn[i]:
                blk["attns"].append(pack_transformer(sd, f"down_blocks.{i}.attentions.{j}.",
                                                     _heads_at(cfg, i), device, _depth_at(cfg, i)))
        if i != len(ch) - 1:
            k = f"down_blocks.{i}.downsamplers.0.conv."
            blk["down"] = Packed(w=pack_conv3x3(sd[k + "weight"], device), b=_f32(sd[k + "bias"], device))
        P["down"].append(blk)
    P["mid"] = Packed(resnets=[res("mid_block.resnets.0.")],
                      attns=[pack_transformer(sd, "mid_block.attentions.0.", _heads_at(cfg, n_lv - 1),
                                              device, _depth_at(cfg, n_lv - 1))])
    P["mid"]["resnets"].append(res("mid_block.resnets.1."))
    P["up"] = []
    rev_attn = list(reversed(cfg.down_attn))
    for i in range(len(ch)):
        blk = Packed(resnets=[], attns=[], up=None)
        for j in range(cfg.layers_per_block + 1):
            blk["resnets"].append(res(f"up_blocks.{i}.resnets.{j}."))
            if rev_attn[i]:
                blk["attns"].append(pack_transformer(sd, f"up_blocks.{i}.attentions.{j}.",
                                                     _heads_at(cfg, n_lv - 1 - i), device,
                                                     _depth_at(cfg, n_lv - 1 - i)))
        if i != len(ch) - 1:
            k = f"up_blocks.{i}.upsamplers.0.conv."
            blk["up"] = Packed(w=pack_upsample_conv3x3(sd[k + "weight"], device), b=_f32(sd[k + "bias"], device))
        P["up"].append(blk)
    # all ResnetBlock2D.time_emb_proj fused into one [sum(cout), temb] matrix: one launch per step
    P["temb_w"] = _bf(torch.cat([sd[r["prefix"] + "time_emb_proj.weight"].float() for r in resnets], 0), device)
    P["temb_b"] = _f32(torch.cat([sd[r["prefix"] + "time_emb_proj.bias"].float() for r in resnets], 0), device)
    P["temb_total"] = P["temb_w"].shape[0]
    P["norm_out_w"], P["norm_out_b"] = _f32(sd["conv_norm_out.weight"], device), _f32(sd["conv_norm_out.bias"], device)
    P["conv_out_w"] = pack_conv3x3(sd["conv_out.weight"], device)
    P["conv_out_b"] = _f32(sd["conv_out.bias"], device)
    P["transformers"] = ([a for b in P["down"] for a in b["attns"]] + P["mid"]["attns"] +
                         [a for b in P["up"] for a in b["attns"]])
    return P


def pack_vae_attention(sd: Dict[str, torch.Tensor], a: str, device) -> Packed:
    """The one-head mid-block attention of the AutoencoderKL encoder and decoder (prefix `a`)."""
    att = Packed()
    att["norm_w"], att["norm_b"] = _f32(sd[a + "group_norm.weight"], device), _f32(sd[a + "group_norm.bias"], device)
    wq, wk, wv, wo = (sd[a + f"{n}.weight"].float() for n in ("to_q", "to_k", "to_v", "to_out.0"))
    bq, bk, bv, bo = (sd[a + f"{n}.bias"].float() for n in ("to_q", "to_k", "to_v", "to_out.0"))
    att["qk_w"] = _bf(torch.cat([wq, wk], 0), device)
    att["qk_b"] = _f32(torch.cat([bq, bk], 0), device)
    att["v_w"] = _bf(wv, device)                   # used as the *activation* operand: V^T = Wv X^T
    att["o_w"] = _bf(wo, device)
    # softmax rows sum to 1  =>  P (V + 1 b_v^T) = P V + b_v^T : fold b_v into the out-proj bias
    att["o_b"] = _f32(bo + wo @ bv, device)
    att["c"] = wq.shape[0]
    return att


def has_vae_encoder(sd: Dict[str, torch.Tensor]) -> bool:
    return "encoder.conv_in.weight" in sd and "quant_conv.weight" in sd


def pack_vae_encoder(sd: Dict[str, torch.Tensor], cfg, device) -> Packed:
    """AutoencoderKL encoder + quant_conv.  conv_in (3 -> C, 3x3) runs as a 1x1 GEMM over the image im2col
    (`dl_pack_image_im2col`): weight [C, 27] with K = (ky*3 + kx)*3 + c, zero-padded to 64.  quant_conv
    (1x1, 2L -> 2L) is applied in fp32 by the latent-packing kernel, like post_quant_conv."""
    P = Packed()
    P["cfg"] = cfg
    d = "encoder."
    w = sd[d + "conv_in.weight"].float()
    P["conv_in_w"] = _bf(torch.nn.functional.pad(w.permute(0, 2, 3, 1).reshape(w.shape[0], -1), (0, 64 - 27)), device)
    P["conv_in_b"] = _f32(sd[d + "conv_in.bias"], device)
    P["down"] = []
    n = len(cfg.block_out_channels)
    for i in range(n):
        blk = Packed(resnets=[pack_resnet(sd, d + f"down_blocks.{i}.resnets.{j}.", device)
                              for j in range(cfg.layers_per_block)], down=None)
        k = d + f"down_blocks.{i}.downsamplers.0.conv."
        if k + "weight" in sd:
            blk["down"] = Packed(w=pack_conv3x3(sd[k + "weight"], device), b=_f32(sd[k + "bias"], device))
        P["down"].append(blk)
    P["mid_res"] = [pack_resnet(sd, d + f"mid_block.resnets.{i}.", device) for i in range(2)]
    P["mid_attn"] = pack_vae_attention(sd, d + "mid_block.attentions.0.", device)
    P["norm_out_w"], P["norm_out_b"] = _f32(sd[d + "conv_norm_out.weight"], device), _f32(sd[d + "conv_norm_out.bias"], device)
    P["conv_out_w"] = pack_conv3x3(sd[d + "conv_out.weight"], device)
    P["conv_out_b"] = _f32(sd[d + "conv_out.bias"], device)
    m = sd["quant_conv.weight"].shape[0]
    P["q_w"] = _f32(sd["quant_conv.weight"].reshape(m, m), device)
    P["q_b"] = _f32(sd["quant_conv.bias"], device)
    return P


def pack_vae_decoder(sd: Dict[str, torch.Tensor], cfg, device) -> Packed:
    P = Packed()
    P["cfg"] = cfg
    # post_quant_conv (1x1, 4->4) is applied in fp32 by the latent-packing kernel
    P["pq_w"] = _f32(sd["post_quant_conv.weight"].reshape(cfg.latent_channels, cfg.latent_channels), device)
    P["pq_b"] = _f32(sd["post_quant_conv.bias"], device)
    d = "decoder."
    P["conv_in_w"] = pack_conv3x3(sd[d + "conv_in.weight"], device, pad_in_to=64)
    P["conv_in_b"] = _f32(sd[d + "conv_in.bias"], device)
    P["mid_res"] = [pack_resnet(sd, d + f"mid_block.resnets.{i}.", device) for i in range(2)]
    P["mid_attn"] = pack_vae_attention(sd, d + "mid_block.attentions.0.", device)
    P["up"] = []
    n_up = len(cfg.block_out_channels)
    for i in range(n_up):
        blk = Packed(resnets=[pack_resnet(sd, d + f"up_blocks.{i}.resnets.{j}.", device)
                              for j in range(cfg.layers_per_block + 1)], up=None)
        k = d + f"up_blocks.{i}.upsamplers.0.conv."
        if k + "weight" in sd:
            blk["up"] = Packed(w=pack_upsample_conv3x3(sd[k + "weight"], device), b=_f32(sd[k + "bias"], device))
        P["up"].append(blk)
    P["norm_out_w"], P["norm_out_b"] = _f32(sd[d + "conv_norm_out.weight"], device), _f32(sd[d + "conv_norm_out.bias"], device)
    P["conv_out_w"] = pack_conv3x3(sd[d + "conv_out.weight"], device)
    P["conv_out_b"] = _f32(sd[d + "conv_out.bias"], device)
    return P
