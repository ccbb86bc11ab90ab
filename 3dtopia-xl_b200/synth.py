"""Synthetic, reproducible parameters / inputs for the hot path (no checkpoints or datasets offline).

Parameter NAMES and SHAPES are the reference's checkpoint contract (SURVEY.md §8b):
  DiT  — /root/reference/models/dit_crossattn.py:111-156 (module tree), attention.py:37-39,83-87,
         utils.py:31-36,85-92
  VAE  — /root/reference/models/vae3d_dib.py:330-367 (Decoder), :429 (post_quant_conv), :270-307 (Encoder), :428 (quant_conv)
Values are drawn from numpy's frozen ``RandomState`` stream so the golden fixtures under
tests/golden/ can be regenerated bit-identically on any box; ``device_state_dict`` draws on the GPU
instead (fast path for full-size benchmarks, values need not match anything).
"""
from __future__ import annotations

import math
from collections import OrderedDict
from typing import Dict, Tuple

import numpy as np
import torch

FULL_DIT = dict(seq_length=2048, in_channels=68, condition_channels=768, hidden_size=1152, depth=28,
                num_heads=16, attn_proj_bias=True, cond_drop_prob=0.1, gradient_checkpointing=False)
FULL_VAE = dict(in_channels=6, latent_channels=1, out_channels=6, down_channels=[32, 256], mid_attention=True,
                up_channels=[256, 32], layers_per_block=2, gradient_checkpointing=False)
# configs/inference_dit.yml:63-65
LATENT_MEAN = [0.0442, -0.0029, -0.0425, -0.0043, -0.4086, -0.2906, -0.7002, -0.0852, -0.4446, -0.6896, -0.7344, -0.3524, -0.5488, -0.4313, -1.1715, -0.0875, -0.6131, -0.3924, -0.7335, -0.3749, 0.4658, -0.0236, 0.8362, 0.3388, 0.0188, 0.5988, -0.1853, 1.1579, 0.6240, 0.0758, 0.9641, 0.6586, 0.6260, 0.2384, 0.7798, 0.8297, -0.6543, -0.4441, -1.3887, -0.0393, -0.9008, -0.8616, -1.7434, -0.1328, -0.8119, -0.8225, -1.8533, -0.0444, -1.0510, -0.5158, -1.1907, -0.5265, 0.2832, 0.6037, 0.5981, 0.5461, 0.4366, 0.4144, 0.7219, 0.5722, 0.5937, 0.5598, 0.9414, 0.7419, 0.2102, 0.3388, 0.4501, 0.5166]
LATENT_STD = [0.0219, 0.3707, 0.3911, 0.3610, 0.7549, 0.7909, 0.9691, 0.9193, 0.8218, 0.9389, 1.1785, 1.0254, 0.6376, 0.6568, 0.7892, 0.8468, 0.8775, 0.7920, 0.9037, 0.9329, 0.9196, 1.1123, 1.3041, 1.0955, 1.2727, 1.6565, 1.8502, 1.7006, 0.8973, 1.0408, 1.2034, 1.2703, 1.0373, 1.0486, 1.0716, 0.9746, 0.7088, 0.8685, 1.0030, 0.9504, 1.0410, 1.3033, 1.5368, 1.4386, 0.6142, 0.6887, 0.9085, 0.9903, 1.0190, 0.9302, 1.0121, 0.9964, 1.1474, 1.2729, 1.4627, 1.1404, 1.3713, 1.6692, 1.8424, 1.5047, 1.1356, 1.2369, 1.3554, 1.1848, 1.1319, 1.0822, 1.1972, 0.9916]


def dit_shapes(in_channels=68, condition_channels=768, hidden_size=1152, depth=28, mlp_ratio=4.0,
               attn_proj_bias=True, cond_drop_prob=0.1, learn_sigma=True, **_) -> "OrderedDict[str, Tuple[int, ...]]":
    D, Dc = hidden_size, condition_channels
    Dm = int(D * mlp_ratio)
    s: "OrderedDict[str, Tuple[int, ...]]" = OrderedDict()
    if cond_drop_prob > 0:
        s["null_cond_embedding"] = (Dc,)
    s["x_embedder.weight"], s["x_embedder.bias"] = (D, in_channels), (D,)
    s["t_embedder.mlp.0.weight"], s["t_embedder.mlp.0.bias"] = (D, 256), (D,)
    s["t_embedder.mlp.2.weight"], s["t_embedder.mlp.2.bias"] = (D, D), (D,)
    for i in range(depth):
        p = f"blocks.{i}."
        for nm, (o, k) in (("crossattn.to_q", (D, D)), ("crossattn.to_k", (D, Dc)), ("crossattn.to_v", (D, Dc))):
            s[p + nm + ".weight"], s[p + nm + ".bias"] = (o, k), (o,)
        s[p + "crossattn.proj.weight"] = (D, D)
        if attn_proj_bias:
            s[p + "crossattn.proj.bias"] = (D,)
        s[p + "attn.qkv.weight"], s[p + "attn.qkv.bias"] = (3 * D, D), (3 * D,)
        s[p + "attn.proj.weight"] = (D, D)
        if attn_proj_bias:
            s[p + "attn.proj.bias"] = (D,)
        s[p + "mlp.fc1.weight"], s[p + "mlp.fc1.bias"] = (Dm, D), (Dm,)
        s[p + "mlp.fc2.weight"], s[p + "mlp.fc2.bias"] = (D, Dm), (D,)
        s[p + "adaLN_modulation.1.weight"], s[p + "adaLN_modulation.1.bias"] = (9 * D, D), (9 * D,)
    oc = in_channels * 2 if learn_sigma else in_channels
    s["final_layer.linear.weight"], s["final_layer.linear.bias"] = (oc, D), (oc,)
    s["final_layer.adaLN_modulation.1.weight"], s["final_layer.adaLN_modulation.1.bias"] = (2 * D, D), (2 * D,)
    return s


def _resnet_shapes(s, p, cin, cout):
    s[p + "norm1.weight"], s[p + "norm1.bias"] = (cin,), (cin,)
    s[p + "conv1.weight"], s[p + "conv1.bias"] = (cout, cin, 3, 3, 3), (cout,)
    s[p + "norm2.weight"], s[p + "norm2.bias"] = (cout,), (cout,)
    s[p + "conv2.weight"], s[p + "conv2.bias"] = (cout, cout, 3, 3, 3), (cout,)
    if cin != cout:
        s[p + "shortcut.weight"], s[p + "shortcut.bias"] = (cout, cin, 1, 1, 1), (cout,)


def vae_decoder_shapes(latent_channels=1, out_channels=6, up_channels=(256, 32), mid_attention=True,
                       layers_per_block=2, **_) -> "OrderedDict[str, Tuple[int, ...]]":
    s: "OrderedDict[str, Tuple[int, ...]]" = OrderedDict()
    c0 = up_channels[0]
    d = "decoder."
    s[d + "conv_in.weight"], s[d + "conv_in.bias"] = (c0, latent_channels, 3, 3, 3), (c0,)
    _resnet_shapes(s, d + "mid_block.nets.0.", c0, c0)
    _resnet_shapes(s, d + "mid_block.nets.1.", c0, c0)
    if mid_attention:
        a = d + "mid_block.attns.0."
        s[a + "norm.weight"], s[a + "norm.bias"] = (c0,), (c0,)
        s[a + "attn.qkv.weight"] = (3 * c0, c0)
        s[a + "attn.proj.weight"], s[a + "attn.proj.bias"] = (c0, c0), (c0,)
    cout = c0
    for u, ch in enumerate(up_channels):
        cin, cout = cout, ch
        for j in range(layers_per_block):
            _resnet_shapes(s, f"{d}up_blocks.{u}.nets.{j}.", cin if j == 0 else cout, cout)
        if u != len(up_channels) - 1:
            s[f"{d}up_blocks.{u}.upsample.weight"], s[f"{d}up_blocks.{u}.upsample.bias"] = (cout, cout, 2, 2, 2), (cout,)
    s[d + "norm_out.weight"], s[d + "norm_out.bias"] = (cout,), (cout,)
    s[d + "conv_out.weight"], s[d + "conv_out.bias"] = (cout, out_channels, 3, 3, 3), (out_channels,)
    s["post_quant_conv.weight"], s["post_quant_conv.bias"] = (latent_channels,) * 2 + (1, 1, 1), (latent_channels,)
    return s


def vae_encoder_shapes(in_channels=1, latent_channels=1, down_channels=(32, 256), mid_attention=True,
                       layers_per_block=2, **_) -> "OrderedDict[str, Tuple[int, ...]]":
    """encoder.* / quant_conv.* keys of VAE (vae3d_dib.py:270-307 Encoder, :428 quant_conv)."""
    s: "OrderedDict[str, Tuple[int, ...]]" = OrderedDict()
    e = "encoder."
    c0 = down_channels[0]
    s[e + "conv_in.weight"], s[e + "conv_in.bias"] = (c0, in_channels, 3, 3, 3), (c0,)
    cout = c0
    for i, ch in enumerate(down_channels):
        cin, cout = cout, ch
        for j in range(layers_per_block):
            _resnet_shapes(s, f"{e}down_blocks.{i}.nets.{j}.", cin if j == 0 else cout, cout)
        if i != len(down_channels) - 1:
            s[f"{e}down_blocks.{i}.downsample.weight"], s[f"{e}down_blocks.{i}.downsample.bias"] = (cout, cout, 3, 3, 3), (cout,)
    _resnet_shapes(s, e + "mid_block.nets.0.", cout, cout)
    _resnet_shapes(s, e + "mid_block.nets.1.", cout, cout)
    if mid_attention:
        a = e + "mid_block.attns.0."
        s[a + "norm.weight"], s[a + "norm.bias"] = (cout,), (cout,)
        s[a + "attn.qkv.weight"] = (3 * cout, cout)
        s[a + "attn.proj.weight"], s[a + "attn.proj.bias"] = (cout, cout), (cout,)
    s[e + "norm_out.weight"], s[e + "norm_out.bias"] = (cout,), (cout,)
    s[e + "conv_out.weight"], s[e + "conv_out.bias"] = (2 * latent_channels, cout, 3, 3, 3), (2 * latent_channels,)
    s["quant_conv.weight"], s["quant_conv.bias"] = (2 * latent_channels,) * 2 + (1, 1, 1), (2 * latent_channels,)
    return s


def _std_for(name: str, shape) -> float:
    if name == "null_cond_embedding":
        return 1.0
    if "adaLN_modulation" in name or name.startswith("final_layer.linear") or name.startswith("t_embedder"):
        return 0.02
    if name.endswith(".bias"):
        return 0.02
    if len(shape) >= 2:
        fan_out = shape[0] * int(np.prod(shape[2:])) if len(shape) > 2 else shape[0]
        fan_in = int(np.prod(shape[1:]))
        if "upsample" in name or "conv_out" in name:   # ConvTranspose3d weight is [in, out, k, k, k]
            fan_in, fan_out = shape[0] * int(np.prod(shape[2:])), shape[1] * int(np.prod(shape[2:]))
        return math.sqrt(2.0 / (fan_in + fan_out))
    return 0.02


def synth_state_dict(shapes: Dict[str, Tuple[int, ...]], seed: int, fp16_roundtrip: bool = True) -> "OrderedDict[str, torch.Tensor]":
    """CPU fp32 tensors from numpy RandomState(seed); optionally rounded through fp16 (the shipped
    checkpoints are fp16: README.md:83-85)."""
    rs = np.random.RandomState(seed)
    sd = OrderedDict()
    for name, shape in shapes.items():
        a = rs.standard_normal(size=shape).astype(np.float32) * np.float32(_std_for(name, shape))
        if ("norm" in name) and name.endswith(".weight"):
            a = a * np.float32(5.0) + np.float32(1.0)      # GroupNorm gains around 1
        t = torch.from_numpy(a)
        sd[name] = t.half().float() if fp16_roundtrip else t
    return sd


def device_state_dict(shapes: Dict[str, Tuple[int, ...]], seed: int, device, dtype=torch.float16) -> "OrderedDict[str, torch.Tensor]":
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    sd = OrderedDict()
    for name, shape in shapes.items():
        t = torch.randn(shape, generator=g, device=device, dtype=torch.float32) * _std_for(name, shape)
        if ("norm" in name) and name.endswith(".weight"):
            t = t * 5.0 + 1.0
        sd[name] = t.to(dtype)
    return sd


def synth_inputs(B: int, N: int, Cin: int, M: int, Dc: int, seed: int = 42):
    """x_T, conditioning tokens: RandomState stand-ins for inference.py:316-317."""
    rs = np.random.RandomState(seed)
    x = torch.from_numpy(rs.standard_normal(size=(B, N, Cin)).astype(np.float32))
    y = torch.from_numpy(rs.standard_normal(size=(B, M, Dc)).astype(np.float32))
    return x, y
