"""Oracle restatement of VAE.encode and the posterior (TEST INFRASTRUCTURE, like oracle/): the encoder half of
/root/reference/models/vae3d_dib.py, built from the decoder oracle's blocks (oracle.vae.resnet_block / volume_attention / _conv).

  * VAE.encode                          vae3d_dib.py:431-435
  * Encoder.forward                     vae3d_dib.py:309-327   (conv_in, down blocks, mid block, GN+SiLU, conv_out)
  * DownBlock._forward                  vae3d_dib.py:176-184   (ResnetBlocks, then Conv3d(k3, s2, p1))
  * quant_conv                          vae3d_dib.py:428
  * DiagonalGaussianDistribution        vae3d_dib.py:50-90

Precision policies as in oracle/vae.py: ``fp32`` and ``fp16`` (the reference under torch.autocast(fp16)).
"""
from __future__ import annotations

import math
from typing import Dict

import torch
import torch.nn.functional as F

from oracle.dit import Policy
from oracle.vae import _conv, _gn, resnet_block, volume_attention

Tensor = torch.Tensor


def encode(sd: Dict[str, Tensor], x: Tensor, precision: str = "fp32", layers_per_block: int = 2, n_down: int = 2,
           stages: dict | None = None) -> Tensor:
    """VAE.encode up to the posterior's parameters: x [P,Cin,8,8,8] -> quant_conv(Encoder(x)) [P,2,4,4,4].  ``stages`` (optional dict)
    receives the activations after conv_in, down_blocks.0 (``down0``), down_blocks.1 (``down1``) and the mid block (``mid``)."""
    pol = Policy(precision)
    sd = {k: v.float() for k, v in sd.items()}
    e = "encoder."
    h = _conv(pol, x.float(), sd[e + "conv_in.weight"], sd[e + "conv_in.bias"], padding=1)
    if stages is not None:
        stages["conv_in"] = h
    for i in range(n_down):
        for j in range(layers_per_block):
            h = resnet_block(sd, f"{e}down_blocks.{i}.nets.{j}.", h, pol)
        if f"{e}down_blocks.{i}.downsample.weight" in sd:
            h = _conv(pol, h, sd[f"{e}down_blocks.{i}.downsample.weight"], sd[f"{e}down_blocks.{i}.downsample.bias"], stride=2, padding=1)
        if stages is not None:
            stages[f"down{i}"] = h
    h = resnet_block(sd, e + "mid_block.nets.0.", h, pol)
    if e + "mid_block.attns.0.norm.weight" in sd:
        h = volume_attention(sd, e + "mid_block.attns.0.", h, pol)
    h = resnet_block(sd, e + "mid_block.nets.1.", h, pol)
    if stages is not None:
        stages["mid"] = h
    h = F.silu(_gn(sd, e + "norm_out.", h))
    h = _conv(pol, h, sd[e + "conv_out.weight"], sd[e + "conv_out.bias"], padding=1)
    return _conv(pol, h, sd["quant_conv.weight"], sd["quant_conv.bias"])


def posterior(parameters: Tensor, deterministic: bool = False) -> dict:
    """DiagonalGaussianDistribution.__init__ (vae3d_dib.py:51-60): mean, clamped logvar, std, var in the parameters' dtype."""
    mean, logvar = torch.chunk(parameters, 2, dim=1)
    logvar = torch.clamp(logvar, -30.0, 20.0)
    std, var = torch.exp(0.5 * logvar), torch.exp(logvar)
    if deterministic:
        var = std = torch.zeros_like(mean)
    return dict(mean=mean, logvar=logvar, std=std, var=var)


def posterior_kl(p: dict, other: dict | None = None, dims=(1, 2, 3, 4)) -> Tensor:
    """DiagonalGaussianDistribution.kl (vae3d_dib.py:67-81), non-deterministic branch."""
    if other is None:
        return 0.5 * torch.mean(torch.pow(p["mean"], 2) + p["var"] - 1.0 - p["logvar"], dim=list(dims))
    return 0.5 * torch.mean(torch.pow(p["mean"] - other["mean"], 2) / other["var"] + p["var"] / other["var"] - 1.0 - p["logvar"] + other["logvar"],
                            dim=list(dims))


def posterior_nll(p: dict, sample: Tensor, dims=(1, 2, 3, 4)) -> Tensor:
    """DiagonalGaussianDistribution.nll (vae3d_dib.py:83-87), non-deterministic branch."""
    return 0.5 * torch.sum(math.log(2.0 * math.pi) + p["logvar"] + torch.pow(sample - p["mean"], 2) / p["var"], dim=list(dims))
