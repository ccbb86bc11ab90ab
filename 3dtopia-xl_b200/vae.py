"""Host-side mirror of the reference's VAE interface, backed by libtpx_b200.

Drop-in for ``models.vae3d_dib.VAE`` (/root/reference/models/vae3d_dib.py:391-453): same constructor kwargs
(configs/inference_dit.yml:31-40), ``load_state_dict(sd['model_state_dict'])`` with the reference key names,
``decode(z[P,1,4,4,4]) -> [P,6,8,8,8]`` in z's dtype, returned as a fresh contiguous tensor (the caller mutates it in
place, inference.py:345-346).
``encode(x[P,6,8,8,8])`` returns a ``DiagonalGaussianDistribution`` (vae3d_dib.py:50-90) in x's dtype and ``forward(x, sample)``
returns ``(decode(z), posterior)`` (:431-453).  The encoder runs on its own C handle, built on the first ``encode`` from the
encoder.* / quant_conv.* tensors ``load_state_dict`` keeps; ``load_checkpoint`` reads the decoder half only, so encoding needs
``load_state_dict(sd['model_state_dict'])``.  Every compute path needs the module on a CUDA device: there is no CPU path.
"""
from __future__ import annotations

import ctypes as C
from collections import OrderedDict
from typing import Optional

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from .synth import vae_decoder_shapes, vae_encoder_shapes


class VAE(nn.Module):
    def __init__(self, in_channels=1, latent_channels=16, out_channels=1, down_channels=(16, 32, 64, 128, 256), mid_attention=True,
                 up_channels=(256, 128, 64, 32, 16), layers_per_block=2, skip_scale=None, gradient_checkpointing=False):
        super().__init__()
        up_channels = tuple(up_channels)
        if not (latent_channels == 1 and up_channels == (256, 32) and mid_attention and layers_per_block == 2 and skip_scale is None):
            raise NotImplementedError("the B200 decoder kernel set covers the released configuration (configs/inference_dit.yml:31-40): "
                                      f"latent_channels=1, up_channels=[256,32], mid_attention, layers_per_block=2; got latent={latent_channels}, "
                                      f"up={list(up_channels)}, mid_attention={mid_attention}, layers={layers_per_block}")
        self.in_channels, self.latent_channels, self.out_channels = in_channels, latent_channels, out_channels
        self.up_channels = up_channels
        self.down_channels, self.mid_attention = tuple(down_channels), mid_attention
        self._shapes = vae_decoder_shapes(latent_channels=latent_channels, out_channels=out_channels, up_channels=up_channels,
                                          mid_attention=mid_attention, layers_per_block=layers_per_block)
        self._anchor = nn.Parameter(torch.zeros(1), requires_grad=False)
        self._sd: Optional["OrderedDict[str, torch.Tensor]"] = None
        self._extra = OrderedDict()   # encoder.* / quant_conv.* tensors, kept only so state_dict() round-trips
        self._handle = None
        self._handle_device = None
        self._ws = {}
        self._enc = None          # encoder handle: created by the first encode, dropped by load_state_dict and device moves
        self._enc_device = None
        self._enc_ws = {}

    def state_dict(self, *args, **kwargs):
        if self._sd is None:
            raise _lib.TpxError("VAE has no parameters yet: load_state_dict first (random initialisation of a decoder is not an inference path)")
        out = OrderedDict(self._extra)
        out.update(self._sd)
        return out

    def load_state_dict(self, state_dict, strict: bool = True, assign: bool = False):
        missing = [k for k in self._shapes if k not in state_dict]
        unexpected = [k for k in state_dict if k not in self._shapes and not k.startswith(("encoder.", "quant_conv."))]
        errs = [f"size mismatch for {k}: copying a param with shape {tuple(state_dict[k].shape)}, expected {tuple(s)}"
                for k, s in self._shapes.items() if k in state_dict and tuple(state_dict[k].shape) != tuple(s)]
        if strict and (missing or unexpected):
            errs.append(f"Missing key(s): {missing[:5]}; unexpected key(s): {unexpected[:5]}")
        if errs:
            raise RuntimeError("Error(s) in loading state_dict for VAE:\n\t" + "\n\t".join(errs))
        self._sd = OrderedDict((k, state_dict[k].detach()) for k in self._shapes if k in state_dict)
        self._extra = OrderedDict((k, v) for k, v in state_dict.items() if k.startswith(("encoder.", "quant_conv.")))
        self._destroy_encoder()
        if self._handle is not None:
            self._ingest()
        return torch.nn.modules.module._IncompatibleKeys(missing, unexpected)

    def load_checkpoint(self, path: str, key: Optional[str] = "model_state_dict"):
        """``vae.load_state_dict(torch.load(path, map_location='cpu')['model_state_dict'])`` (inference.py:257-258) from a memory-mapped
        file: only decoder.* / post_quant_conv.* tensors are read and uploaded (the encoder half of the checkpoint is never touched, so
        ``encode`` after this raises; load the full ``sd['model_state_dict']`` with ``load_state_dict`` to encode)."""
        try:
            ck = torch.load(path, map_location="cpu", mmap=True, weights_only=True)
        except (RuntimeError, ValueError, TypeError):
            ck = torch.load(path, map_location="cpu", weights_only=True)
        sd = ck[key] if key is not None else ck
        return self.load_state_dict(OrderedDict((k, v) for k, v in sd.items() if not k.startswith(("encoder.", "quant_conv."))))

    def _apply(self, fn, recurse=True):
        out = super()._apply(fn, recurse)
        dev = self._anchor.device
        if self._enc is not None and self._enc_device != dev:
            self._destroy_encoder()
        if dev.type == "cuda" and (self._handle is None or self._handle_device != dev):
            self._create_handle(dev)
        return out

    def _create_handle(self, dev):
        lib = _lib.lib()
        self._destroy_handle()
        cfg = _lib.VaeConfig(self.latent_channels, self.out_channels, self.up_channels[0], self.up_channels[1], 8)
        h = C.c_void_p()
        with torch.cuda.device(dev):
            _lib.check(lib.tpx_vae_create(C.byref(cfg), C.byref(h)), "tpx_vae_create")
        self._handle, self._handle_device = h, dev
        self._ws.clear()
        if self._sd is not None:
            self._ingest()

    def _ingest(self):
        lib = _lib.lib()
        dev = self._handle_device
        with torch.cuda.device(dev):
            st = _lib.stream_ptr()
            keep = []
            for k, v in self._sd.items():
                t = v.detach()
                if t.dtype not in (torch.float16, torch.float32):
                    t = t.float()
                t = t.to(dev, non_blocking=True).contiguous()
                keep.append(t)
                shape = (C.c_int64 * t.dim())(*t.shape)
                _lib.check(lib.tpx_vae_set_weight(self._handle, k.encode(), t.data_ptr(), _lib.dtype_tag(t), shape, t.dim(), st), f"set_weight({k})")
            _lib.check(lib.tpx_vae_finalize(self._handle, st), "tpx_vae_finalize")
            torch.cuda.current_stream().synchronize()

    def _destroy_handle(self):
        if self.__dict__.get("_handle") is not None:
            try:
                _lib.load_library().tpx_vae_destroy(self._handle)
            except Exception:
                pass
            self.__dict__["_handle"] = None      # not nn.Module.__setattr__: this also runs at interpreter shutdown

    def _destroy_encoder(self):
        if self.__dict__.get("_enc") is not None:
            try:
                _lib.load_library().tpx_vae_encoder_destroy(self._enc)
            except Exception:
                pass
            self.__dict__["_enc"] = None
        self.__dict__.get("_enc_ws", {}).clear()

    def __del__(self):
        self._destroy_encoder()
        self._destroy_handle()

    def decode(self, x: torch.Tensor) -> torch.Tensor:
        """VAE.decode (vae3d_dib.py:437-440)."""
        if self._handle is None:
            raise _lib.TpxError("VAE is not on a CUDA device: call .to('cuda') first (this implementation has no CPU path)")
        if self._sd is None:
            raise _lib.TpxError("VAE.decode before load_state_dict")
        if x.dim() != 5 or tuple(x.shape[1:]) != (self.latent_channels, 4, 4, 4):
            raise ValueError(f"z must be [P,{self.latent_channels},4,4,4], got {tuple(x.shape)}")
        lib = _lib.lib()
        dev = self._handle_device
        z = x.detach().to(dev)
        if z.dtype not in (torch.float16, torch.float32):
            z = z.float()
        z = z.contiguous()
        P = z.shape[0]
        out = torch.empty(P, self.out_channels, 8, 8, 8, dtype=z.dtype, device=dev)
        if P == 0:
            return out
        with torch.cuda.device(dev):
            nbytes = lib.tpx_vae_workspace_bytes(self._handle, P)
            ws = self._ws.get(P)
            if ws is None:
                self._ws.clear()
                ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=dev)
                self._ws[P] = ws
            base = (ws.data_ptr() + 255) & ~255
            _lib.check(lib.tpx_vae_decode(self._handle, z.data_ptr(), _lib.dtype_tag(z), out.data_ptr(), _lib.dtype_tag(out), P, base, nbytes,
                                          _lib.stream_ptr()), "tpx_vae_decode")
        return out

    def _encoder(self):
        """The encoder handle, built from the encoder.* / quant_conv.* tensors of the last load_state_dict on first use."""
        if self._enc is not None:
            return self._enc
        if self.down_channels != (32, 256) or not self.mid_attention:
            raise NotImplementedError("the B200 encoder kernel set covers the released configuration (configs/inference_dit.yml:31-40): "
                                      f"down_channels=[32,256] with mid_attention; got down={list(self.down_channels)}, "
                                      f"mid_attention={self.mid_attention}")
        if self._sd is None:
            raise _lib.TpxError("VAE.encode before load_state_dict")
        shapes = vae_encoder_shapes(in_channels=self.in_channels, latent_channels=self.latent_channels, down_channels=self.down_channels,
                                    mid_attention=self.mid_attention)
        for k, shp in shapes.items():
            if k not in self._extra:
                raise _lib.TpxError(f"VAE.encode: encoder key '{k}' missing from the loaded state_dict (load_checkpoint reads the decoder half "
                                    "only; use load_state_dict(sd['model_state_dict']) to encode)")
            if tuple(self._extra[k].shape) != tuple(shp):
                raise _lib.TpxError(f"VAE.encode: size mismatch for {k}: loaded {tuple(self._extra[k].shape)}, expected {tuple(shp)}")
        lib = _lib.lib()
        dev = self._handle_device
        cfg = _lib.VaeEncoderConfig(self.in_channels, self.latent_channels, self.down_channels[0], self.down_channels[1], 8)
        h = C.c_void_p()
        with torch.cuda.device(dev):
            _lib.check(lib.tpx_vae_encoder_create(C.byref(cfg), C.byref(h)), "tpx_vae_encoder_create")
            try:
                st = _lib.stream_ptr()
                keep = []
                for k in shapes:
                    t = self._extra[k].detach()
                    if t.dtype not in (torch.float16, torch.float32):
                        t = t.float()
                    t = t.to(dev, non_blocking=True).contiguous()
                    keep.append(t)
                    shape = (C.c_int64 * t.dim())(*t.shape)
                    _lib.check(lib.tpx_vae_encoder_set_weight(h, k.encode(), t.data_ptr(), _lib.dtype_tag(t), shape, t.dim(), st), f"set_weight({k})")
                _lib.check(lib.tpx_vae_encoder_finalize(h, st), "tpx_vae_encoder_finalize")
                torch.cuda.current_stream().synchronize()
            except Exception:
                lib.tpx_vae_encoder_destroy(h)
                raise
        self._enc, self._enc_device = h, self._anchor.device
        return h

    def _check_cuda(self, what: str):
        if self._anchor.device.type != "cuda" or self._handle is None:
            raise NotImplementedError(f"VAE.{what} needs the module on a CUDA device (.to('cuda')): this implementation has no CPU path")

    def _workspace(self, cache: dict, nbytes: int, P: int):
        ws = cache.get(P)
        if ws is None:
            cache.clear()
            ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=self._handle_device)
            cache[P] = ws
        return (ws.data_ptr() + 255) & ~255

    def _prepare_input(self, x: torch.Tensor) -> torch.Tensor:
        if x.dim() != 5 or tuple(x.shape[1:]) != (self.in_channels, 8, 8, 8):
            raise ValueError(f"x must be [P,{self.in_channels},8,8,8], got {tuple(x.shape)}")
        t = x.detach().to(self._handle_device)
        if t.dtype not in (torch.float16, torch.float32):
            t = t.float()
        return t.contiguous()

    def encode_stage(self, x: torch.Tensor, stage: int) -> torch.Tensor:
        """The encoder's activation after stage 1 conv_in, 2 down_blocks.0, 3 down_blocks.1 or 4 mid_block, as fp16 NCDHW (parity aid)."""
        self._check_cuda("encode_stage")
        h = self._encoder()
        t = self._prepare_input(x)
        P = t.shape[0]
        S, Cc = (8, self.down_channels[0]) if stage == 1 else (4, self.down_channels[0] if stage == 2 else self.down_channels[1])
        out = torch.empty(P, S, S, S, Cc, dtype=torch.float16, device=self._handle_device)
        if P:
            lib = _lib.lib()
            with torch.cuda.device(self._handle_device):
                nbytes = lib.tpx_vae_encoder_workspace_bytes(h, P)
                base = self._workspace(self._enc_ws, nbytes, P)
                _lib.check(lib.tpx_vae_encode_stage(h, t.data_ptr(), _lib.dtype_tag(t), P, stage, out.data_ptr(), base, nbytes, _lib.stream_ptr()),
                           "tpx_vae_encode_stage")
        return out.permute(0, 4, 1, 2, 3)

    def encode(self, x: torch.Tensor) -> "DiagonalGaussianDistribution":
        """VAE.encode (vae3d_dib.py:431-435): x [P, in_channels, 8, 8, 8] fp32 / fp16 -> posterior over [P, latent, 4, 4, 4] in x's dtype."""
        self._check_cuda("encode")
        h = self._encoder()
        t = self._prepare_input(x)
        P = t.shape[0]
        params = torch.empty(P, 2 * self.latent_channels, 4, 4, 4, dtype=t.dtype, device=self._handle_device)
        if P:
            lib = _lib.lib()
            with torch.cuda.device(self._handle_device):
                nbytes = lib.tpx_vae_encoder_workspace_bytes(h, P)
                base = self._workspace(self._enc_ws, nbytes, P)
                _lib.check(lib.tpx_vae_encode(h, t.data_ptr(), _lib.dtype_tag(t), params.data_ptr(), _lib.dtype_tag(params), P, base, nbytes,
                                              _lib.stream_ptr()), "tpx_vae_encode")
        return DiagonalGaussianDistribution(params)

    def forward(self, x, sample=True):
        """VAE.forward (vae3d_dib.py:442-453): (decode(z), posterior), z = posterior.sample() or posterior.mode()."""
        self._check_cuda("forward")
        p = self.encode(x)
        z = p.sample() if sample else p.mode()
        return self.decode(z), p


class DiagonalGaussianDistribution:
    """vae3d_dib.py:50-90.  The fields come from one tpx_vae_posterior launch over ``parameters`` (a CUDA fp32 / fp16 tensor
    [B, 2C, ...]); ``mean`` is a view of its first half along dim 1, as torch.chunk gives it."""

    def __init__(self, parameters, deterministic=False):
        if not (isinstance(parameters, torch.Tensor) and parameters.is_cuda):
            raise NotImplementedError("DiagonalGaussianDistribution needs CUDA parameters: this implementation has no CPU path")
        if parameters.dim() < 2 or parameters.shape[1] % 2 != 0:
            raise ValueError(f"parameters must be [B, 2C, ...], got {tuple(parameters.shape)}")
        self.parameters = parameters
        self.mean, lv_view = torch.chunk(parameters, 2, dim=1)
        self.deterministic = deterministic
        src = parameters.detach().contiguous()
        B = parameters.shape[0]
        half = lv_view.numel() // B if B else 0
        self.logvar = torch.empty_like(lv_view, memory_format=torch.contiguous_format)
        self.std = torch.empty_like(self.logvar)
        self.var = torch.empty_like(self.logvar)
        if self.logvar.numel():
            lib = _lib.lib()
            with torch.cuda.device(parameters.device):
                _lib.check(lib.tpx_vae_posterior(src.data_ptr(), _lib.dtype_tag(src), B, half, 1 if deterministic else 0, self.logvar.data_ptr(),
                                                 self.std.data_ptr(), self.var.data_ptr(), _lib.stream_ptr()), "tpx_vae_posterior")

    def sample(self):
        sample = torch.randn(self.mean.shape, device=self.parameters.device, dtype=self.parameters.dtype)
        return self.mean + self.std * sample

    def kl(self, other=None, dims=[1, 2, 3, 4]):
        if self.deterministic:
            return torch.Tensor([0.0])
        if other is None:
            return 0.5 * torch.mean(torch.pow(self.mean, 2) + self.var - 1.0 - self.logvar, dim=dims)
        return 0.5 * torch.mean(torch.pow(self.mean - other.mean, 2) / other.var + self.var / other.var - 1.0 - self.logvar + other.logvar, dim=dims)

    def nll(self, sample, dims=[1, 2, 3, 4]):
        if self.deterministic:
            return torch.Tensor([0.0])
        logtwopi = np.log(2.0 * np.pi)
        return 0.5 * torch.sum(logtwopi + self.logvar + torch.pow(sample - self.mean, 2) / self.var, dim=dims)

    def mode(self):
        return self.mean
