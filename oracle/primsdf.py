"""Oracle restatement of the PrimSDF point query (TEST INFRASTRUCTURE — see oracle/__init__.py).

Restates /root/reference/models/primsdf.py:
  * PrimSDF.prim_weight       :104-109  (inf-norm box weights, normalised by sum + 1e-6)
  * PrimSDF.grid_sample_feat  :65-102   (trilinear sample, align_corners=True, of the primitives with w > 0; at
                                          inference the SDF of uncovered points is approximated from the nearest voxel of
                                          the nearest primitive)
  * PrimSDF.forward           :52-63    (sdf raw; tex / mat clipped to [0,1])
Dense O(points x prims) torch math, for small problem sizes.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F


def fixture_scene(seed: int, K: int = 96, S: int = 8, n: int = 4000, dim_feat: int = 6):
    """The seeded scene of tests/golden/primsdf.npz (tests/golden/make_golden.py), rebuilt instead of stored: numpy
    RandomState(seed) draws, in this order, srt [K,4] (scale in [0.05, 0.25], centre in [-0.8, 0.8]^3), feat [K, dim_feat*S^3]
    standard normal and n points in [-1, 1]^3.  -> (srt, feat, pts), float32 arrays."""
    rs = np.random.RandomState(seed)
    srt = np.concatenate([rs.uniform(0.05, 0.25, size=(K, 1)), rs.uniform(-0.8, 0.8, size=(K, 3))], axis=1).astype(np.float32)
    feat = rs.standard_normal(size=(K, dim_feat * S ** 3)).astype(np.float32)
    pts = rs.uniform(-1, 1, size=(n, 3)).astype(np.float32)
    return srt, feat, pts


def local_grid(S: int) -> torch.Tensor:
    xx = torch.linspace(-1, 1, S)
    mx, my, mz = torch.meshgrid(xx, xx, xx, indexing="ij")
    return torch.stack((mz, my, mx), dim=-1).reshape(-1, 3)           # primsdf.py:38-41


def query(x: torch.Tensor, srt: torch.Tensor, feat: torch.Tensor, S: int = 8, dim_feat: int = 6, inference: bool = True):
    """x [n,3]; srt [K,4] = (scale, tx, ty, tz); feat [K, dim_feat*S^3] channel-major.  Returns dict sdf/tex/mat."""
    pos, scale = srt[:, 1:4], srt[:, 0:1]
    local = (x[:, None, :] - pos[None]) / scale[None]
    w = F.relu(1 - torch.norm(local, p=float("inf"), dim=-1))
    w = w / (w.sum(-1, keepdim=True) + 1e-6)
    ib, ip = torch.where(w > 0)
    pts = local[ib, ip].reshape(-1, 1, 1, 1, 3)
    vol = feat[ip].reshape(-1, dim_feat, S, S, S)
    samp = F.grid_sample(vol, pts, mode="bilinear", padding_mode="zeros", align_corners=True).reshape(-1, dim_feat)
    out = torch.zeros(x.shape[0], dim_feat, dtype=x.dtype, device=x.device)
    out.index_add_(0, ib, samp * w[ib, ip][:, None])
    if inference:
        miss = w.sum(1) <= 0
        if miss.any():
            xm = x[miss]
            near = torch.norm(xm[:, None, :] - pos[None], p=2, dim=-1).argmin(1)
            cand = pos[near][:, None, :] + scale[near][..., None] * local_grid(S).to(x)[None]
            dist, vi = torch.norm(xm[:, None, :] - cand, p=2, dim=-1).min(1)
            sdf = feat[:, : S ** 3][near, vi]
            out[miss, 0] = sdf + dist * torch.sign(sdf)
    return {"sdf": out[:, 0:1], "tex": out[:, 1:4].clip(0.0, 1.0), "mat": out[:, 4:6].clip(0.0, 1.0)}
