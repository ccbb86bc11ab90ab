#!/usr/bin/env python
"""Generate tests/golden/ref_fp16.npz: what tests/test_gpu_ref_fp16.py compares the CUDA path with.

Runs THE REFERENCE'S OWN MODULES (staged unmodified under oracle/_ref by oracle/stage_ref.py; the xformers attention restated
by oracle/refmods.py) on a B200, under torch.autocast('cuda', fp16) and in fp32 with TF32 off, over the inputs the test builds
(its block_inputs / full_inputs / vae_inputs).  Needs a GPU and the staged reference:

    python oracle/stage_ref.py && python tests/golden/make_ref_fp16_golden.py [OUT]     # OUT defaults to tests/golden/ref_fp16.npz

Stored, to stay well under 1 MB: a fixed sample of every fp16 output (every 32nd token of the DiT outputs, every 128th token
of each of the 25 DDIM samples, every 256th primitive of the VAE decode, also in fp32), the reference's fp16-vs-fp32
relative L2 over each whole tensor, and float64 fingerprints of the GPU-drawn DiT weights and inputs.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import test_gpu_ref_fp16 as T                     # noqa: E402
from gpu_util import rel_l2                       # noqa: E402
from oracle import refmods                        # noqa: E402
from tpxl_b200 import synth                       # noqa: E402

DEV = T.DEV
DIT_TOKENS = np.arange(0, 2048, 32)
TRAJ_TOKENS = np.arange(0, 2048, 128)
VAE_PRIMS = np.arange(0, 2048, 256)


def _sample(t, idx, dim):
    return t.index_select(dim, torch.from_numpy(idx).to(t.device)).cpu().numpy()


def main(out):
    if not refmods.available():
        raise SystemExit("oracle/_ref is not staged: run python oracle/stage_ref.py where the reference checkout exists")
    torch.set_grad_enabled(False)
    T._no_tf32()
    fx = dict(dit_tokens=DIT_TOKENS, traj_tokens=TRAJ_TOKENS, vae_prims=VAE_PRIMS,
              made_on=f"{torch.cuda.get_device_name(DEV)}, torch {torch.__version__}")
    fp32 = dict(precision_dtype=torch.float32, enable_amp=False)

    cfg, sd, x, y, t = T.block_inputs()
    fx["block_inputs"] = T.fingerprint(sd, x, y)
    ref = refmods.build_dit(cfg, sd, DEV)
    for tag, fn in (("fwd", lambda **kw: ref.forward(x, t, y, **kw)), ("cfg", lambda **kw: ref.forward_with_cfg(x, t, y, cfg_scale=6.0, **kw))):
        r16, r32 = fn(**T.KW), fn(**fp32)
        fx[f"block_{tag}16"], fx[f"block_{tag}_noise"] = _sample(r16, DIT_TOKENS, 1), rel_l2(r16, r32)
    del ref, sd

    cfg, sd, x, y = T.full_inputs()
    fx["full_inputs"] = T.fingerprint(sd, x, y)
    ref = refmods.build_dit(cfg, sd, DEV)
    del sd
    t = torch.tensor([960], device=DEV)
    for tag, fn in (("fwd", lambda **kw: ref.forward(x, t, y, **kw)), ("cfg", lambda **kw: ref.forward_with_cfg(x, t, y, cfg_scale=6.0, **kw))):
        r16, r32 = fn(**T.KW), fn(**fp32)
        fx[f"full_{tag}16"], fx[f"full_{tag}_noise"] = _sample(r16, DIT_TOKENS, 1), rel_l2(r16, r32)
    rdiff = refmods.load().create_diffusion("ddim25", noise_schedule="squaredcos_cap_v2", diffusion_steps=1000, parameterization="v")
    traj = {}
    for tag, kw in (("16", T.KW), ("32", fp32)):
        traj[tag] = [s["sample"].clone() for s in rdiff.ddim_sample_loop_progressive(ref.forward_with_cfg, x.shape, x, clip_denoised=False,
                                                                                     model_kwargs=dict(y=y, cfg_scale=6.0, **kw), progress=False, device=DEV)]
    fx["traj16"] = np.stack([_sample(s, TRAJ_TOKENS, 1) for s in traj["16"]])
    fx["traj_noise"] = np.array([rel_l2(a, b) for a, b in zip(traj["16"], traj["32"])])
    del ref, traj
    torch.cuda.empty_cache()

    sd, z = T.vae_inputs()
    ref = refmods.build_vae(synth.FULL_VAE, sd, DEV)
    r32 = torch.cat([ref.decode(z[i:i + 256]) for i in range(0, 2048, 256)])
    with torch.autocast("cuda", dtype=torch.float16):
        r16 = torch.cat([ref.decode(z[i:i + 256]) for i in range(0, 2048, 256)])
    fx["vae16"], fx["vae32"], fx["vae_noise"] = _sample(r16, VAE_PRIMS, 0), _sample(r32, VAE_PRIMS, 0), rel_l2(r16.float(), r32)

    np.savez_compressed(out, **fx)
    print(fx["made_on"], "->", out, f"{os.path.getsize(out)} bytes")
    for k, v in fx.items():
        if k.endswith("_noise"):
            print(f"  {k}: ref16_vs_ref32 = {np.max(v):.3e}")
        elif isinstance(v, np.ndarray) and v.ndim > 1:
            print(f"  {k}: {v.shape} {v.dtype}")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden", "ref_fp16.npz"))
