"""GPU: the CUDA path against THE REFERENCE'S OWN MODULES run on a B200 under ``torch.autocast('cuda', fp16)`` — the contract
north_star's tolerance is stated against (models/dit_crossattn.py:197, inference.py:339).

The reference's outputs are stored in ``tests/golden/ref_fp16.npz``: tests/golden/make_ref_fp16_golden.py ran the reference's
unmodified modules (staged by oracle/stage_ref.py, xformers restated by oracle/refmods.py) on a B200 over the inputs built
below, in fp16 autocast and in fp32 (TF32 off).  The fixture keeps a fixed sample of each fp16 output (every 32nd token of a
DiT output, every 128th token of each trajectory step, every 256th primitive of the VAE decode; the fp32 output too for the
VAE) and the reference's own fp16-vs-fp32 distance over the whole tensor.  Every test prints (relative L2):

    ours_vs_ref16     this repo's kernels vs the reference under CUDA autocast fp16, on the stored sample   <- the parity number
    oracle16_vs_ref16 the oracle's hand-written fp16 policy vs the real autocast, on the stored sample
    ref16_vs_ref32    the reference's own fp16 path vs its own fp32 path, whole tensor                      <- the contract's own noise

Tolerances.  A single forward without guidance must meet north_star's 1e-3 outright.  With CFG 6 the guidance arithmetic
``u + 6 (c - u)`` amplifies the fp16 rounding noise of BOTH implementations (the reference's own fp16 path then sits several
1e-3 from its fp32 path), so there the bound is the contract's own measured noise: ours_vs_ref16 <= 1.25 x ref16_vs_ref32
(two independent fp16 roundings of the same fp32 function differ by about sqrt(2) x their distance to it) and never
looser than 5e-3.

The weights and inputs of the DiT cases are drawn on the GPU; each case first checks them against fingerprints stored with
the fixture, so a changed random stream fails as such instead of as a parity error.
"""
import os

import numpy as np
import pytest
import torch

import oracle
import tpxl_b200
from tpxl_b200 import synth
from gpu_util import rel_l2

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
KW = dict(precision_dtype=torch.float16, enable_amp=True)
FIXTURE = "ref_fp16.npz"


def _no_tf32():
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False


# ---- inputs (shared with tests/golden/make_ref_fp16_golden.py) -------------------------------------------------------
def block_inputs():
    """One block at the shipped width (N=2048, D=1152, 16x72, M=1370): cfg, fp16 weights, x_T, conditioning, t."""
    cfg = dict(synth.FULL_DIT, depth=1)
    sd = synth.device_state_dict(synth.dit_shapes(**cfg), 201, DEV, torch.float16)
    g = torch.Generator(device=DEV).manual_seed(202)
    x, y = torch.randn(1, 2048, 68, generator=g, device=DEV), torch.randn(1, 1370, 768, generator=g, device=DEV)
    return cfg, sd, x, y, torch.tensor([600], device=DEV)


def full_inputs():
    """The shipped architecture (28 blocks), synthetic fp16 weights: cfg, weights, x_T, conditioning."""
    sd = synth.device_state_dict(synth.dit_shapes(**synth.FULL_DIT), 211, DEV, torch.float16)
    g = torch.Generator(device=DEV).manual_seed(212)
    x, y = torch.randn(1, 2048, 68, generator=g, device=DEV), torch.randn(1, 1370, 768, generator=g, device=DEV)
    return synth.FULL_DIT, sd, x, y


def vae_inputs():
    """config #4: decoder weights and 2048 primitive latents (numpy RandomState streams, drawn on the host)."""
    sd = synth.synth_state_dict(synth.vae_decoder_shapes(**synth.FULL_VAE), 221)
    rs = np.random.RandomState(222)
    z = torch.from_numpy((rs.standard_normal(size=(2048, 64)) * np.array(synth.LATENT_STD[4:]) + np.array(synth.LATENT_MEAN[4:])).astype(np.float32)).reshape(2048, 1, 4, 4, 4)
    return sd, z.to(DEV)


def fingerprint(sd, *tensors):
    """float64 sum of every weight and input tensor."""
    return np.array([float(v.double().sum()) for v in (*sd.values(), *tensors)])


def _check_inputs(g, key, sd, *tensors):
    np.testing.assert_allclose(fingerprint(sd, *tensors), g[key], rtol=1e-9, atol=0,
                               err_msg=f"the inputs differ from those {FIXTURE} was made from: the GPU random stream changed")


# ---- the tests --------------------------------------------------------------------------------------------------------
def _ours(cfg, sd):
    m = tpxl_b200.DiT(**{k: v for k, v in cfg.items() if k != "gradient_checkpointing"})
    m.load_state_dict(sd)
    return m.to(DEV).eval()


def _ref(g, key):
    return torch.from_numpy(g[key]).to(DEV).float()


def _report(tag, **r):
    print(f"[ref-fp16] {tag}: " + "  ".join(f"{k}={v:.3e}" for k, v in r.items()))
    return r


@pytest.fixture(scope="module")
def golden(golden_dir):
    return np.load(os.path.join(golden_dir, FIXTURE))


def test_one_full_width_block_forward_and_cfg(golden):
    """One block at the shipped width: forward and forward_with_cfg."""
    _no_tf32()
    g = golden
    cfg, sd, x, y, t = block_inputs()
    _check_inputs(g, "block_inputs", sd, x, y)
    m = _ours(cfg, sd)
    tok = torch.from_numpy(g["dit_tokens"]).to(DEV)
    sdf = {k: v.float() for k, v in sd.items()}
    with torch.no_grad():
        o = m.forward(x, t, y, **KW).float()[:, tok]
        o16 = oracle.dit.forward(sdf, x, t, y, 16, "fp16")[:, tok]
        oc = m.forward_with_cfg(x, t, y, cfg_scale=6.0, **KW).float()[:, tok]
        oc16 = oracle.dit.forward_with_cfg(sdf, x, t, y, 6.0, 16, "fp16")[:, tok]
    r16, c16 = _ref(g, "block_fwd16"), _ref(g, "block_cfg16")
    a = _report("1 block forward", ours_vs_ref16=rel_l2(o, r16), oracle16_vs_ref16=rel_l2(o16, r16), ref16_vs_ref32=float(g["block_fwd_noise"]))
    b = _report("1 block cfg=6", ours_vs_ref16=rel_l2(oc, c16), oracle16_vs_ref16=rel_l2(oc16, c16), ref16_vs_ref32=float(g["block_cfg_noise"]))
    assert a["ours_vs_ref16"] < 1e-3 and a["oracle16_vs_ref16"] < 1e-3
    assert b["ours_vs_ref16"] < max(1e-3, 1.25 * b["ref16_vs_ref32"]) and b["ours_vs_ref16"] < 5e-3


@pytest.fixture(scope="module")
def full(golden):
    """This repo's DiT at the shipped architecture (28 blocks) on the fixture's inputs."""
    _no_tf32()
    cfg, sd, x, y = full_inputs()
    _check_inputs(golden, "full_inputs", sd, x, y)
    m = _ours(cfg, sd)
    del sd
    yield m, x, y
    del m
    torch.cuda.empty_cache()


def test_full_depth_forward_and_cfg(golden, full):
    g = golden
    m, x, y = full
    t = torch.tensor([960], device=DEV)
    tok = torch.from_numpy(g["dit_tokens"]).to(DEV)
    with torch.no_grad():
        o = m.forward(x, t, y, **KW).float()[:, tok]
        oc = m.forward_with_cfg(x, t, y, cfg_scale=6.0, **KW).float()[:, tok]
    a = _report("28 blocks forward", ours_vs_ref16=rel_l2(o, _ref(g, "full_fwd16")), ref16_vs_ref32=float(g["full_fwd_noise"]))
    b = _report("28 blocks cfg=6", ours_vs_ref16=rel_l2(oc, _ref(g, "full_cfg16")), ref16_vs_ref32=float(g["full_cfg_noise"]))
    assert a["ours_vs_ref16"] < max(1e-3, 1.25 * a["ref16_vs_ref32"]) and a["ours_vs_ref16"] < 3e-3
    assert b["ours_vs_ref16"] < max(1e-3, 1.25 * b["ref16_vs_ref32"]) and b["ours_vs_ref16"] < 5e-3


def test_ddim25_trajectory_config2(golden, full):
    """Config #2 as a trajectory: the reference's own sampler driving the reference's DiT under autocast, 25 DDIM steps, CFG 6,
    against this repo's sampler driving this repo's DiT, same x_T and conditioning (inference.py:313-325)."""
    g = golden
    m, x, y = full
    odiff = tpxl_b200.create_diffusion("ddim25", noise_schedule="squaredcos_cap_v2", diffusion_steps=1000, parameterization="v")
    with torch.no_grad():
        mine = [s["sample"].clone() for s in odiff.ddim_sample_loop_progressive(m.forward_with_cfg, x.shape, x, clip_denoised=False,
                                                                                model_kwargs=dict(y=y, cfg_scale=6.0, **KW), progress=False, device=DEV)]
    t16, noise = _ref(g, "traj16"), [float(v) for v in g["traj_noise"]]
    tok = torch.from_numpy(g["traj_tokens"]).to(DEV)
    assert len(mine) == len(t16) == len(noise) == 25
    per_step = [rel_l2(a[:, tok], b) for a, b in zip(mine, t16)]
    r = _report("DDIM-25 trajectory", final_ours_vs_ref16=per_step[-1], max_ours_vs_ref16=max(per_step), final_ref16_vs_ref32=noise[-1],
                max_ref16_vs_ref32=max(noise))
    assert all(torch.isfinite(s).all() for s in mine)
    assert r["max_ours_vs_ref16"] < max(1e-3, 1.25 * r["max_ref16_vs_ref32"]) and r["max_ours_vs_ref16"] < 1e-2


def test_vae_decode_2048_primitives(golden):
    """config #4: VAE.decode of 2048 primitive latents.  The reference invokes it in fp32 (inference.py:337-340); under autocast it
    is the fp16 path.  Ours computes fp16 tensor-core convolutions for either input dtype; all 2048 primitives are decoded in one
    call and the fixture's primitives are compared."""
    _no_tf32()
    g = golden
    sd, z = vae_inputs()
    vae = tpxl_b200.VAE(**synth.FULL_VAE)
    vae.load_state_dict(sd)
    vae = vae.to(DEV)
    idx = torch.from_numpy(g["vae_prims"]).to(DEV)
    with torch.no_grad():
        o = vae.decode(z)
        assert o.shape == (2048, 6, 8, 8, 8)
        o = o[idx]
        o16 = vae.decode(z.half()).float()[idx]
    r16, r32 = _ref(g, "vae16"), _ref(g, "vae32")
    r = _report(f"VAE decode 2048 prims ({len(idx)} compared)", ours_vs_ref16=rel_l2(o, r16), ref16_vs_ref32=float(g["vae_noise"]),
                ours_vs_ref32=rel_l2(o, r32), ours_half_io_vs_ref16=rel_l2(o16, r16))
    per_prim = ((o - r32).flatten(1).norm(dim=1) / r32.flatten(1).norm(dim=1).clamp_min(1e-20))
    print(f"[ref-fp16] VAE per-primitive ours_vs_ref32: max={float(per_prim.max()):.3e} median={float(per_prim.median()):.3e}")
    assert r["ours_vs_ref32"] < max(1e-3, 1.5 * r["ref16_vs_ref32"]) and r["ours_vs_ref32"] < 5e-3
    assert r["ours_vs_ref16"] < max(1e-3, 1.5 * r["ref16_vs_ref32"])
    assert float(per_prim.max()) < 2e-2
