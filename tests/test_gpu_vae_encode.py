"""GPU: VAE.encode / VAE.forward and the encoder's kernels against F.conv3d / torch fp32, the oracle and the reference fixtures.

Tolerance: the encoder computes with fp16 tensor-core inputs, fp32 accumulation and fp32 GroupNorm statistics, one fp16 rounding
per layer (DESIGN §5); against the fp32 reference, relative L2 <= 1e-2 and within 2.5x the distance of the reference's own
fp16-autocast run (oracle fp16 policy, and the stored autocast run of tests/golden/make_vae_encode_fp16_golden.py)."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import oracle
import tpxl_b200
from tpxl_b200 import _lib, synth
from gpu_util import linear, rel_l2, st
import vae_encode_oracle as E

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ENC_SEED, DEC_SEED = 211, 103          # tests/golden/make_vae_encode_golden.py
FP16_FIXTURE = "vae_encode_fp16.npz"
FP16_PRIMS = np.arange(0, 2048, 128)


def _pack(w):   # [Cout,Cin,3,3,3] -> [Cout, 27*Cin], k = tap*Cin + ci
    return w.permute(0, 2, 3, 4, 1).reshape(w.shape[0], -1).contiguous()


def full_sd(enc_seed=ENC_SEED, dec_seed=DEC_SEED):
    sd = synth.synth_state_dict(synth.vae_decoder_shapes(**synth.FULL_VAE), dec_seed)
    sd.update(synth.synth_state_dict(synth.vae_encoder_shapes(**synth.FULL_VAE), enc_seed))
    return sd


def make_vae(sd):
    vae = tpxl_b200.VAE(**synth.FULL_VAE)
    vae.load_state_dict(sd)
    return vae.to(DEV)


def glue_inputs(P, seed):
    """P primitives in the range the sample -> decode glue hands the VAE: sdf * 5 and (rgb, material) * 2 - 1 (CPU, reproducible)."""
    rs = np.random.RandomState(seed)
    sdf = np.tanh(rs.standard_normal(size=(P, 1, 8, 8, 8)) * 0.5) * 0.8 * 5
    feat = rs.uniform(0.0, 1.0, size=(P, 5, 8, 8, 8)) * 2 - 1
    return torch.from_numpy(np.concatenate([sdf, feat], axis=1).astype(np.float32))


def fp16_inputs():
    """Shared with tests/golden/make_vae_encode_fp16_golden.py: synthetic weights and a 2048-primitive batch."""
    return full_sd(231, 232), glue_inputs(2048, 233)


def fingerprint(sd, *tensors):
    return np.array([float(v.double().sum()) for v in (*sd.values(), *tensors)])


# ---- kernels -------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("P", [1, 3, 2048])
def test_conv3d_stride2(P):
    g = torch.Generator(device=DEV).manual_seed(100 + P)
    x = torch.randn(P, 8, 8, 8, 32, generator=g, device=DEV).half()
    w = (torch.randn(32, 32, 3, 3, 3, generator=g, device=DEV) * (27 * 32) ** -0.5).half()
    b = torch.randn(32, generator=g, device=DEV).half()
    out = torch.empty(P, 4, 4, 4, 32, dtype=torch.float16, device=DEV)
    _lib.check(_lib.lib().tpx_conv3d_k3_s2(x.data_ptr(), _pack(w).data_ptr(), b.data_ptr(), out.data_ptr(), P, 32, 32, st()))
    ref = F.conv3d(x.float().permute(0, 4, 1, 2, 3), w.float(), b.float(), stride=2, padding=1).permute(0, 2, 3, 4, 1)
    torch.cuda.synchronize()
    assert rel_l2(out.float(), ref) < 2e-3


@pytest.mark.parametrize("P", [3, 5])
def test_conv3d_4cube_32_to_256(P):
    g = torch.Generator(device=DEV).manual_seed(200 + P)
    x = torch.randn(P, 4, 4, 4, 32, generator=g, device=DEV).half()
    w = (torch.randn(256, 32, 3, 3, 3, generator=g, device=DEV) * (27 * 32) ** -0.5).half()
    b = torch.randn(256, generator=g, device=DEV).half()
    out = torch.empty(P, 4, 4, 4, 256, dtype=torch.float16, device=DEV)
    _lib.check(_lib.lib().tpx_conv3d_k3(x.data_ptr(), _pack(w).data_ptr(), b.data_ptr(), None, 1.0, out.data_ptr(), P, 4, 32, 256, st()))
    ref = F.conv3d(x.float().permute(0, 4, 1, 2, 3), w.float(), b.float(), padding=1).permute(0, 2, 3, 4, 1)
    torch.cuda.synchronize()
    assert rel_l2(out.float(), ref) < 2e-3


@pytest.mark.parametrize("M", [64, 3 * 64, 2048 * 64])
def test_shortcut_k32_n256(M):
    g = torch.Generator(device=DEV).manual_seed(M)
    A = torch.randn(M, 32, generator=g, device=DEV).half()
    W = (torch.randn(256, 32, generator=g, device=DEV) * 32 ** -0.5).half()
    b = torch.randn(256, generator=g, device=DEV).half()
    out = linear(A, W, b, tile_n=256)
    torch.cuda.synchronize()
    assert rel_l2(out.float(), A.float() @ W.float().t() + b.float()) < 2e-3


@pytest.mark.parametrize("P", [1, 3, 2048])
def test_groupnorm_4cube_32ch(P):
    g = torch.Generator(device=DEV).manual_seed(300 + P)
    x = (torch.randn(P, 64, 32, generator=g, device=DEV) * 3 + 1).half()
    gamma = (torch.randn(32, generator=g, device=DEV) * 5 + 1).half()
    beta = torch.randn(32, generator=g, device=DEV).half()
    out = torch.empty_like(x)
    _lib.check(_lib.lib().tpx_groupnorm_silu(x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), P, 64, 32, 32, 1e-5, 1, out.data_ptr(), st()))
    xr = x.float().permute(0, 2, 1).reshape(P, 32, 4, 4, 4)
    ref = F.silu(F.group_norm(xr, 32, gamma.float(), beta.float(), eps=1e-5)).reshape(P, 32, 64).permute(0, 2, 1)
    torch.cuda.synchronize()
    assert rel_l2(out.float(), ref) < 2e-3


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
def test_pack_and_input_conv(dtype):
    sd = full_sd()
    vae = make_vae(sd)
    x = glue_inputs(5, 7).to(DEV).to(dtype)
    got = vae.encode_stage(x, 1)
    ref = F.conv3d(x.half().float(), sd["encoder.conv_in.weight"].to(DEV).half().float(), sd["encoder.conv_in.bias"].to(DEV).half().float(), padding=1)
    assert got.shape == (5, 32, 8, 8, 8)
    assert rel_l2(got.float(), ref) < 2e-3


def test_conv_out_with_quant_conv_epilogue():
    """norm_out, conv_out and the folded quant_conv on the encoder's own mid-block output, against torch fp32."""
    sd = full_sd()
    vae = make_vae(sd)
    x = glue_inputs(3, 8).to(DEV)
    mid = vae.encode_stage(x, 4).float()
    params = vae.encode(x).parameters
    s = {k: v.to(DEV) for k, v in sd.items()}
    h = F.silu(F.group_norm(mid, 32, s["encoder.norm_out.weight"], s["encoder.norm_out.bias"], eps=1e-5))
    h = F.conv3d(h.half().float(), s["encoder.conv_out.weight"].half().float(), s["encoder.conv_out.bias"].half().float(), padding=1)
    ref = F.conv3d(h.half().float(), s["quant_conv.weight"].half().float(), s["quant_conv.bias"].half().float())
    assert rel_l2(params, ref) < 2e-3


# ---- encode against the fixtures -----------------------------------------------------------------------------------------------
def test_encode_against_reference_fixture(golden_dir):
    g = np.load(os.path.join(golden_dir, "vae_encode.npz"))
    sd = full_sd()
    vae = make_vae(sd)
    x = torch.from_numpy(g["x"]).to(DEV)
    with torch.no_grad():
        p32 = vae.encode(x)
        p16 = vae.encode(x.half())
        o16 = E.encode({k: v.to(DEV) for k, v in sd.items()}, x, "fp16")
    o16p = E.posterior(o16)
    ref = {k: torch.from_numpy(g[k]).to(DEV) for k in ("parameters", "mean", "logvar", "std")}
    assert p32.parameters.dtype == torch.float32 and p16.parameters.dtype == torch.float16 and p32.parameters.shape == (4, 2, 4, 4, 4)
    for name, p in (("fp32", p32), ("fp16", p16)):
        for f in ("parameters", "std"):
            ours = rel_l2(getattr(p, f).float(), ref[f])
            bound = 2.5 * rel_l2(o16 if f == "parameters" else o16p["std"], ref[f]) + 1e-4
            print(f"{name} input, {f}: ours vs ref32 {ours:.3e}, bound {bound:.3e}")
            assert ours <= 1e-2 and ours <= bound, (name, f)
        assert getattr(p, "mean").dtype == p.parameters.dtype and p.logvar.dtype == p.parameters.dtype
    for i, k in ((1, "conv_in"), (2, "down0"), (3, "down1"), (4, "mid")):
        got = vae.encode_stage(x, i).float()
        r = rel_l2(got, torch.from_numpy(g["stage_" + k]).to(DEV).float())
        print(f"stage {k}: {r:.3e}")
        assert r < 1e-2, k


def test_encode_against_autocast_fixture(golden_dir):
    path = os.path.join(golden_dir, FP16_FIXTURE)
    if not os.path.exists(path):
        pytest.skip(f"{FP16_FIXTURE} not generated yet: run tests/golden/make_vae_encode_fp16_golden.py on a B200")
    g = np.load(path)
    sd, x = fp16_inputs()
    np.testing.assert_allclose(fingerprint(sd, x), g["inputs"], rtol=1e-9, atol=0)
    vae = make_vae(sd)
    with torch.no_grad():
        p = vae.encode(x.to(DEV))
    idx = torch.from_numpy(FP16_PRIMS).to(DEV)
    for f in ("parameters", "std"):
        ours = rel_l2(getattr(p, f).index_select(0, idx), torch.from_numpy(g[f + "32"]).to(DEV))
        ref16 = rel_l2(torch.from_numpy(g[f + "16"]).float(), torch.from_numpy(g[f + "32"]))
        print(f"{f}: ours vs ref32 {ours:.3e}; ref16 vs ref32 {ref16:.3e} (sample), {float(g[f + '_noise']):.3e} (whole batch)")
        assert ours <= 2.5 * ref16 + 1e-4


def test_logvar_clamp():
    sd = full_sd()
    sd["quant_conv.weight"] = sd["quant_conv.weight"].clone()
    sd["quant_conv.weight"][1] *= 400.0          # the logvar row: the clamp acts at both ends for a visible share
    vae = make_vae(sd)
    x = glue_inputs(64, 9).to(DEV)
    with torch.no_grad():
        p = vae.encode(x)
        ref = E.posterior(E.encode({k: v.to(DEV) for k, v in sd.items()}, x, "fp32"))
    lo, hi = float((p.logvar == -30).float().mean()), float((p.logvar == 20).float().mean())
    print(f"clamped low {lo:.3f}, high {hi:.3f}")
    assert lo > 0.05 and hi > 0.05
    assert rel_l2(p.logvar, ref["logvar"]) < 1e-2
    assert rel_l2(p.mean, ref["mean"]) < 1e-2
    both = ((ref["logvar"] == -30) | (ref["logvar"] == 20)) & (p.logvar == ref["logvar"])
    torch.testing.assert_close(p.std[both], ref["std"][both], rtol=1e-6, atol=0)
    torch.testing.assert_close(p.var[both], ref["var"][both], rtol=1e-6, atol=0)


def test_posterior_and_rng():
    vae = make_vae(full_sd())
    x = glue_inputs(6, 10).to(DEV)
    for dtype in (torch.float32, torch.float16):
        p = vae.encode(x.to(dtype))
        torch.manual_seed(1234)
        s = p.sample()
        torch.manual_seed(1234)
        n = torch.randn(p.mean.shape, device=DEV, dtype=dtype)
        assert torch.equal(s, p.mean + p.std * n)
        d = tpxl_b200.vae.DiagonalGaussianDistribution(p.parameters, deterministic=True)
        assert not d.std.any() and not d.var.any() and torch.equal(d.logvar, p.logvar)
        assert torch.equal(d.kl(), torch.Tensor([0.0])) and torch.equal(d.nll(s), torch.Tensor([0.0]))
    p = vae.encode(x)
    ref = E.posterior(p.parameters)
    for f in ("mean", "logvar", "std", "var"):
        assert rel_l2(getattr(p, f), ref[f]) < 1e-6, f
    q = vae.encode(glue_inputs(6, 11).to(DEV))
    assert rel_l2(p.kl(), E.posterior_kl(ref)) < 1e-5
    assert rel_l2(p.kl(q), E.posterior_kl(ref, E.posterior(q.parameters))) < 1e-5
    s = p.sample()
    assert rel_l2(p.nll(s), E.posterior_nll(ref, s)) < 1e-5


def test_forward():
    vae = make_vae(full_sd())
    x = glue_inputs(5, 12).to(DEV)
    with torch.no_grad():
        out, post = vae.forward(x, sample=False)
        again = vae.decode(vae.encode(x).mode())
        out_s, post_s = vae(x)
        out16, post16 = vae(x.half(), sample=False)
    assert torch.equal(out, again)
    assert out.shape == (5, 6, 8, 8, 8) and out.dtype == torch.float32 and isinstance(post, tpxl_b200.vae.DiagonalGaussianDistribution)
    assert out_s.shape == out.shape and post_s.parameters.shape == (5, 2, 4, 4, 4)
    assert out16.dtype == torch.float16 and post16.parameters.dtype == torch.float16


def test_encode_full_batch_properties():
    """2048 primitives: finite, deterministic, primitive-wise independent, and 256 strided primitives against the oracle."""
    sd = full_sd(71, 72)
    vae = make_vae(sd)
    x = glue_inputs(2048, 73).to(DEV)
    with torch.no_grad():
        full = vae.encode(x).parameters
        again = vae.encode(x).parameters
        part = vae.encode(x[1000:1007].contiguous()).parameters
        sub = x[3::8].contiguous()
        ref = E.encode({k: v.to(DEV) for k, v in sd.items()}, sub, "fp32")
    assert torch.isfinite(full).all() and torch.equal(full, again)
    assert torch.equal(part, full[1000:1007])
    got = full[3::8]
    per_prim = (got - ref).flatten(1).norm(dim=1) / ref.flatten(1).norm(dim=1).clamp_min(1e-20)
    print("256 strided primitives vs oracle fp32: rel-L2", rel_l2(got, ref), "worst primitive", float(per_prim.max()))
    assert rel_l2(got, ref) < 1e-2 and float(per_prim.max()) < 3e-2


def test_decode_unchanged_by_encoder_handle():
    vae = make_vae(full_sd())
    z = torch.randn(37, 1, 4, 4, 4, device=DEV)
    before = vae.decode(z)
    vae.encode(glue_inputs(9, 13).to(DEV))
    assert vae._enc is not None
    assert torch.equal(vae.decode(z), before)


def test_error_paths():
    sd = full_sd()
    vae = make_vae(sd)
    with pytest.raises(ValueError):
        vae.encode(torch.zeros(1, 6, 4, 4, 4, device=DEV))
    with pytest.raises(ValueError):
        vae.encode(torch.zeros(1, 5, 8, 8, 8, device=DEV))
    p = vae.encode(torch.zeros(0, 6, 8, 8, 8, device=DEV))
    assert p.parameters.shape == (0, 2, 4, 4, 4) and p.std.shape == (0, 1, 4, 4, 4) and p.sample().shape == (0, 1, 4, 4, 4)
    bad = dict(sd)
    del bad["encoder.down_blocks.1.nets.0.shortcut.weight"]
    vae.load_state_dict(bad)                             # load_state_dict accepts what it accepted before ...
    assert vae._enc is None                              # ... and drops the encoder handle
    with pytest.raises(_lib.TpxError, match="encoder.down_blocks.1.nets.0.shortcut.weight"):
        vae.encode(torch.zeros(1, 6, 8, 8, 8, device=DEV))
    bad = dict(sd)
    bad["encoder.conv_out.weight"] = torch.zeros(2, 256, 1, 1, 1)
    vae.load_state_dict(bad)
    with pytest.raises(_lib.TpxError, match="encoder.conv_out.weight"):
        vae.encode(torch.zeros(1, 6, 8, 8, 8, device=DEV))
    other = tpxl_b200.VAE(**dict(synth.FULL_VAE, down_channels=[16, 32]))
    other.load_state_dict(sd)
    other = other.to(DEV)
    with pytest.raises(NotImplementedError, match="down_channels"):
        other.encode(torch.zeros(1, 6, 8, 8, 8, device=DEV))


def test_device_move_drops_encoder_handle():
    vae = make_vae(full_sd())
    x = glue_inputs(4, 14).to(DEV)
    a = vae.encode(x).parameters
    vae = vae.cpu()
    assert vae._enc is None
    with pytest.raises(NotImplementedError):
        vae.encode(x)
    vae = vae.to(DEV)
    assert torch.equal(vae.encode(x).parameters, a)
