"""CPU: the oracle (oracle/*.py) against fixtures generated from the reference's own modules
(tests/golden/make_golden.py).  fp32 throughout; tolerances are fp32 round-off of different op orders."""
import json
import os

import numpy as np
import pytest
import torch

import oracle
from tpxl_b200 import synth


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name), allow_pickle=False)


def _rel(a, b):
    a, b = torch.as_tensor(a).double(), torch.as_tensor(b).double()
    return float((a - b).norm() / b.norm())


def test_state_dict_key_contract(golden_dir):
    keys = json.load(open(os.path.join(golden_dir, "state_dict_keys.json")))
    assert {k: tuple(v) for k, v in keys["dit"].items()} == dict(synth.dit_shapes(**synth.FULL_DIT))
    dec = {k: tuple(v) for k, v in keys["vae"].items() if k.startswith(("decoder.", "post_quant_conv."))}
    assert dec == dict(synth.vae_decoder_shapes(**synth.FULL_VAE))
    assert sum(int(np.prod(v)) for v in keys["dit"].values()) == 909_426_568 or True  # informational


@pytest.mark.parametrize("tag", ["dit_tiny", "dit_cfg1"])
def test_dit_forward_matches_reference(golden_dir, tag):
    g = _load(golden_dir, tag + ".npz")
    cfg = json.loads(str(g["cfg"]))
    sd = synth.synth_state_dict(synth.dit_shapes(**cfg), int(g["seed"]))
    B = g["forward"].shape[0]
    x, y = synth.synth_inputs(B, cfg["seq_length"], cfg["in_channels"], int(g["M"]), cfg["condition_channels"], int(g["seed"]) + 1000)
    t = torch.from_numpy(g["t"])
    with torch.no_grad():
        assert _rel(oracle.dit.t_embedder(sd, t), g["t_emb"]) < 1e-6
        out, blocks = oracle.dit.forward(sd, x, t, y, cfg["num_heads"], "fp32", return_blocks=True)
        assert _rel(out, g["forward"]) < 2e-5
        if g["blocks"].size:
            for i, b in enumerate(blocks):
                assert _rel(b, g["blocks"][i]) < 1e-5, f"block {i}"
        cfg_out = oracle.dit.forward_with_cfg(sd, x, t, y, 6.0, cfg["num_heads"], "fp32")
        assert _rel(cfg_out, g["forward_with_cfg"]) < 2e-5


def test_uncond_cross_attention_collapse(golden_dir):
    """SURVEY §8a a8: with an all-null context the cross-attention output is proj(to_v(null)) for every query."""
    g = _load(golden_dir, "dit_tiny.npz")
    cfg = json.loads(str(g["cfg"]))
    sd = synth.synth_state_dict(synth.dit_shapes(**cfg), int(g["seed"]))
    x = torch.randn(2, 8, cfg["hidden_size"])
    y = sd["null_cond_embedding"].expand(2, 24, -1)
    pol = oracle.dit.Policy("fp32")
    full = oracle.dit.cross_attention(sd, "blocks.1.crossattn.", x, y, cfg["num_heads"], pol)
    const = oracle.dit.uncond_cross_constant(sd, 1)
    assert (full - const).abs().max() < 1e-5


def test_fp16_policy_close_to_fp32(golden_dir):
    g = _load(golden_dir, "dit_tiny.npz")
    cfg = json.loads(str(g["cfg"]))
    sd = synth.synth_state_dict(synth.dit_shapes(**cfg), int(g["seed"]))
    x, y = synth.synth_inputs(2, cfg["seq_length"], cfg["in_channels"], int(g["M"]), cfg["condition_channels"], int(g["seed"]) + 1000)
    out16 = oracle.dit.forward_with_cfg(sd, x, torch.from_numpy(g["t"]), y, 6.0, cfg["num_heads"], "fp16")
    r = _rel(out16, g["forward_with_cfg"])
    assert 0 < r < 1e-2


def test_schedule_tables_and_timestep_maps(golden_dir):
    g = _load(golden_dir, "sampler.npz")
    for k, stride in ((25, 40), (50, 20), (100, 10), (200, 5)):
        s = oracle.diffusion.Schedule(f"ddim{k}")
        assert s.timestep_map == list(range(0, 1000, stride))
        assert np.array_equal(np.array(s.timestep_map), g[f"map_ddim{k}"])           # integer contract: exact
        np.testing.assert_allclose(s.alphas_cumprod, g[f"acp_ddim{k}"], rtol=1e-13, atol=0)
    full = oracle.diffusion.Schedule("")
    np.testing.assert_allclose(full.alphas_cumprod, g["acp_full"], rtol=1e-13)
    lin = oracle.diffusion.Schedule("ddim50", noise_schedule="linear")
    assert lin.timestep_map == list(g["map_linear_ddim50"])
    np.testing.assert_allclose(lin.alphas_cumprod, g["acp_linear_ddim50"], rtol=1e-12)
    np.testing.assert_allclose(full.betas, g["betas_full"], rtol=1e-12)
    assert np.array_equal(np.array(oracle.diffusion.Schedule("10").timestep_map), g["map_sec10"])
    s = oracle.diffusion.Schedule("ddim25")
    for nm in ("posterior_log_variance_clipped", "posterior_mean_coef1", "posterior_mean_coef2", "sqrt_recipm1_alphas_cumprod"):
        np.testing.assert_allclose(getattr(s, nm), g[nm + "_ddim25"], rtol=1e-12)


def _tiny_model(golden_dir):
    g = _load(golden_dir, "dit_tiny.npz")
    cfg = json.loads(str(g["cfg"]))
    sd = synth.synth_state_dict(synth.dit_shapes(**cfg), int(g["seed"]))
    x, y = synth.synth_inputs(2, cfg["seq_length"], cfg["in_channels"], int(g["M"]), cfg["condition_channels"], 2101)
    return (lambda xx, tt: oracle.dit.forward_with_cfg(sd, xx, tt, y, 6.0, cfg["num_heads"], "fp32")), x


def test_ddim_trajectory_matches_reference(golden_dir):
    g = _load(golden_dir, "sampler.npz")
    model, x = _tiny_model(golden_dir)
    s = oracle.diffusion.Schedule("ddim25")
    with torch.no_grad():
        traj = list(oracle.diffusion.sample_loop(s, model, x, ddim=True))
    assert len(traj) == 25
    for i, o in enumerate(traj):
        assert _rel(o["sample"], g["ddim25_samples"][i]) < 5e-5, i
        assert _rel(o["pred_xstart"], g["ddim25_x0"][i]) < 5e-5, i
    torch.manual_seed(7)
    with torch.no_grad():
        last = list(oracle.diffusion.sample_loop(s, model, x, ddim=True, eta=0.5, step_noise=torch.randn_like))[-1]
    assert _rel(last["sample"], g["ddim25_eta05_final"]) < 5e-5


def test_ddpm_trajectory_matches_reference(golden_dir):
    g = _load(golden_dir, "sampler.npz")
    model, x = _tiny_model(golden_dir)
    s = oracle.diffusion.Schedule("10")
    torch.manual_seed(7)
    with torch.no_grad():
        traj = list(oracle.diffusion.sample_loop(s, model, x, ddim=False, step_noise=torch.randn_like))
    for i, o in enumerate(traj):
        assert _rel(o["sample"], g["ddpm10_samples"][i]) < 5e-5, i


def test_sampler_with_clip_denoised_matches_reference(golden_dir):
    """clip_denoised=True is the default of every sampling entry point of the reference (gaussian_diffusion.py:399,442,487,536,656); the
    fixture replays seeded model outputs through the REFERENCE sampler with the clamp of process_xstart (:310-315) active on ~30 % of
    the entries (tests/golden/make_sampler_clip_golden.py).  With the model replayed, the oracle's arithmetic is the reference's op for op."""
    g = _load(golden_dir, "sampler_clip.npz")
    x_T = torch.from_numpy(g["x_T"])
    assert 0.1 < float(g["clamped_fraction"]) < 0.6

    def replay(outs):
        it = iter(torch.from_numpy(outs))
        return lambda xx, tt: next(it)

    s25, s10 = oracle.diffusion.Schedule("ddim25"), oracle.diffusion.Schedule("10")
    traj = list(oracle.diffusion.sample_loop(s25, replay(g["outs25"]), x_T, ddim=True, clip_denoised=True))
    for i, o in enumerate(traj):
        assert float(o["pred_xstart"].abs().max()) <= 1.0
        assert _rel(o["pred_xstart"], g["ddim25_x0"][i]) < 1e-6 and _rel(o["sample"], g["ddim25_samples"][i]) < 1e-6, i
    torch.manual_seed(11)
    traj = list(oracle.diffusion.sample_loop(s25, replay(g["outs25"]), x_T, ddim=True, eta=0.5, clip_denoised=True, step_noise=torch.randn_like))
    assert max(_rel(o["sample"], g["ddim25_eta05_samples"][i]) for i, o in enumerate(traj)) < 1e-6
    torch.manual_seed(12)
    traj = list(oracle.diffusion.sample_loop(s10, replay(g["outs10"]), x_T, ddim=False, clip_denoised=True, step_noise=torch.randn_like))
    for i, o in enumerate(traj):
        assert _rel(o["pred_xstart"], g["ddpm10_x0"][i]) < 1e-6 and _rel(o["sample"], g["ddpm10_samples"][i]) < 1e-6, i
    # and the fixture does see the clamp: the unclamped oracle leaves it
    plain = list(oracle.diffusion.sample_loop(s25, replay(g["outs25"]), x_T, ddim=True, clip_denoised=False))
    assert _rel(plain[0]["pred_xstart"], g["ddim25_x0"][0]) > 1e-2


@pytest.mark.parametrize("par", ["eps", "xstart"])
def test_sampler_eps_and_xstart_parameterisations_match_reference(golden_dir, par):
    """The oracle under create_diffusion's other parameterisations against the reference sampler on replayed model outputs
    (tests/golden/make_sampler_param_golden.py): 25-step DDIM with and without the clamp, 10-step DDPM."""
    g = _load(golden_dir, "sampler_param.npz")
    x_T = torch.from_numpy(g["x_T"])

    def replay(outs):
        it = iter(torch.from_numpy(outs))
        return lambda xx, tt: next(it)

    s25, s10 = oracle.diffusion.Schedule("ddim25"), oracle.diffusion.Schedule("10")
    for clip in (False, True):
        tag = f"{par}_ddim25" + ("_clip" if clip else "")
        traj = list(oracle.diffusion.sample_loop(s25, replay(g["outs25"]), x_T, ddim=True, clip_denoised=clip, parameterization=par))
        for i, o in enumerate(traj):
            assert _rel(o["pred_xstart"], g[tag + "_x0"][i]) < 1e-6 and _rel(o["sample"], g[tag + "_samples"][i]) < 1e-6, (clip, i)
    torch.manual_seed(21)
    traj = list(oracle.diffusion.sample_loop(s10, replay(g["outs10"]), x_T, ddim=False, step_noise=torch.randn_like, parameterization=par))
    assert max(_rel(o["sample"], g[f"{par}_ddpm10_samples"][i]) for i, o in enumerate(traj)) < 1e-6
    other = "xstart" if par == "eps" else "eps"          # the fixture tells the parameterisations apart
    wrong = list(oracle.diffusion.sample_loop(s25, replay(g["outs25"]), x_T, ddim=True, parameterization=other))
    assert _rel(wrong[0]["sample"], g[f"{par}_ddim25_samples"][0]) > 1e-2


def test_vae_decode_matches_reference(golden_dir):
    g = _load(golden_dir, "vae_decode.npz")
    sd = synth.synth_state_dict(synth.vae_decoder_shapes(**synth.FULL_VAE), 103)
    stages = {}
    with torch.no_grad():
        out = oracle.vae.decode(sd, torch.from_numpy(g["z"]), "fp32", stages=stages)
    assert out.shape == (4, 6, 8, 8, 8)
    assert _rel(out, g["out"]) < 2e-5
    for k, v in stages.items():
        ref = g["stage_" + k]
        got = np.array([float(v.double().mean()), float(v.double().abs().mean()), float(v.double().std())])
        np.testing.assert_allclose(got, ref, rtol=2e-4, atol=1e-6, err_msg=k)
    assert _rel(stages["up1"][0, :, 3, 4, :], g["stage_up1_slice"]) < 2e-5
    assert _rel(stages["mid"][1, :8], g["stage_mid_slice"]) < 2e-5
    out16 = oracle.vae.decode(sd, torch.from_numpy(g["z"]), "fp16")
    assert 0 < _rel(out16, g["out"]) < 2e-2


def test_latent_slicing_and_voxel_packing_contract():
    """inference.py:328-348 index contract: latent 0:4 | 4:68; decoded voxels packed channel-major."""
    s = torch.arange(2 * 3 * 68, dtype=torch.float32).reshape(2, 3, 68)
    srt, feat = oracle.vae.denormalise_latents(s, torch.zeros(68), torch.ones(68))
    assert srt.shape == (2, 3, 4) and feat.shape == (2, 3, 64)
    assert torch.equal(srt[1, 2], s[1, 2, :4]) and torch.equal(feat[0, 1], s[0, 1, 4:])
    dec = torch.zeros(3, 6, 8, 8, 8)
    dec[:, 0] = 5.0
    dec[:, 1:] = 1.0
    dec[2, 3, 1, 2, 3] = 3.0
    packed = oracle.vae.pack_decoded(dec, 1, 3)
    assert packed.shape == (1, 3, 3072)
    assert torch.all(packed[0, :, :512] == 1.0)                # sdf channel first, /5
    assert packed[0, 2, 3 * 512 + 1 * 64 + 2 * 8 + 3] == 2.0   # (3+1)/2 at channel-major offset


def test_primsdf_query_matches_reference(golden_dir):
    """oracle/primsdf.py against the reference PrimSDF.forward (models/primsdf.py:52-109) on 96 primitives / 4000 points."""
    fx = np.load(os.path.join(golden_dir, "primsdf.npz"))
    srt, feat, x = (torch.from_numpy(a) for a in oracle.primsdf.fixture_scene(int(fx["seed"])))
    got = oracle.primsdf.query(x, srt, feat, S=8, dim_feat=6, inference=True)
    assert 0 < int(fx["covered"].sum()) < len(x)                     # both branches are exercised
    for k in ("sdf", "tex", "mat"):
        np.testing.assert_allclose(got[k].numpy(), fx[k], rtol=1e-5, atol=1e-6, err_msg=k)
    # training mode leaves uncovered points at zero (primsdf.py:82)
    tr = oracle.primsdf.query(x, srt, feat, inference=False)
    assert float(tr["sdf"][~torch.from_numpy(fx["covered"])].abs().max()) == 0.0


def test_dit_full_width_block_matches_reference(golden_dir):
    """The shipped width (D 1152, 16 heads x 72, 2048 tokens, 1370 context tokens) with one block, against the reference's own
    output: the logits scale q.k/72, the 9-way modulation split and the head layout at the real sizes."""
    g = _load(golden_dir, "dit_full1.npz")
    cfg = json.loads(str(g["cfg"]))
    assert cfg["hidden_size"] == 1152 and cfg["num_heads"] == 16 and cfg["seq_length"] == 2048 and cfg["depth"] == 1
    sd = synth.synth_state_dict(synth.dit_shapes(**cfg), int(g["seed"]))
    x, y = synth.synth_inputs(1, cfg["seq_length"], cfg["in_channels"], int(g["M"]), cfg["condition_channels"], int(g["seed"]) + 1000)
    t = torch.from_numpy(g["t"])
    with torch.no_grad():
        out = oracle.dit.forward(sd, x, t, y, cfg["num_heads"], "fp32")
        assert _rel(out[:, ::8], g["forward"]) < 2e-5            # the fixture keeps every 8th token of both outputs
        cfg_out = oracle.dit.forward_with_cfg(sd, x, t, y, 6.0, cfg["num_heads"], "fp32")
        assert _rel(cfg_out[:, ::8], g["forward_with_cfg"]) < 2e-5


def test_oracle_respacing_matches_reference(golden_dir):
    fx = _load(golden_dir, "sampler.npz")
    cases = json.loads(str(fx["space_cases"]))
    for spec, want in cases.items():
        if want == "ValueError":
            with pytest.raises(ValueError):
                oracle.diffusion.kept_timesteps(1000, spec)
        else:
            assert sorted(oracle.diffusion.kept_timesteps(1000, spec)) == want, spec


def test_dinov2_encoder_matches_reference(golden_dir):
    """oracle/dinov2.py against the reference's own Dinov2Wrapper('dinov2_vitb14_reg') (image_dinov2.py:44-61) with synthetic
    weights: full 518 x 518 input (every 6th output token stored), per-block statistics, and a 224 x 224 input through the
    bicubic antialiased Resize."""
    g = _load(golden_dir, "dinov2.npz")
    sd = oracle.dinov2.synth_weights(int(g["seed"]))
    rs = np.random.RandomState(int(g["img_seed"]))
    yy, xx = np.meshgrid(np.linspace(0, 1, 518), np.linspace(0, 1, 518), indexing="ij")
    img = np.stack([127 + 100 * np.sin(6 * xx + 2 * yy), 127 + 100 * np.cos(5 * yy), 255 * xx * yy], -1) + 12 * rs.standard_normal((518, 518, 3))
    img = np.clip(img, 0, 255).astype(np.float32)[None]
    with torch.no_grad():
        out, blocks = oracle.dinov2.forward(sd, torch.from_numpy(img), return_blocks=True)
        assert tuple(out.shape) == (1, 1370, 768)
        assert _rel(out[:, ::6], g["out"]) < 2e-5
        stats = np.array([[float(b.double().mean()), float(b.double().abs().mean()), float(b.double().std())] for b in blocks])
        np.testing.assert_allclose(stats, g["block_stats"], rtol=1e-4, atol=1e-6)
        assert _rel(blocks[0][0, :8, :16], g["block0_slice"]) < 1e-5 and _rel(blocks[11][0, 5:13, :16], g["block11_slice"]) < 2e-5
        small = np.ascontiguousarray(np.clip(img[:, ::2, ::2][:, :224, :224], 0, 255))
        assert _rel(oracle.dinov2.forward(sd, torch.from_numpy(small))[:, ::24], g["out_small"]) < 2e-5


def test_raymarch_restatement_agrees_with_the_reference_torch_marcher():
    """oracle.raymarch.raymarch (the CUDA kernel's structure: per-warp hit lists, start at the first hit, accumulated steps) against
    oracle.raymarch.raymarch_dense (the reference's own pure-PyTorch ray-marcher, mvpraymarch.py:391-475): same image up to the
    step-placement differences of the two formulations (a ray enters a box at most one step apart)."""
    import torch
    from oracle import raymarch as rmo
    g = torch.Generator().manual_seed(11)
    K, S, H, W, volradius, dt = 12, 4, 16, 16, 50.0, 1.0
    pos = (torch.rand(K, 3, generator=g) - 0.5) * 0.8
    scale = 1.0 / (0.15 + 0.1 * torch.rand(K, 1, generator=g)).repeat(1, 3)
    rot = torch.eye(3)[None].repeat(K, 1, 1)
    tpl = torch.rand(K, S, S, S, 4, generator=g)
    tpl[..., :3] *= 255.0
    tpl[..., 3] *= 20.0
    RT = torch.tensor([[[1.0, 0, 0, 0], [0, -1.0, 0, 0], [0, 0, -1.0, 3.0 * volradius]]])
    Kc = torch.tensor([[[1.2 * W, 0, W / 2], [0, 1.2 * W, H / 2], [0, 0, 1.0]]])
    cam = rmo.convert_camera_parameters(RT, Kc)
    raypos, raydir, tmm = rmo.compute_raydirs(cam["campos"], cam["camrot"], torch.diagonal(cam["focal"], dim1=1, dim2=2), cam["princpt"], H, W, volradius)
    a = rmo.raymarch(raypos[0], raydir[0], dt / volradius, tmm[0], tpl, pos, rot, scale)
    b = rmo.raymarch_dense(raypos[0], raydir[0], dt / volradius, tmm[0], tpl, pos, rot, scale)
    assert float(b[..., 3].max()) > 0.3
    rel = float((a - b).norm() / b.norm())
    assert rel < 2e-2, rel


def test_raymarch_oracle_matches_the_reference_torch_marcher_fixture(golden_dir):
    """tests/golden/raymarch_ref.npz holds the image the REFERENCE's own pure-PyTorch ray-marcher (the block its gradcheck script runs
    against the CUDA kernel, mvpraymarch.py:391-475) produced for a seeded scene; tests/golden/make_raymarch_golden.py executed that
    block from /root/reference on the CPU.  Both oracle restatements are held to it: `raymarch_dense` (the same algorithm) tightly,
    `raymarch` (the CUDA kernel's structure, which the GPU test compares the kernel with) up to float rounding on this scene, whose
    rays carry their own [tmin, tmax] so the two formulations take the same steps."""
    import torch
    from oracle import raymarch as rmo
    d = np.load(os.path.join(golden_dir, "raymarch_ref.npz"))
    t = lambda k: torch.from_numpy(d[k])[0]      # noqa: E731  (one batch element)
    args = (t("raypos"), t("raydir"), float(d["stepsize"]), t("tminmax"), t("template_chlast"), t("primpos"), t("primrot"), t("primscale"),
            float(d["fadescale"]), float(d["fadeexp"]))
    ref = t("rayrgba")
    assert float((ref[..., 3] > 0).float().mean()) > 0.5 and float((ref[..., 3] >= 1 - 1e-6).float().mean()) > 0.1   # covered and saturating rays
    dense = rmo.raymarch_dense(*args)
    assert float((dense - ref).abs().max()) < 5e-6, float((dense - ref).abs().max())
    kern = rmo.raymarch(*args)
    assert float((kern - ref).abs().max()) < 2e-5, float((kern - ref).abs().max())


def test_inference_glue_matches_the_reference_statements(golden_dir):
    """tests/golden/inference_glue.npz: `recon_param` as the REFERENCE's own statements (inference.py:328-348, executed from
    /root/reference by tests/golden/make_inference_glue_golden.py with an index-revealing stand-in for vae.decode) produce it, for both
    settings of perchannel_norm and two latent_nf.  The oracle restatement — which the CUDA glue kernels are held to on the GPU — must
    reproduce it bit for bit (same eager fp32 ops on the CPU)."""
    import torch
    d = np.load(os.path.join(golden_dir, "inference_glue.npz"))

    def fake_decode(z):
        n = z.shape[0]
        base = torch.arange(n * 6 * 512, dtype=torch.float32).reshape(n, 6, 8, 8, 8)
        return base * 1e-3 - 3.0 + z.reshape(n, -1).sum(1).reshape(n, 1, 1, 1, 1)

    sample, mean, std = (torch.from_numpy(d[k]) for k in ("sample", "latent_mean", "latent_std"))
    prims = sample.shape[1] // 68
    n = 0
    for key in d.files:
        if not key.startswith("recon_param_"):
            continue
        pc = key.split("_pc")[1][0] == "1"
        nf = float(key.split("_nf")[1])
        got = oracle.vae.inference_glue(sample.clone().reshape(sample.shape[0], prims, 68), fake_decode, mean, std, nf, pc)
        assert torch.equal(got, torch.from_numpy(d[key])), key
        n += 1
    assert n == 4

