#!/usr/bin/env python
"""Generate the golden fixtures under tests/golden/ by IMPORTING THE REFERENCE'S OWN MODULES.

Run in the build container only (needs /root/reference; it does not exist on the GPU box):

    python tests/golden/make_golden.py

The reference has no tests / golden vectors for this path (SURVEY.md §4), so these fixtures are how the
oracle (oracle/*.py) is pinned.  The reference modules are imported unchanged; the single un-vendored
dependency on the path, ``xformers.ops`` (attention.py:17), is provided as an in-memory module that
restates its contract: memory_efficient_attention(q,k,v) = softmax(q k^T * Dh^-1/2) v over
[B,N,H,Dh] tensors; unbind = torch.unbind.

Weights / inputs come from numpy RandomState streams (``synth.py``) so tests can rebuild them.
Outputs are the reference's fp32 CPU results (autocast('cuda') is inert on CPU).
"""
import importlib.util
import json
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
REF = "/root/reference"
OUT = os.path.join(ROOT, "tests", "golden")


def _load_synth():
    spec = importlib.util.spec_from_file_location("tpx_synth", os.path.join(ROOT, "3dtopia-xl_b200", "synth.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _install_xformers_shim():
    import torch.nn.functional as F

    def memory_efficient_attention(q, k, v, attn_bias=None, p=0.0, scale=None):
        assert attn_bias is None and p == 0.0
        o = F.scaled_dot_product_attention(q.transpose(1, 2), k.transpose(1, 2), v.transpose(1, 2), scale=scale)
        return o.transpose(1, 2)

    xf = types.ModuleType("xformers")
    ops = types.ModuleType("xformers.ops")
    ops.memory_efficient_attention = memory_efficient_attention
    ops.unbind = torch.unbind
    xf.ops = ops
    sys.modules["xformers"], sys.modules["xformers.ops"] = xf, ops


def main():
    synth = _load_synth()
    _install_xformers_shim()
    sys.path.insert(0, REF)
    from models.dit_crossattn import DiT            # noqa: E402
    from models.vae3d_dib import VAE                # noqa: E402
    from models.diffusion import create_diffusion   # noqa: E402
    torch.set_grad_enabled(False)
    torch.set_num_threads(os.cpu_count())

    # ---- key / shape contract of the FULL config (configs/inference_dit.yml) -------------------------
    with torch.device("meta"):
        full = DiT(**synth.FULL_DIT)
        vfull = VAE(**synth.FULL_VAE)
    keys = {"dit": {k: list(v.shape) for k, v in full.state_dict().items()},
            "vae": {k: list(v.shape) for k, v in vfull.state_dict().items()}}
    assert {k: tuple(v) for k, v in keys["dit"].items()} == dict(synth.dit_shapes(**synth.FULL_DIT))
    dec = {k: tuple(v) for k, v in keys["vae"].items() if k.startswith(("decoder.", "post_quant_conv."))}
    assert dec == dict(synth.vae_decoder_shapes(**synth.FULL_VAE)), "decoder key/shape contract drifted"
    json.dump(keys, open(os.path.join(OUT, "state_dict_keys.json"), "w"), indent=0, sort_keys=True)

    # ---- DiT: tiny config (per-block outputs) and config #1 (N=256, D=384, depth 4, 16 heads) ----------
    for tag, cfg, M, seed in (
        ("dit_tiny", dict(seq_length=32, in_channels=12, condition_channels=48, hidden_size=64, depth=2,
                          num_heads=4, attn_proj_bias=True, cond_drop_prob=0.1, gradient_checkpointing=False), 24, 101),
        ("dit_cfg1", dict(seq_length=256, in_channels=68, condition_channels=768, hidden_size=384, depth=4,
                          num_heads=16, attn_proj_bias=True, cond_drop_prob=0.1, gradient_checkpointing=False), 1370, 102),
        # the shipped width (D=1152, 16 heads x 72, N=2048, M=1370) with ONE block: pins the 1/72 logits scale, the 9-way
        # modulation split and the head layout at the real sizes
        ("dit_full1", dict(synth.FULL_DIT, depth=1), 1370, 104),
    ):
        sd = synth.synth_state_dict(synth.dit_shapes(**cfg), seed)
        model = DiT(**cfg).eval()
        model.load_state_dict(sd, strict=True)
        B = 2 if tag == "dit_tiny" else 1
        x, y = synth.synth_inputs(B, cfg["seq_length"], cfg["in_channels"], M, cfg["condition_channels"], seed + 1000)
        t = torch.tensor([960, 40][:B], dtype=torch.int64)
        hooks, blocks = [], []
        for blk in model.blocks:
            hooks.append(blk.register_forward_hook(lambda m, i, o: blocks.append(o.clone())))
        fwd = model.forward(x, t, y)
        for h in hooks:
            h.remove()
        cfg_out = model.forward_with_cfg(x, t, y, cfg_scale=6.0)
        if tag == "dit_full1":        # keep the fixture under 1 MB: every 8th token of both outputs
            fwd, cfg_out = fwd[:, ::8], cfg_out[:, ::8]
        np.savez_compressed(os.path.join(OUT, tag + ".npz"), cfg=json.dumps(cfg), M=M, seed=seed, t=t.numpy(),
                            forward=fwd.numpy(), forward_with_cfg=cfg_out.numpy(),
                            blocks=np.stack([b.numpy() for b in blocks]) if tag == "dit_tiny" else np.zeros(0),
                            t_emb=model.t_embedder(t).numpy())
        print(tag, "forward", tuple(fwd.shape), float(fwd.abs().mean()), "cfg", float(cfg_out.abs().mean()))
        if tag == "dit_tiny":
            tiny_model, tiny_cfg, tiny_M = model, cfg, M

    # ---- sampler: schedule tables, timestep maps, and trajectories through the reference sampler -------
    fx = {}
    for k in (25, 50, 100, 200):
        d = create_diffusion(timestep_respacing=f"ddim{k}", noise_schedule="squaredcos_cap_v2", diffusion_steps=1000, parameterization="v")
        fx[f"map_ddim{k}"] = np.array(d.timestep_map)
        fx[f"acp_ddim{k}"] = d.alphas_cumprod
    d0 = create_diffusion(timestep_respacing="", noise_schedule="squaredcos_cap_v2", diffusion_steps=1000, parameterization="v")
    fx["acp_full"] = d0.alphas_cumprod
    fx["betas_full"] = d0.betas
    d10 = create_diffusion(timestep_respacing="10", noise_schedule="squaredcos_cap_v2", diffusion_steps=1000, parameterization="v")
    fx["map_sec10"] = np.array(d10.timestep_map)
    d25 = create_diffusion(timestep_respacing="ddim25", noise_schedule="squaredcos_cap_v2", diffusion_steps=1000, parameterization="v")
    for nm in ("posterior_log_variance_clipped", "posterior_mean_coef1", "posterior_mean_coef2", "sqrt_recipm1_alphas_cumprod"):
        fx[nm + "_ddim25"] = getattr(d25, nm)
    x, y = synth.synth_inputs(2, tiny_cfg["seq_length"], tiny_cfg["in_channels"], tiny_M, tiny_cfg["condition_channels"], 2101)
    kw = dict(y=y, cfg_scale=6.0, precision_dtype=torch.float16, enable_amp=True)
    traj = [o for o in d25.ddim_sample_loop_progressive(tiny_model.forward_with_cfg, x.shape, x, clip_denoised=False,
                                                        model_kwargs=kw, progress=False, device="cpu")]
    fx["ddim25_samples"] = np.stack([o["sample"].numpy() for o in traj])
    fx["ddim25_x0"] = np.stack([o["pred_xstart"].numpy() for o in traj])
    torch.manual_seed(7)
    traj = [o for o in d25.ddim_sample_loop_progressive(tiny_model.forward_with_cfg, x.shape, x, clip_denoised=False,
                                                        model_kwargs=kw, progress=False, device="cpu", eta=0.5)]
    fx["ddim25_eta05_final"] = traj[-1]["sample"].numpy()
    torch.manual_seed(7)
    traj = [o for o in d10.p_sample_loop_progressive(tiny_model.forward_with_cfg, x.shape, x, clip_denoised=False,
                                                     model_kwargs=kw, progress=False, device="cpu")]
    fx["ddpm10_samples"] = np.stack([o["sample"].numpy() for o in traj])
    dl = create_diffusion(timestep_respacing="ddim50", noise_schedule="linear", diffusion_steps=1000, parameterization="v")
    fx["acp_linear_ddim50"] = dl.alphas_cumprod
    fx["map_linear_ddim50"] = np.array(dl.timestep_map)
    # respacing strings through the reference's own space_timesteps (respace.py:12-62), incl. the cases it rejects
    from models.diffusion.respace import space_timesteps
    cases = {}
    for spec in ("ddim10", "ddim20", "ddim40", "ddim125", "ddim500", "ddim1000", "ddim600", "ddim999", "1", "7", "250", "1000", "10,10,5", "1,1,1,1",
                 "3,0,7", "400,300,200", "2000", "334,334,334"):
        try:
            cases[spec] = sorted(int(v) for v in space_timesteps(1000, spec))
        except ValueError:
            cases[spec] = "ValueError"
    fx["space_cases"] = json.dumps(cases)
    np.savez_compressed(os.path.join(OUT, "sampler.npz"), **fx)
    print("sampler", fx["map_ddim25"][:4], fx["ddim25_samples"].shape)

    # ---- VAE decode (shipped channel config, 4 primitives) ---------------------------------------------
    sd = synth.synth_state_dict(synth.vae_decoder_shapes(**synth.FULL_VAE), 103)
    vae = VAE(**synth.FULL_VAE).eval()
    missing, unexpected = vae.load_state_dict(sd, strict=False)
    assert not unexpected and all(m.startswith(("encoder.", "quant_conv.")) for m in missing)
    rs = np.random.RandomState(1103)
    z = torch.from_numpy((rs.standard_normal(size=(4, 64)) * np.array(synth.LATENT_STD[4:]) + np.array(synth.LATENT_MEAN[4:])).astype(np.float32)).reshape(4, 1, 4, 4, 4)
    stages = {}
    dec_ = vae.decoder
    h = dec_.conv_in(vae.post_quant_conv(z)); stages["conv_in"] = h
    h = dec_.mid_block.nets[0](h)
    h = dec_.mid_block.attns[0](h); stages["mid_attn"] = h
    h = dec_.mid_block.nets[1](h); stages["mid"] = h
    h = dec_.up_blocks[0](h); stages["up0"] = h
    h = dec_.up_blocks[1](h); stages["up1"] = h
    out = vae.decode(z)
    np.savez_compressed(os.path.join(OUT, "vae_decode.npz"), z=z.numpy(), out=out.numpy(),
                        **{"stage_" + k: np.array([float(v.double().mean()), float(v.double().abs().mean()), float(v.double().std())]) for k, v in stages.items()},
                        stage_up1_slice=stages["up1"][0, :, 3, 4, :].numpy(), stage_mid_slice=stages["mid"][1, :8].numpy())
    print("vae", tuple(out.shape), float(out.abs().mean()))

    # ---- PrimSDF point query (SURVEY §8f-1): the reference class, with `trimesh` (imported but unused on this path) stubbed
    sys.modules.setdefault("trimesh", types.ModuleType("trimesh"))
    from models.primsdf import PrimSDF              # noqa: E402
    sys.path.insert(0, ROOT)
    import oracle                                                            # noqa: E402  (scene / weight synthesis shared with the tests)
    srt, feat, pts = oracle.primsdf.fixture_scene(1104)
    K, S = srt.shape[0], 8
    m = PrimSDF(num_prims=K, dim_feat=6, prim_shape=S).eval()
    m.srt_param.data = torch.from_numpy(srt)
    m.feat_param.data = torch.from_numpy(feat)
    preds = m(torch.from_numpy(pts))
    covered = (m.prim_weight(torch.from_numpy(pts)).sum(1) > 0).numpy()
    np.savez_compressed(os.path.join(OUT, "primsdf.npz"), seed=1104, covered=covered,
                        sdf=preds["sdf"].numpy(), tex=preds["tex"].numpy(), mat=preds["mat"].numpy())
    print("primsdf", int(covered.sum()), "of", len(pts), "points covered")

    # ---- DINOv2 ViT-B/14-reg encoder (SURVEY §8f-2): the reference wrapper, random weights instead of the hub download --------
    from models.conditioner.image_dinov2 import Dinov2Wrapper               # noqa: E402
    import models.conditioner.dinov2.hub.backbones as bb                     # noqa: E402
    Dinov2Wrapper._build_dinov2 = staticmethod(lambda model_name, modulation_dim=None, pretrained=True:
                                               getattr(bb, model_name)(modulation_dim=modulation_dim, pretrained=False))
    enc = Dinov2Wrapper("dinov2_vitb14_reg", freeze=True).eval()
    sd = oracle.dinov2.synth_weights(105)
    assert {k: tuple(v.shape) for k, v in enc.state_dict().items()} == {k: tuple(v.shape) for k, v in sd.items()}, "DINOv2 key/shape contract drifted"
    assert list(enc.state_dict().keys()) == list(sd.keys())
    enc.load_state_dict(sd, strict=True)
    rs = np.random.RandomState(1105)
    # a smooth synthetic picture + noise, 0..255, the 518 x 518 the pipeline feeds (configs/inference_dit.yml:18-19)
    yy, xx = np.meshgrid(np.linspace(0, 1, 518), np.linspace(0, 1, 518), indexing="ij")
    img = np.stack([127 + 100 * np.sin(6 * xx + 2 * yy), 127 + 100 * np.cos(5 * yy), 255 * xx * yy], -1) + 12 * rs.standard_normal((518, 518, 3))
    img = np.clip(img, 0, 255).astype(np.float32)[None]
    blocks = []
    hooks = [b.register_forward_hook(lambda m_, i_, o_: blocks.append(o_.clone())) for b in enc.model.blocks]
    out = enc(torch.from_numpy(img))
    for h in hooks:
        h.remove()
    small = np.clip(img[:, ::2, ::2][:, :224, :224], 0, 255)                # a 224 x 224 picture: exercises Resize(518, bicubic)
    out_small = enc(torch.from_numpy(np.ascontiguousarray(small)))
    np.savez_compressed(os.path.join(OUT, "dinov2.npz"), seed=105, img_seed=1105, out=out.numpy()[:, ::6], out_small=out_small.numpy()[:, ::24],
                        block_stats=np.array([[float(b.double().mean()), float(b.double().abs().mean()), float(b.double().std())] for b in blocks]),
                        block0_slice=blocks[0][0, :8, :16].numpy(), block11_slice=blocks[11][0, 5:13, :16].numpy())
    print("dinov2", tuple(out.shape), float(out.abs().mean()), float(out_small.abs().mean()))


if __name__ == "__main__":
    main()
