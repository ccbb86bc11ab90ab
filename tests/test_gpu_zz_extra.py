"""GPU: the rarely-taken paths of the tcgen05
attention kernel (lazy rescale of O in TMEM, redo of a tile against a new row maximum, row sums across rescales) and one block
at the shipped width against the reference fixture.  Kept in their own module, collected after the validated ones."""
import pytest
import torch

from tpxl_b200 import _lib
from gpu_util import rel_l2, st

pytestmark = pytest.mark.gpu   # promoted to plain tests: all five passed on a B200 at the end of round 1 (GPUTEST_r01.json)


def test_full_width_block_against_reference_fixture(golden_dir):
    """One block at the shipped width against the reference's own fp32 output (tests/golden/dit_full1.npz)."""
    import json
    import os

    import numpy as np

    import oracle
    import tpxl_b200
    from tpxl_b200 import synth
    g = np.load(os.path.join(golden_dir, "dit_full1.npz"))
    cfg = json.loads(str(g["cfg"]))
    sd = synth.synth_state_dict(synth.dit_shapes(**cfg), int(g["seed"]))
    x, y = synth.synth_inputs(1, cfg["seq_length"], cfg["in_channels"], int(g["M"]), cfg["condition_channels"], int(g["seed"]) + 1000)
    t = torch.from_numpy(g["t"])
    kw = {k: v for k, v in cfg.items() if k != "gradient_checkpointing"}
    m = tpxl_b200.DiT(**kw)
    m.load_state_dict(sd)
    m = m.to("cuda:0").eval()
    with torch.no_grad():
        out = m.forward(x.cuda(), t.cuda(), y.cuda(), torch.float16, True)
        out_cfg = m.forward_with_cfg(x.cuda(), t.cuda(), y.cuda(), cfg_scale=6.0, precision_dtype=torch.float16, enable_amp=True)
        sdd = {k: v.cuda() for k, v in sd.items()}
        o16_cfg = oracle.dit.forward_with_cfg(sdd, x.cuda(), t.cuda(), y.cuda(), 6.0, cfg["num_heads"], "fp16")
    ref, ref_cfg = torch.from_numpy(g["forward"]).cuda(), torch.from_numpy(g["forward_with_cfg"]).cuda()
    r = dict(ours_vs_ref32=rel_l2(out.float()[:, ::8], ref), cfg_ours_vs_ref32=rel_l2(out_cfg.float()[:, ::8], ref_cfg),
             cfg_oracle16_vs_ref32=rel_l2(o16_cfg[:, ::8], ref_cfg), cfg_ours_vs_oracle16=rel_l2(out_cfg.float(), o16_cfg))
    print(r)
    assert r["ours_vs_ref32"] < 1e-2 and r["cfg_ours_vs_ref32"] < 1e-2
    assert r["cfg_ours_vs_oracle16"] < 3e-3
    assert r["cfg_ours_vs_ref32"] < 4 * r["cfg_oracle16_vs_ref32"] + 5e-4      # no further from fp32 than the fp16 contract itself


def test_dinov2_encoder_against_reference_fixture(golden_dir):
    """The DINOv2 ViT-B/14-reg mirror (built from the DiT kernels + tpx_gelu_erf) against the reference wrapper's fp32 output.
    Tolerance 5e-3 relative L2: fp16-input GEMMs against an fp32 reference (the CPU emulation of the same contract sits at ~1e-3)."""
    import importlib
    import os

    import numpy as np

    import oracle
    d = importlib.import_module("tpxl_b200.dinov2")
    g = np.load(os.path.join(golden_dir, "dinov2.npz"))
    sd = oracle.dinov2.synth_weights(int(g["seed"]))
    rs = np.random.RandomState(int(g["img_seed"]))
    yy, xx = np.meshgrid(np.linspace(0, 1, 518), np.linspace(0, 1, 518), indexing="ij")
    img = np.stack([127 + 100 * np.sin(6 * xx + 2 * yy), 127 + 100 * np.cos(5 * yy), 255 * xx * yy], -1) + 12 * rs.standard_normal((518, 518, 3))
    img = np.clip(img, 0, 255).astype(np.float32)[None]
    m = d.Dinov2Wrapper("dinov2_vitb14_reg", freeze=True)
    m.load_state_dict(sd)
    m = m.to("cuda:0").eval()
    with torch.no_grad():
        out = m(torch.from_numpy(img).cuda())
        small = np.ascontiguousarray(np.clip(img[:, ::2, ::2][:, :224, :224], 0, 255))
        out_small = m(torch.from_numpy(small).cuda())
        two = m(torch.from_numpy(np.concatenate([img, img[:, ::-1].copy()], 0)).cuda())        # batch of 2: per-picture token blocks
    torch.cuda.synchronize()
    assert out.shape == (1, 1370, 768) and out.dtype == torch.float32
    r = dict(full=rel_l2(out[:, ::6], torch.from_numpy(g["out"]).cuda()), small=rel_l2(out_small[:, ::24], torch.from_numpy(g["out_small"]).cuda()),
             batch=rel_l2(two[0:1], out))
    print(r)
    assert r["full"] < 5e-3 and r["small"] < 5e-3
    assert r["batch"] < 1e-4                                   # the same picture gives the same tokens whatever shares the batch
                                                               # (tile widths depend on the row count, so not necessarily bit-identical)


@pytest.mark.parametrize("B,H,Nq,Nk,growth", [(1, 2, 256, 1024, 0.0), (1, 2, 384, 1370, 0.6), (2, 1, 128, 640, -0.5)])
def test_attention_tcgen05_peaky_logits(B, H, Nq, Nk, growth):
    """Logits with a standard deviation of ~8 (and key norms that grow or shrink from one 128-key tile to the next), so the
    running row maximum jumps past the kernel's lazy-rescale threshold (2^8) between tiles: exercises the rescale of O in
    TMEM, the redo of a tile against the new maximum, and the tensor-core row sums across rescales."""
    Dh, DhP = 72, 80
    NkPad = (Nk + 7) // 8 * 8
    g = torch.Generator(device="cuda").manual_seed(Nq * 11 + Nk)
    q = torch.zeros(B, H, Nq, DhP, dtype=torch.float16, device="cuda")
    k = torch.zeros(B, H, Nk, DhP, dtype=torch.float16, device="cuda")
    v = torch.zeros(B, H, Nk, DhP, dtype=torch.float16, device="cuda")
    q[..., :Dh] = (torch.randn(B, H, Nq, Dh, generator=g, device="cuda") * 8).half()
    tile = torch.arange(Nk, device="cuda") // 128
    kscale = (1.0 + growth * tile.float()).clamp_min(0.2) if growth >= 0 else (1.0 + (-growth) * (tile.max() - tile).float())
    k[..., :Dh] = (torch.randn(B, H, Nk, Dh, generator=g, device="cuda") * kscale[None, None, :, None]).half()
    v[..., :Dh] = torch.randn(B, H, Nk, Dh, generator=g, device="cuda").half()
    vT = torch.zeros(B, H, DhP, NkPad, dtype=torch.float16, device="cuda")
    vT[..., :Nk] = v.transpose(-1, -2)
    out = torch.full((B, Nq, H * Dh), 9.0, dtype=torch.float16, device="cuda")
    scale = Dh ** -0.5
    _lib.check(_lib.lib().tpx_attention_tc(q.data_ptr(), k.data_ptr(), vT.data_ptr(), out.data_ptr(), B, H, Nq, Nk, NkPad, Dh, scale, st()))
    s = torch.matmul(q.float(), k.float().transpose(-1, -2)) * scale
    jumps = (s.reshape(B, H, Nq, -1)[..., : (Nk // 128) * 128].reshape(B, H, Nq, -1, 128).amax(-1).diff(dim=-1) * 1.4427 > 8).any()
    assert growth < 0 or bool(jumps), "the inputs were meant to force a rescale"
    ref = torch.matmul(torch.softmax(s, -1), v.float())[..., :Dh].permute(0, 2, 1, 3).reshape(B, Nq, H * Dh)
    torch.cuda.synchronize()
    assert torch.isfinite(out.float()).all()
    assert rel_l2(out.float(), ref) < 2e-3
    assert (out.float() - ref).abs().max() < 2e-2
