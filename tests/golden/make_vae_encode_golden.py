#!/usr/bin/env python
"""Generate tests/golden/vae_encode.npz by IMPORTING THE REFERENCE'S OWN VAE (models/vae3d_dib.py), as make_golden.py does.

Run in the build container only (needs /root/reference; it does not exist on the GPU box):

    python tests/golden/make_vae_encode_golden.py

Weights: synthetic encoder (RandomState 211) and decoder (RandomState 103, the decoder of vae_decode.npz) tensors from synth.py.
Inputs: 4 primitives whose features lie where the sample -> decode glue puts them (sdf * 5, (rgb, material) * 2 - 1): the
reference decoder's output for seeded latents drawn with the released per-channel latent statistics.
Stored: the input; the activations after conv_in, down_blocks.0, down_blocks.1 and the mid block (fp16, to stay small); the
posterior's parameters, mean, logvar and std; forward(x, sample=False)[0].  All fp32 CPU results of the reference.
Rerunning reproduces the file.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

from make_golden import REF, _install_xformers_shim, _load_synth   # noqa: E402

OUT = os.path.join(HERE, "vae_encode.npz")
P = 4
ENC_SEED, DEC_SEED, Z_SEED = 211, 103, 212


def main():
    synth = _load_synth()
    _install_xformers_shim()
    sys.path.insert(0, REF)
    from models.vae3d_dib import VAE                # noqa: E402
    torch.set_grad_enabled(False)
    torch.set_num_threads(os.cpu_count())

    sd = synth.synth_state_dict(synth.vae_decoder_shapes(**synth.FULL_VAE), DEC_SEED)
    sd.update(synth.synth_state_dict(synth.vae_encoder_shapes(**synth.FULL_VAE), ENC_SEED))
    vae = VAE(**synth.FULL_VAE).eval()
    missing, unexpected = vae.load_state_dict(sd, strict=True)
    assert not missing and not unexpected

    rs = np.random.RandomState(Z_SEED)
    z = rs.standard_normal(size=(P, 64)) * np.array(synth.LATENT_STD[4:]) + np.array(synth.LATENT_MEAN[4:])
    x = vae.decode(torch.from_numpy(z.astype(np.float32)).reshape(P, 1, 4, 4, 4)).contiguous()

    enc = vae.encoder
    stages = {}
    h = enc.conv_in(x); stages["conv_in"] = h
    h = enc.down_blocks[0](h); stages["down0"] = h
    h = enc.down_blocks[1](h); stages["down1"] = h
    h = enc.mid_block(h); stages["mid"] = h
    post = vae.encode(x)
    out, p2 = vae.forward(x, sample=False)
    assert torch.equal(p2.parameters, post.parameters)
    np.savez_compressed(OUT, x=x.numpy(), parameters=post.parameters.numpy(), mean=post.mean.numpy(), logvar=post.logvar.numpy(),
                        std=post.std.numpy(), forward_out=out.numpy(), **{"stage_" + k: v.half().numpy() for k, v in stages.items()})
    print(OUT, os.path.getsize(OUT), "bytes; x range", float(x.min()), float(x.max()), "logvar range", float(post.logvar.min()),
          float(post.logvar.max()))


if __name__ == "__main__":
    main()
