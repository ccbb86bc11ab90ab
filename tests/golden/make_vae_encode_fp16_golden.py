#!/usr/bin/env python
"""Generate tests/golden/vae_encode_fp16.npz: what tests/test_gpu_vae_encode.py::test_encode_against_autocast_fixture compares with.

Runs THE REFERENCE'S OWN VAE.encode (staged unmodified under oracle/_ref by oracle/stage_ref.py) on a B200, under
torch.autocast('cuda', fp16) and in fp32 with TF32 off, over the test's fp16_inputs() (2048 primitives).  Needs a GPU and the
staged reference:

    python oracle/stage_ref.py && python tests/golden/make_vae_encode_fp16_golden.py [OUT]

Stored: parameters and std of every 128th primitive from both runs, the fp16-vs-fp32 relative L2 of parameters and std over the
whole batch, and float64 fingerprints of the weights and inputs.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import test_gpu_vae_encode as T                   # noqa: E402
from gpu_util import rel_l2                       # noqa: E402
from oracle import refmods                        # noqa: E402
from tpxl_b200 import synth                       # noqa: E402

DEV = T.DEV


def main(out):
    if not refmods.available():
        raise SystemExit("oracle/_ref is not staged: run python oracle/stage_ref.py where the reference checkout exists")
    torch.set_grad_enabled(False)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    sd, x = T.fp16_inputs()
    fx = dict(inputs=T.fingerprint(sd, x), prims=T.FP16_PRIMS, made_on=f"{torch.cuda.get_device_name(DEV)}, torch {torch.__version__}")
    ref = refmods.build_vae(synth.FULL_VAE, sd, DEV)
    xd = x.to(DEV)
    p32 = ref.encode(xd)
    with torch.autocast("cuda", dtype=torch.float16):
        p16 = ref.encode(xd)
    idx = torch.from_numpy(T.FP16_PRIMS).to(DEV)
    for f in ("parameters", "std"):
        a, b = getattr(p16, f), getattr(p32, f)
        fx[f + "16"], fx[f + "32"] = a.index_select(0, idx).cpu().numpy(), b.index_select(0, idx).cpu().numpy()
        fx[f + "_noise"] = np.array(rel_l2(a.float(), b))
    np.savez_compressed(out, **fx)
    print(fx["made_on"], "->", out, f"{os.path.getsize(out)} bytes", {k: float(v) for k, v in fx.items() if k.endswith("_noise")},
          "dtype16", p16.parameters.dtype)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden", "vae_encode_fp16.npz"))
