"""CPU: the VAE encoder's host contract — the oracle restatement against the reference's own encode (vae_encode.npz), the
encoder key / shape contract, the state_dict round trip with encoder keys, the paths that refuse to run without a CUDA module,
and the C-ABI table of the encoder entry points."""
import importlib
import json
import os
import re

import numpy as np
import pytest
import torch

import oracle
import tpxl_b200
from tpxl_b200 import _lib, synth
import vae_encode_oracle as E

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ENC_SEED, DEC_SEED = 211, 103     # tests/golden/make_vae_encode_golden.py
NEW_SYMBOLS = ["tpx_vae_encoder_create", "tpx_vae_encoder_destroy", "tpx_vae_encoder_set_weight", "tpx_vae_encoder_finalize",
               "tpx_vae_encoder_workspace_bytes", "tpx_vae_encode", "tpx_vae_encode_stage", "tpx_vae_posterior", "tpx_conv3d_k3_s2"]


def rel(a, b):
    a, b = torch.as_tensor(a).double(), torch.as_tensor(b).double()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def full_sd():
    sd = synth.synth_state_dict(synth.vae_decoder_shapes(**synth.FULL_VAE), DEC_SEED)
    sd.update(synth.synth_state_dict(synth.vae_encoder_shapes(**synth.FULL_VAE), ENC_SEED))
    return sd


def test_oracle_encode_matches_reference_fixture(golden_dir):
    g = np.load(os.path.join(golden_dir, "vae_encode.npz"))
    sd = full_sd()
    x = torch.from_numpy(g["x"])
    stages = {}
    params = E.encode(sd, x, "fp32", stages=stages)
    post = E.posterior(params)
    for k in ("parameters", "mean", "logvar", "std"):
        got = params if k == "parameters" else post[k]
        assert rel(got, torch.from_numpy(g[k])) <= 2e-5, k
    for k, v in stages.items():                       # stored as fp16
        assert rel(v, torch.from_numpy(g["stage_" + k]).float()) <= 1e-3, k
    out = oracle.vae.decode(sd, post["mean"], "fp32")  # forward(x, sample=False)[0] = decode(mode())
    assert rel(out, torch.from_numpy(g["forward_out"])) <= 2e-5


def test_oracle_posterior_clamp_and_deterministic():
    p = torch.tensor([[1.0, -2.0, -40.0, 25.0]]).reshape(1, 4, 1, 1, 1)
    post = E.posterior(p)
    assert post["logvar"].flatten().tolist() == [-30.0, 20.0]
    torch.testing.assert_close(post["std"], torch.exp(0.5 * post["logvar"]))
    d = E.posterior(p, deterministic=True)
    assert not d["std"].any() and not d["var"].any()


def test_encoder_key_contract(golden_dir):
    keys = json.load(open(os.path.join(golden_dir, "state_dict_keys.json")))["vae"]
    enc = {k: tuple(v) for k, v in keys.items() if k.startswith(("encoder.", "quant_conv."))}
    assert len(enc) == 65
    assert dict(synth.vae_encoder_shapes(**synth.FULL_VAE)) == enc


def test_state_dict_round_trip_with_encoder_keys(tmp_path):
    sd = full_sd()
    v = tpxl_b200.VAE(**synth.FULL_VAE)
    res = v.load_state_dict(sd)
    assert not res.missing_keys and not res.unexpected_keys
    out = v.state_dict()
    assert set(out) == set(sd)
    enc = [k for k in out if k.startswith(("encoder.", "quant_conv."))]
    assert len(enc) == 65 and all(torch.equal(out[k], sd[k]) for k in enc)
    # load_checkpoint stays decode-only: the encoder half of a checkpoint is not read
    path = tmp_path / "vae.pt"
    torch.save({"model_state_dict": sd}, path)
    w = tpxl_b200.VAE(**synth.FULL_VAE)
    w.load_checkpoint(str(path))
    assert not any(k.startswith(("encoder.", "quant_conv.")) for k in w.state_dict())


def test_no_cpu_path():
    v = tpxl_b200.VAE(**synth.FULL_VAE)
    v.load_state_dict(full_sd())
    with pytest.raises(NotImplementedError, match="CUDA"):
        v.encode(torch.zeros(1))                     # raised before the input is looked at
    with pytest.raises(NotImplementedError, match="CUDA"):
        v.forward(torch.zeros(1))
    with pytest.raises(NotImplementedError):
        v.encode(None)
    with pytest.raises(NotImplementedError):
        tpxl_b200.vae.DiagonalGaussianDistribution(torch.zeros(1, 2, 4, 4, 4))
    # an encoder layout outside the kernel set still constructs (the constructor is unchanged); encode refuses it
    other = tpxl_b200.VAE(**dict(synth.FULL_VAE, down_channels=[16, 32]))
    with pytest.raises(NotImplementedError):
        other.encode(torch.zeros(1, 6, 8, 8, 8))


def test_install_resolves_posterior_class():
    tpxl_b200.install()
    m = importlib.import_module("models.vae3d_dib")
    assert m.DiagonalGaussianDistribution is tpxl_b200.vae.DiagonalGaussianDistribution


def test_abi_table_lists_encoder_symbols():
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "tpx.h")).read(), flags=re.S)
    declared = set(re.findall(r"\b(tpx_[a-z0-9_]+)\s*\(", src))
    for n in NEW_SYMBOLS:
        assert n in declared and n in _lib.SIGNATURES, n
    hdr = open(os.path.join(ROOT, "include", "tpx.h")).read()
    for cite in ("vae3d_dib.py:270-327", "vae3d_dib.py:51-60", "vae3d_dib.py:431-433"):
        assert cite in hdr


def test_library_exports_encoder_symbols():
    import __graft_entry__
    __graft_entry__._load_build_module().build()
    lib = _lib.load_library()
    for n in NEW_SYMBOLS:
        assert hasattr(lib, n), n
    # argument validation happens before any CUDA call
    assert lib.tpx_vae_encoder_workspace_bytes(None, 8) == 0
    assert lib.tpx_vae_encode(None, None, 0, None, 0, 1, None, 0, None) == -1 and b"null" in lib.tpx_last_error()
    assert lib.tpx_vae_posterior(None, 0, 1, 64, 0, None, None, None, None) == -1 and b"null" in lib.tpx_last_error()
    assert lib.tpx_vae_encoder_create(None, None) == -1


def test_stride2_conv_kernel_is_tcgen05_and_tma():
    """The stride-2 convolution is its own gemm_tc_kernel instantiation (AMODE_CONV3_S2 = 2) with tensor-core MMAs and TMA loads."""
    import subprocess
    import __graft_entry__
    __graft_entry__._load_build_module().build()
    obj = os.path.join(ROOT, "3dtopia-xl_b200", "build", "gemm_tc.o")
    sass = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True).stdout
    funcs = {f.split("\n", 1)[0]: f for f in re.split(r"\n\s*Function : ", sass)[1:]}
    s2 = [body for name, body in funcs.items() if "gemm_tc_kernelILi32ELi32ELi2ELi0E" in name]
    assert len(s2) == 1
    for mnem in ("UTCHMMA", "UTMALDG", "LDTM"):
        assert mnem in s2[0], mnem
