"""Time tpxl_b200.VAE.encode on 2048 primitives next to VAE.decode, and split one profiled encode by kernel class.

    python tools/vae_encode_perf.py [min_seconds]      # default: a timed window of at least 1 s per measurement

The encode input (2048 x 6 x 8^3 fp16 = 12.6 MB) fits the 126 MB L2, so before every timed pass a 256 MB scratch buffer is
overwritten (L2 flush, outside the timed interval): the numbers are cold-L2 pass times, summed over a window of >= 1 s.
Work is counted from the layer shapes below (2 * MACs), F_enc = 3.638 TFLOP per 2048 primitives.  The card's name, power limit
and SM clock limit are read in the same process and printed with the numbers.
"""
import ctypes as C
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch                                    # noqa: E402

import tpxl_b200                                # noqa: E402
from tpxl_b200 import _lib, synth               # noqa: E402

P = 2048
DEV = "cuda:0"
CLASSES = ["gemm", "attention", "ln", "gemv", "elementwise", "conv_gemm", "groupnorm", "vae_misc"]


def encoder_flop(P, cin=6, c0=32, c1=256, lat2=2, heads=8):
    """2 * multiply-adds of every convolution / linear / attention product of Encoder + quant_conv, per the released shapes."""
    v8, v4 = 512, 64
    conv = lambda vox, ci, co, k=27: 2 * vox * ci * co * k
    f = conv(v8, cin, c0)                                         # conv_in
    f += 4 * conv(v8, c0, c0)                                     # down_blocks.0: two ResnetBlocks
    f += conv(v4, c0, c0)                                         # downsample (stride 2: 4^3 outputs)
    f += conv(v4, c0, c1) + conv(v4, c1, c1) + conv(v4, c0, c1, 1)   # down_blocks.1.nets.0 (+ 1x1 shortcut)
    f += 2 * conv(v4, c1, c1)                                     # down_blocks.1.nets.1
    f += 4 * conv(v4, c1, c1)                                     # mid ResnetBlocks
    f += 2 * v4 * c1 * 3 * c1 + 2 * v4 * c1 * c1 + 2 * 2 * v4 * v4 * c1   # attention: qkv, proj, QK^T and PV
    f += conv(v4, c1, lat2) + conv(v4, lat2, lat2, 1)             # conv_out, quant_conv
    return P * f


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def timed(fn, flush, min_s):
    """Mean device time of fn() per pass with a cold L2, over a window of at least min_s seconds."""
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    n, tot, tot_flush, t0 = 0, 0.0, 0.0, time.perf_counter()
    while time.perf_counter() - t0 < min_s or n < 10:
        ev[0].record(); flush(); ev[1].record(); fn(); ev[2].record()
        torch.cuda.synchronize()
        tot_flush += ev[0].elapsed_time(ev[1]); tot += ev[1].elapsed_time(ev[2]); n += 1
    return tot / n, n


def main():
    min_s = float(sys.argv[1]) if len(sys.argv) > 1 else 1.0
    assert torch.cuda.is_available(), "needs the B200"
    sd = synth.device_state_dict(synth.vae_decoder_shapes(**synth.FULL_VAE), 1, DEV, torch.float32)
    sd.update(synth.device_state_dict(synth.vae_encoder_shapes(**synth.FULL_VAE), 2, DEV, torch.float32))
    vae = tpxl_b200.VAE(**synth.FULL_VAE)
    vae.load_state_dict(sd)
    vae = vae.to(DEV)
    g = torch.Generator(device=DEV).manual_seed(3)
    x = torch.randn(P, 6, 8, 8, 8, generator=g, device=DEV).half()
    z = torch.randn(P, 1, 4, 4, 4, generator=g, device=DEV).half()
    scratch = torch.empty(256 << 20, dtype=torch.uint8, device=DEV)
    flush = lambda: scratch.fill_(1)
    with torch.no_grad():
        for _ in range(3):
            vae.encode(x); vae.decode(z)
        torch.cuda.synchronize()
        enc_ms, n_enc = timed(lambda: vae.encode(x), flush, min_s)
        dec_ms, n_dec = timed(lambda: vae.decode(z), flush, min_s)
        lib = _lib.lib()
        split = {}
        for name, fn in (("encode", lambda: vae.encode(x)), ("decode", lambda: vae.decode(z))):
            flush(); torch.cuda.synchronize()
            lib.tpx_profile_begin()
            fn()
            ms = (C.c_float * 8)(); cnt = (C.c_int64 * 8)()
            lib.tpx_profile_end(ms, cnt)
            split[name] = {CLASSES[i]: dict(ms=round(ms[i], 4), launches=int(cnt[i])) for i in range(8) if cnt[i]}
    F_enc = encoder_flop(P)
    res = dict(card=card(), primitives=P, input_dtype="fp16", l2="flushed before every pass (256 MB overwrite, not timed)",
               encode_ms=round(enc_ms, 4), encode_passes=n_enc, decode_ms=round(dec_ms, 4), decode_passes=n_dec,
               F_enc_tflop=round(F_enc / 1e12, 4), encode_tflops=round(F_enc / (enc_ms * 1e-3) / 1e12, 1),
               profiled_split_ms=split)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
