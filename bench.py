#!/usr/bin/env python
"""bench.py — DiT denoising steps/sec (2048 primitive tokens, CFG x2) on N B200s, plus VAE decode ms.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): image-conditioned DDIM, CFG 6, 2048 tokens x 1370 context tokens, fp16, ONE
sample per GPU.  A *step* is one `forward_with_cfg` (two sequences) + the sampler update.  Synthetic weights of the
shipped architecture and synthetic inputs of the shipped shapes (no checkpoints or images exist offline).

  value    steps/s, whole job: inputs already in HBM, device-timed (CUDA events on the launch stream), max over ranks.  The timestep
           embedding + adaLN modulation rows of the schedule are computed once per image (DiT.set_timesteps, what the sampling loops do)
           INSIDE the timed region — every 25 steps — and `timestep_table` reports their cost and the rate without the hoist.
  e2e      the same through the public API from HOST buffers: every step copies x_t from pinned host memory, runs
           forward_with_cfg + the update, and reads x_{t-1} back to pinned host memory; the per-image conditioning
           upload and K/V hoist are inside the timed region too.
  roofline tcgen05 GEMM kernel family: algorithmic FLOPs of the GEMMs in a step / their summed device time, measured
           live with per-launch CUDA events (a separate profiled pass of the same steps); peak from MEASURED_PEAKS.json.
  cpu_baseline / --impl reference: the staged reference modules (oracle/_ref; the oracle port only if they are absent), fp32, host cores.

  --dump-outputs DIR  after the timed steps, rank 0 writes what the last timed step returned to its caller as DIR/<name>.npy (float32):
           model_output (forward_with_cfg), sample and pred_xstart (the sampler update); with --config 5, sample and recon_param of the
           last generation.  Weights and inputs are seeded, so two builds run with the same arguments can be compared output for output.
           Past 64 MB in all, each array is replaced by the same share of its elements, flattened, at sorted positions drawn from a fixed seed.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True        # the benchmark writes nothing into the tree it runs from (which may be read-only)

METRIC = "DiT steps/sec (2048 prim tokens, CFG x2)"
UNIT = "steps/s"
N_TOK, M_CTX, D, H, L, DC, CIN = 2048, 1370, 1152, 16, 28, 768, 68
CFG_SCALE = 6.0
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}


# ---- algorithmic work (SURVEY.md §8d term table; FLOPs = 2*MACs, per sequence of 2048 tokens) ----------------------
def flops_terms():
    g = lambda m, n, k: 2.0 * m * n * k
    per_block = dict(
        adaln=g(1, 9 * D, D), ca_q=g(N_TOK, D, D), ca_k=g(M_CTX, D, DC), ca_v=g(M_CTX, D, DC), ca_qk=g(N_TOK, M_CTX, D), ca_pv=g(N_TOK, M_CTX, D),
        ca_proj=g(N_TOK, D, D), sa_qkv=g(N_TOK, 3 * D, D), sa_qk=g(N_TOK, N_TOK, D), sa_pv=g(N_TOK, N_TOK, D), sa_proj=g(N_TOK, D, D),
        fc1=g(N_TOK, 4 * D, D), fc2=g(N_TOK, D, 4 * D))
    embed_final = g(N_TOK, D, CIN) + g(1, D, 256) + g(1, D, D) + g(1, 2 * D, D) + g(N_TOK, 2 * CIN, D)
    return per_block, embed_final


def f_step_algorithmic() -> float:
    pb, ef = flops_terms()
    return 2 * (L * sum(pb.values()) + ef)            # 6.343e12


def f_step_executed() -> dict:
    """What the build actually executes per step: cross K/V hoisted out of the step, the null half skips cross-attention."""
    pb, ef = flops_terms()
    gemm_cond = pb["ca_q"] + pb["ca_proj"]
    gemm_both = pb["sa_qkv"] + pb["sa_proj"] + pb["fc1"] + pb["fc2"]
    gemm = L * (gemm_cond + 2 * gemm_both) + 2 * 2.0 * N_TOK * 2 * CIN * D
    attn = L * (pb["ca_qk"] + pb["ca_pv"] + 2 * (pb["sa_qk"] + pb["sa_pv"]))
    return {"gemm": gemm, "attention": attn, "total": gemm + attn}


F_VAE = 4.593e12   # SURVEY.md §8a a14: 2242.8 MFLOP per primitive x 2048
DUMP_BYTES = 64_000_000


def dump_outputs(dirname: str, tensors: dict) -> None:
    """--dump-outputs: each tensor as <dirname>/<name>.npy in float32; over DUMP_BYTES in all, a fixed seeded sample of each."""
    import numpy as np
    arrays = {k: v.detach().float().cpu().numpy() for k, v in tensors.items()}
    total = sum(a.nbytes for a in arrays.values())
    budget = DUMP_BYTES - 1024 * len(arrays)                     # room for the .npy headers
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        if total > budget:
            keep = a.size * budget // total
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(dirname, name + ".npy"), a)
    print(f"[bench] wrote {', '.join(arrays)} to {dirname}" + (" (sampled)" if total > budget else ""), file=sys.stderr, flush=True)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return {k: float(d[k]) for k in FALLBACK_PEAKS if k in d} | {"source": "measured (MEASURED_PEAKS.json)"}
        except Exception:
            pass
    return dict(FALLBACK_PEAKS, source="fallback (B200_PROFILING.md)")


# ---- clocks sampler -------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def mark(self):
        return len(self.rows)

    def stop(self, start_idx=0):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()          # exact PID we started
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        rows = [r.split(", ") for r in self.rows[start_idx:] if r.count(",") >= 6] or [r.split(", ") for r in self.rows if r.count(",") >= 6]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = [float(r[0]) for r in rows]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for j, n in enumerate(names) if any(r[3 + j].strip().lower().startswith("active") for r in rows)]
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": float(rows[0][1]), "power_w_max": max(float(r[2]) for r in rows),
                "samples": len(rows), "reasons": reasons}


# ---- reference arm / cpu baseline: the reference's own modules on the host cores -------------------------------------
def _cpu_step_fn():
    """-> (step_fn, kind, what).  step_fn() runs ONE whole DDIM step of configs[1] on the host cores in fp32: the full 28-block
    forward_with_cfg (2 sequences x 2048 tokens x 1370 context tokens) + the sampler update — no depth extrapolation.

    kind "reference": the UNMODIFIED reference modules staged under oracle/_ref (oracle/stage_ref.py; DiT from
    models/dit_crossattn.py driven by models/diffusion's own ddim_sample_loop_progressive, xformers restated with SDPA) — on a
    CPU torch.autocast('cuda') disables itself, so this is the reference's fp32 arithmetic.  kind "port": the oracle port
    (oracle/dit.py + oracle/diffusion.py), used only when oracle/_ref is not staged."""
    import torch
    from tpxl_b200 import synth
    torch.set_grad_enabled(False)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(1, N_TOK, CIN, generator=g)
    y = torch.randn(1, M_CTX, DC, generator=g)
    try:
        from oracle import refmods
        have_ref = refmods.available()
    except Exception:
        have_ref = False
    if have_ref:
        import warnings
        warnings.filterwarnings("ignore", message=".*Disabling autocast.*")
        ref = refmods.load()
        with torch.device("meta"):
            model = ref.DiT(**synth.FULL_DIT)
        model = model.to_empty(device="cpu").eval()
        for prm in model.parameters():
            prm.normal_(0.0, 0.02, generator=g)
        diffusion = ref.create_diffusion("ddim25", noise_schedule="squaredcos_cap_v2", diffusion_steps=1000, parameterization="v")
        kw = dict(y=y, cfg_scale=CFG_SCALE, precision_dtype=torch.float16, enable_amp=True)      # inference.py:318-320
        state = {"it": None}

        def step():
            if state["it"] is None:
                state["it"] = iter(diffusion.ddim_sample_loop_progressive(model.forward_with_cfg, x.shape, x, clip_denoised=False, model_kwargs=kw,
                                                                          progress=False, device="cpu"))
            try:
                next(state["it"])
            except StopIteration:                      # more than 25 steps requested: start another image
                state["it"] = None
                step()
        return step, "reference", "reference DiT.forward_with_cfg (28 blocks) + reference ddim_sample per step, fp32 on the host cores (oracle/_ref)"
    import oracle
    sd = {k: torch.randn(s, generator=g) * 0.02 for k, s in synth.dit_shapes(**synth.FULL_DIT).items()}
    sched = oracle.diffusion.Schedule("ddim25")
    state = {"i": 24, "x": x}

    def step():
        t = torch.tensor([sched.timestep_map[state["i"]]])
        out = oracle.dit.forward_with_cfg(sd, state["x"], t, y, CFG_SCALE, H, "fp32")
        state["x"] = oracle.diffusion.ddim_step(sched, state["x"], out, state["i"])["sample"]
        state["i"] = state["i"] - 1 if state["i"] > 0 else 24
    return step, "port", "oracle port (oracle/dit.py forward_with_cfg, 28 blocks, + oracle/diffusion.py ddim_step) per step, fp32 on the host cores"


def _pick_threads() -> int:
    """torch's CPU GEMMs do not always scale to every hardware thread of a large host: try all / half / 32 threads on one MLP-sized
    fp32 GEMM (4096 x 1152 x 4608) and keep the fastest.  Returns the thread count now in effect."""
    import torch
    ncpu = os.cpu_count() or 1
    a, b = torch.randn(4096, D), torch.randn(D, 4 * D)
    best = (float("inf"), ncpu)
    for nt in sorted({ncpu, max(1, ncpu // 2), min(ncpu, 32)}, reverse=True):
        torch.set_num_threads(nt)
        a @ b
        t0 = time.perf_counter()
        for _ in range(3):
            a @ b
        dt = time.perf_counter() - t0
        if dt < best[0]:
            best = (dt, nt)
    torch.set_num_threads(best[1])
    return best[1]


def cpu_steps(n_warm: int, n_timed: int, budget_s: float):
    """Times whole reference steps on all host cores.  Stops early (never below 3 timed steps when n_timed >= 3) once `budget_s`
    is spent.  -> dict(value steps/s, per-step seconds, cores, kind, what)."""
    import torch
    cores = _pick_threads()
    step, kind, what = _cpu_step_fn()
    t_begin = time.perf_counter()
    for _ in range(n_warm):
        step()
    per = []
    floor = min(3, n_timed)
    for i in range(n_timed):
        t0 = time.perf_counter()
        step()
        per.append(time.perf_counter() - t0)
        spent = time.perf_counter() - t_begin
        if len(per) >= floor and spent + statistics.mean(per) > budget_s:
            break
    total = sum(per)
    return {"value": len(per) / total, "per_step_s": per, "total_s": total, "cores": cores, "kind": kind, "what": what}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # one untimed step pages the 3.6 GB of fp32 parameters in and spins the thread pool up; then whole steps are timed
    n_warm = min(max(args.warmup, 0), 1)
    r = cpu_steps(n_warm=n_warm, n_timed=args.steps, budget_s=float("inf"))      # exactly --steps timed steps
    n = len(r["per_step_s"])
    sample = f"{n} whole steps timed ({r['what']}); requested --steps {args.steps} --warmup {args.warmup}, {n_warm} untimed warm-up step(s), no extrapolation"
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": n, "warmup": n_warm,
            "ms_per_step": 1000.0 / r["value"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": {"workload": "configs[1]: image-cond DDIM-25 step, CFG 6, 2048 tokens x 1370 ctx tokens, 1 sample (2 sequences per forward), "
                                   "the reference's own modules in fp32 on the host cores"},
            "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": sample},
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
            "extrapolated": False, "same_config": True, "measured_blocks": L}
    print(json.dumps(line), flush=True)


# ---- our arm -----------------------------------------------------------------------------------------------------------
def _note(msg):
    if os.environ.get("TPX_BENCH_VERBOSE"):
        print(f"[bench] {msg}", file=sys.stderr, flush=True)


def run_ours(args):
    import torch
    import tpxl_b200
    from tpxl_b200 import _lib, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    lib = _lib.lib()
    K, W = args.steps, max(args.warmup, 3)

    # model (random init of the shipped architecture), one sample per GPU, noise/conditioning drawn like inference.py:313-317
    sd = synth.device_state_dict(synth.dit_shapes(**synth.FULL_DIT), 1234, dev, torch.float16)
    model = tpxl_b200.DiT(**synth.FULL_DIT)
    model.load_state_dict(sd)
    model = model.to(dev).eval()
    del sd
    g = torch.Generator().manual_seed(42 + rank)
    _ = torch.randn(1, N_TOK, 1, 4, 4, 4, generator=g)
    BS = args.samples_per_gpu
    x_host = torch.randn(BS, N_TOK, CIN, generator=g).pin_memory()
    y_host = torch.randn(BS, M_CTX, DC, generator=torch.Generator().manual_seed(43 + rank)).pin_memory()
    respacing = "ddim25"
    diffusion = tpxl_b200.create_diffusion(respacing, noise_schedule="squaredcos_cap_v2", diffusion_steps=1000, parameterization="v")
    diffusion.match_reference_rng = True
    nT = diffusion.num_timesteps
    t_all = torch.tensor(diffusion.timestep_map, dtype=torch.int64, device=dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    tmap = [int(v) for v in diffusion.timestep_map]
    hoist = os.environ.get("TPX_BENCH_HOIST_T", "1") != "0"     # 0: every forward recomputes the timestep MLP + adaLN pass (A/B switch)

    def begin_image():
        # what SpacedDiffusion's loops do at the start of every sampling run: the timestep embedding + adaLN modulation rows of the
        # schedule's 25 timesteps in one go (DiT.set_timesteps).  force=True: recomputed for every image, inside the timed regions.
        if hoist:
            model.set_timesteps(tmap, force=True)

    last = {}                                                   # what the latest step returned to its caller (--dump-outputs)

    def one_step(x, y, i, use_table=True):
        t = t_all[i % nT].expand(BS).contiguous()
        out = model.forward_with_cfg(x, t, y, cfg_scale=CFG_SCALE, precision_dtype=torch.float16, enable_amp=True,
                                     t_host=tmap[i % nT] if (hoist and use_table) else None)
        noise = torch.randn_like(x)
        step = diffusion._step(True, x, out, i % nT, 0.0, False, noise)
        last.update(step, model_output=out)
        return step["sample"]

    _note("model ready")
    # ---- device-resident timing ("value") ----
    x = x_host.to(dev)
    y = y_host.to(dev)
    with torch.no_grad():
        begin_image()
        for i in range(W):
            x = one_step(x, y, nT - 1 - i)
        barrier()
        clocks = ClockSampler(local) if rank == 0 else None
        mark = clocks.mark() if clocks else 0
        l0 = lib.tpx_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for i in range(K):
            if i % nT == 0:
                begin_image()                               # once per image (25 steps), inside the timed region
            x = one_step(x, y, nT - 1 - (i % nT))
        e1.record()
        barrier()
        launches = lib.tpx_launch_count() - l0
        ms_dev = e0.elapsed_time(e1)
        clock_info = clocks.stop(mark) if clocks else None
        outputs = dict(last)                                    # the last timed step's results (the later legs take new steps)

        _note(f"value leg done: {ms_dev:.2f} ms")
        # the same K steps with every forward recomputing the timestep MLP + adaLN pass (what the table replaces): in-run A/B, not a headline
        ms_plain = None
        if hoist:
            p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            p0.record()
            for i in range(K):
                x = one_step(x, y, nT - 1 - (i % nT), use_table=False)
            p1.record()
            barrier()
            ms_plain = p0.elapsed_time(p1)
        # ---- end to end from host buffers ("e2e") ----
        x_pin_out = torch.empty_like(x_host).pin_memory()
        xd = torch.empty(BS, N_TOK, CIN, device=dev)
        for i in range(2):
            xd.copy_(x_host, non_blocking=True)
            x_pin_out.copy_(one_step(xd, y, nT - 1 - i), non_blocking=True)
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        f0.record()
        y_e2e = y_host.to(dev, non_blocking=True)          # per-image conditioning upload + K/V hoist inside the timed region
        cur = x_host
        for i in range(K):
            if i % nT == 0:
                begin_image()
            xd.copy_(cur, non_blocking=True)
            x_pin_out.copy_(one_step(xd, y_e2e, nT - 1 - (i % nT)), non_blocking=True)
            torch.cuda.current_stream().synchronize()      # the host consumes the step result (progressive preview, inference.py:325)
            cur = x_pin_out
        f1.record()
        barrier()
        ms_e2e = f0.elapsed_time(f1)
        h2d = x_host.numel() * 4 + 8 + (y_host.numel() * 4) / K
        d2h = x_host.numel() * 4

        _note(f"e2e leg done: {ms_e2e:.2f} ms")
        # ---- the per-image timestep table on its own (device time of one DiT.set_timesteps over the schedule) ----
        ts_ms = None
        if hoist:
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            g0.record()
            begin_image()
            g1.record()
            torch.cuda.synchronize()
            ts_ms = g0.elapsed_time(g1)
        # ---- per-kernel-class device time (roofline leg): same steps, every launch bracketed by events ----
        nprof = min(K, 5)
        ms_cls, n_cls = (C.c_float * 8)(), (C.c_int64 * 8)()
        _lib.check(lib.tpx_profile_begin())
        for i in range(nprof):
            x = one_step(x, y, nT - 1 - i)
        _lib.check(lib.tpx_profile_end(ms_cls, n_cls))
        ms_cls = [v / nprof for v in ms_cls]
        n_cls = [int(v) // nprof for v in n_cls]

        _note("profile leg done")
        # ---- VAE decode of 2048 primitives (config #4), fp16 in/out ----
        vae_ms = None
        if rank == 0 and not args.no_vae:
            vsd = synth.device_state_dict(synth.vae_decoder_shapes(**synth.FULL_VAE), 1236, dev, torch.float16)
            vae = tpxl_b200.VAE(**synth.FULL_VAE)
            vae.load_state_dict(vsd)
            vae = vae.to(dev)
            z = (torch.randn(2048, 64, generator=torch.Generator().manual_seed(44)) * torch.tensor(synth.LATENT_STD[4:]) + torch.tensor(synth.LATENT_MEAN[4:])).reshape(2048, 1, 4, 4, 4).to(dev).half()
            for _ in range(3):
                vae.decode(z)
            torch.cuda.synchronize()
            v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            v0.record()
            for _ in range(5):
                vae.decode(z)
            v1.record()
            torch.cuda.synchronize()
            vae_ms = v0.elapsed_time(v1) / 5
            _lib.check(lib.tpx_profile_begin())
            vae.decode(z)
            vms, vn = (C.c_float * 8)(), (C.c_int64 * 8)()
            _lib.check(lib.tpx_profile_end(vms, vn))
            vae_cls = {"conv_gemm_ms": vms[5], "gemm_ms": vms[0], "groupnorm_ms": vms[6], "attention_ms": vms[1], "other_ms": vms[7]}
            # ---- config #2 as the user runs it: PrimXPipeline = DDIM-25 (CFG 6) + a13 + VAE.decode + a15 -> recon_param; and the
            # progressive variant (inference.py:325-349: previews at steps 0/10/20/24) with and without side-stream decode overlap
            pipe = tpxl_b200.PrimXPipeline(model, vae, latent_mean=synth.LATENT_MEAN, latent_std=synth.LATENT_STD, latent_nf=1.0, cfg_scale=CFG_SCALE, ddim_steps=25)
            xs, ys = x_host[:1].to(dev), y[:1].contiguous()

            def timed(fn, reps=3):
                # best of `reps` single runs after one warm-up run: the serial / overlapped previews differ by a few ms out of ~220,
                # less than the run-to-run spread of an average over two runs
                fn()
                torch.cuda.synchronize()
                best = float("inf")
                for _ in range(reps):
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    fn()
                    b.record()
                    torch.cuda.synchronize()
                    best = min(best, a.elapsed_time(b))
                return best

            t_final = timed(lambda: pipe(ys, xs))
            t_ser = timed(lambda: [0 for _ in pipe.sample_progressive(ys, xs, preview_every=10, overlap=False)])
            t_ovl = timed(lambda: [0 for _ in pipe.sample_progressive(ys, xs, preview_every=10, overlap=True)])
            pipe_info = {"workload": "configs[1] end to end: DDIM-25, CFG 6, + latent split + VAE decode (2048 prims, fp32 io) + primvolume pack, 1 sample",
                         "ms_per_sample": t_final, "samples_per_s": 1e3 / t_final,
                         "progressive_4_previews_ms": {"serial": t_ser, "side_stream_overlap": t_ovl, "hidden_ms": t_ser - t_ovl}}

    _note("vae leg done")
    # max over ranks
    t = torch.tensor([ms_dev, ms_e2e], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        gathered = [torch.empty_like(x) for _ in range(world)] if rank == 0 else None
        dist.gather(x, gathered, dst=0)                     # final latents to rank 0 over NCCL/NVLink (0.56 MB per sample)
    ms_dev, ms_e2e = float(t[0]), float(t[1])
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)

    peaks = load_peaks()
    # Both measured peaks are reported.  The timed loop is a fraction of a second at ~1.95 GHz (not the power-throttled regime the
    # sustained figure was taken in), so the BURST figure is the denominator of `frac`; `frac_sustained` is given beside it.
    peak_tf = peaks["bf16_tflops"]
    peak_sus = peaks["bf16_tflops_sustained"]
    steps_per_s = world * K / (ms_dev / 1e3)          # one step advances all BS local samples
    sample_steps_per_s = steps_per_s * BS
    fx = {k: v * BS for k, v in f_step_executed().items()}      # per step of this GPU (BS samples advance together)
    gemm_ms = ms_cls[0]
    gemm_tf = fx["gemm"] / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
    attn_tf = fx["attention"] / (ms_cls[1] / 1e3) / 1e12 if ms_cls[1] > 0 else 0.0
    step_ms_prof = sum(ms_cls)
    traffic = None
    import glob
    cands = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_gemm_traffic.json")))
    tp = cands[-1] if cands else ""
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    line = {
        "metric": METRIC, "value": steps_per_s, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_dev / K,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp16", "data": "synthetic",
        "config": {"workload": f"configs[1]: image-cond DDIM-25 step, CFG 6, 2048 tokens x 1370 ctx tokens, fp16, {BS} sample{'s' if BS > 1 else ''} per GPU ({2 * BS} sequences per forward)",
                   "samples_per_gpu": BS, "respacing": respacing, "cfg_scale": CFG_SCALE, "parallelism": f"dp{world} ({BS} sample{'s' if BS > 1 else ''} per GPU, no collective in the step loop)",
                   "l2": "each step streams 1.8 GB of fp16 weights (> 126 MB L2), so no separate L2 flush is needed"},
        "e2e": {"value": world * K / (ms_e2e / 1e3), "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
        "gpu_launches": int(launches),
        "sample_steps_per_s": sample_steps_per_s,
        "clocks": clock_info,
        "roofline": {"bound": "tensor", "kernel": "gemm_tc_kernel + gemm_tc2_kernel (tcgen05/TMA GEMM family incl. the cta_group::2 pair-tile kernel, all DiT linears)", "achieved": gemm_tf, "peak": peak_tf,
                     "unit": "TFLOP/s", "frac": gemm_tf / peak_tf if peak_tf else None, "frac_sustained": gemm_tf / peak_sus if peak_sus else None,
                     "peak_sustained": peak_sus, "traffic": traffic, "peak_source": peaks["source"] + ": burst bf16 (= fp16 rate) for `peak`/`frac`, sustained beside it",
                     "traffic_source": "profile constant: dram__bytes_read+write per launch from the latest committed ncu --set full capture (" + os.path.basename(tp) + "), not a live counter",
                     "flops_per_step": fx["gemm"], "launches_per_step": n_cls[0], "ms_per_step": gemm_ms,
                     "share_of_step": gemm_ms / step_ms_prof if step_ms_prof else None},
        "attention": {"kernel": "attention_tc_p_kernel (tcgen05 flash attention, S/O in TMEM, software-pipelined softmax warps)", "achieved": attn_tf, "unit": "TFLOP/s", "frac": attn_tf / peak_tf if peak_tf else None, "frac_sustained": attn_tf / peak_sus if peak_sus else None,
                      "ms_per_step": ms_cls[1], "launches_per_step": n_cls[1], "share_of_step": ms_cls[1] / step_ms_prof if step_ms_prof else None},
        "step_breakdown_ms": {"gemm": ms_cls[0], "attention": ms_cls[1], "ln_modulate": ms_cls[2], "gemv_embed": ms_cls[3], "cfg_sampler": ms_cls[4]},
        "timestep_table": ({"hoisted": True, "timesteps": nT, "ms_per_image": ts_ms, "ms_per_step_amortised": ts_ms / nT,
                            "steps_per_s_per_gpu_without_hoist": K / (ms_plain / 1e3),
                            "note": "timestep MLP + adaLN modulation of the schedule's timesteps computed once per image (DiT.set_timesteps, inside the "
                                    "timed regions of value and e2e); a step reads its row, so step_breakdown_ms.gemv_embed holds the token embedder only"}
                           if ts_ms is not None else {"hoisted": False}),
        "step_utilisation": {"F_step_algorithmic": BS * f_step_algorithmic(), "F_step_executed": fx["total"],
                             "frac_of_peak_algorithmic": steps_per_s / world * BS * f_step_algorithmic() / 1e12 / peak_tf,
                             "frac_of_peak_executed": steps_per_s / world * fx["total"] / 1e12 / peak_tf, "peak": peak_tf, "peak_kind": "burst"},
    }
    if vae_ms is not None:
        line["pipeline"] = pipe_info
        line["vae_decode"] = {"ms": vae_ms, "primitives": 2048, "dtype": "fp16", "achieved_tflops": F_VAE / (vae_ms / 1e3) / 1e12,
                              "frac": F_VAE / (vae_ms / 1e3) / 1e12 / peaks["bf16_tflops"], "peak": peaks["bf16_tflops"], "breakdown_ms": vae_cls}
    if not args.no_cpu and world >= 1:
        try:
            r = cpu_steps(n_warm=1, n_timed=2, budget_s=40.0)
            line["cpu_baseline"] = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"],
                                    "sample": f"{len(r['per_step_s'])} whole steps after 1 warm-up ({r['what']}): " + ", ".join(f"{v:.2f} s" for v in r["per_step_s"])}
        except Exception as ex:  # never lose the GPU line over the CPU leg
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {ex}"}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


# ---- configs[4] (config #5): end-to-end DDIM-100 + VAE decode, 4 samples per GPU -----------------------------------------
def run_config5(args):
    """BASELINE.json configs[4]: batch = 32 over 8 GPUs = 4 samples per GPU in one forward (8 sequences under CFG), DDIM 100 steps,
    then a13 + VAE.decode + a15 of every sample (PrimXPipeline).  A *step* here is one whole generation of the rank's 4 samples;
    value = samples/s over all ranks (weak scaling: 4 samples per GPU whatever N is).  No collective inside the timed region."""
    import torch
    import tpxl_b200
    from tpxl_b200 import _lib, synth
    world, rank, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    lib = _lib.lib()
    BS, STEPS = args.samples_per_gpu if args.samples_per_gpu > 1 else 4, args.ddim
    K, W = max(args.steps, 1), max(args.warmup, 1)
    sd = synth.device_state_dict(synth.dit_shapes(**synth.FULL_DIT), 1234, dev, torch.float16)
    model = tpxl_b200.DiT(**synth.FULL_DIT)
    model.load_state_dict(sd)
    model = model.to(dev).eval()
    del sd
    vae = tpxl_b200.VAE(**synth.FULL_VAE)
    vae.load_state_dict(synth.device_state_dict(synth.vae_decoder_shapes(**synth.FULL_VAE), 1236, dev, torch.float16))
    vae = vae.to(dev)
    pipe = tpxl_b200.PrimXPipeline(model, vae, latent_mean=synth.LATENT_MEAN, latent_std=synth.LATENT_STD, latent_nf=1.0, cfg_scale=CFG_SCALE, ddim_steps=STEPS)
    noise = tpxl_b200.shard.draw_noise(world * BS, N_TOK, CIN, seed=42)[tpxl_b200.shard.assigned(world * BS, world, rank)].pin_memory()
    y_host = torch.randn(BS, M_CTX, DC, generator=torch.Generator().manual_seed(43 + rank)).pin_memory()
    out_host = torch.empty(BS, N_TOK, 4 + 6 * 512).pin_memory()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def generation():          # host buffers in, host buffers out: this IS the end-to-end path
        y = y_host.to(dev, non_blocking=True)
        x = noise.to(dev, non_blocking=True)
        res = pipe(y, x)
        out_host.copy_(res["recon_param"], non_blocking=True)
        return res

    for _ in range(W):
        generation()
    barrier()
    clocks = ClockSampler(local) if rank == 0 else None
    mark = clocks.mark() if clocks else 0
    l0 = lib.tpx_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(K):
        res = generation()
    e1.record()
    barrier()
    launches = lib.tpx_launch_count() - l0
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    clock_info = clocks.stop(mark) if clocks else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"sample": res["sample"], "recon_param": out_host})
    # split of one generation: the DDIM loop alone vs decode + glue
    y, x = y_host.to(dev), noise.to(dev)
    d = pipe.make_diffusion()
    a, b, c = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    torch.cuda.synchronize()
    a.record()
    with torch.no_grad():
        for smp in d.ddim_sample_loop_progressive(model.forward_with_cfg, x.shape, x, clip_denoised=False, model_kwargs=pipe._model_kwargs(y), device=dev):
            pass
        b.record()
        pipe.decode_latents(smp["sample"])
    c.record()
    torch.cuda.synchronize()
    loop_ms, dec_ms = a.elapsed_time(b), b.elapsed_time(c)
    if dist is not None:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    if rank == 0:
        peaks = load_peaks()
        t = float(ms[0]) / 1e3
        sps = world * BS * K / t
        flops = BS * (STEPS * f_step_executed()["total"] + F_VAE)            # executed tensor-core FLOPs of one generation on one GPU
        tf = flops * K / t / 1e12
        line = {"metric": "samples/s, end-to-end DDIM-%d + VAE decode (CFG 6, 2048 prims), %d samples per GPU" % (STEPS, BS), "value": sps, "unit": "samples/s",
                "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": float(ms[0]) / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "fp16", "data": "synthetic",
                "config": {"workload": "configs[4]: DDIM-%d + VAE decode, batch %d = %d samples per GPU x %d GPUs, CFG 6 (8 sequences per forward)" % (STEPS, world * BS, BS, world),
                           "samples_per_gpu": BS, "parallelism": f"dp{world} (samples sharded s mod G, no collective in the loop)",
                           "l2": "each forward streams 1.8 GB of fp16 weights (> 126 MB L2)"},
                "e2e": {"value": sps, "unit": "samples/s", "h2d_bytes_per_step": int(noise.numel() * 4 + y_host.numel() * 4), "d2h_bytes_per_step": int(out_host.numel() * 4)},
                "gpu_launches": int(launches), "clocks": clock_info,
                "roofline": {"bound": "tensor", "kernel": "whole generation (DiT steps + VAE decode), executed FLOPs", "achieved": tf, "peak": peaks["bf16_tflops"],
                             "peak_sustained": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s", "frac": tf / peaks["bf16_tflops"],
                             "frac_sustained": tf / peaks["bf16_tflops_sustained"], "traffic": None, "peak_source": peaks["source"]},
                "split_ms": {"ddim_loop": loop_ms, "decode_and_glue": dec_ms, "per_dit_step": loop_ms / STEPS, "dit_sample_steps_per_s": BS * STEPS / (loop_ms / 1e3)}}
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=25)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-vae", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--samples-per-gpu", type=int, default=1, help="B per GPU (config #5 uses 4); the headline config is 1")
    ap.add_argument("--config", type=int, default=2, choices=[2, 5], help="2 = BASELINE configs[1] (the headline: DiT steps/s); 5 = configs[4] "
                    "(end-to-end DDIM-100 + VAE decode, 4 samples per GPU, samples/s; here --steps counts whole generations)")
    ap.add_argument("--ddim", type=int, default=100, help="DDIM steps of --config 5")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy (float32, rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the CUDA path; the reference arm has other weights and inputs")
    # The contract is ONE JSON line on stdout.  Native libraries write there too (NCCL prints its version banner to fd 1 when
    # NCCL_DEBUG=VERSION is set on the box), so fd 1 is pointed at stderr for the whole run and the result line goes to the
    # saved descriptor.
    try:
        sys.stdout.flush()
        real_fd = os.dup(1)
        os.dup2(2, 1)
        sys.stdout = os.fdopen(real_fd, "w", buffering=1)
    except OSError:
        pass                                      # unusual descriptor set-up: keep the plain stdout
    if args.impl == "reference":
        run_reference(args)
    elif args.config == 5:
        if "--steps" not in sys.argv:
            args.steps = 2
        run_config5(args)
    else:
        run_ours(args)
    sys.stdout.flush()


if __name__ == "__main__":
    main()
