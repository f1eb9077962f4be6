#!/usr/bin/env python
"""bench.py -- denoised-latents/sec (+ rendered-views/sec) of the LN3Diff generation hot path.

Workload (BASELINE.json configs[1]): DiT-L/2 T23D tri-latent, 250-step Euler-EDM + VanillaCFG(6.5)
(the shipped sampler, sgm/configs/txt2img-clipl-compat.yaml:47-60), batch = 8 prompts per GPU
(16 DiT samples per forward), bf16 tensor-core GEMMs / fp32 residual + sampler state.
One "step" = one full pass of the hot path over one batch: 250 denoising steps for 8 latents.
Independent prompts shard across GPUs with no data-path collective (weak scaling); the finished
latents are all-gathered once per step (tiny).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

`--impl reference` times the reference algorithm's CPU path (the oracle port of the reference's
Python modules) on a bounded sample of the same workload.

`--dump-outputs DIR` writes what the last timed step returned, the denoised latents of the batch
(all ranks' latents after the gather), as DIR/latents.npy in float32.  The inputs are drawn from
fixed seeds, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ARCH = "DiT-L/2"
PROMPTS_PER_GPU = 8
DENOISE_STEPS = 250
CFG_SCALE = 6.5
FLOPS_PER_FORWARD_PER_SAMPLE = 0.613e12  # SURVEY.md section 8d (T23D DiT-L/2, MAC = 2 FLOP), as the reference computes it
# what this implementation executes per sample-forward: the context K/V projection is hoisted out of the loop
# (-0.32 GF/layer) and the zero-embedding CFG half skips its cross-attention q GEMM / FMHA / out GEMM
# (-3.46 GF/layer for half of the samples): 24 x (25.18 + 21.72) / 2 GF + 1 GF of embedders / final layer
FLOPS_EXECUTED_PER_FORWARD_PER_SAMPLE = 0.564e12


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--denoise-steps", type=int, default=DENOISE_STEPS, help=argparse.SUPPRESS)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the latents of the last timed step to DIR/latents.npy (float32)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs is only available with --impl ours")
    return a


def workload_config(n_gpus):
    return {"workload": "configs[1]: DiT-L/2 T23D tri-latent (12x32x32), EulerEDM 250 steps + VanillaCFG 6.5, "
                        "8 prompts/GPU (16 samples/forward)",
            "arch": ARCH, "denoise_steps": DENOISE_STEPS, "cfg_scale": CFG_SCALE,
            "prompts_per_gpu": PROMPTS_PER_GPU, "global_batch": PROMPTS_PER_GPU * n_gpus,
            "parallelism": f"prompt-sharded x{n_gpus} (replicated weights, no data-path collective)",
            "l2": "inputs larger than L2: 1.1 GB of bf16 weights stream through every forward",
              "adaln": "one modulation row per step shared by the batch, all 250 steps' rows computed in one pass per "
                       "sampling run (same arithmetic, bit-identical latents; LN3_SHARED_MODULATION=0 disables)",
              "uncond_cross_attention": "closed form for the zero-embedding CFG half (identical context tokens -> "
                                        "uniform softmax -> to_out(v_row)); LN3_UNCOND_CLOSED_FORM=0 disables"}


# ------------------------------------------------------------------ CPU reference arm / baseline
def host_cores() -> int:
    from ln3diff_b200.utils import host_cores as hc
    return hc()


# bounded samples of one Euler-EDM+CFG denoising step, largest first: (name, prompts, forwards, layers)
REF_SAMPLES = (("1 of 250 Euler-EDM+CFG steps for 1 prompt (2 DiT-L/2 fp32 forwards: uncond + cond)", 2, 24),
               ("1 of the 2 CFG forwards of 1 of 250 steps for 1 prompt (1 DiT-L/2 fp32 forward)", 1, 24),
               ("6 of the 24 blocks of 1 of the 2 CFG forwards of 1 of 250 steps for 1 prompt", 1, 6))
REF_BUDGET_S = 360.0          # whole `--impl reference` run (driver: "ends within a few minutes")


class CpuReference:
    """The oracle port of the DiT-L/2 denoising step on the host cores.  The model state is built ONCE;
    `step(level)` times one bounded sample and returns (latents/s extrapolated to the full 250-step job for
    one prompt, seconds).  Extrapolation is linear in blocks x forwards x steps (every block costs the same;
    embedders / final layer are < 0.2 % of a forward)."""

    def __init__(self, threads=None):
        import torch
        from oracle import dit as odit
        from ln3diff_b200.utils import build_t23d
        self.torch, self.odit = torch, odit
        self.cores = threads or host_cores()
        torch.set_num_threads(self.cores)
        m = build_t23d(ARCH)
        self.sd = {k: v.float() for k, v in m.state_dict().items()}
        del m
        g = torch.Generator().manual_seed(41)
        self.x = torch.randn(1, 12, 32, 32, generator=g)
        self.ctx = torch.cat([torch.zeros(1, 77, 768), torch.randn(1, 77, 768, generator=g)], 0)   # (uc, c)
        from oracle import samplers as osmp
        self.table = osmp.legacy_ddpm_sigmas(1000, append_zero=False, flip=True)
        self.sigmas = osmp.legacy_ddpm_sigmas(DENOISE_STEPS)
        self.osmp = osmp

    def step(self, level=0):
        torch, osmp = self.torch, self.osmp
        _, forwards, layers = REF_SAMPLES[level]
        t0 = time.perf_counter()
        with torch.no_grad():
            xx = self.x * torch.sqrt(1.0 + self.sigmas[0] ** 2.0)
            s = torch.ones(1) * self.sigmas[0]
            xin, sin = torch.cat([xx] * 2), torch.cat([s] * 2)
            sq = self.table[osmp.sigma_to_idx(sin, self.table)]
            sq4 = sq[:, None, None, None]
            sel = slice(0, 2) if forwards == 2 else slice(1, 2)
            net = self.odit.dit_t23d_forward(self.sd, ARCH, (xin / (sq4 ** 2 + 1.0) ** 0.5)[sel],
                                             osmp.sigma_to_idx(sq, self.table)[sel], self.ctx[sel],
                                             first_blocks=None if layers == 24 else layers)
            if forwards == 2:
                den = net * (-sq4) + xin
                x_u, x_c = den.chunk(2)
                d = (xx - (x_u + CFG_SCALE * (x_c - x_u))) / s[:, None, None, None]
                xx = xx + (self.sigmas[1] - s)[:, None, None, None] * d
        dt = time.perf_counter() - t0
        per_step = dt * (2 / forwards) * (24 / layers)       # one full CFG denoising step for one prompt
        return 1.0 / (per_step * DENOISE_STEPS), dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t_all = time.perf_counter()
    ref = CpuReference()
    n_iter = args.warmup + args.steps
    # the first pass (cold caches, thread pool start-up) picks the largest sample that keeps the whole run
    # inside REF_BUDGET_S; it is not one of the counted iterations
    level = 0
    _, dt0 = ref.step(0)
    while level + 1 < len(REF_SAMPLES):
        _, fw, ly = REF_SAMPLES[level]
        if dt0 * (fw / 2) * (ly / 24) * n_iter <= REF_BUDGET_S - (time.perf_counter() - t_all):
            break
        level += 1
    vals = []
    for i in range(n_iter):
        v, dt = ref.step(level)
        if i >= args.warmup:
            vals.append((v, dt))
    value = sum(v for v, _ in vals) / len(vals)
    ms = 1e3 * sum(dt for _, dt in vals) / len(vals)
    sample = REF_SAMPLES[level][0] + " per bench step; latents/s extrapolated linearly in blocks x forwards x steps x prompts"
    line = {"impl": "reference", "metric": "denoised-latents/sec", "value": value, "unit": "latents/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(args.gpus),
            "cpu_baseline": {"value": value, "unit": "latents/s", "cores": ref.cores, "kind": "port",
                             "sample": sample},
            "e2e": {"value": value, "unit": "latents/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "wall_s": time.perf_counter() - t_all}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------ clocks sampler
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons, pw = [], [], set(), []
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------ GPU reference leg (eager PyTorch)
def gpu_reference_leg(torch, dev, state_dict, B, nsteps, randn_d, ctx_d):
    """The reference's GPU arithmetic (stock eager PyTorch under bf16 autocast: cuBLAS + SDPA-flash, the
    reference's per-step recomputation and sampler launches left in; baseline/torch_eager.py) on the same
    B200, same workload, timed BEFORE the repo's arm in the same process (SURVEY.md 8d timing protocol).
    Bounded sample: `sample_steps` of the 250 denoising steps for the full 8-prompt batch, 3 repeats after a
    warm-up, extrapolated linearly in steps (every step launches the same kernels on the same shapes)."""
    from baseline.torch_eager import EagerDiT, euler_edm_cfg_steps
    sample_steps = 20
    m = EagerDiT(depth=24, dim=1024, heads=16, ctx_dim=768).to(dev).load_mirror_state_dict(state_dict).eval()
    uc = torch.zeros_like(ctx_d)
    run = lambda: euler_edm_cfg_steps(m, randn_d, ctx_d, uc, nsteps, CFG_SCALE, first_steps=sample_steps)
    run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 3
    e0.record()
    for _ in range(reps):
        run()
    e1.record()
    torch.cuda.synchronize()
    ms_step = e0.elapsed_time(e1) / reps / sample_steps
    del m
    torch.cuda.empty_cache()
    return {"value": B / (ms_step * nsteps / 1e3), "unit": "latents/s", "ms_per_denoise_step": ms_step,
            "kind": "port", "impl": "baseline/torch_eager.py: eager PyTorch, bf16 autocast, cuBLAS GEMMs + "
                                    "F.scaled_dot_product_attention, the reference's module structure and sgm sampler",
            "sample": f"{sample_steps} of {nsteps} Euler-EDM+CFG steps for {B} prompts x {reps} repeats, "
                      "extrapolated linearly in steps"}


# ------------------------------------------------------------------ our arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    from ln3diff_b200 import _lib, ops, pipeline
    from ln3diff_b200.utils import build_ae_decoder, build_t23d, orbit_cameras

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py --impl ours needs a CUDA GPU (no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n_gpus = world
    B = PROMPTS_PER_GPU
    nsteps = args.denoise_steps

    model = build_t23d(ARCH, seed=0, device=dev)
    # identical-seed inputs as the reference engine draws them (CPU generator, then moved):
    # one global randn for all prompts, sliced per rank (SURVEY.md section 8e)
    g = torch.Generator().manual_seed(41)
    randn_all = torch.randn(B * n_gpus, 12, 32, 32, generator=g)
    ctx_all = torch.randn(B * n_gpus, 77, 768, generator=g)
    sl = slice(rank * B, (rank + 1) * B)
    randn_h = randn_all[sl].contiguous().pin_memory()
    ctx_h = ctx_all[sl].contiguous().pin_memory()
    out_h = torch.empty(B, 12, 32, 32).pin_memory()
    randn_d, ctx_d = randn_h.to(dev), ctx_h.to(dev)
    uc_d = torch.zeros_like(ctx_d)

    # ---- the reference's GPU path first (same process, same box), then ours
    gpu_ref = None
    if rank == 0 and n_gpus == 1:
        try:
            gpu_ref = gpu_reference_leg(torch, dev, model.state_dict(), B, nsteps, randn_d, ctx_d)
        except Exception as e:  # noqa
            gpu_ref = {"error": repr(e)}

    model.prepare()
    tables = pipeline.edm_cfg_tables(nsteps, CFG_SCALE, B, dev)
    gathered = torch.empty(n_gpus * B, 12, 32, 32, device=dev) if world > 1 else None
    last = {}

    def one_step_device():
        lat = pipeline.sample_t23d(model, randn_d, {"crossattn": ctx_d}, {"crossattn": uc_d}, nsteps,
                                   CFG_SCALE, tables)
        if world > 1:
            dist.all_gather_into_tensor(gathered, lat)
        last["latents"] = gathered if world > 1 else lat
        return lat

    def one_step_e2e():
        # the public pipeline call with HOST inputs: H2D of noise + prompt embeddings, the per-prompt-batch
        # conditioning (context projection, all layers' K/V), 250 steps, D2H of the latents
        x = randn_h.to(dev, non_blocking=True)
        c = ctx_h.to(dev, non_blocking=True)
        lat = pipeline.sample_t23d(model, x, {"crossattn": c}, {"crossattn": torch.zeros_like(c)}, nsteps,
                                   CFG_SCALE, tables)
        out_h.copy_(lat, non_blocking=True)
        return lat

    def timed(fn, k, w):
        for _ in range(w):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = _lib.launch_count()
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item(), _lib.launch_count() - l0

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    ms_total, launches = timed(one_step_device, args.steps, args.warmup)
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "latents.npy"), last["latents"].float().cpu().numpy())
    ms_step = ms_total / args.steps
    value = B * n_gpus / (ms_step / 1e3)

    ms_e2e_total, _ = timed(one_step_e2e, args.steps, 1)
    e2e_value = B * n_gpus / (ms_e2e_total / args.steps / 1e3)

    # ---- BASELINE configs[4] (SURVEY 8d config 5), every rank: 32 prompts/GPU -> 250-step sampling ->
    #      VAE decode -> 24 views at 256x256 -> uint8 frames -> NCCL all-gather of the frames (151 MB/rank)
    c5 = None
    try:
        P5, V5, R5 = 32, 24, 256
        dec = build_ae_decoder("DiT2-L/2", device=dev)
        cams5 = orbit_cameras(V5).to(dev)
        g5 = torch.Generator().manual_seed(43)
        c5_all = {"crossattn": torch.randn(P5 * n_gpus, 77, 768, generator=g5)}
        uc5_all = {"crossattn": torch.zeros(P5 * n_gpus, 77, 768)}
        run5 = lambda steps: pipeline.generate_sharded(model, dec, c5_all, uc5_all, cams5, seed=41, num_steps=steps,
                                                       scale=CFG_SCALE, resolution=R5, batch=P5)
        run5(3)                                   # warm-up: workspaces, the 64-sample graph, NCCL buffers
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        o5 = run5(nsteps)
        e1.record()
        torch.cuda.synchronize()
        ms5 = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms5, op=dist.ReduceOp.MAX)
        ms5 = ms5.item()
        # stage split on this rank (un-overlapped, informational)
        lat5 = o5["latents"]
        e0.record()
        r5 = pipeline.decode_and_render(dec, lat5, cams5, R5)
        e1.record()
        torch.cuda.synchronize()
        ms5_render = e0.elapsed_time(e1)
        c5 = {"rendered_views_per_s": P5 * n_gpus * V5 / (ms5 / 1e3), "latents_per_s": P5 * n_gpus / (ms5 / 1e3),
              "ms": ms5, "prompts_per_gpu": P5, "views_per_prompt": V5, "res": R5, "denoise_steps": nsteps,
              "samples_per_forward": 2 * P5, "decode_render_ms_per_gpu": ms5_render,
              "gather": "all_gather_into_tensor of uint8 HWC frames on a side stream" if world > 1 else "none (1 GPU)",
              "gather_bytes_per_rank": o5["gather_bytes_per_rank"],
              "frames_shape": list(o5["frames_all"].shape), "frames_checksum": int(o5["frames_all"][::7, ::5].sum().item()),
              "what": "BASELINE configs[4] / SURVEY 8d config 5 through pipeline.generate_sharded: global CPU noise "
                      "draw sliced per rank -> sample_t23d -> decode_and_render -> frame sink -> NCCL all-gather"}
        del o5, r5, lat5, dec
        torch.cuda.empty_cache()
    except Exception as e:  # noqa
        c5 = {"error": repr(e)}
        if world > 1:
            raise

    line = None
    if rank == 0:
        # ---- roofline of the dominant kernel (tcgen05 GEMM): instrumented pass over one forward,
        # CUDA events around every GEMM launch on the launching stream.
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks = json.load(f)
        except Exception:
            pass
        peak_tf = peaks.get("bf16_tflops_sustained")
        peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)"
        if not peak_tf:
            peak_tf, peak_src = 1400.0, "fallback (B200_PROFILING.md sustained ~1.4 PFLOP/s)"
        ev, flops = [], []
        real_gemm = ops.gemm

        def gemm_probe(a, w, *a_, **kw):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = real_gemm(a, w, *a_, **kw)
            e1.record()
            ev.append((e0, e1))
            flops.append(2.0 * a.shape[0] * a.shape[1] * w.shape[0])
            return r

        x2 = torch.randn(2 * B, 12, 32, 32, device=dev)
        ctx2 = torch.cat([uc_d, ctx_d], 0)
        os.environ["LN3_CUDA_GRAPH"] = "0"      # eager launches so that every GEMM can be bracketed by events
        try:
            model(x2, tables["t_idx"][0], ctx2, in_scale=tables["c_in"][0])
            torch.cuda.synchronize()
            ops.gemm = gemm_probe
            model(x2, tables["t_idx"][1], ctx2, in_scale=tables["c_in"][1])
            torch.cuda.synchronize()
        finally:
            ops.gemm = real_gemm
            os.environ.pop("LN3_CUDA_GRAPH", None)
        big = [(f, e0.elapsed_time(e1)) for f, (e0, e1) in zip(flops, ev) if f > 1e10]
        gemm_ms = sum(t for _, t in big)
        gemm_fl = sum(f for f, _ in big)
        achieved = gemm_fl / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
        traffic, traffic_src = None, None
        try:   # dram bytes of the dominant launch from this round's `ncu --set full` capture (tools/summarize_ncu.py)
            with open(os.path.join(ROOT, "profiles", "r2_gemm_traffic.json")) as f:
                tj = json.load(f)
            traffic, traffic_src = tj["dram_bytes_per_launch"], tj["source"]
        except Exception:
            pass
        roofline = {"kernel": "ln3::gemm2_bf16_kernel (tcgen05 cta_group::2, 256x256x64 per CTA pair, fused epilogues)",
                    "bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                    "frac": achieved / peak_tf, "peak_source": peak_src,
                    "traffic": traffic, "traffic_source": traffic_src,
                    "launches_measured": len(big), "avg_launch_us": 1e3 * gemm_ms / max(len(big), 1),
                    "flops_per_launch_avg": gemm_fl / max(len(big), 1),
                    "note": "events add launch gaps; gemm share of the forward in profiles/"}
        model_tf = FLOPS_EXECUTED_PER_FORWARD_PER_SAMPLE * 2 * B * nsteps / (ms_step / 1e3) / 1e12
        model_tf_ref = FLOPS_PER_FORWARD_PER_SAMPLE * 2 * B * nsteps / (ms_step / 1e3) / 1e12

        # ---- second headline quantity: rendered views/sec of the fused ray-march kernel
        views = None
        try:
            gg = torch.Generator().manual_seed(4)
            n_obj, V = 4, 16
            planes = (5 * torch.randn(n_obj, 3, 32, 128, 128, generator=gg)).to(dev)
            osg = [torch.randn(64, 32, generator=gg), torch.randn(64, generator=gg) * 0.1,
                   torch.randn(4, 64, generator=gg), torch.randn(4, generator=gg) * 0.1]
            osg[3][0] += 2.0
            osg = tuple(t.to(dev) for t in osg)
            pcl = ops.planes_to_channels_last(planes)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

            def time_render(res, tf32, nv):
                cams = orbit_cameras(nv).repeat(n_obj, 1).to(dev)
                M = res * res
                nc = torch.rand(n_obj * nv, M, 64, device=dev)
                nf = torch.rand(n_obj * nv, M, 64, device=dev)
                o, d = ops.generate_rays(cams, res)
                for _ in range(2):
                    ops.render_views(pcl, o, d, nc, nf, osg, views_per_obj=nv, mlp_tf32=tf32)
                torch.cuda.synchronize()
                e0.record()
                for _ in range(3):
                    ops.render_views(pcl, o, d, nc, nf, osg, views_per_obj=nv, mlp_tf32=tf32)
                e1.record()
                torch.cuda.synchronize()
                return e0.elapsed_time(e1) / 3

            rms, rms32 = time_render(128, True, V), time_render(128, False, V)
            rms256 = time_render(256, True, 8)
            views = {"value": n_obj * V / (rms / 1e3), "unit": "views/s", "res": 128, "views": n_obj * V,
                     "samples_per_ray": "64+64", "ms": rms,
                     "mlp": "TF32 tensor-core OSG MLP (product default; pixels within 1e-4 rel-L2 of fp32)",
                     "exact_fp32_mlp_views_per_s": n_obj * V / (rms32 / 1e3),
                     "views_per_s_256": n_obj * 8 / (rms256 / 1e3),
                     "flops_per_s_T": 0.70e6 * 128 * 128 * n_obj * V / (rms / 1e3) / 1e12,
                     "data": "synthetic planes 5*randn, explicit noise (SURVEY.md 8d config 3 render-only)"}
        except Exception as e:  # noqa
            views = {"error": repr(e)}

        # ---- VAE decode (DiT2-L/2 + conv upsampler) throughput: latent -> channels-last tri-plane
        vae = None
        try:
            dec = build_ae_decoder("DiT2-L/2", device=dev)
            lat8 = torch.randn(B, 12, 32, 32, device=dev)
            for _ in range(2):
                dec.decode_to_channels_last(lat8, in_mul=0.96806)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                dec.decode_to_channels_last(lat8, in_mul=0.96806)
            e1.record()
            torch.cuda.synchronize()
            dms = e0.elapsed_time(e1) / 3
            vae = {"value": B / (dms / 1e3), "unit": "latents/s", "batch": B, "ms": dms,
                   "what": "latent (12,32,32) -> tri-plane (3,128,128,32): PatchEmbedTriplane + DiT2-L/2 + SD conv decoder"}
            # BASELINE configs[2]: 64 denoised latents -> decode -> 16 views each at 128x128, through the
            # public pipeline call (device RNG for the sampler noise), 8 latents per call
            cams16 = orbit_cameras(16).to(dev)
            lat64 = torch.randn(64, 12, 32, 32, device=dev)
            pipeline.decode_and_render(dec, lat64[:8], cams16, 128)
            torch.cuda.synchronize()
            e0.record()
            for i0 in range(0, 64, 8):
                pipeline.decode_and_render(dec, lat64[i0:i0 + 8], cams16, 128)
            e1.record()
            torch.cuda.synchronize()
            c2ms = e0.elapsed_time(e1)
            vae["configs2_decode_render"] = {"value": 64 * 16 / (c2ms / 1e3), "unit": "views/s", "latents": 64,
                                             "views_per_latent": 16, "res": 128, "ms": c2ms,
                                             "what": "VAE decode + fused ray march, 64 latents x 16 views (BASELINE configs[2])"}
            del dec
        except Exception as e:  # noqa
            vae = {"error": repr(e)}

        # ---- BASELINE configs[3] on this rank's shard: I23D flow matching, 50-point Euler ODE + CFG 4.0,
        #      DiT-PixArt-L/2 with DINO/CLIP tokens, 8 images per GPU (16 samples per forward)
        i23d = None
        try:
            from ln3diff_b200.transport import Sampler, create_transport
            from ln3diff_b200.utils import build_i23d
            mi = build_i23d("DiT-PixArt-L/2", device=dev)
            gi = torch.Generator(device=dev).manual_seed(7)
            zi = torch.randn(B, 12, 32, 32, device=dev, generator=gi)
            ci = {"vector": torch.randn(B, 768, device=dev, generator=gi),
                  "crossattn": torch.randn(B, 256, 2048, device=dev, generator=gi)}
            cti = {k: torch.cat([v, torch.zeros_like(v)]) for k, v in ci.items()}
            fn = Sampler(create_transport(snr_type="lognorm")).sample_ode(sampling_method="euler", num_steps=50)
            run = lambda: fn(torch.cat([zi, zi]), mi.forward_with_cfg, context=cti, cfg_scale=4.0)
            run()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run()
            e1.record()
            torch.cuda.synchronize()
            ims = e0.elapsed_time(e1)
            i23d = {"value": B / (ims / 1e3), "unit": "latents/s", "images_per_gpu": B, "ode_points": 50, "cfg_scale": 4.0,
                    "ms": ims, "what": "BASELINE configs[3] shard: DiT-PixArt-L/2 sample_ode('euler', 50) + forward_with_cfg "
                                       "(49 network evaluations of 16 samples), through the transport mirror "
                                       "(every forward replays the model's cached CUDA graph)"}
            del mi
        except Exception as e:  # noqa
            i23d = {"error": repr(e)}

        # ---- mesh-extraction lattice: 192^3 point queries (triplane_decode_grid) on one object
        grid = None
        try:
            gen = torch.Generator(device=dev).manual_seed(5)
            pl = torch.randn(1, 3, 128, 128, 32, device=dev, generator=gen)
            osg_w = (torch.randn(64, 32, device=dev, generator=gen), torch.zeros(64, device=dev),
                     torch.randn(4, 64, device=dev, generator=gen), torch.zeros(4, device=dev))
            for _ in range(2):
                ops.query_points(pl, osg_w, grid_size=192)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                ops.query_points(pl, osg_w, grid_size=192)
            e1.record()
            torch.cuda.synchronize()
            gms = e0.elapsed_time(e1) / 3
            grid = {"value": 192 ** 3 / (gms / 1e3) / 1e6, "unit": "Mpoints/s", "ms_per_192cubed_grid": gms,
                    "what": "tri-plane gather + OSG decoder on the 192^3 mesh-extraction lattice (one launch)"}
        except Exception as e:  # noqa
            grid = {"error": repr(e)}

        # ---- mesh export tail: device marching cubes on a 192^3 density lattice (SURVEY 8f-2)
        mc = None
        try:
            gx = torch.linspace(-1, 1, 192, device=dev)
            dens = 10.0 * (0.7 - torch.sqrt(gx[:, None, None] ** 2 + gx[None, :, None] ** 2 + gx[None, None, :] ** 2)).contiguous()
            for _ in range(2):
                mv, mf = ops.marching_cubes(dens, 0.0)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(5):
                mv, mf = ops.marching_cubes(dens, 0.0)
            e1.record()
            torch.cuda.synchronize()
            mms = e0.elapsed_time(e1) / 5
            mc = {"value": 192 ** 3 / (mms / 1e3) / 1e6, "unit": "Mcells/s", "ms_per_192cubed_grid": mms,
                  "vertices": int(mv.shape[0]), "faces": int(mf.shape[0]),
                  "what": "ln3_marching_cubes_count + _emit incl. the size read-back (mcubes.marching_cubes replacement)"}
        except Exception as e:  # noqa
            mc = {"error": repr(e)}

        # ---- conditioner towers (SURVEY 8f-1): CLIP-L text (T23D), OpenCLIP ViT-L/14 + DINOv2 ViT-L/14-reg (I23D), random init
        cond = None
        try:
            from ln3diff_b200.sgm.modules.encoders.modules import (FrozenCLIPEmbedder, FrozenDinov2ImageEmbedder,
                                                                   FrozenOpenCLIPImageEmbedder)

            def _time(fn, n=5):
                for _ in range(2):
                    fn()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(n):
                    fn()
                e1.record()
                torch.cuda.synchronize()
                return e0.elapsed_time(e1) / n
            ids = torch.randint(3, 49000, (8, 77), generator=torch.Generator().manual_seed(9))
            ids[:, 30:] = 49407
            te = FrozenCLIPEmbedder(device=dev, always_return_pooled=True, random_init=True)
            t_ms = _time(lambda: te(ids))
            del te
            img8 = torch.rand(8, 3, 224, 224, generator=torch.Generator().manual_seed(10)).to(dev) * 2 - 1
            ce = FrozenOpenCLIPImageEmbedder(device=dev, output_tokens=True, random_init=True)
            de = FrozenDinov2ImageEmbedder(device=dev, random_init=True)
            i_ms = _time(lambda: (ce(img8), de(img8)))
            del ce, de
            cond = {"clip_text_prompts_per_s": 8 / t_ms * 1e3, "i23d_images_per_s": 8 / i_ms * 1e3,
                    "ms_per_8_prompts": t_ms, "ms_per_8_images_clip_plus_dino": i_ms,
                    "what": "frozen conditioner towers on the tcgen05 GEMM / FMHA kernels, 8 prompts or images per call"}
        except Exception as e:  # noqa
            cond = {"error": repr(e)}

        cpu = None
        if n_gpus == 1:
            try:
                ref = CpuReference()
                ref.step(0)                        # cold pass (thread pool, page faults)
                v, dt = ref.step(0)
                cpu = {"value": v, "unit": "latents/s", "cores": ref.cores, "kind": "port",
                       "sample": f"{REF_SAMPLES[0][0]} ({dt:.1f} s); latents/s extrapolated linearly in steps x prompts"}
                del ref
            except Exception as e:  # noqa
                cpu = {"error": repr(e)}
        line = {"metric": "denoised-latents/sec", "value": value, "unit": "latents/s", "n_gpus": n_gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": workload_config(n_gpus),
                "e2e": {"value": e2e_value, "unit": "latents/s",
                        "h2d_bytes_per_step": randn_h.numel() * 4 + ctx_h.numel() * 4,
                        "d2h_bytes_per_step": out_h.numel() * 4},
                "gpu_launches": int(launches), "clocks": clk, "roofline": roofline,
                "ms_per_denoise_step": ms_step / nsteps,
                "model_tflops": model_tf, "model_tflops_reference_flop_count": model_tf_ref,
                "gpu_reference": gpu_ref,
                "vs_gpu_reference": (value / gpu_ref["value"]) if gpu_ref and "value" in gpu_ref else None,
                "config5_sharded_generation": c5,
                "rendered_views": views, "vae_decode": vae, "i23d_flow": i23d, "point_queries": grid, "marching_cubes": mc, "conditioners": cond,
                "cpu_baseline": cpu}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
