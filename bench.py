#!/usr/bin/env python
"""Benchmark of the hot path: 512x512 (64x64 latent), 50-step PLMS, grounded generation with classifier-free
guidance 7.5 -> images / second  (BASELINE.json `metric`; default workload = configs[1]: SD-1.4 box+text, batch 4 per
GPU, bf16).

    python bench.py --gpus 1 --steps 3 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --preset 3|4|5 ...          # the other BASELINE.json configs (text+image / inpaint / keypoint)
    python bench.py --global-batch 16 ...       # strong scaling: the global batch is fixed and sharded over the ranks
    python bench.py --sweep                     # every BASELINE config + the keypoint batch sweep, one JSON line each
    python bench.py --impl reference ...        # the reference's own PLMSSampler + UNetModel on the host cores
    python bench.py --dump-outputs DIR ...      # also write the last timed step's final latent(s) to DIR/*.npy
    python bench.py --per-op-json FILE ...      # also write the kernel pass's per-op times to FILE

One "step" = one full `PLMSSampler.sample(S=50)` of one batch = 102 UNet forwards per image (cond + uncond
x (50 + 1)); weights are seeded random of the SD-1.4 + GLIGEN architecture (no checkpoints offline), inputs
are synthetic CLIP/grounding embeddings (SURVEY 8d).  `value` times the loop with inputs already resident in
HBM; `e2e` times the same public call with inputs in pinned HOST memory and the final latent read back.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from functools import partial

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from gligen_b200 import synth  # noqa: E402
from gligen_b200.spec import NAMED_CONFIGS, flops_per_forward, synthetic_state_dict  # noqa: E402

UNIT = "images/s"
DUMP_BYTES = 64 * 10 ** 6          # --dump-outputs: bound on the arrays of all ranks together
# BASELINE.json configs[1..4] (configs[0] is the reference's CPU plumbing case: a parity test, not a bench line)
PRESETS = {
    2: dict(config="sd14_box_text", batch=4, alpha_type="1,0,0", what="box+text"),
    3: dict(config="sd14_box_text_image", batch=8, alpha_type="1,0,0", what="box+text+image"),
    4: dict(config="sd14_inpaint_box_text", batch=8, alpha_type="0.3,0,0.7", what="inpainting box+text"),      # 16 over 2 GPUs
    5: dict(config="sd14_keypoint", batch=4, alpha_type="1,0,0", what="keypoint"),
}


def parse(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--preset", type=int, default=0, choices=[0, 2, 3, 4, 5], help="BASELINE.json config number (1-based)")
    ap.add_argument("--config", default="sd14_box_text")
    ap.add_argument("--batch", type=int, default=4, help="images per GPU per step (weak scaling)")
    ap.add_argument("--global-batch", type=int, default=0, help="strong scaling: total images per step, sharded over the ranks")
    ap.add_argument("--max-objs", type=int, default=30)
    ap.add_argument("--plms-steps", type=int, default=50)
    ap.add_argument("--guidance", type=float, default=7.5)
    ap.add_argument("--alpha-type", default="1,0,0", help="scheduled sampling stages, e.g. 0.3,0,0.7 (gligen_inference default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernel-pass", action="store_true")
    ap.add_argument("--sweep", action="store_true", help="all BASELINE configs + keypoint batch sweep (1 GPU); one JSON line each")
    ap.add_argument("--ref-budget-s", type=float, default=200.0, help="reference arm: wall-clock budget that sizes its bounded sample")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the final latent of the last timed step as DIR/<name>.npy (float32)")
    ap.add_argument("--per-op-json", metavar="FILE", default=None,
                    help="write the kernel pass's per-op GPU times, flops and bytes to FILE (scripts/summarize_profiles.py reads them)")
    args = ap.parse_args(argv)
    if args.preset:
        pr = PRESETS[args.preset]
        given = argv if argv is not None else sys.argv
        args.config = pr["config"]
        if "--alpha-type" not in given:
            args.alpha_type = pr["alpha_type"]
        if "--batch" not in given:
            args.batch = pr["batch"]
    return args


def metric_name(cfg_name):
    what = {"sd14_box_text": "box+text", "sd14_box_text_image": "box+text+image", "sd14_inpaint_box_text": "inpainting box+text",
            "sd14_keypoint": "keypoint"}.get(cfg_name, cfg_name)
    return f"512x512 50-step PLMS {what} images/sec"


def algorithmic_flops_per_image(cfg, G, S, atype, use_cfg=True):
    """F_alg (SURVEY 8d): forwards with the fuser on count F(G), forwards at scale == 0 count F without the
    fuser; step 0 evaluates twice (improved Euler).  Unpadded 2*MAC only."""
    from gligen_b200.pipeline import alpha_generator
    alphas = alpha_generator(S, atype)
    per = 2 if use_cfg else 1
    f_on, f_off = flops_per_forward(cfg, G, True), flops_per_forward(cfg, G, False)
    total = 0.0
    for i, a in enumerate(alphas):
        n = per * (2 if i == 0 else 1)
        total += n * (f_on if a != 0 else f_off)
    return total


def workload_string(cfg_name, cfg, args, B, atype):
    G = cfg.tokens_per_sample(args.max_objs) if cfg.tokenizer != "keypoint" else cfg.max_persons * 17
    return (f"SD-1.4 GLIGEN {cfg_name}, 64x64 latent, PLMS {args.plms_steps} + CFG {args.guidance}, batch {B}/GPU, G={G}, alpha_type={atype}")


# ------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU with NVML every 100 ms while running."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz, self._stop = [], set(), None, threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:                                                  # pragma: no cover
            self.nv, self.err = None, str(e)
        self.th = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": "nvmlClocksEventReasonHwSlowdown", "hw_thermal_slowdown": "nvmlClocksEventReasonHwThermalSlowdown",
                 "sw_thermal_slowdown": "nvmlClocksEventReasonSwThermalSlowdown", "sw_power_cap": "nvmlClocksEventReasonSwPowerCap"}
        legacy = {"hw_slowdown": "nvmlClocksThrottleReasonHwSlowdown", "hw_thermal_slowdown": "nvmlClocksThrottleReasonHwThermalSlowdown",
                  "sw_thermal_slowdown": "nvmlClocksThrottleReasonSwThermalSlowdown", "sw_power_cap": "nvmlClocksThrottleReasonSwPowerCap"}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k in names:
                    bit = getattr(nv, names[k], None) or getattr(nv, legacy[k], 0)
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.1)

    def start(self):
        if self.nv is not None:
            self.th.start()

    def stop(self):
        self._stop.set()
        if self.nv is not None and self.th.is_alive():
            self.th.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# ------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's own CPU implementation of the path on the host cores
# ------------------------------------------------------------------------------------------------------
def _thread_candidates():
    """Thread counts worth trying for the CPU arm, ascending: 16, 32, the physical cores, all logical CPUs (torch's
    intra-op parallelism over 100+ hyper-threads is far slower than over a few dozen cores for these layer sizes:
    measured on the B200 host 49 s per forward at 128 threads against 5.4 s at 32)."""
    n = os.cpu_count() or 1
    cand = {n, min(32, n), min(16, n)}
    try:
        import psutil
        cand.add(psutil.cpu_count(logical=False) or n)
    except Exception:
        pass
    return sorted(cand)


class _Enough(Exception):
    pass


def run_reference(args):
    """`--impl reference`: the UNMODIFIED reference code (oracle/_ref archive, or /root/reference where it exists) -
    its PLMSSampler driving its UNetModel, fp32 on the host cores, all usable threads.  One "step" is ONE guided sampler
    evaluation (cond + uncond UNet forward of the batch) taken from inside a real `PLMSSampler.sample` call; the image
    rate follows from the 51 evaluations a 50-step image needs.  The bounded sample: the batch is the product arm's batch
    when `--steps + --warmup` evaluations of it fit `--ref-budget-s`, else the largest batch that does (CPU time is
    linear in the batch; the line says which).  Falls back to the oracle port (kind "port") when no reference is available."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    cfg = NAMED_CONFIGS[args.config]
    atype = [float(v) for v in args.alpha_type.split(",")]
    S = args.plms_steps
    n_eval = S + 1
    sd = synthetic_state_dict(cfg, seed=0)
    kind = "reference"
    try:
        from oracle import ref_harness as RH
        RH.mount()
    except Exception as e:                                                       # no archive on this box: oracle port
        kind, RH = "port", None
        print(f"[bench] reference archive unavailable ({e}); timing the oracle port", file=sys.stderr)

    # ---- thread-count calibration on one B=1 forward (smallest first; stop once clearly slower)
    inp1 = synth.make_inputs(cfg, 1, args.max_objs, seed=2)
    ts1 = torch.tensor([981])
    if kind == "reference":
        model = RH.ref_model(cfg)
        model.load_state_dict(sd, strict=True)
        one = lambda: RH.run_reference_forward(cfg, model, inp1, ts1, 1.0, True)
    else:
        from oracle import unet_oracle as UO
        model = None
        one = lambda: UO.unet_forward(cfg, sd, inp1["x"], ts1, inp1["context"], inp1["grounding_input"], 1.0,
                                      None if not cfg.inpaint_mode else torch.zeros(1, 5, cfg.image_size, cfg.image_size))

    def timed_one():
        t0 = time.perf_counter(); one(); return time.perf_counter() - t0

    cands = _thread_candidates()
    torch.set_num_threads(cands[0])
    timed_one()                                   # warm-up: page in the weights
    best_n, best_t = cands[0], None
    for n in cands:
        torch.set_num_threads(n)
        t = timed_one()
        if best_t is None or t < best_t:
            best_n, best_t = n, t
        elif t > 1.5 * best_t:
            break
    torch.set_num_threads(best_n)
    cores, t_fw1 = best_n, best_t

    # ---- bounded sample: K + W guided evaluations (2 forwards each) at batch b
    K, W = max(1, args.steps), max(0, args.warmup)
    b = args.batch
    while b > 1 and (K + W) * 2 * t_fw1 * b > args.ref_budget_s:
        b -= 1
    if kind == "reference":
        inp = synth.make_inputs(cfg, b, args.max_objs, seed=100)
        stamps = []
        orig_forward = model.forward

        def hooked(input):
            out = orig_forward(input)
            stamps.append(time.perf_counter())
            if len(stamps) >= 2 * (K + W) + 1:
                raise _Enough()
            return out

        model.forward = hooked
        stamps.append(time.perf_counter())
        import contextlib
        try:
            # the real sampler loop; enough PLMS steps that K + W evaluations happen, aborted by the hook afterwards
            with contextlib.redirect_stdout(sys.stderr):          # the reference prints; stdout carries only the JSON line
                S_ref = min(d for d in (2, 4, 5, 8, 10, 20, 25, 40, 50, 100, 125, 200, 250, 500, 1000) if d >= min(K + W, 1000))   # 1000 % S == 0 (util.py:58-60)
                RH.run_reference_sampler(cfg, sd, inp, "plms", S_ref, atype, args.guidance, "cpu", None, model=model, verbose=False)
        except _Enough:
            pass
        model.forward = orig_forward
        pair = [(stamps[2 * i + 2] - stamps[2 * i]) for i in range((len(stamps) - 1) // 2)]
        timed = pair[W:W + K] if len(pair) >= W + K else pair[-K:]
        t_pair = float(np.mean(timed))
        sample = (f"{len(timed)} guided evaluations (cond + uncond forward, fp32) of the reference UNetModel at batch {b}, taken inside a real "
                  f"reference PLMSSampler.sample call after {W} warm-up evaluations; x{n_eval} evaluations per {S}-step image")
    else:
        times = [timed_one() for _ in range(K)]
        b = 1
        t_pair = 2 * float(np.mean(times))
        sample = f"{K} timed B=1 fp32 UNet forwards of the oracle port (reference algorithm, torch CPU ops), x{2 * n_eval} forwards/image"
    value = b / (n_eval * t_pair)
    line = {"impl": "reference", "metric": metric_name(args.config), "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": K,
            "warmup": W, "ms_per_step": t_pair * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_string(args.config, cfg, args, args.batch, atype), "forwards_per_image": 2 * n_eval,
                       "reference_batch": b, "sample": sample},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    return line


def cpu_baseline_subprocess(args):
    """cpu_baseline of the product line: the reference arm on a small bounded sample, in a fresh process (this one has
    the drop-in `ldm` imported; the reference's own `ldm` must be mounted in a clean interpreter)."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "2", "--warmup", "1", "--ref-budget-s", "45",
           "--config", args.config, "--batch", str(args.batch), "--max-objs", str(args.max_objs), "--plms-steps", str(args.plms_steps),
           "--alpha-type", args.alpha_type, "--guidance", str(args.guidance)]
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    env["CUDA_VISIBLE_DEVICES"] = ""
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
        for ln in reversed(r.stdout.strip().splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)["cpu_baseline"]
        return {"error": (r.stderr or r.stdout)[-300:]}
    except Exception as e:                                                       # pragma: no cover
        return {"error": str(e)}


# ------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------
def kernel_pass(model, N, n_ctx, B, reps=4):
    """Per-op GPU time of ONE 2B-row forward: (kind -> [flops, bytes, ms, launches]).  Every op of the plan is captured
    `reps` times into its own CUDA graph and the replay is timed with CUDA events on the launching stream: a python-driven
    launch costs 6-13 us of host time, more than many of these kernels run, so event pairs around eager calls would
    measure the host (round 1 did; the per-op numbers of small kernels were inflated)."""
    eng = model.engine()
    ops = eng.ops
    P = eng._plan(2 * B, N, n_ctx)
    fuser_on = eng.scale != 0.0
    steps = [(n, fn) for n, fu, st, fn in P.steps if (fuser_on or not fu) and not st]
    ops.trace = []
    for name, fn in steps:                              # eager warm-up pass (also records the algorithmic work per op)
        fn()
    torch.cuda.synchronize()
    trace, ops.trace = ops.trace, None
    times = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for name, fn in steps:
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(reps):
                fn()
        g.replay()
        torch.cuda.synchronize()
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1) / reps)
        del g
    agg, per_op = {}, []
    for (name, _), (kind, fl, by), ms in zip(steps, trace, times):
        a = agg.setdefault(kind, [0.0, 0.0, 0.0, 0])
        a[0] += fl; a[1] += by; a[2] += ms; a[3] += 1
        per_op.append((name, kind, fl, by, ms))
    return agg, per_op


def run_ours(args, world, rank, local_rank, dev, quiet_extras=False):
    from ldm.models.diffusion.ldm import LatentDiffusion
    from ldm.models.diffusion.plms import PLMSSampler
    from gligen_b200.pipeline import alpha_generator, build_model, sampler_inputs, set_alpha_scale

    cfg = NAMED_CONFIGS[args.config]
    atype = [float(v) for v in args.alpha_type.split(",")]
    S = args.plms_steps
    strong = args.global_batch > 0
    if strong:
        from gligen_b200.dist import shard_range
        lo, hi = shard_range(args.global_batch, rank, world)
        B = hi - lo
    else:
        B = args.batch
    cfg, model = build_model(cfg, dev, load_weights=False)
    sd = None
    if rank == 0 or world == 1:
        sd = synthetic_state_dict(cfg, seed=0)
        model.load_state_dict(sd)
    t_bc = time.perf_counter()
    sent = model.broadcast_packed_weights(src=0)         # frozen weights: once, packed bf16 arena over NCCL / NVLink
    torch.cuda.synchronize()
    t_bc = time.perf_counter() - t_bc
    diffusion = LatentDiffusion(linear_start=0.00085, linear_end=0.012, timesteps=1000).to(dev)
    sampler = PLMSSampler(diffusion, model, alpha_generator_func=partial(alpha_generator, type=atype), set_alpha_scale=set_alpha_scale)
    if any(a == 0 for a in alpha_generator(S, atype)) and not cfg.inpaint_mode:
        os.chdir(os.path.join(ROOT, "tests", "golden"))       # SD_input_conv_weight_bias.pth is read CWD-relative

    # per-rank synthetic inputs, generated on the host
    Bh = max(B, 1)
    host = synth.make_inputs(cfg, Bh, args.max_objs, seed=100 + rank)
    pinned = {k: v.pin_memory() for k, v in host.items() if isinstance(v, torch.Tensor)}
    pinned_batch = {k: v.pin_memory() for k, v in host["batch"].items()}
    shape = (Bh, cfg.in_channels, cfg.image_size, cfg.image_size)
    h2d = sum(v.numel() * v.element_size() for v in list(pinned.values()) + list(pinned_batch.values()))
    d2h = Bh * cfg.in_channels * cfg.image_size ** 2 * 4
    resident = {k: v.to(dev) for k, v in pinned.items()}
    resident_batch = {k: v.to(dev) for k, v in pinned_batch.items()}
    out_host = torch.empty(shape, dtype=torch.float32).pin_memory()

    def one_image_batch(from_host: bool):
        if B == 0:
            return None
        if from_host:
            t = {k: v.to(dev, non_blocking=True) for k, v in pinned.items()}
            bt = {k: v.to(dev, non_blocking=True) for k, v in pinned_batch.items()}
        else:
            t, bt = resident, resident_batch
        input, mask, x0 = sampler_inputs(cfg, model, t, bt)
        lat = sampler.sample(S=S, shape=shape, input=input, uc=t["uc"], guidance_scale=args.guidance, mask=mask, x0=x0)
        if from_host:
            out_host.copy_(lat, non_blocking=True)
        return lat

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    last = [None]

    def timed(n, from_host):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            last[0] = one_image_batch(from_host)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    eng = model.engine()
    import contextlib
    _quiet = contextlib.redirect_stdout(sys.stderr)       # "First conv layer is not restorable ..." (inpaint) belongs on stderr here
    _quiet.__enter__()
    for _ in range(args.warmup):
        one_image_batch(False)
    # the inpainting sampler draws q_sample noise from the global generator: a fixed seed here makes the timed steps'
    # inputs identical from run to run, whatever the code before this point drew
    torch.manual_seed(1234)
    clocks = ClockSampler(local_rank)
    clocks.start()
    l0 = eng.kernel_launches
    ms = timed(args.steps, False)
    launches = eng.kernel_launches - l0 + (args.steps * (S + 1) if B else 0)          # + the fused sampler-update kernels
    clk = clocks.stop()
    final_latent = last[0].float().cpu() if last[0] is not None else None
    one_image_batch(True)
    ms_e2e = timed(args.steps, True)
    _quiet.__exit__(None, None, None)

    total_images = (args.global_batch if strong else world * B) * args.steps
    value = total_images / (ms / 1e3)
    e2e = total_images / (ms_e2e / 1e3)
    G = cfg.max_persons * 17 if cfg.tokenizer == "keypoint" else cfg.tokens_per_sample(args.max_objs)
    f_img = algorithmic_flops_per_image(cfg, G, S, atype)
    line = None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
        peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if peaks else "fallback 1.4 PFLOP/s sustained (of fallback)"
        roof = {"bound": "tensor", "unit": "TFLOP/s", "peak": peak_tf, "peak_source": peak_src, "traffic": None}
        kernel_shares = None
        if not args.no_kernel_pass and B > 0:
            set_alpha_scale(model, 1.0 if atype[0] > 0 else 0.0)
            model._sync_scales(eng)
            N = resident_batch["points"].shape[1] if cfg.tokenizer == "keypoint" else resident_batch["boxes"].shape[1]
            agg, per_op = kernel_pass(model, N, resident["uc"].shape[1], min(B, eng.MAX_ROWS // 2))       # one chunk's plan
            tot_ms = sum(a[2] for a in agg.values())
            tc = [agg.get(k, [0, 0, 0, 0]) for k in ("gemm", "conv3x3")]
            tc_fl, tc_ms, tc_n = tc[0][0] + tc[1][0], tc[0][2] + tc[1][2], tc[0][3] + tc[1][3]
            kernel_shares = {k: {"ms": round(a[2], 4), "share": round(a[2] / tot_ms, 4), "launches": a[3],
                                 "tflops": round(a[0] / (a[2] * 1e-3) / 1e12, 1) if a[0] and a[2] else None,
                                 "gbs": round(a[1] / (a[2] * 1e-3) / 1e9, 1) if a[1] and a[2] else None} for k, a in agg.items()}
            # dominant kernel = gemm_tc_kernel (linear + 1x1 + implicit 3x3 conv): algorithmic flops per launch
            # / average CUDA-event launch duration, both from this live pass
            roof.update({"kernel": "gemm_tc_kernel (tcgen05 GEMM + implicit-GEMM conv3x3)",
                         "achieved": tc_fl / (tc_ms * 1e-3) / 1e12, "frac": tc_fl / (tc_ms * 1e-3) / 1e12 / peak_tf,
                         "flops_per_launch": tc_fl / max(tc_n, 1), "avg_launch_ms": tc_ms / max(tc_n, 1), "launches_per_forward": tc_n,
                         "forward_ms_sum_of_ops": tot_ms, "op_timing": "each op replayed from its own CUDA graph (GPU time, no host issue time)"})
            if args.per_op_json and not quiet_extras:
                os.makedirs(os.path.dirname(args.per_op_json), exist_ok=True)
                with open(args.per_op_json, "w") as f:
                    json.dump([dict(name=n, kind=k, gflop=fl / 1e9, mbytes=by / 1e6, ms=m) for n, k, fl, by, m in per_op], f)
        for tname in ("r2_gemm_dram_traffic.json", "r1_gemm_dram_traffic.json"):
            tpath = os.path.join(ROOT, "profiles", tname)
            if os.path.exists(tpath):                  # measured with ncu (bench.py cannot run under a profiler itself)
                tr = json.load(open(tpath))
                roof["traffic"] = tr["dram_bytes_read_per_launch"] + tr["dram_bytes_write_per_launch"]
                roof["traffic_note"] = ("dram__bytes_read.sum + dram__bytes_write.sum per gemm_tc_kernel launch, mean of "
                                        f"{tr['launches']} launches (profiles/{tname}); algorithmic minimum "
                                        f"{tr['algorithmic_bytes_per_launch']:.3g} B/launch - L2 (126 MB) keeps producer->consumer activations off DRAM")
                break
        roof["whole_step_achieved"] = f_img * value / world / 1e12
        roof["whole_step_frac"] = roof["whole_step_achieved"] / peak_tf
        cpu = None
        if not args.no_cpu_baseline and world == 1 and not quiet_extras:          # reported at N = 1 only (rank 0's host cores)
            cpu = cpu_baseline_subprocess(args)
        line = {"metric": metric_name(args.config), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
                "dtype": "bf16", "data": "synthetic",
                "config": {"workload": workload_string(args.config, cfg, args, B if not strong else f"{args.global_batch} global / {world}", atype),
                           "forwards_per_image": 2 * (S + 1), "cfg_batching": "cond+uncond as one 2B pass",
                           "parallelism": f"dp{world} (sample sharding, no per-step collective)",
                           "l2": "working set (2.1 GB bf16 weights + activations) >> 126 MB L2; no explicit flush",
                           "weights_broadcast": {"bytes": sent, "seconds": round(t_bc, 3), "what": "packed bf16 arena + fp32 vectors"} if world > 1 else None,
                           "algorithmic_tflop_per_image": f_img / 1e12},
                "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / args.steps},
                "gpu_launches": int(launches), "clocks": clk, "roofline": roof, "cpu_baseline": cpu, "kernel_shares": kernel_shares}
    del sampler, model, eng
    torch.cuda.empty_cache()
    return line, final_latent


def dump_outputs(dirname, arrays, budget):
    """Write each tensor of `arrays` as dirname/<name>.npy in float32.  When they hold more than `budget` bytes in all,
    each is replaced by the same fraction of its elements, flattened, at indices drawn from a fixed seed."""
    os.makedirs(dirname, exist_ok=True)
    total = 4 * sum(t.numel() for t in arrays.values())
    for name, t in arrays.items():
        a = t.float().cpu().numpy()
        if total > budget:
            keep = a.size * budget // total
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(dirname, name + ".npy"), a)


def main():
    args = parse()
    if args.impl == "reference" and args.dump_outputs:
        raise SystemExit("--dump-outputs writes what the timed GPU path computed: it needs --impl ours")
    if args.impl == "reference":
        line = run_reference(args)
        if line is not None:
            print(json.dumps(line))
        return
    for k in ("dump_outputs", "per_op_json"):                        # run_ours changes the working directory
        if getattr(args, k):
            setattr(args, k, os.path.abspath(getattr(args, k)))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl=ours) needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)"
    cwd = os.getcwd()
    suffix = f"_rank{rank}" if world > 1 else ""
    outputs = {}
    if args.sweep:
        # every BASELINE.json config at its own batch + the keypoint batch sweep (config 5), short runs; one line each
        cases = [dict(preset=2), dict(preset=2, alpha_type="0.3,0,0.7"), dict(preset=3), dict(preset=4)]
        cases += [dict(preset=5, batch=b) for b in (1, 2, 4, 8, 16, 32, 64)]
        for i, c in enumerate(cases):
            a = parse(["--preset", str(c["preset"]), "--steps", str(args.steps), "--warmup", str(args.warmup), "--gpus", str(args.gpus)] +
                      (["--batch", str(c["batch"])] if "batch" in c else []) + (["--alpha-type", c["alpha_type"]] if "alpha_type" in c else []))
            if "batch" in c:
                a.batch = c["batch"]
            a.no_kernel_pass = args.no_kernel_pass
            os.chdir(cwd)
            line, lat = run_ours(a, world, rank, local_rank, dev, quiet_extras=True)
            if lat is not None:
                outputs[f"sweep{i:02d}_latent{suffix}"] = lat
            if line is not None:
                line["sweep"] = True
                print(json.dumps(line), flush=True)
    else:
        line, lat = run_ours(args, world, rank, local_rank, dev)
        if lat is not None:
            outputs["latent" + suffix] = lat
        if line is not None:
            print(json.dumps(line))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs, DUMP_BYTES // world)
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
