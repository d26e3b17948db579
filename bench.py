#!/usr/bin/env python
"""bench.py -- edits/s of the FreeFine hot path on B200 (BASELINE.json metric), one JSON line on rank 0.

    python bench.py --gpus N --steps K --warmup W            # our arm (N>1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's CPU path (oracle port)

Workload (`config.workload`): BASELINE.json configs[1] -- SD1.5 2-D geometric edits (move + rotate + scale) at 512x512,
50-step DDIM schedule, 8 edits per stream batch per GPU, synthetic images / masks / transforms (freefine_b200/synth.py),
random-init SD1.5-shaped stand-in UNet (diffusers and the checkpoint are not available: no network).  A "step" is one
batch of 8 whole edits: coarse warp+blend -> DDIM inversion (UNet x n_inv, 16 streams) -> TCA sampling with local CFG
and masked DDPM steps (UNet x n_samp, 32 streams) -> decode.  Default n_inv = n_samp = 50 (`--start-step 0`); the
reference's GeoBench-2D default skips the first 35 schedule steps (`--start-step 35`, 15+15 UNet calls).

`value`   : whole-job edits/s with the inputs already resident in HBM (CUDA-event timed, max over ranks).
`e2e`     : the same through FreeFinePipeline.FreeFine_generation_batch with HOST buffers (pinned uint8 images and
            masks in, uint8 images out), copies inside the timed region.
`roofline`: the dominant kernel (ff_attn_masked_kv on the S=4096, d=40 TCA layers): algorithmic FLOPs per launch
            (freefine_b200.plans.algorithmic_flops) / mean launch duration from CUDA-event pairs recorded around every
            launch inside the timed region, against the measured bf16 peak of MEASURED_PEAKS.json.
`cpu_baseline`: the CPU restatement of the reference path (oracle/ff_pipeline_cpu.py, kind "port": the reference is
            Python that needs diffusers and cannot travel to the GPU box) timed on the host cores on a bounded sample
            (one inversion UNet step + one sampling UNet step of one 512x512 edit), extrapolated to a whole edit.
`rooflines`: (N=1) every kernel alone after the timed region -- HBM-bound kernels on L2-exceeding batches, one attention
            launch per SD1.5 layer shape (freefine_b200/roofline.py) -- so that the fractions of DESIGN.md are driver-run.
`gpu_active_frac`: sum of kernel durations / wall span of one step (CUPTI through torch.profiler).
`parity`  : (N=1) final-latent relative L2 of golden whole edits (tests/golden, made by the UNMODIFIED reference) run in
            this process on the UNet path that was timed, and on the fp32 UNet body.
`secondary`: (N=1) short measurements of the GeoBench-2D default schedule (start_step 35), of 768^2 / start_step 15
            (BASELINE.json configs[4] shape) and of the fp32 UNet body (`--unet-dtype fp32` arm), same code path.
`gpu_launches`: launches of OUR kernels inside the timed region (per C-ABI entry in `gpu_launches_by_entry`);
            `library_gemm_launches_by_entry` lists apart the entries that launch library code (ff_linear_bias_residual = one
            cuBLASLt GEMM with bias epilogue + beta*C).  `config.cudnn_benchmark`: torch.backends.cudnn.benchmark is on by
            default (fixed convolution shapes, tuned inside the warm-up steps; `--no-cudnn-benchmark` for the A/B).
`--sweep M`: BASELINE.json configs[2]: M edits sharded i mod W (DistributedSampler order, tail padding included), batches of
            `--edits`, final latents gathered over NCCL inside the timed region; strong scaling, reported as `sweep`.
`--dump-outputs DIR`: the images the last timed batch returned, DIR/images.npy (float32); the inputs depend only on the
            arguments (seeded synthetic edits, seeded stand-in weights), so two builds compare output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "edits/s @512^2 50-step SD1.5 (FreeFine 2-D geometric edit)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--edits", type=int, default=8, help="edits per stream batch per GPU")
    ap.add_argument("--res", type=int, default=512)
    ap.add_argument("--num-step", type=int, default=50)
    ap.add_argument("--start-step", type=int, default=0)
    ap.add_argument("--preset", default="sd15")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--channels-last", action="store_true", help="run the (library) UNet body in channels_last")
    ap.add_argument("--no-cudnn-benchmark", dest="cudnn_benchmark", action="store_false",
                    help="A/B: leave torch.backends.cudnn.benchmark off (default on: the convolution shapes are fixed, the "
                         "auto-tuner runs inside the warm-up steps; measured +1.8 %% on the full schedule)")
    ap.add_argument("--cudnn-benchmark", dest="cudnn_benchmark", action="store_true", help=argparse.SUPPRESS)
    ap.set_defaults(cudnn_benchmark=True)
    ap.add_argument("--plain-unet", action="store_true",
                    help="A/B only: eager NCHW UNet body instead of the channels-last fast path (csrc/unet_glue.cu)")
    ap.add_argument("--unet-dtype", default="bf16", choices=["bf16", "fp32"],
                    help="fp32: UNet body in fp32 (TF32 off) -- the arm whose whole-edit parity meets the 1e-2 north-star")
    ap.add_argument("--sweep", type=int, default=0, help="config 3: that many edits sharded over the ranks + final gather")
    ap.add_argument("--no-extras", action="store_true", help="skip rooflines / parity / secondary measurements")
    ap.add_argument("--active-frac-steps", type=int, default=4,
                    help="schedule steps of the batch run under CUPTI for gpu_active_frac (4 = quick default; the batch "
                         "boundaries weigh 12x more there than in the full 50-step schedule -- pass 50 for the real figure)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the edited images of the last timed batch to DIR/images.npy "
                         "(float32, [edits,H,W,3], 0..255; a fixed seeded sample of the pixels beyond 64 MB) so that two "
                         "builds can be compared output for output on identical inputs")
    args = ap.parse_args()
    if args.dump_outputs and args.sweep:
        ap.error("--dump-outputs applies to the batch benchmark, not to --sweep")
    return args


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, name, arr):
    """arr -> out_dir/<name>.npy as float32; above DUMP_BYTES a seeded sample of the flattened values (the same
    elements for the same shape, so runs with the same arguments stay comparable)."""
    import numpy as np
    a = np.asarray(arr, dtype=np.float32)
    cap = DUMP_BYTES // a.itemsize
    if a.size > cap:
        idx = np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))
        a = a.reshape(-1)[idx]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), a)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1392.3), d.get("bf16_tflops", 1639.8), "measured (MEASURED_PEAKS.json)"
    return 1400.0, 1590.0, "fallback (B200_PROFILING.md)"


# -------------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's algorithm restated on the CPU (oracle port), bounded sample
# -------------------------------------------------------------------------------------------------------------------
def cpu_sample(args, n_samples=1):
    """Times one inversion UNet step (2 streams) + one TCA sampling step (4 streams) of one edit on the host cores.
    Returns (edits_per_s, seconds_per_sample list, cores)."""
    import numpy as np
    import torch
    from freefine_b200 import coarse_edit, synth
    from freefine_b200.standin import build_standin
    from oracle.ff_pipeline_cpu import OraclePipeline
    from oracle import ff_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    cores = torch.get_num_threads()
    e = synth.make_edit(0, args.res)
    pipe = OraclePipeline(build_standin(args.preset))
    m = e["mask"]
    n_inv = n_samp = args.num_step - args.start_step
    times = []
    for _ in range(n_samples):
        t0 = time.perf_counter()
        # coarse edit as the reference does it (cv2 on the CPU: vis_utils.py:210-274), inside the timed sample
        coarse, tgt255, _ = O.re_edit_2d(e["image"], m, e["edit_param"], e["image"])
        inv = pipe.invert(coarse, e["image"], args.num_step, args.start_step, max_steps=1)
        t1 = time.perf_counter()
        inv_full = [inv[-1]] * (n_inv + 1)
        pipe.sample(inv_full, e["prompt"], tgt255, m, np.zeros_like(m), (args.res, args.res), args.num_step, args.start_step,
                    args.num_step, 7.5, 1.0, "tca", True, tgt255, True, 0.0, max_steps=1)
        t2 = time.perf_counter()
        times.append((t1 - t0, t2 - t1))
    t_inv = sum(t[0] for t in times) / len(times)
    t_samp = sum(t[1] for t in times) / len(times)
    return 1.0 / (n_inv * t_inv + n_samp * t_samp), times, cores, t_inv, t_samp


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = max(1, args.steps)
    warm = 1 if args.warmup > 0 else 0
    t0 = time.perf_counter()
    v, times, cores, t_inv, t_samp = cpu_sample(args, n_samples=warm + n)
    # drop the warm-up sample
    tt = times[warm:]
    t_inv = sum(t[0] for t in tt) / len(tt)
    t_samp = sum(t[1] for t in tt) / len(tt)
    n_calls = args.num_step - args.start_step
    v = 1.0 / (n_calls * (t_inv + t_samp))
    sample = (f"{warm} warm-up + {n} timed samples of [coarse edit (cv2) + 1 inversion UNet step (2 streams) + 1 TCA sampling step "
              f"(4 streams)] of one {args.res}x{args.res} edit, fp32, extrapolated x{n_calls} (t_inv={t_inv:.2f}s t_samp={t_samp:.2f}s); "
              "the port evaluates the 7-pass closed form of the TCA layer, cheaper than the 12 materialised-mask passes of the "
              "reference itself, so a GPU/CPU ratio taken against it is conservative")
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "edits/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * args.edits / v, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, reference=True),
            "cpu_baseline": {"value": v, "unit": "edits/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "edits/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.perf_counter() - t0}
    _emit(line)


def ncu_traffic(sq, skv, d, B):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from the committed `ncu --set full` capture
    (profiles/r2b_attn_ncu_summary.txt: the same launch shape, S=4096 d=40 32 streams, run alone by profiles/attn_case.py);
    {} when the dominant launch of this run has another shape or the summary is absent."""
    here = os.path.dirname(os.path.abspath(__file__))
    path = next((q for q in (os.path.join(here, "profiles", f) for f in ("r2b_attn_ncu_summary.txt", "r2_attn_ncu_summary.txt", "r1_attn_ncu_summary.txt"))
                 if os.path.exists(q)), None)
    if (sq, skv, d, B) != (4096, 4096, 40, 32) or path is None:
        return {}
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    tot = 0.0
    for line in open(path):
        f = line.split()
        if len(f) >= 3 and f[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum") and f[2] in unit:
            tot += float(f[1]) * unit[f[2]]
    if tot <= 0:
        return {}
    return {"traffic": tot, "traffic_unit": "bytes per launch (DRAM read + write, ncu --set full)",
            "traffic_source": "profiles/" + os.path.basename(path) + " (static: one ncu --set full capture of the same launch shape)"}


def workload_config(args, reference=False):
    n = args.num_step - args.start_step
    fp32 = reference or getattr(args, "unet_dtype", "bf16") == "fp32"
    which = "configs[1]" if args.res == 512 else "configs[4] shape"
    if fp32:
        body = "plain PyTorch forward, fp32" + ("" if reference else ", TF32 off")
    elif getattr(args, "plain_unet", False):
        body = "eager NCHW (A/B)"
    else:
        body = "channels-last fast path: cuDNN/cuBLAS + fused GroupNorm/SiLU, bias+residual, GEGLU, LayerNorm kernels"
    return {"workload": f"{which}: SD1.5 2D geometric edit (move/rotate/scale) {args.res}x{args.res}, {args.num_step}-step "
                        f"schedule, batch {args.edits} per GPU",
            "resolution": args.res, "edits_per_step_per_gpu": args.edits, "num_step": args.num_step,
            "start_step": args.start_step, "unet_calls_per_edit": f"{n} inversion (2 streams) + {n} sampling (4 streams)",
            "method": "tca", "guidance_scale": 7.5, "eta": 1.0, "use_auto_draw": True, "reduce_inp_artifacts": True,
            "network": f"random-init SD1.5-shaped stand-in UNet ({args.preset}), {'fp32' if fp32 else 'bf16'}",
            "unet_body": body,
            "cudnn_benchmark": bool(getattr(args, "cudnn_benchmark", True)),
            "l2": "working set per step (UNet weights 1.7 GB + activations) exceeds the 126 MB L2; no explicit flush",
            "parallelism": "independent edits, one model replica per GPU, no collective on the hot path"}


# -------------------------------------------------------------------------------------------------------------------
# clocks
# -------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.p = None

    def __enter__(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                       "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None
        return self

    def __exit__(self, *a):
        self.result = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        for ln in out.splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            sm.sort()
            self.result = {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# -------------------------------------------------------------------------------------------------------------------
# our arm
# -------------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from freefine_b200 import _lib, coarse_edit, ops, plans, synth
    from freefine_b200 import dist as ffdist
    from freefine_b200.pipeline import Attention_Modulator, FreeFinePipeline, register_attention_control
    from freefine_b200.standin import build_standin

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product has no CPU path; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()
    if args.cudnn_benchmark:
        torch.backends.cudnn.benchmark = True
    if args.plain_unet:
        import freefine_b200.standin as _standin
        _standin.FAST_PATH = False

    def set_tf32(on):
        torch.backends.cuda.matmul.allow_tf32 = on
        torch.backends.cudnn.allow_tf32 = on

    def make_pipe(dtype, preset=None):
        parts = build_standin(preset or args.preset, device=dev, dtype=dtype)
        if args.channels_last:
            parts.unet.to(memory_format=torch.channels_last)
        controller = Attention_Modulator(start_layer=10)
        pipe = FreeFinePipeline.from_parts(parts, controller, device=dev)
        register_attention_control(pipe, controller)
        pipe.modify_unet_forward()
        return pipe

    main_dtype = torch.float32 if args.unet_dtype == "fp32" else torch.bfloat16
    set_tf32(args.unet_dtype != "fp32")
    pipe = make_pipe(main_dtype)

    def settings(num_step, start_step):
        return dict(guidance_scale=7.5, eta=1.0, end_step=num_step, num_step=num_step, start_step=start_step,
                    method_type="tca", use_auto_draw=True, reduce_inp_artifacts=True, end_scale=0.0)

    def thetas_for(b, R):
        return torch.tensor(np.stack([coarse_edit.cv2_theta(coarse_edit.edit_matrix(b["masks"][i], b["edit_params"][i]), R, R)
                                      for i in range(len(b["edit_params"]))]), dtype=torch.float32)

    def host_batch(first, E, R):
        b = synth.make_batch(first, E, R)
        b["images_pin"] = torch.from_numpy(b["images"]).pin_memory()
        b["masks_pin"] = torch.from_numpy(b["masks"]).pin_memory()
        return b

    def to_dev(b, R):
        return dict(images=b["images_pin"].to(dev), masks=b["masks_pin"].to(dev), thetas=thetas_for(b, R).to(dev),
                    prompts=b["prompts"])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def run_device(p_, b_dev, kw):
        return p_.FreeFine_generation_batch(b_dev["images"], b_dev["masks"], None, b_dev["prompts"], thetas=b_dev["thetas"], **kw)

    def run_host(p_, b, kw):
        # the call a user makes: host buffers in, host images out; bounding boxes -> 2x3 matrices -> thetas are computed
        # inside (host work of the public API), H2D / D2H copies inside
        return p_.FreeFine_generation_batch(b["images_pin"], b["masks_pin"], b["edit_params"], b["prompts"], **kw)

    def timed_device(p_, E, R, kw, warmup, steps, first=0):
        """edits/s of this rank-set with device-resident inputs: `warmup` untimed + `steps` timed batches of E edits."""
        hb = [host_batch(first + ((s * world + rank) * E), E, R) for s in range(warmup + steps)]
        db = [to_dev(b, R) for b in hb]
        for s in range(warmup):
            run_device(p_, db[s], kw)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for s in range(warmup, warmup + steps):
            out = run_device(p_, db[s], kw)
        e1.record()
        barrier()
        t = max_over_ranks(e0.elapsed_time(e1) / 1e3)
        return world * E * steps / t, t, hb, db, out

    E, R = args.edits, args.res
    kw = settings(args.num_step, args.start_step)
    total_steps = args.warmup + args.steps

    # =========================================================================================================
    # config 3: M edits sharded i mod W, final latents gathered over NCCL inside the timed region (strong scaling)
    # =========================================================================================================
    if args.sweep > 0:
        M = args.sweep
        mine = ffdist.shard_indices(M, rank, world)                      # DistributedSampler order incl. the tail padding
        batches = [mine[i:i + E] for i in range(0, len(mine), E)]
        hb = []
        for ids in batches:                                              # synthetic inputs of MY edits, pinned host memory
            es = [synth.make_edit(i, R) for i in ids]
            hb.append(dict(images_pin=torch.from_numpy(np.stack([e["image"] for e in es])).pin_memory(),
                           masks_pin=torch.from_numpy(np.stack([e["mask"] for e in es])).pin_memory(),
                           edit_params=[e["edit_param"] for e in es], prompts=[e["prompt"] for e in es]))
        wb = host_batch(10 ** 6, E, R)
        for _ in range(max(args.warmup, 3)):                             # warm-up on edits outside the sweep
            run_host(pipe, wb, kw)
        barrier()
        ops.COUNTS.clear()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        with ClockSampler(local) as clk:
            e0.record()
            lat = []
            for b in hb:
                _, l = pipe.FreeFine_generation_batch(b["images_pin"], b["masks_pin"], b["edit_params"], b["prompts"],
                                                      return_latents=True, **kw)
                lat.append(l.view(len(b["prompts"]), 2, *l.shape[1:])[:, 0])     # the edit stream's final latents
            local_lat = torch.cat(lat).contiguous()
            gathered = ffdist.gather_results(local_lat, mine, M)              # ONE all-gather of [ceil(M/W),4,h,w] per rank
            checksum = float(gathered.double().abs().sum().item())           # D2H read of the gathered result
            e1.record()
            barrier()
        t = max_over_ranks(max(e0.elapsed_time(e1) / 1e3, time.perf_counter() - t0))
        if rank == 0:
            n_run = len(mine) * world
            line = {"metric": METRIC, "value": M / t, "unit": "edits/s", "n_gpus": world, "steps": len(batches), "warmup": max(args.warmup, 3),
                    "ms_per_step": 1e3 * t / max(len(batches), 1), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                    "dtype": args.unet_dtype, "data": "synthetic", "config": dict(workload_config(args),
                    workload=f"configs[2]: GeoBench-2d-shaped synthetic sweep of {M} independent {R}x{R} edits sharded i mod W over "
                             f"{world} GPU(s), batches of {E}, final latents gathered (all_gather_into_tensor) + read on the host"),
                    "clocks": clk.result, "gpu_launches": int(sum(v for k, v in ops.COUNTS.items() if k not in ops.LIBRARY_ENTRIES)),
                    "e2e": {"value": M / t, "unit": "edits/s", "h2d_bytes_per_step": int(hb[0]["images_pin"].nbytes + hb[0]["masks_pin"].nbytes),
                            "d2h_bytes_per_step": int(E * R * R * 3)},
                    "sweep": {"edits": M, "edits_run_incl_tail_padding": n_run, "gathered_shape": list(gathered.shape),
                              "gathered_abs_sum": checksum, "finite": bool(torch.isfinite(gathered).all().item()), "seconds": t}}
            _emit(line)
        if world > 1:
            dist.destroy_process_group()
        return

    # =========================================================================================================
    # A: inputs resident in HBM
    # =========================================================================================================
    host = [host_batch((s * world + rank) * E, E, R) for s in range(total_steps)]
    dev_batches = [to_dev(b, R) for b in host]
    for s in range(args.warmup):
        run_device(pipe, dev_batches[s], kw)
    barrier()
    ops.COUNTS.clear()
    prof = []
    ops.PROFILE = prof
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        ev0.record()
        for s in range(args.warmup, total_steps):
            out = run_device(pipe, dev_batches[s], kw)
        ev1.record()
        barrier()
    ops.PROFILE = None
    t_dev = max_over_ranks(ev0.elapsed_time(ev1) / 1e3)
    # hand-written kernels only: ff_linear_bias_residual is a cuBLASLt GEMM behind the C ABI (library code), listed apart
    counts = {k: v for k, v in ops.COUNTS.items() if k not in ops.LIBRARY_ENTRIES}
    library_counts = {k: v for k, v in ops.COUNTS.items() if k in ops.LIBRARY_ENTRIES}
    launches = int(sum(counts.values()))
    value = world * E * args.steps / t_dev
    finite = bool(torch.isfinite(out.float()).all().item())
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, "images" if world == 1 else f"images_rank{rank}", out.cpu().numpy())

    # ---- roofline of the dominant kernel + every attention shape of the step, from the event pairs of the timed region
    groups = {}
    for r in prof:
        ms = r["ev0"].elapsed_time(r["ev1"])
        key = (r["s_q"], r["s_kv"], r["d"], r["B"], id(r["plan"]))
        g = groups.setdefault(key, dict(ms=0.0, n=0, rec=r))
        g["ms"] += ms
        g["n"] += 1
    attn_ms_total = sum(g["ms"] for g in groups.values())
    by_shape = {}
    for key, g in groups.items():
        sh = key[:4]
        b = by_shape.setdefault(sh, dict(ms=0.0, n=0, flops=0.0))
        rec = g["rec"]
        plan = rec["plan"]
        pop = rec["popcount"].cpu().numpy() if rec["popcount"] is not None else None
        fl = plans.algorithmic_flops(plan, rec["s_q"], rec["s_kv"], rec["d"], pop) if plan is not None else 0.0
        b["ms"] += g["ms"]
        b["n"] += g["n"]
        b["flops"] += fl * g["n"]
    sustained, burst, peak_src = peaks()
    in_run = []
    for (sq, skv, d, B), dg in sorted(by_shape.items(), key=lambda kv: -kv[1]["ms"]):
        ach = dg["flops"] / (dg["ms"] / 1e3) / 1e12 if dg["ms"] > 0 else 0.0
        in_run.append({"kernel": "ff_attn_masked_kv", "size": f"S_q={sq} S_kv={skv} d={d} streams={B}", "launches": dg["n"],
                       "avg_launch_ms": dg["ms"] / max(dg["n"], 1), "achieved": ach, "unit": "TFLOP/s", "peak": sustained,
                       "frac": ach / sustained, "share_of_step": dg["ms"] / (t_dev * 1e3)})
    dom = max(by_shape.items(), key=lambda kv: kv[1]["ms"])
    (sq, skv, d, B), dg = dom
    achieved = dg["flops"] / (dg["ms"] / 1e3) / 1e12 if dg["ms"] > 0 else 0.0
    roofline = {"bound": "tensor", "kernel": f"ff_attn_masked_kv (S_q={sq}, S_kv={skv}, d={d}, streams={B})",
                "achieved": achieved, "peak": sustained, "unit": "TFLOP/s", "frac": achieved / sustained,
                "peak_source": peak_src + ", bf16_tflops_sustained (kernel timed inside a long step)",
                "frac_of_burst_peak": achieved / burst, "launches": dg["n"],
                "avg_launch_ms": dg["ms"] / max(dg["n"], 1),
                "algorithmic_gflop_per_launch": dg["flops"] / max(dg["n"], 1) / 1e9,
                "share_of_step": dg["ms"] / (t_dev * 1e3), "all_attention_share_of_step": attn_ms_total / (t_dev * 1e3),
                "traffic": None}
    roofline.update(ncu_traffic(sq, skv, d, B))

    # =========================================================================================================
    # B: end to end through the public API with host buffers
    # =========================================================================================================
    e2e = None
    if not args.no_e2e:
        run_host(pipe, host[0], kw)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for s in range(args.warmup, total_steps):
            o = run_host(pipe, host[s], kw)
        e1.record()
        barrier()
        t_host = max_over_ranks(max(e0.elapsed_time(e1) / 1e3, time.perf_counter() - t0))
        h2d = int(host[0]["images"].nbytes + host[0]["masks"].nbytes + E * 6 * 4)
        d2h = int(o.nbytes)
        e2e = {"value": world * E * args.steps / t_host, "unit": "edits/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "includes": "host-side bounding boxes -> 2x3 matrices -> thetas, H2D of images / masks / thetas, D2H of the uint8 results"}

    # =========================================================================================================
    # extras (N = 1 only): gpu_active_frac, per-kernel rooflines, parity, secondary configurations
    # =========================================================================================================
    extras = {}
    if world == 1 and not args.no_extras:
        from freefine_b200 import roofline as RF, selfcheck
        t_x = time.perf_counter()
        try:
            extras["gpu_active_frac"] = RF.gpu_active_frac(lambda: run_device(pipe, dev_batches[args.warmup], settings(args.num_step, max(args.start_step, args.num_step - args.active_frac_steps))))
            if extras["gpu_active_frac"]:
                n_af = args.num_step - max(args.start_step, args.num_step - args.active_frac_steps)
                extras["gpu_active_frac"]["step"] = (f"one batch with the last {n_af} schedule steps ({n_af} inversion + {n_af} sampling UNet "
                                                     f"calls) incl. the per-batch coarse edit / mask prep / VAE boundaries")
        except Exception as e:
            extras["gpu_active_frac"] = {"frac": None, "error": str(e)[:200]}
        del dev_batches[:]
        torch.cuda.empty_cache()
        hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", 6650.0) if os.path.exists(
            os.path.join(ROOT, "MEASURED_PEAKS.json")) else 6650.0
        try:
            extras["rooflines"] = RF.hbm_rooflines(dev, hbm_peak) + RF.attention_rooflines(dev, burst)
            extras["rooflines_note"] = ("each kernel alone after the timed region: HBM-bound kernels on L2-exceeding batches (CUDA-graph "
                                        "replays, 3 warm-ups, best of 5) vs the measured copy peak; attention per layer shape vs the "
                                        "BURST bf16 peak (kernel timed in isolation); in-run attention rows (`rooflines_in_run`) vs the sustained peak; the HBM "
                                        "denominator is the measured COPY bandwidth (1 read : 1 write), so a read-heavy kernel at the HBM limit "
                                        "(ff_geglu: 2 reads : 1 write) can show a fraction slightly above 1")
        except Exception as e:
            extras["rooflines"] = [{"error": str(e)[:300]}]
        # ---- parity of whole edits against the reference goldens, on the timed UNet path and on the fp32 body
        par = {"tolerance_north_star": 1e-2, "reference": "tests/golden/{pipeline,config1}.npz: latents of the UNMODIFIED reference (CPU fp32), "
               "tiny stand-in UNet with SD1.5 head dims", "cases": []}
        try:
            for dt_name, dt in (("fp32", torch.float32), ("bf16", torch.bfloat16)):
                set_tf32(False)
                for name in ("sched50_ss35", "sched50_full"):
                    tp = make_pipe(dt, "tiny")
                    r = selfcheck.run_golden_edit(tp, name)
                    par["cases"].append({"case": name, "unet_body": dt_name, "final_latent_rel_l2": r["final_rel_l2"],
                                         "inverted_latent_rel_l2": r["inverted_rel_l2"], "schedule_steps": r["n_latents"] - 1})
                tp = make_pipe(dt, "tiny")
                r = selfcheck.run_config1(tp)
                par["cases"].append({"case": "config1 (Examples/Editing/2D/bear, +60 px, 10-step, 512x512)", "unet_body": dt_name,
                                     "final_latent_rel_l2": r["final_rel_l2"], "inverted_latent_rel_l2": r["inverted_rel_l2"],
                                     "coarse_mask_bit_exact": r["coarse_mask_bit_exact"]})
            par["timed_path"] = args.unet_dtype
            par["note"] = ("the fp32 UNet body meets the 1e-2 north-star tolerance; the bf16 body (the default timed path) is a lower "
                           "network precision than the fp32 reference and does not (see DESIGN.md 2)")
        except Exception as e:
            par["error"] = str(e)[:300]
        extras["parity"] = par
        set_tf32(args.unet_dtype != "fp32")
        # ---- secondary configurations (short: 3 warm-ups + 2 timed batches each)
        sec = []
        try:
            v, t, *_ = timed_device(pipe, E, 512, settings(50, 35), 3, 2, first=5000)
            sec.append({"config": "configs[1] with the reference's GeoBench-2D default start_step=35 (15 + 15 UNet calls), 512x512, batch %d" % E,
                        "unet_body": args.unet_dtype, "value": v, "unit": "edits/s"})
            v, t, *_ = timed_device(pipe, 4, 768, settings(50, 15), 3, 2, first=6000)
            sec.append({"config": "configs[4] shape: 768x768 (96x96 latents, S=9216 self-attention), start_step=15 (35 + 35 UNet calls), batch 4",
                        "unet_body": args.unet_dtype, "value": v, "unit": "edits/s"})
            other = torch.float32 if args.unet_dtype == "bf16" else torch.bfloat16
            del pipe
            torch.cuda.empty_cache()
            set_tf32(other != torch.float32)
            p2 = make_pipe(other)
            v, t, *_ = timed_device(p2, E, 512, settings(50, 35), 3, 2, first=7000)
            sec.append({"config": "configs[1], start_step=35, 512x512, batch %d" % E, "unet_body": "fp32 (TF32 off)" if other == torch.float32 else "bf16",
                        "value": v, "unit": "edits/s"})
            del p2
        except Exception as e:
            sec.append({"error": str(e)[:300]})
        extras["secondary"] = sec
        extras["extras_wall_s"] = time.perf_counter() - t_x

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, times, cores, t_inv, t_samp = cpu_sample(args, n_samples=1)
        n = args.num_step - args.start_step
        cpu = {"value": v, "unit": "edits/s", "cores": cores, "kind": "port",
               "sample": f"coarse edit (cv2) + 1 inversion UNet step (2 streams, {t_inv:.1f}s) + 1 TCA sampling step (4 streams, {t_samp:.1f}s) of one "
                         f"{R}x{R} edit on the host cores (oracle/ff_pipeline_cpu.py, fp32), extrapolated x{n}; the port evaluates the "
                         "7-pass closed form of the TCA layer (the reference materialises 12 masked passes), so the ratio is conservative"}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "edits/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": 1e3 * t_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": args.unet_dtype, "data": "synthetic", "config": workload_config(args), "clocks": clk.result,
                "e2e": e2e, "gpu_launches": launches, "gpu_launches_by_entry": counts, "library_gemm_launches_by_entry": library_counts,
                "roofline": roofline,
                "rooflines_in_run": in_run, "cpu_baseline": cpu, "output_finite": finite}
        line.update(extras)
        _emit(line)
    if world > 1:
        dist.destroy_process_group()


_JSON_OUT = sys.stdout


def _emit(line: dict):
    """The ONE JSON line of the contract, on the process's original stdout."""
    _JSON_OUT.write(json.dumps(line) + "\n")
    _JSON_OUT.flush()


def main():
    global _JSON_OUT
    args = parse()
    # library chatter (e.g. the "NCCL version ..." banner some NCCL_DEBUG settings print on stdout) must not precede
    # the JSON line: file descriptor 1 is pointed at stderr for the whole run, the JSON goes to a dup of the real stdout
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
