#!/usr/bin/env python
"""bench.py -- denoised frames/sec of the Hallo denoising hot path on B200 (contract: see the task prompt).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--size 64] [--frames 16]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A "step" is one denoising step of one 16-frame window at 512x512 (BASELINE.json configs[1]): UNet3D forward on
the CFG batch (2, 4, 16, 64, 64) + CFG combine + DDIM update, fp16 storage / fp32 accumulate, random-init weights,
synthetic inputs.  metric = 16 frames / (40 steps x time per step).  N > 1: the window is sharded over
(CFG half x frame group) ranks (strong scaling); the temporal K/V all-gather and the CFG exchange are inside the
timed region.  Timing: CUDA events around exactly K graph replays, barrier + synchronize on both sides, max over
ranks.  The per-step activation working set (several GB) is far larger than the 126 MB L2, so no explicit flush
is needed between steps.

--impl reference and the `cpu_baseline` object of the default run time the reference's algorithm on the host cores
through the oracle restatement (oracle/port.py, fp32, pinned to the unmodified reference at 1.7e-6): `cpu_baseline` is
ONE measured forward of the full 16-frame window; the reference arm times exactly K sample steps (see
run_reference_arm) -- both are measurements, nothing is extrapolated.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "denoised frames/sec at 512x512, 16-frame window, 40 DDIM steps"
UNIT = "frames/s"
N_DDIM = 40


def load_peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return dict(burst=p["bf16_tflops"], sustained=p["bf16_tflops_sustained"], hbm=p["hbm_gbs"], src="measured")
    except Exception:
        return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def dump_outputs(path: str, arrays: dict, limit: int) -> None:
    """Writes each tensor as float32 `path`/<name>.npy.  A tensor larger than its share of `limit` bytes is replaced by a
    fixed seeded sample of its flattened elements, so that runs with the same arguments stay comparable."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    n_max = (limit - 4096 * len(arrays)) // 4 // len(arrays)
    for name, t in arrays.items():
        a = t.detach().float().cpu()
        if a.numel() > n_max:
            a = a.reshape(-1)[torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:n_max].sort().values]
        np.save(os.path.join(path, name + ".npy"), a.numpy())


def plan_shard(rank: int, world: int, n_frames: int):
    from hallo_b200.dist import plan_shard as ps
    return ps(rank, world, n_frames)


# ------------------------------------------------------------------------------------------------ CPU reference arm
def _cpu_forward_seconds(size: int, f: int, reps: int = 1):
    """Wall time of ONE UNet3D forward of the CFG batch (2, 4, f, size, size) through the oracle port (fp32, all host
    threads, F.scaled_dot_product_attention like the reference's AttnProcessor2_0); returns the list of `reps` times."""
    from hallo_b200.spec import UNetConfig
    from hallo_b200.synth import synth_inputs, synth_state_dict
    from oracle import port
    port.USE_SDPA = True
    cfg = UNetConfig()
    if not hasattr(_cpu_forward_seconds, "sd"):
        _cpu_forward_seconds.sd = synth_state_dict(cfg, seed=0)
    inp = synth_inputs(cfg, size, size, f, seed=42)
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        port.unet_forward(_cpu_forward_seconds.sd, cfg, inp)
        out.append(time.perf_counter() - t0)
    return out


def run_cpu_baseline(size: int, frames: int):
    """`cpu_baseline` of the default run: ONE real forward of the full window (all `frames` frames of the CFG batch) of
    the reference's algorithm on the host cores -- a measurement, not an extrapolation (about 50 s on 16 cores, less on
    bigger hosts).  frames/s = frames / (40 steps x that forward)."""
    from hallo_b200.synth import host_threads
    cores = host_threads()
    torch.set_num_threads(cores)
    t = _cpu_forward_seconds(size, frames, 1)[0]
    return dict(value=frames / (N_DDIM * t), unit=UNIT, cores=cores, kind="port",
                sample=f"one measured UNet3D forward of the full CFG batch (2,4,{frames},{size},{size}) in fp32 via "
                       f"oracle/port.py: {t:.1f} s on {cores} threads; x{N_DDIM} steps per window (no extrapolation)",
                seconds_per_forward=t)


def run_reference_arm(size: int, frames: int, K: int, Wm: int):
    """`--impl reference`: the reference's algorithm on the host cores, W warm-up + exactly K timed steps.  A full-window
    forward costs ~50 s on 16 cores, so K of them would take a quarter of an hour; each timed step is therefore one
    forward of a BOUNDED sample of the same workload -- the same CFG batch, latent size, motion frames and weights with
    `fs` of the window's frames, fs chosen so that the whole run stays within a few minutes -- and
    value = fs / (40 x seconds per sample step).  ms_per_step is the MEASURED time of a sample step (so steps x ms_per_step
    is the real timed region).  The fixed per-forward cost (weight traffic, the 2 motion frames) is amortised over fewer
    frames in the sample, so this under-reports the CPU by ~15-20 %; one real full-window forward is timed as well when
    the step budget allows and reported next to it (`full_window`)."""
    from hallo_b200.synth import host_threads
    cores = host_threads()
    torch.set_num_threads(cores)
    n = K + Wm
    fs = min(frames, 4 if n <= 8 else (2 if n <= 30 else 1))
    _cpu_forward_seconds(size, fs, Wm) if Wm > 0 else None
    t0 = time.perf_counter()
    ts = _cpu_forward_seconds(size, fs, K)
    total = time.perf_counter() - t0
    t_step = total / K
    full = None
    if n <= 30 and fs < frames:
        tf = _cpu_forward_seconds(size, frames, 1)[0]
        full = {"seconds_per_forward": tf, "value": frames / (N_DDIM * tf), "frames": frames}
    return dict(value=fs / (N_DDIM * t_step), unit=UNIT, cores=cores, kind="port", ms_per_step=t_step * 1e3,
                sample_frames=fs, full_window=full, step_seconds=[round(x, 3) for x in ts],
                sample=f"each step = one UNet3D forward of the CFG batch (2,4,{fs},{size},{size}) (a {fs}-of-{frames}-frame "
                       f"sample of the window, same weights / latent size / motion frames) in fp32 via oracle/port.py on "
                       f"{cores} threads: {t_step:.2f} s per step measured over {K} steps")


# ------------------------------------------------------------------------------------------------ configs[4]: clip e2e
def run_clip(args, rank, world, dev, dt, config):
    """End-to-end frames/s of a clip: N sequential 16-frame windows with 2 motion frames handed from window to window,
    every component on the path (random-init SD-1.5 VAE, engine-backed ReferenceNet, conditioning encoders, the 40-step
    denoising loop, decode), host tensors in, host video out.  One untimed warm-up window (graph capture, cuDNN plans)."""
    import torch.distributed as dist
    from hallo_b200.animate.face_animate import FaceAnimatePipeline
    from hallo_b200.driver import ClipAnimator, process_audio_emb
    from hallo_b200.models.audio_proj import AudioProjModel
    from hallo_b200.models.face_locator import FaceLocator
    from hallo_b200.models.image_proj import ImageProjModel
    from hallo_b200.models.unet_2d_condition import UNet2DConditionModel
    from hallo_b200.models.unet_3d import UNet3DConditionModel
    from hallo_b200.models.vae import AutoencoderKL
    from hallo_b200.scheduler import DDIMScheduler
    from hallo_b200.spec import HALLO_UNET_KWARGS, SD15_UNET_CONFIG, UNetConfig
    from hallo_b200.synth import mask_levels, synth_audio_proj_state_dict
    cfg = UNetConfig()
    H = W = args.size * 8
    cl = args.frames
    torch.manual_seed(0)
    # parameters are created uninitialised on the device and filled from device-drawn random-init weights: nothing of the
    # 1.5 G + 0.86 G parameters is drawn or held on the host (8 ranks share one box)
    from hallo_b200.models.unet_3d import empty_weights
    from hallo_b200.spec import param_spec_2d
    from hallo_b200.synth import synth_state_dict_device
    with empty_weights(dev, dt):
        unet = UNet3DConditionModel.from_config(SD15_UNET_CONFIG, **HALLO_UNET_KWARGS)
        refnet = UNet2DConditionModel.from_config(SD15_UNET_CONFIG)
    unet.load_state_dict(synth_state_dict_device(cfg, dev, seed=0), strict=True)
    refnet.load_state_dict(synth_state_dict_device(cfg, dev, seed=1, spec=param_spec_2d(cfg)), strict=True)
    torch.cuda.empty_cache()
    vae = AutoencoderKL().to(memory_format=torch.channels_last)
    fl_ = FaceLocator(conditioning_embedding_channels=320)
    torch.nn.init.normal_(fl_.conv_out.weight, std=0.02)                      # de-zeroed so the branch is live
    ip = ImageProjModel(cross_attention_dim=768, clip_embeddings_dim=512, clip_extra_context_tokens=4)
    ap_ = AudioProjModel()
    ap_.load_state_dict(synth_audio_proj_state_dict(), strict=True)
    sched = DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="linear", clip_sample=False, steps_offset=1,
                          prediction_type="v_prediction", rescale_betas_zero_snr=True, timestep_spacing="trailing")
    pipe = FaceAnimatePipeline(vae=vae, reference_unet=refnet, denoising_unet=unet, face_locator=fl_, scheduler=sched,
                               image_proj=ip)
    pipe.to(device=dev, dtype=dt)
    ap_ = ap_.to(dev, dt)
    g = torch.Generator().manual_seed(42)
    n_win = args.windows
    audio = process_audio_emb(torch.randn((n_win + 1) * cl, 12, 768, generator=g))
    masks = [torch.rand(1, L, generator=g) for L in mask_levels(args.size, args.size)]
    kw = dict(source_image_pixels=torch.rand(3, H, W, generator=g) * 2 - 1, source_image_face_region=torch.rand(3, H, W, generator=g),
              source_image_face_emb=torch.randn(512, generator=g), source_image_full_mask=masks, source_image_face_mask=masks,
              source_image_lip_mask=masks, width=W, height=H, num_inference_steps=N_DDIM, guidance_scale=3.5)
    anim = ClipAnimator(pipe, ap_, clip_length=cl, n_motion_frames=cfg.n_motion_frames)
    anim(audio_emb=audio[:cl], **kw)                                          # warm-up window
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    video = anim(audio_emb=audio[cl:], **kw)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    dt_s = time.perf_counter() - t0
    if world > 1:
        tmax = torch.tensor([dt_s], device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dt_s = float(tmax)
    phases = {}
    for wt in anim.window_timings:
        for k, v in wt.items():
            phases[k] = phases.get(k, 0.0) + v / len(anim.window_timings)
    eng = unet.engine(args.size, args.size, cl, pipe._window_shard(cl))
    if rank == 0:
        line = {"metric": "end-to-end frames/sec, sliding 16-frame windows with 2 motion-frame overlap (BASELINE.json configs[4])",
                "value": video.shape[1] / dt_s, "unit": UNIT, "n_gpus": world, "windows": n_win, "frames": int(video.shape[1]),
                "seconds": dt_s, "higher_is_better": True, "dtype": args.dtype, "data": "synthetic",
                "config": {"workload": f"{n_win} windows x {cl} frames at {W}x{H}, {N_DDIM} DDIM steps, host in -> host out; "
                                       "a 30 s clip is 47 windows (750 frames padded to 752)", **config},
                "ms_per_window_by_phase": {k: round(v, 2) for k, v in phases.items()},
                "video_finite": bool(torch.isfinite(video).all())}
        print(json.dumps(line), flush=True)
    if world > 1:
        eng.graph = None
        torch.cuda.synchronize()
        if eng.arena is not None:
            eng.arena.close()
        dist.barrier()
        if eng.px and eng.arena is None:                 # NCCL work captured in the graph: see orderly_exit() in main()
            sys.stdout.flush()
            os._exit(0)
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ GPU arm
def kineto_report(eng, path, replays=3):
    """Warm, in-graph kernel durations (CUPTI activity records of `replays` graph replays): per kernel name the
    count / mean / total per step, how much of the step no kernel was running (launch gaps + dependency stalls), and
    -- in `path`.seq -- the kernels of one replay in launch order with their grids, next to the op sequence of one
    eager step (`path`.ops: one line per hallo_b200.ops call, same order) so that durations can be matched to shapes."""
    import tempfile
    from torch.profiler import ProfilerActivity, profile
    from hallo_b200 import ops
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(replays):
            eng.step()
        torch.cuda.synchronize()
    tmp = tempfile.mktemp(suffix=".json")
    prof.export_chrome_trace(tmp)
    trace = json.load(open(tmp))
    os.remove(tmp)
    ks = sorted(((e["ts"], e["ts"] + e["dur"], e["name"], e.get("args", {}).get("grid"))
                 for e in trace.get("traceEvents", []) if e.get("cat") == "kernel"), key=lambda t: t[0])
    if not ks:
        open(path, "w").write("no kernel records (CUPTI unavailable?)\n")
        return
    span = ks[-1][1] - ks[0][0]
    busy, gaps, cur_end = 0.0, [], ks[0][0]
    agg = {}
    shorten = lambda name: name.split("(")[0].replace("void hb::", "")[:70]
    for a, b, name, _ in ks:
        if a > cur_end:
            gaps.append(a - cur_end)
        busy += max(0.0, b - max(a, cur_end))
        cur_end = max(cur_end, b)
        c = agg.setdefault(shorten(name), [0, 0.0])
        c[0] += 1
        c[1] += b - a
    with open(path, "w") as f:
        f.write(f"{replays} graph replays: span {span / replays / 1e3:.3f} ms/step, kernels busy {busy / replays / 1e3:.3f} ms/step, "
                f"idle {(span - busy) / replays / 1e3:.3f} ms/step in {len(gaps) // replays} gaps "
                f"(median gap {sorted(gaps)[len(gaps) // 2] if gaps else 0:.2f} us), {len(ks) // replays} kernels/step\n")
        for name, (n, t) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
            f.write(f"  {t / replays / 1e3:8.3f} ms/step  x{n // replays:4d}  {t / n:8.2f} us each  {name}\n")
    per = len(ks) // replays
    with open(path + ".seq", "w") as f:
        for a, b, name, grid in ks[per:2 * per]:
            f.write(f"{b - a:9.2f} us  grid {grid}  {shorten(name)}\n")
    # the same step, eager, to list the ops in launch order (their event timings are not used)
    ops.PROFILE = []
    g, eng.graph = eng.graph, None
    eng.step()
    torch.cuda.synchronize()
    names = [name for name, _, _ in ops.PROFILE]
    ops.PROFILE = None
    eng.graph = g
    open(path + ".ops", "w").write("\n".join(names) + "\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--size", type=int, default=64, help="latent side (64 = 512x512)")
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--dtype", default="f16", choices=["f16", "bf16"], help="storage / tensor-core input type (configs[3]: bf16)")
    ap.add_argument("--windows", type=int, default=0, metavar="N",
                    help="BASELINE.json configs[4]: end-to-end frames/s of N sliding 16-frame windows through the whole "
                         "pipeline (VAE, ReferenceNet, conditioning, denoising, decode, motion-frame hand-off), host to host")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--profiler-range", action="store_true",
                    help="wrap ONE eager denoising step in cudaProfilerStart/Stop and exit (for `ncu --profile-from-start off`: "
                         "the launch list then holds exactly the step's kernels, not the set-up's)")
    ap.add_argument("--profile-ops", action="store_true", help="print a per-op time table of one eager forward")
    ap.add_argument("--kineto", default="", metavar="FILE",
                    help="after the timed run, trace 3 graph replays with torch.profiler (CUPTI) and write the per-kernel "
                         "in-graph durations and the idle gaps between kernels to FILE (diagnostic, not a bench value)")
    ap.add_argument("--emulate-shard", type=int, default=0, metavar="R",
                    help="single GPU: run the workload of ONE rank of an R-rank job (cond half, first frame group, no "
                         "collectives) -- for ncu / op profiles of the sharded shapes; the JSON line is marked invalid")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write the latents the last timed step returned (float32, [1, 4, frames, "
                         "size, size]) to DIR/latents.npy, or each rank's frames to DIR/latents_rank<r>.npy; weights and "
                         "inputs are seeded, so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.windows > 0 or args.profiler_range):
        ap.error("--dump-outputs writes the outputs of the timed denoising steps of the GPU run")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    K, Wm = args.steps, max(args.warmup, 0)
    which = {64: "configs[1]", 96: "configs[3]"}.get(args.size, "non-standard size")
    config = {"workload": f"{args.size * 8}x{args.size * 8}, {args.frames}-frame window, CFG batch 2, "
                          f"{N_DDIM}-step DDIM ({which})", "latent": [2, 4, args.frames, args.size, args.size],
              "parallelism": f"frame-shard (both CFG halves per rank) over {world} rank(s)",
              "l2": "per-step working set >> 126 MB L2, no explicit flush"}

    if args.impl == "reference":
        if rank != 0:
            return
        r = run_reference_arm(args.size, args.frames, K, Wm)
        line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
                "steps": K, "warmup": Wm, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "sample_frames", "full_window")},
                "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (hallo_b200 has no CPU path); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from hallo_b200 import lib, ops
    from hallo_b200.engine import DenoiseEngine, PackedWeights
    from hallo_b200.flops import spatial_attention_flops, unet_forward_flops
    from hallo_b200.scheduler import DDIMScheduler
    from hallo_b200.spec import UNetConfig
    from hallo_b200.synth import synth_inputs, synth_state_dict_device

    peaks = load_peaks()
    cfg = UNetConfig()
    dt = torch.float16 if args.dtype == "f16" else torch.bfloat16
    if args.windows > 0:
        return run_clip(args, rank, world, dev, dt, config)
    from hallo_b200.synth import host_threads
    torch.set_num_threads(max(1, host_threads() // world))
    try:
        sd = synth_state_dict_device(cfg, dev, seed=0)   # random-init weights, drawn on the GPU (identical on every rank)
    except Exception as e:                               # set-up only: same distributions from the host streams
        print(f"# rank {rank}: on-device weight synthesis failed ({type(e).__name__}: {e}); drawing on the host", file=sys.stderr)
        from hallo_b200.synth import synth_state_dict
        sd = synth_state_dict(cfg, seed=0)
    W = PackedWeights(sd, cfg, dev, dt)
    del sd
    inp = synth_inputs(cfg, args.size, args.size, args.frames, seed=42)
    shard = plan_shard(rank, world, args.frames)
    if args.emulate_shard > 1 and world == 1:
        from hallo_b200.dist import shard_layout
        from hallo_b200.engine import Shard
        halves, frames_ = shard_layout(args.emulate_shard, args.frames)[0]
        shard = Shard(halves=halves, frames=frames_, emulate_group=args.emulate_shard)
        config["emulated_rank_of"] = args.emulate_shard
    eng = DenoiseEngine(W, args.size, args.size, args.frames, shard)
    # record the kernel-selection switches this line was measured with (defaults = the kernels that won their hardware A/B runs)
    try:
        config["switches"] = {n: lib.get_option(n) for n in ("gemm_tepi", "gemm_1cta", "gemm_fill", "attn_occ2", "attn_poly",
                                                              "attn_v1", "xattn_tc", "tattn_mma", "gn_fused")}
    except Exception:
        pass
    if world > 1:
        config["temporal_exchange"] = ("frame<->pixel swap around each motion module, fused into the producing kernels' "
                                       "stores over peer memory + flag barriers" if shard.exchange == "peer"
                                       else "frame<->pixel swap around each motion module, NCCL all_to_all_single")
    sch = DDIMScheduler()
    sch.set_timesteps(N_DDIM)

    # host-side (pinned) copies of everything a window needs: the e2e leg pays their H2D
    def pin(t):
        return t.to(dt if t.is_floating_point() and t.dtype != torch.float16 else t.dtype).contiguous().pin_memory()

    # a rank only needs its own frames of the per-frame tensors: slice on the host, so the e2e leg's H2D is the shard's
    fr = list(shard.frames)
    rows = [b * args.frames + g for b in (0, 1) for g in fr]
    host = dict(encoder_hidden_states=pin(inp["encoder_hidden_states"]), audio_embedding=pin(inp["audio_embedding"][:, fr]),
                mask_cond_fea=pin(inp["mask_cond_fea"][:, :, fr]), full_mask=[pin(m[rows]) for m in inp["full_mask"]],
                face_mask=[pin(m[rows]) for m in inp["face_mask"]], lip_mask=[pin(m[rows]) for m in inp["lip_mask"]])
    # the K/V banks are NOT a host input: in the pipeline the ReferenceNet produces them on the device once per window
    # (hallo_b200/refnet.py -> reader.update); they are resident before the timed region, like the weights
    banks_dev = {k: v.to(dev) for k, v in inp["banks"].items()}
    lat_host = inp["sample"][:1, :, list(shard.frames)].float().contiguous().pin_memory()
    lat_back = torch.empty_like(lat_host).pin_memory()

    def window_bytes():
        n = sum(t.numel() * t.element_size() for t in [host["encoder_hidden_states"], host["audio_embedding"], host["mask_cond_fea"]])
        n += sum(t.numel() * t.element_size() for k in ("full_mask", "face_mask", "lip_mask") for t in host[k])
        return n

    def begin_window_from_host():
        d = {k: (v.to(dev, non_blocking=True) if torch.is_tensor(v) else
                 ([t.to(dev, non_blocking=True) for t in v] if isinstance(v, list) else
                  {kk: t.to(dev, non_blocking=True) for kk, t in v.items()})) for k, v in host.items()}
        eng.begin_window(motion_scale=inp["motion_scale"], local_frames=True, banks=banks_dev, **d)

    begin_window_from_host()
    eng.set_schedule(sch.timesteps.tolist(), sch.coef_table(), 3.5)
    eng.latents.copy_(lat_host.to(dev))
    lib.launch_count(reset=True)
    if args.profiler_range:
        eng.step()                                   # warm-up (allocates every buffer)
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        eng.step()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        print(json.dumps({"profiler_range": "one eager denoising step", "launches": lib.launch_count(reset=True) // 2}))
        return
    if args.no_graph:
        eng.step()
        launches_per_step = lib.launch_count(reset=True)
    else:
        try:
            eng.capture()
            launches_per_step = lib.launch_count(reset=True) // 2  # capture() runs the step twice (warm-up + capture)
        except Exception as e:                                     # e.g. a collective that refuses stream capture
            print(f"# rank {rank}: CUDA-graph capture failed ({type(e).__name__}: {e}); stepping eagerly", file=sys.stderr)
            eng.graph = None
            torch.cuda.synchronize()
            lib.launch_count(reset=True)
            eng.step()
            launches_per_step = lib.launch_count(reset=True)
        config["cuda_graph"] = eng.graph is not None
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        import torch.distributed as dist
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    # ---------------- device-resident timing: value ----------------
    eng.latents.copy_(lat_host.to(dev))
    eng.step_idx.zero_()
    for _ in range(Wm):
        eng.step()
    barrier()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        eng.step()
    e1.record()
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"latents" if world == 1 else f"latents_rank{rank}": eng.latents}, (64 << 20) // world)
    ms_step = ms_total / K
    fps = args.frames / (N_DDIM * ms_step * 1e-3)

    # ---------------- end-to-end through host buffers: e2e ----------------
    # One window through the engine's public entry points with HOST inputs.  A window = one set-up (window tensors
    # H2D from pinned memory + the hoisted K/V projections, `begin_window`) followed by N_DDIM denoising steps, so the
    # set-up cost is charged at 1/N_DDIM per step whatever --steps is; every timed step additionally pays the H2D of
    # its latents from pinned memory and the D2H of the updated latents.
    barrier()
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    t2 = torch.cuda.Event(enable_timing=True)
    t0.record()
    begin_window_from_host()
    t1.record()
    eng.step_idx.zero_()
    for _ in range(K):
        eng.latents.copy_(lat_host, non_blocking=True)
        eng.step()
        lat_back.copy_(eng.latents, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        lat_host.copy_(lat_back)
    t2.record()
    barrier()
    setup_ms = max_over_ranks(t0.elapsed_time(t1))
    e2e_ms = setup_ms / N_DDIM + max_over_ranks(t1.elapsed_time(t2)) / K
    e2e_fps = args.frames / (N_DDIM * e2e_ms * 1e-3)
    h2d = lat_host.numel() * 4 + window_bytes() // N_DDIM
    d2h = lat_back.numel() * 4

    if args.kineto and rank == 0:
        kineto_report(eng, args.kineto)

    # ---------------- optional per-op table: one eager step on EVERY rank (the collectives need all of them) ----------------
    prof_saved = None
    if args.profile_ops:
        ops.PROFILE = []
        eng.graph_saved, eng.graph = eng.graph, None
        eng.step()
        torch.cuda.synchronize()
        prof_saved = [(name, a.elapsed_time(b_)) for name, a, b_ in ops.PROFILE]
        ops.PROFILE = None
        eng.graph = eng.graph_saved
        barrier()

    # ---------------- N > 1: the sharded run must reproduce the unsharded engine (collective; rank 0 holds the answer) ----
    shard_err = None
    if world > 1:
        from hallo_b200.dist import sharded_vs_unsharded
        try:
            shard_err = sharded_vs_unsharded(eng, inp, steps=2, use_graph=eng.graph is not None)
        except Exception as e:                               # never costs the bench line; the failure is reported in it
            shard_err = f"check failed: {type(e).__name__}: {e}"

    def orderly_exit():
        """Graphs first (a live graph holding NCCL work is what hung destroy_process_group in round 1), then the peer
        mappings, then the process group."""
        import torch.distributed as dist
        eng.graph = None
        torch.cuda.synchronize()
        if eng.arena is not None:
            eng.arena.close()
        dist.barrier()
        if eng.px and eng.arena is None:
            # NCCL exchange captured into the CUDA graph: destroy_process_group() still blocks for minutes after the graph
            # object is dropped (measured again in round 2: profiles/r2e_summary.txt, exit 124) -- leave hard, as round 1 did
            sys.stdout.flush()
            sys.stderr.flush()
            os._exit(0)
        dist.destroy_process_group()

    if rank != 0:
        if world > 1:
            orderly_exit()
        return

    # ---------------- roofline of the dominant kernel (fused spatial + reference-KV attention, L0) ----------------
    fl = unet_forward_flops(cfg, args.size, args.size, args.frames)
    L0, C0 = args.size * args.size, cfg.block_out_channels[0]
    Bl = eng.B
    qkv = torch.randn(Bl * L0, 3 * C0, device=dev, dtype=dt)
    kvr = torch.randn(2 * L0, 2 * C0, device=dev, dtype=dt)
    o = torch.empty(Bl * L0, C0, device=dev, dtype=dt)
    ridx = eng.window["ref_index"]
    n_cond = int((ridx >= 0).sum())
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ts = []
    for i in range(6):
        flush.zero_()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        ops.attention(qkv[:, :C0], qkv[:, C0:2 * C0], qkv[:, 2 * C0:], o, heads=cfg.heads, L=L0, kref=kvr[:, :C0],
                      vref=kvr[:, C0:], ref_index=ridx)
        a1.record()
        torch.cuda.synchronize()
        if i >= 2:
            ts.append(a0.elapsed_time(a1))
    attn_ms = sum(ts) / len(ts)
    attn_flops = spatial_attention_flops(L0, C0, n_cond, Bl - n_cond)
    achieved = attn_flops / (attn_ms * 1e-3) / 1e12
    traffic, traffic_src = None, None
    try:   # dram__bytes_read.sum + dram__bytes_write.sum of this kernel from the committed ncu --set full capture
        ns = [e for e in json.load(open(os.path.join(ROOT, "profiles", "r2_ncu_summaries.json"))) if e["name"] == "attn"][0]
        if args.size == 64 and Bl == 32 and args.dtype == "f16":
            traffic, traffic_src = ns["traffic_bytes"], "profiles/r2_ncu_summaries.json (ncu --set full, same kernel and shape)"
    except Exception:
        pass
    roofline = {"kernel": "attn2_tc_kernel<D=40> (spatial self-attention + in-kernel reference-KV concat, L0)",
                "bound": "tensor", "achieved": achieved, "peak": peaks["burst"], "unit": "TFLOP/s",
                "frac": achieved / peaks["burst"], "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": f"bf16 burst, {peaks['src']}",
                "ms_per_launch": attn_ms, "algorithmic_flops_per_launch": attn_flops,
                "whole_step": {"achieved": fl["total"] * world / world / (ms_step * 1e-3) / 1e12 / world,
                               "peak": peaks["sustained"], "frac": fl["total"] / (ms_step * 1e-3) / 1e12 / world / peaks["sustained"],
                               "unit": f"TFLOP/s per GPU ({fl['total'] / 1e12:.2f} TFLOP algorithmic per forward)"}}

    if prof_saved is not None:
        agg, byname = {}, {}
        for name, ms_ in prof_saved:
            kind = name.split(" ")[0]
            agg.setdefault(kind, [0.0, 0])
            agg[kind][0] += ms_
            agg[kind][1] += 1
            byname.setdefault(name, [0.0, 0])
            byname[name][0] += ms_
            byname[name][1] += 1
        tot = sum(v[0] for v in agg.values())
        print("# top shapes (eager, includes ~10 us launch gap each):", file=sys.stderr)
        for k, v in sorted(byname.items(), key=lambda kv: -kv[1][0])[:32]:
            print(f"#     {k:44s} {v[0]:8.3f} ms x{v[1]:3d}  {1e3 * v[0] / v[1]:8.1f} us each", file=sys.stderr)
        print(f"# per-op breakdown of one eager step on rank 0 ({tot:.2f} ms summed)", file=sys.stderr)
        for k, v in sorted(agg.items(), key=lambda kv: -kv[1][0]):
            print(f"#   {k:22s} {v[0]:9.3f} ms  {100 * v[0] / tot:5.1f} %  x{v[1]}", file=sys.stderr)

    # second roofline the north star asks for: the L0 3x3 conv of the ResNet blocks (implicit GEMM on tcgen05), timed
    # live like the attention kernel; informational (the graded `roofline` object stays the attention kernel)
    roofline_conv = None
    try:
        hh = args.size
        xc = torch.randn(Bl, hh, hh, C0, device=dev, dtype=dt)
        wc = torch.randn(C0, 9 * C0, device=dev, dtype=dt) * 0.01
        oc = torch.empty(Bl * hh * hh, C0, device=dev, dtype=dt)
        tc_ = []
        for i in range(6):
            flush.zero_()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            ops.conv3x3(xc, wc, oc)
            a1.record()
            torch.cuda.synchronize()
            if i >= 2:
                tc_.append(a0.elapsed_time(a1))
        conv_ms = sum(tc_) / len(tc_)
        conv_flops = 2.0 * Bl * hh * hh * 9 * C0 * C0
        conv_tf = conv_flops / (conv_ms * 1e-3) / 1e12
        roofline_conv = {"kernel": f"gemm_tc_kernel<CONV> 3x3 {C0}->{C0} at {hh}x{hh}, {Bl} frames", "bound": "tensor",
                         "achieved": conv_tf, "peak": peaks["burst"], "unit": "TFLOP/s", "frac": conv_tf / peaks["burst"],
                         "ms_per_launch": conv_ms, "algorithmic_flops_per_launch": conv_flops}
        del xc, wc, oc
    except Exception as e:                                   # informational only: never costs the bench line
        roofline_conv = {"error": f"{type(e).__name__}: {e}"}

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu = run_cpu_baseline(args.size, args.frames)
        cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}

    line = {"metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": args.dtype,
            "data": "synthetic", "config": config, "clocks": clk,
            "e2e": {"value": e2e_fps, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": e2e_ms, "window_setup_ms": setup_ms,
                    "note": "window set-up (H2D of the window's host inputs -- audio tokens, masks, face-locator feature, image tokens "
                            "-- + hoisted projections; the ReferenceNet banks are device-produced, not a host input) charged at "
                            "1/40 per step"},
            "gpu_launches": int(launches_per_step * K), "launches_per_step": int(launches_per_step),
            "roofline": roofline, "roofline_conv": roofline_conv, "cpu_baseline": cpu}
    if world > 1:
        line["sharded_vs_unsharded_rel_l2"] = shard_err
        line["sharded_vs_unsharded_note"] = ("final latents of 2 denoising steps, all ranks gathered, against the unsharded "
                                             "engine on rank 0 (same weights); run-to-run noise of one plan is ~1e-3")
    print(json.dumps(line), flush=True)
    if world > 1:
        orderly_exit()


if __name__ == "__main__":
    main()
