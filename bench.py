#!/usr/bin/env python
"""bench.py — UNet sampler steps/s at 1024x1024 bs=1 (BASELINE.json metric), SDXL base, synthetic weights.

  python bench.py --gpus N --steps K --warmup W            our arm (libsdxl_b200.so, sm_100a kernels)
  python bench.py --impl reference --gpus N --steps K ...  CPU arm: the restated oracle on the host cores
  torchrun --nproc-per-node N bench.py --gpus N ...        one process per GPU, prompt-sharded replicas

  ... --workload image|refiner|inpaint                     whole images through sdxl_sample_latent (BASELINE configs 3, 4, 5)
  ... --dump-outputs DIR                                   also write the last timed step's result (rank 0) as DIR/latent.npy

A "step" = one iteration of the reference's sampler loop body (src/model/stablediffusion/mod.rs:406-429):
alpha lookups, forward_diffuser (conditional + unconditional UNet evaluation, CFG combine) and the DDIM
update — i.e. 2 UNet forwards at latent 128x128. Workload = BASELINE.json configs[1] (base, 1024x1024,
n=30 => 31 iterations per image, cfg 7.5, bs=1); with N>1 every rank runs its own image (configs[2]-style
prompt sharding, no in-step collective) and `value` is the whole-job steps/s.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "stable-diffusion-xl-burn_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "unet_sampler_steps_per_sec_1024x1024_bs1"
UNIT = "steps/s"
HW = 1024
N_STEPS = 30          # => 31 iterations (SURVEY D6)
GUIDANCE = 7.5
N_CTX = 77


def read_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            p = json.load(fh)
        return {"tflops": float(p["bf16_tflops_sustained"]), "tflops_burst": float(p["bf16_tflops"]), "hbm_gbs": float(p["hbm_gbs"]),
                "src": "measured (MEASURED_PEAKS.json: cuBLAS bf16 sustained, 1350 MHz under the 1 kW cap; burst = best of 10)"}
    except Exception:
        return {"tflops": 1400.0, "tflops_burst": 1590.0, "hbm_gbs": 6650.0, "src": "fallback (B200_PROFILING.md: ~1.4 PFLOP/s sustained, 1.59 burst)"}


def read_parity():
    """Final-latent parity of the CUDA path against the oracle at BASELINE's own configs (tests/test_fullsize_parity_gpu.py on a
    B200; committed copy of the test's output)."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_parity.json")) as fh:
            d = json.load(fh)
        c2 = d.get("config2_1024_31it_cfg7.5", {})
        return {"final_latent_rel": c2.get("rel_err"), "bound": 1e-3, "config": "SDXL base 1024x1024, 31 iterations, cfg 7.5 vs CPU f32 oracle (parity unpinned: the reference cannot be built)",
                "all": {k: v.get("rel_err") for k, v in d.items() if isinstance(v, dict) and "rel_err" in v}, "source": "profiles/r2_parity.json"}
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = max(mx, float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def dump_outputs(directory, **arrays):
    """`--dump-outputs`: what the timed path returned in its last step, one float32 .npy per array, so that two builds run with
    the same arguments (hence the same seeded inputs) can be compared output for output."""
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(directory, f"{name}.npy"), t.detach().float().cpu().numpy())


def make_conditioning(rank: int, device):
    """SURVEY 8(d) config 2/3: N(0,1) conditioning, seeds 10r+{1..4}."""
    import sdxl_b200
    g = lambda s: torch.Generator().manual_seed(10 * rank + s)  # noqa: E731
    return sdxl_b200.Conditioning(
        context_full=torch.randn(1, N_CTX, 2048, generator=g(1)).half(), unconditional_context_full=torch.randn(N_CTX, 2048, generator=g(2)).half(),
        channel_context=torch.randn(1, 2816, generator=g(3)).half(), unconditional_channel_context=torch.randn(2816, generator=g(4)).half(),
        resolution=(HW, HW))


# --------------------------------------------------------------------------------------------------
# CPU arm / cpu_baseline: the restated oracle (oracle/unet_oracle.py) on the host cores
# --------------------------------------------------------------------------------------------------
def host_cores() -> int:
    """Cores this process may actually use: min(os.cpu_count, affinity mask, cgroup v2 quota)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per))))
    except Exception:
        pass
    return n


def pick_threads() -> int:
    """Thread count that actually maximises f32 GEMM throughput on this host (containers often expose more
    logical CPUs than they may use; oversubscribing libtorch's pool is catastrophically slow)."""
    lim = host_cores()
    cands = sorted({c for c in (4, 8, 16, 32, 48, 64, 96, 128, lim) if c <= lim})
    a = torch.randn(1536, 1536)
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        a @ a
        t0 = time.perf_counter()
        for _ in range(3):
            a @ a
        dt = time.perf_counter() - t0
        if dt < best_t * 0.95:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def cpu_forward_seconds(weights_f32, latent_hw: int, reps: int, threads: int):
    from oracle import unet_oracle as O
    import sdxl_b200
    torch.set_num_threads(threads)
    cfg = sdxl_b200.SDXL_BASE
    x = torch.randn(1, 4, latent_hw, latent_hw, generator=torch.Generator().manual_seed(0))
    ctx = torch.randn(1, N_CTX, 2048, generator=torch.Generator().manual_seed(1)).half().float()
    y = torch.randn(1, 2816, generator=torch.Generator().manual_seed(3)).half().float()
    ts = []
    with torch.no_grad():
        for _ in range(reps):
            t0 = time.perf_counter()
            O.unet_forward(cfg, weights_f32, x, torch.tensor([999]), ctx, y)
            ts.append(time.perf_counter() - t0)
    return ts


def run_reference_arm(args, rank: int, world: int):
    """`--impl reference`: the reference's CPU path cannot be built here (Rust + un-vendored burn/tch crates, no cargo), so this arm
    times the line-by-line f32 restatement (kind "port") with all host threads: REAL 1024x1024 forwards (the conditional branch
    of a sampler step; a step is two of them), as many of the requested steps as fit a ~4 minute budget."""
    if rank != 0:
        return
    import sdxl_b200
    from oracle import unet_oracle as O
    cores = pick_threads()
    t0 = time.perf_counter()
    w = O.to_f32(sdxl_b200.synth_weights(sdxl_b200.SDXL_BASE, seed=0, device="cpu"))
    gen_s = time.perf_counter() - t0
    cal = cpu_forward_seconds(w, 32, 1, cores)[0]            # one 256x256 forward: calibration only
    est_full = cal * (6.7612 / 0.4278)
    budget = 230.0
    n_fit = int(budget / max(est_full, 1e-3))
    total_req = args.steps + args.warmup
    if n_fit >= 2:
        n_run = min(total_req, n_fit)
        n_warm = min(args.warmup, 1) if n_run > 1 else 0
        ts = cpu_forward_seconds(w, 128, n_run, cores)[n_warm:]
        fwd_s = statistics.mean(ts)
        sample = (f"{len(ts)} timed (+{n_warm} warm-up) conditional-branch UNet forwards at 1024x1024 (latent 128x128), f32, {cores} threads; "
                  f"one sampler step = 2 such forwards; {total_req} steps were requested, the rest are not run (bounded sample)")
        same = True
    else:   # even one real forward does not fit: scaled 256x256 forward, labelled as such
        ts = cpu_forward_seconds(w, 32, 3, cores)[1:]
        fwd_s = statistics.mean(ts) * (6.7612 / 0.4278)
        sample = "UNet forwards at 256x256 scaled by the algorithmic FLOP ratio 15.80 (a 1024x1024 forward does not fit the time budget on this host)"
        same = False
    ms_step = 2.0 * fwd_s * 1e3  # a sampler step = 2 forwards (the reference always runs both, mod.rs:523-541)
    value = 1e3 / ms_step
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "SDXL base UNet sampler step (cfg, 2 forwards), 1024x1024, bs=1, restated oracle on host cores (libtorch CPU kernels) — not the reference binary",
                   "weights": "synthetic N(0,1/fan_in), seed 0", "weight_gen_s": round(gen_s, 1), "measured_at_full_size": same,
                   "forward_seconds": fwd_s},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------
def run_ours(args, rank: int, local_rank: int, world: int):
    import sdxl_b200
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    cfg = sdxl_b200.SDXL_BASE
    ctx = sdxl_b200.Context(local_rank)
    # weights: rank 0 generates the pack on its GPU, one NCCL broadcast, every rank re-lays it out locally
    t0 = time.perf_counter()
    from sdxl_b200 import sharding
    pack = sdxl_b200.build_pack(sdxl_b200.synth_weights(cfg, seed=0, device=str(dev))) if rank == 0 else None
    comm = None
    if world > 1:
        # the C ABI's own multi-GPU load: sdxl_unet_load_broadcast (one flat ncclBroadcast inside the library); torch.distributed
        # only carries the NCCL unique id and the max-over-ranks reduction of the timings
        comm = sharding.nccl_comm_init(rank, world, dev)
    torch.cuda.synchronize()
    diffuser = sdxl_b200.Diffuser(ctx, cfg, pack, nccl_comm=comm, rank=rank, root=0)
    ctx.synchronize()
    load_s = time.perf_counter() - t0
    cpu_pack = pack.cpu() if (rank == 0 and world == 1 and not args.no_cpu_baseline and args.workload == "step") else None
    refiner = None
    if args.workload == "refiner":
        rpack = sdxl_b200.build_pack(sdxl_b200.synth_weights(sdxl_b200.SDXL_REFINER, seed=2, device=str(dev))) if rank == 0 else None
        refiner = sdxl_b200.Diffuser(ctx, sdxl_b200.SDXL_REFINER, rpack, nccl_comm=comm, rank=rank, root=0)
        ctx.synchronize()
        del rpack
    del pack
    torch.cuda.empty_cache()
    if args.workload != "step":
        return run_images(args, rank, local_rank, world, ctx, diffuser, refiner, dist, comm, load_s)

    cond = make_conditioning(rank, dev)
    diffuser.sampler_begin(cond, GUIDANCE)
    ts = sdxl_b200.ddim_timesteps(N_STEPS)  # 31 timesteps
    step_size = 1000 // N_STEPS
    lat_n = 4 * (HW // 8) * (HW // 8)
    state = {"i": 0, "img": 0}

    def new_image():
        noise = ctx.randn(lat_n, seed=rank, subsequence=state["img"]).reshape(1, 4, HW // 8, HW // 8)
        diffuser.sampler_set_latent(noise)
        state["img"] += 1

    def one_step():
        i = state["i"] % len(ts)
        if i == 0 and state["i"] > 0:
            new_image()  # next image of this rank's prompt shard
        t = ts[i]
        diffuser.sampler_step(t, t - step_size if t >= step_size else -1)
        state["i"] += 1

    new_image()
    for _ in range(args.warmup):
        one_step()
    ctx.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- e2e: same step through the host-buffer entry point (H2D latent in, D2H latent out, every step). Wall clock per step;
    # the value is built on the MEDIAN step (the box's host cores are shared: a single preemption of tens of ms inside a 0.2 s
    # region would otherwise halve the number; the mean is reported beside it). Runs before the clock sampler's nvidia-smi starts.
    host_lat = torch.randn(1, 4, HW // 8, HW // 8).pin_memory()
    e2e_steps = args.steps
    for _ in range(2):
        diffuser.sampler_step_host(999, 999 - step_size, host_lat)
    barrier()
    e2e_times = []
    for k in range(e2e_steps):
        t = ts[k % len(ts)]
        w0 = time.perf_counter()
        diffuser.sampler_step_host(t, t - step_size if t >= step_size else -1, host_lat)   # returns after the D2H copy and a stream sync
        e2e_times.append((time.perf_counter() - w0) * 1e3)
        if not torch.isfinite(host_lat).all():
            host_lat.normal_()
    e2e_ms = sharding.max_over_ranks(statistics.median(e2e_times), dev)
    e2e_mean_ms = sharding.max_over_ranks(sum(e2e_times) / len(e2e_times), dev)
    e2e_value = world * 1e3 / e2e_ms
    new_image()
    for _ in range(2):
        one_step()
    ctx.synchronize()

    # ---- device-timed region: K steps, CUDA events on the ctx stream ----
    sampler = ClockSampler(local_rank)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    launches0 = ctx.launch_count
    sampler.start()
    torch.cuda.nvtx.range_push("timed")
    e0.record(ctx.stream)
    for _ in range(args.steps):
        one_step()
    e1.record(ctx.stream)
    ctx.synchronize()
    torch.cuda.nvtx.range_pop()
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, latent=diffuser.sampler_get_latent(torch.empty(1, 4, HW // 8, HW // 8)))
    ms_total = e0.elapsed_time(e1)
    launches = ctx.launch_count - launches0
    ms_step = sharding.max_over_ranks(ms_total, dev) / args.steps   # timing rule: max over ranks of the device time
    value = world * 1e3 / ms_step

    if rank != 0:
        if world > 1:
            dist.barrier()
            sharding.nccl_comm_destroy(comm)
            dist.destroy_process_group()
        return

    # ---- per-kernel roofline (rank 0): CUDA-event time of every launch of one step's plan ----
    prof = diffuser.profile_plan()
    prof = diffuser.profile_plan()  # second pass: warm
    if args.dump_ops:
        diffuser.profile_dump(args.dump_ops)
    peaks = read_peaks()
    ig = prof["igemm_tcgen05"]
    step_flops = diffuser.plan_flops
    exec_flops = diffuser.plan_flops_executed
    total_prof_ms = sum(v["ms"] for v in prof.values())
    # The eager per-launch event times do not add up to the graph step (launch gaps in, PDL overlap out): the kernel's time INSIDE
    # the timed step is taken as its share of the eager profile times the measured step (the ncu launch list under profiles/ gives
    # the same share).
    share = ig["ms"] / total_prof_ms
    ig_ms_in_step = share * ms_step
    ach = ig["flops"] / (ig_ms_in_step * 1e-3) / 1e12
    ach_eager = ig["flops"] / (ig["ms"] * 1e-3) / 1e12
    at = prof.get("attention_tcgen05")
    whole = step_flops / (ms_step * 1e-3) / 1e12
    roofline = {
        "bound": "tensor", "achieved": ach, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": ach / peaks["tflops"],
        "frac_vs_burst": ach / peaks["tflops_burst"], "peak_burst": peaks["tflops_burst"],
        # dram__bytes_read+write of the largest igemm launch (FF-in GEGLU, M=2048 N=10240 K=1280; algorithmic bytes
        # 26.2 MB weights + 5.2 MB activations in + 21 MB out) from the ncu --set full capture under profiles/
        "traffic": 32.63e6, "traffic_unit": "bytes/launch (ncu --set full, profiles/r2_ncu_full_igemm.csv: FF-in GEGLU launch, 31.57 MB read + 1.05 MB written, tensor pipe 72.3 % active; algorithmic operand bytes 31.4 MB: the weights stream once)",
        "kernel": "igemm_pair_kernel / igemm_kernel (tcgen05 implicit GEMM: all Linear + conv of the step)",
        "peak_source": peaks["src"],
        "how": "algorithmic FLOPs of the step's igemm launches / (their share of an eager CUDA-event profile of the same plan x the measured graph step)",
        "achieved_eager_events": ach_eager,
        "kernel_share_of_step": share, "kernel_ms_in_step": ig_ms_in_step,
        "launches_per_step": ig["launches"],
        "whole_step": {"tflops": whole, "frac": whole / peaks["tflops"], "frac_vs_burst": whole / peaks["tflops_burst"], "flops_per_step": step_flops,
                       "executed_flops": exec_flops,
                       "note": "flops_per_step is the algorithmic figure (SURVEY 8(d) rule: includes the K/V projections hoisted to set_conditioning and the "
                               "upsample convs at 9 taps); executed_flops is what the step's tensor-core launches issue (hoisted work out, phase-decomposed "
                               "upsample convs at 4 taps, channel / key padding in)"},
        "by_kernel_ms_eager": {k: round(v["ms"], 4) for k, v in prof.items()},
        "by_kernel_ms_in_step": {k: round(v["ms"] / total_prof_ms * ms_step, 4) for k, v in prof.items()},
        "attention_tflops": (at["flops"] / (at["ms"] / total_prof_ms * ms_step * 1e-3) / 1e12) if at else None,
    }

    # ---- cpu_baseline (rank 0, N=1 only): bounded sample of the same workload on the host cores ----
    cpu_baseline = None
    if cpu_pack is not None:
        try:
            from oracle import unet_oracle as O
            cores = pick_threads()
            w32 = {}
            import struct
            raw = cpu_pack.numpy()
            n = struct.unpack_from("<I", raw, 8)[0]
            for i in range(n):
                name, dtype, ndim, s0, s1, s2, s3, off, nb = struct.unpack_from("<120sII4QQQ", raw, 24 + 176 * i)
                shape = [s0, s1, s2, s3][:ndim]
                w32[name.rstrip(b"\0").decode()] = cpu_pack[off:off + nb].view(torch.float16).reshape(shape).float()
            del cpu_pack
            cal = cpu_forward_seconds(w32, 32, 1, cores)[0]
            if cal * 15.8 < 40.0:
                fwd = cpu_forward_seconds(w32, 128, 1, cores)[0]
                sample = "one conditional-branch UNet forward at 1024x1024 (1 of the 62 forwards of config 2), f32, all host threads; step = 2 forwards"
            else:
                fwd = cal * (6.7612 / 0.4278)
                sample = "one UNet forward at 256x256 scaled by the algorithmic FLOP ratio 15.80 (a 1024x1024 forward would exceed the time bound); step = 2 forwards"
            cpu_baseline = {"value": 1.0 / (2.0 * fwd), "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "forward_seconds": fwd}
        except Exception as ex:  # the baseline must never take the bench line down
            cpu_baseline = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {ex!r}"}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "config": {"workload": "SDXL base 1024x1024, n=30 (31 DDIM iterations/image), cfg=7.5, bs=1 per GPU; step = CFG-batched UNet eval (2 forwards) + CFG + DDIM update",
                   "parallelism": f"replicas x{world} (prompt-sharded, NCCL weight broadcast at load, no in-step collective)",
                   "weights": "synthetic N(0,1/fan_in) f16, seed 0, 2.5675 B params", "l2": "per-step working set = 5.1 GB of weights >> 126 MB L2 (no flush needed)",
                   "forwards_per_sec": 2 * value, "images_per_sec_unet_only": value / len(ts), "load_seconds": round(load_s, 2),
                   "accumulate": "f32 (operands f16, residual stream / norms / softmax / sampler f32)"},
        "clocks": clocks, "gpu_launches": int(launches),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": lat_n * 4 + 4, "d2h_bytes_per_step": lat_n * 4, "steps": e2e_steps, "ms_per_step_median": e2e_ms, "ms_per_step_mean": e2e_mean_ms,
                "how": "sdxl_sampler_step_host: pinned host latent -> device, CFG step, latent -> host, stream sync; wall clock per step, value = 1 / median step (mean beside it)"},
        "roofline": roofline,
        "parity": read_parity(),
    }
    if cpu_baseline is not None:
        line["cpu_baseline"] = cpu_baseline
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        sharding.nccl_comm_destroy(comm)
        dist.destroy_process_group()


# --------------------------------------------------------------------------------------------------
# whole-image workloads (BASELINE configs 3, 4, 5) through the library's own sampler entry point
# --------------------------------------------------------------------------------------------------
def run_images(args, rank, local_rank, world, ctx, base, refiner, dist, comm, load_s):
    """One "step" = one whole image of this rank's prompt shard through sdxl_sample_latent (sampler_begin's conditioning hoist,
    the full DDIM loop, final latent). image: n=50 (config 3). refiner: base n=30 (31 iterations) + refine_latent(step_start 800,
    n=50) = 10 refiner iterations (config 4). inpaint: n=100 with per-step re-noising of the reference + mask blend (config 5)."""
    import sdxl_b200
    from sdxl_b200 import sharding
    dev = torch.device("cuda", local_rank)
    wl = args.workload
    cond = make_conditioning(rank, dev)
    g = lambda s: torch.Generator().manual_seed(10 * rank + s)  # noqa: E731
    rcond = None
    if wl == "refiner":
        rc, ry = torch.randn(1, N_CTX, 1280, generator=g(5)).half(), torch.randn(1, 2560, generator=g(6)).half()
        rcond = sdxl_b200.Conditioning(context_open_clip=rc, channel_context_refiner=ry, unconditional_context_open_clip=rc[0], unconditional_channel_context_refiner=ry[0],
                                       resolution=(HW, HW))
    ref = mask = None
    if wl == "inpaint":
        ref = torch.randn(1, 4, HW // 8, HW // 8, generator=g(7)).to(dev)
        mask = torch.zeros(1, 4, HW // 8, HW // 8, dtype=torch.bool)
        mask[:, :, :25] = True   # 200 px / 8
        mask = mask.to(dev)
    n_steps = {"image": 50, "refiner": 30, "inpaint": 100}[wl]
    iters = {"image": 50, "refiner": 31 + 10, "inpaint": 100}[wl]
    state = {"img": 0}

    def one_image(host=False):
        seed = 1000 * rank + state["img"]
        state["img"] += 1
        if wl == "image":
            return base.sample_latent(cond, GUIDANCE, n_steps, seed=seed, host=host)
        if wl == "refiner":
            lat = base.sample_latent(cond, GUIDANCE, n_steps, seed=seed)
            return refiner.refine_latent(lat, rcond, GUIDANCE, 800, 50, seed=seed + 500)
        return base.sample_latent_with_inpainting(cond, GUIDANCE, n_steps, ref, mask, seed=seed)

    for _ in range(max(1, min(args.warmup, 2))):
        one_image()
    ctx.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    launches0 = ctx.launch_count
    sampler.start()
    e0.record(ctx.stream)
    for _ in range(args.steps):
        out = one_image()
    e1.record(ctx.stream)
    ctx.synchronize()
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, latent=out)
    ms_img = sharding.max_over_ranks(e0.elapsed_time(e1), dev) / args.steps
    value = world * 1e3 / ms_img
    launches = ctx.launch_count - launches0
    # e2e: conditioning and result in host memory (the call a `sample` binary makes), wall clock
    e2e = None
    if wl == "image":
        one_image(host=True)
        barrier()
        w0 = time.perf_counter()
        n = max(2, min(args.steps, 4))
        for _ in range(n):
            out = one_image(host=True)
        e2e_ms = sharding.max_over_ranks((time.perf_counter() - w0) * 1e3 / n, dev)
        lat_b = 4 * (HW // 8) * (HW // 8) * 4
        cond_b = 2 * (N_CTX * 2048 + 2816) * 2
        e2e = {"value": world * 1e3 / e2e_ms, "unit": "images/s", "h2d_bytes_per_step": cond_b, "d2h_bytes_per_step": lat_b,
               "how": "sdxl_sample_latent with host conditioning / host latent out (on_host=1), stream sync, wall clock"}
        assert torch.isfinite(out).all()
    if rank == 0:
        peaks = read_peaks()
        fl_img = {"image": 50 * 13.5224e12, "refiner": 31 * 13.5224e12 + 10 * 7.2860e12, "inpaint": 100 * 13.5224e12}[wl]
        tf = fl_img / (ms_img * 1e-3) / 1e12
        line = {
            "metric": f"images_per_sec_1024x1024_{wl}", "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_img, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {"workload": {"image": "BASELINE config 3: SDXL base 1024x1024, n=50 (50 DDIM iterations), cfg 7.5, one image per GPU per step, UNet only (no CLIP / VAE)",
                                    "refiner": "BASELINE config 4: SDXL base n=30 (31 iterations, cfg 7.5) + refiner refine_latent(step_start 800, n 50) = 10 iterations, one image per GPU per step",
                                    "inpaint": "BASELINE config 5: SDXL base inpainting 1024x1024, mask = top 25 latent rows (200 px), n=100, cfg 7.5, seeded per-step noise"}[wl],
                       "parallelism": f"replicas x{world} (prompt-sharded, sdxl_unet_load_broadcast at load, no in-step collective)",
                       "iterations_per_image": iters, "sampler_steps_per_sec": value * iters, "load_seconds": round(load_s, 2),
                       "l2": "per-step working set = 5.1 GB of weights >> 126 MB L2 (no flush needed)"},
            "clocks": clocks, "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "achieved": tf, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": tf / peaks["tflops"], "frac_vs_burst": tf / peaks["tflops_burst"],
                         "flops_per_image": fl_img, "kernel": "whole image (all launches)", "peak_source": peaks["src"]},
        }
        if e2e:
            line["e2e"] = e2e
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        sharding.nccl_comm_destroy(comm)
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=31)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="step", choices=["step", "image", "refiner", "inpaint"],
                    help="step (default): BASELINE metric, sampler steps/s at 1024^2 bs=1; image / refiner / inpaint: whole images (configs 3 / 4 / 5)")
    ap.add_argument("--dump-ops", default=None, help="write a per-launch CSV of one step (CUDA-event times)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write the final latent of the last one (rank 0, float32) as DIR/latent.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")
    if args.warmup < 3 and args.workload == "step":
        args.warmup = 3
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under torch.distributed.run
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", os.environ.get("MASTER_PORT", "29541"), os.path.abspath(__file__), "--gpus", str(args.gpus), "--steps", str(args.steps),
               "--warmup", str(args.warmup), "--workload", args.workload] + (["--no-cpu-baseline"] if args.no_cpu_baseline else []) \
            + (["--dump-outputs", os.path.abspath(args.dump_outputs)] if args.dump_outputs else [])
        sys.exit(subprocess.call(cmd))
    run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
