#!/usr/bin/env python
"""Benchmark of the ResShift denoising hot path (BASELINE.json metric: 256x256 x4-SR images/sec at 15
steps; ms/denoise-step).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch: the full T=15-step residual-shift sampling loop
(denoiser forward + p_sample update per step) for a batch of 16 latents of 64x64 (= sixteen 256x256 x4-SR
images), BASELINE config 2 (`realsr_swinunet_realesrgan256_journal.yaml` with steps=15), random-init
weights, synthetic inputs.  N > 1 (torchrun, one rank per GPU): every rank owns 16 images (weak scaling,
config 3 = 128 images on 8 GPUs); rank 0 broadcasts the weights over NCCL once (untimed set-up,
`resshift_b200.parallel.broadcast_state_dict`) and the result shards are all-gathered inside the timed step
(`resshift_b200.parallel.gather_shards`).  Every rank uses the SAME seed, like the reference
(sampler.py:59-64): the global batch is drawn once, rank r takes slice r, and the per-step noise is identical
on every rank — so the sharded run can be checked bit for bit (`shard_parity`).

Printed JSON (one line, rank 0): see README/DESIGN.md.  `value` = images/s with inputs resident in HBM
(CUDA-graph replay of the loop); `e2e` = the same through the C-ABI host-buffer entry point
(`rs_sampler_run_host`: pinned host -> device copies of z_y, the T+1 noise tensors and the LQ image, the
loop, device -> host copy of the final latent, all inside the timed region).
Extra keys: `gpu_library_baseline` (the oracle port of the reference moved to CUDA under fp16 autocast = the
cuDNN / cuBLAS regime of reference sampler.py:185, informational), `other_configs` (BASELINE configs 1, 4, 5),
`shard_parity` (N > 1), `cpu_baseline`.
"""
from __future__ import annotations

import argparse
import ctypes as C
import csv
import json
import math
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

# SURVEY.md §8(d): algorithmic 2*MACs per image per denoise step, hook-counted on the reference
GF_PER_IMAGE_STEP = {"realsr": 101.32e9, "inpaint": 102.72e9, "faceir": 107.37e9}
T_STEPS = 15
BATCH_PER_GPU = 16


def _peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"tensor_tflops": float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1590.0))),
                "hbm_gbs": float(d.get("hbm_gbs", 6650.0)), "source": "MEASURED_PEAKS.json (sustained bf16 cuBLAS)"}
    return {"tensor_tflops": 1400.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md: ~1.4 PF sustained)"}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=3)
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows for i in range(4) if len(r) > 2 + i and r[2 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


def log(msg):
    print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


# --------------------------------------------------------------------------------------------------
# host cores: what this process may really use (cgroup CPU quota AND scheduler affinity)
# --------------------------------------------------------------------------------------------------
def host_threads() -> dict:
    aff = len(os.sched_getaffinity(0))
    quota = None
    try:
        txt = Path("/sys/fs/cgroup/cpu.max").read_text().split()
        if txt and txt[0] != "max":
            quota = float(txt[0]) / float(txt[1])
    except Exception:
        try:   # cgroup v1
            q = int(Path("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read_text())
            per = int(Path("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read_text())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    usable = aff if quota is None else max(1, min(aff, int(math.floor(quota + 1e-6))))
    return {"threads": usable, "affinity_cpus": aff, "cgroup_cpu_quota": quota, "os_cpu_count": os.cpu_count()}


def cpu_reference_images_per_s(steps_T: int, n_images: int, repeats: int):
    """The reference's algorithm for this path on the host cores: the CPU oracle (a torch fp32 restatement of
    UNetModelSwin.forward + p_sample, pinned to reference-generated goldens).  Thread count = what the cgroup quota and
    the affinity mask allow (both are printed); one untimed warm-up, then the MIN over `repeats` runs."""
    import torch
    from oracle import diffusion_oracle as do
    from oracle import unet_oracle as uo
    from resshift_b200.config import preset
    from resshift_b200.weights import random_state_dict
    ht = host_threads()
    ucfg, dcfg = preset("realsr_journal", steps_T)
    sd = random_state_dict(ucfg, 0)
    tabs = do.schedule_tables(do.eta_schedule(dcfg.steps, dcfg.min_noise_level, dcfg.etas_end, dcfg.kappa,
                                              dcfg.schedule_kwargs["power"]), dcfg.kappa)
    g = torch.Generator().manual_seed(12345)
    y = torch.rand(n_images, 3, 64, 64, generator=g) * 2 - 1
    noises = [torch.randn(n_images, 3, 64, 64, generator=g) for _ in range(steps_T + 1)]
    # thread count: every CPU the cgroup quota / affinity mask grants, or fewer when that is faster for this batch-1
    # workload (SMT siblings, NUMA): one timed forward per candidate after a warm-up, the fastest wins and is reported
    usable = ht["threads"]
    cand = sorted({usable, max(1, usable // 2), min(usable, 32), min(usable, 16)}, reverse=True)
    t_zero = torch.zeros(n_images, dtype=torch.long)
    trial = {}
    for c in cand:
        torch.set_num_threads(c)
        uo.unet_forward(sd, ucfg, y, t_zero, lq=y)                                   # warm-up (thread pool, allocator)
        t0 = time.perf_counter()
        uo.unet_forward(sd, ucfg, y, t_zero, lq=y)
        trial[c] = time.perf_counter() - t0
    best = min(trial, key=trial.get)
    torch.set_num_threads(best)
    ht = dict(ht, threads=best, usable_cpus=usable, forward_seconds_by_threads={str(k): round(v, 4) for k, v in trial.items()})
    times = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        do.p_sample_loop(lambda x, t: uo.unet_forward(sd, ucfg, x, t, lq=y), y, noises, tabs, dcfg.kappa)
        times.append(time.perf_counter() - t0)
    return n_images / min(times), times, ht


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    per_step, ht = [], None
    for i in range(args.warmup + args.steps):
        ips, times, ht = cpu_reference_images_per_s(T_STEPS, 1, 1)
        if i >= args.warmup:
            per_step.append(times[0])
    sec = min(per_step)
    val = 1.0 / sec
    line = {
        "impl": "reference", "metric": "256x256 x4 SR images/sec (15 steps), denoising hot path", "value": val,
        "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "ms_per_denoise_step": sec * 1e3 / T_STEPS,
        "config": {"workload": "realsr 64x64 latent (256x256 x4 SR), 15 steps, random-init weights; bounded sample: "
                               "1 image per step on the host CPU", "batch": 1},
        "cpu_baseline": {"value": val, "unit": "images/s", "cores": ht["threads"], "kind": "port", "host": ht,
                         "all_step_seconds": per_step,
                         "sample": "1 image x 15 denoise steps per timed step, min over the timed steps (oracle port of the "
                                   "reference, torch fp32 CPU; threads = best of {all, 1/2, 32, 16} CPUs the cgroup quota / affinity mask grant)"},
        "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# informational: the reference's regime on the same GPU (eager PyTorch, fp16 autocast -> cuDNN / cuBLAS kernels)
# --------------------------------------------------------------------------------------------------
def gpu_library_baseline(B: int, T: int, dev):
    import torch
    from oracle import diffusion_oracle as do
    from oracle import unet_oracle as uo
    from resshift_b200.config import preset
    from resshift_b200.weights import random_state_dict
    ucfg, dcfg = preset("realsr_journal", T)
    sd = {k: v.to(dev) for k, v in random_state_dict(ucfg, 0).items()}
    tabs = do.schedule_tables(do.eta_schedule(dcfg.steps, dcfg.min_noise_level, dcfg.etas_end, dcfg.kappa,
                                              dcfg.schedule_kwargs["power"]), dcfg.kappa)
    g = torch.Generator(device=dev).manual_seed(12345)
    y = torch.rand(B, 3, 64, 64, device=dev, generator=g) * 2 - 1
    noises = [torch.randn(B, 3, 64, 64, device=dev, generator=g) for _ in range(T + 1)]

    def loop():
        with torch.autocast("cuda", dtype=torch.float16):
            return do.p_sample_loop(lambda x, t: uo.unet_forward(sd, ucfg, x, t, lq=y), y, noises, tabs, dcfg.kappa)
    loop()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for _ in range(3):
        e0.record()
        loop()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    best = min(ms)
    return {"value": B / (best * 1e-3), "unit": "images/s", "ms_per_denoise_step": best / T, "batch": B,
            "what": "oracle port of the reference (functional torch ops: F.conv2d / F.group_norm / matmul / softmax) on the "
                    "same GPU, eager, torch.autocast(fp16) as reference sampler.py:185 — cuDNN / cuBLAS kernels, "
                    "min of 3 loops after one warm-up, CUDA events; device-resident inputs",
            "all_ms": ms}


VQ_F4_GFLOP_PER_IMAGE = 1020.0      # SURVEY.md §8(f) rank 1: VQ-GAN f4 encode + decode of one 256x256 image, 2*MACs


def e2e_with_bookends(B: int, dev, steps: int, world: int = 1):
    """images/s of the complete x4 super-resolution of B 64x64 uint8 images -> B 256x256 uint8 images on one GPU,
    through ResShiftSampler (this package's native denoiser, VQ-GAN f4 and edge kernels), host buffers at both ends."""
    import torch
    from resshift_b200.config import preset
    from resshift_b200.sampler import ResShiftSampler, make_configs
    from resshift_b200.vq_arch import random_vq_state_dict, vq_preset
    from resshift_b200.weights import random_state_dict
    ucfg, dcfg = preset("realsr_journal", T_STEPS)
    vcfg = vq_preset("f4")
    ae = {"target": "ldm.models.autoencoder.VQModelTorch", "params": vcfg.to_kwargs(), "ckpt_path": random_vq_state_dict(vcfg, 0)}
    s = ResShiftSampler(make_configs(ucfg, dcfg, autoencoder=ae, state_dict=random_state_dict(ucfg, 0)), sf=4, use_amp=True,
                        chop_size=64, chop_stride=64, chop_bs=1, padding_offset=16, seed=12345)
    g = torch.Generator().manual_seed(2024)
    h_in = torch.randint(0, 256, (B, 64, 64, 3), dtype=torch.uint8, generator=g).pin_memory()
    h_out = torch.empty(B, 256, 256, 3, dtype=torch.uint8).pin_memory()

    def step():
        d_in = h_in.to(dev, non_blocking=True)
        out = s._process_u8(d_in, noise_repeat=False, bgr=True)
        if world > 1:            # the final gather of north_star: uint8 [B/G, 256, 256, 3] shards over NCCL / NVLink
            from resshift_b200 import parallel
            allout = parallel.gather_shards(out, world * B)
            out = allout[:B]
        h_out.copy_(out, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3 / steps
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    # stage breakdown with CUDA events (device-resident, one run each after the warm-up above)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    d_in = h_in.to(dev)
    lq = torch.empty(B, 3, 64, 64, device=dev)
    from resshift_b200 import _lib
    _lib.check(_lib.lib.rs_op_ingest_u8(d_in.data_ptr(), B, 64, 64, 3, lq.data_ptr(), _lib.current_stream()))
    diff, ae_m, model = s.base_diffusion, s.autoencoder, s.model
    ev[0].record()
    z_y = diff.encode_first_stage(lq, ae_m, up_sample=True)
    ev[1].record()
    z = diff.sample_latent(z_y, model, {"lq": lq})
    ev[2].record()
    img = ae_m.decode(z)
    ev[3].record()
    torch.cuda.synchronize()
    enc_ms, loop_ms, dec_ms = ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[2].elapsed_time(ev[3])
    peaks = _peaks()
    vq_tflops = B * VQ_F4_GFLOP_PER_IMAGE * 1e9 / ((enc_ms + dec_ms) * 1e-3) / 1e12
    return {"value": world * B / (ms * 1e-3), "unit": "images/s", "ms_per_step": ms, "batch": B, "n_gpus": world,
            "h2d_bytes_per_step": int(h_in.numel()), "d2h_bytes_per_step": int(h_out.numel()),
            "stage_ms": {"bicubic_plus_vq_encode": enc_ms, "denoise_loop_15_steps_incl_noise_draw": loop_ms, "quantise_plus_vq_decode": dec_ms},
            "vq_roofline": {"bound": "tensor", "achieved": vq_tflops, "peak": peaks["tensor_tflops"], "unit": "TFLOP/s",
                            "frac": vq_tflops / peaks["tensor_tflops"],
                            "note": "VQ-GAN f4 encode + decode, 1.02 TFLOP per 256x256 image (SURVEY.md §8f), CUDA events around both"},
            "what": "uint8 [B,64,64,3] pinned host -> H2D -> ingest -> bicubic x4 -> VQ-GAN f4 encode -> 15-step loop (CUDA graph) -> "
                    "quantise + decode -> uint8 emit -> D2H [B,256,256,3]; random-init weights; wall clock per batch",
            "nan": bool(torch.isnan(img).any().item())}


def newest_ncu_summary():
    """(traffic bytes per GEMM launch, tensor-pipe % per kernel, file) from the newest profiles/*_ncu_full_summary.csv."""
    files = sorted((ROOT / "profiles").glob("*_ncu_full_summary.csv"), key=lambda p: p.stat().st_mtime)
    # prefer the highest round / session tag in the name (mtime is not preserved by git)
    def tag(p):
        import re
        m = re.match(r"r(\d+)_s(\d+)_", p.name)
        return (int(m.group(1)), int(m.group(2))) if m else (0, 0)
    files = sorted(files, key=tag)
    if not files:
        return None, None, None
    f = files[-1]
    rows = list(csv.reader(f.open()))
    hdr = rows[0]
    try:
        i_name, i_rd, i_wr = hdr.index("Kernel Name"), hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
        i_tp = hdr.index("sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active")
    except ValueError:
        return None, None, f.name
    units = rows[1]
    scale = {"Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0, "Gbyte": 1e9}
    tot, n, tp = 0.0, 0, {}
    for r in rows[2:]:
        if len(r) <= max(i_rd, i_wr, i_tp) or not r[i_name]:
            continue
        if "conv_gemm" in r[i_name] or "mlp_fused" in r[i_name] or "swin" in r[i_name]:
            tot += float(r[i_rd]) * scale.get(units[i_rd], 1.0) + float(r[i_wr]) * scale.get(units[i_wr], 1.0)
            n += 1
            tp.setdefault(r[i_name], []).append(float(r[i_tp]))
    tp = {k: round(sum(v) / len(v), 1) for k, v in tp.items()}
    return (tot / n if n else None), tp, f.name


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir: Path, arrays: dict):
    """Writes what the timed path returned in its last step as <out_dir>/<name>.npy (float32), so that two builds run
    with the same arguments (same seeded inputs) can be compared output for output.  An output larger than
    DUMP_MAX_BYTES in all keeps a fixed, seeded sample of its images (leading axis)."""
    import numpy as np
    out_dir.mkdir(parents=True, exist_ok=True)
    total = sum(a.numel() * 4 for a in arrays.values())
    for name, a in arrays.items():
        a = a.detach().float().cpu().numpy()
        if total > DUMP_MAX_BYTES:
            n = a.shape[0]
            keep = max(1, int(n * DUMP_MAX_BYTES // total))
            a = a[np.sort(np.random.default_rng(0).choice(n, keep, replace=False))]
        np.save(out_dir / f"{name}.npy", np.ascontiguousarray(a, dtype=np.float32))
    log(f"outputs of the last timed step written to {out_dir}")


def run_gpu(args):
    import faulthandler
    faulthandler.dump_traceback_later(900, exit=True)
    import torch
    import torch.distributed as dist
    from resshift_b200 import _lib
    from resshift_b200 import parallel
    from resshift_b200.config import preset
    from resshift_b200.models.script_util import create_gaussian_diffusion
    from resshift_b200.models.unet import UNetModelSwin
    from resshift_b200.weights import random_state_dict

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group(backend="nccl", init_method="env://", device_id=dev)

    B = args.batch
    stream = torch.cuda.current_stream().cuda_stream

    def build(name, steps, bcast=True):
        ucfg, dcfg = preset(name, steps)
        dcfg.sf = 1       # the loop works on the latent; the bicubic + VQ bookends are outside the hot path
        model = UNetModelSwin(**ucfg.to_kwargs())
        if rank == 0:
            model.load_state_dict(random_state_dict(ucfg, 0))
        model = model.cuda().eval()
        if world > 1 and bcast:     # ONE NCCL broadcast of all weights as a flat buffer, untimed set-up
            parallel.broadcast_state_dict({k: p.data for k, p in model.named_parameters()}, src=0)
        return ucfg, model, create_gaussian_diffusion(**dcfg.to_kwargs())

    ucfg, model, diff = build("realsr_journal", T_STEPS)
    T = diff.num_timesteps

    # same seed on every rank (reference sampler.py:59-64): global batch drawn once, rank r owns slice r; the per-step
    # noise tensors have the shard's shape and are therefore identical on every rank
    g = torch.Generator(device=dev).manual_seed(12345)
    z_all = torch.rand(world * B, 3, 64, 64, device=dev, generator=g) * 2 - 1
    noises = torch.randn(T + 1, B, 3, 64, 64, device=dev, generator=g)
    s0, s1 = parallel.shard_range(world * B, world, rank)
    z_y = z_all[s0:s1].contiguous()
    lq = z_y.clone()
    out = torch.empty_like(z_y)
    sampler = diff.native_sampler(model, B, 64, 64)
    plan = model.plan(B, 64, 64)
    launches_per_forward = _lib.lib.rs_plan_num_launches(plan.handle)
    launches_per_loop = T * (launches_per_forward - 6 + 1) + 2      # per step: body + p_sample; + prior + pack
    gathered = {}

    def one_step(use_graph=True):
        _lib.check(_lib.lib.rs_sampler_run(sampler, z_y.data_ptr(), noises.data_ptr(), lq.data_ptr(), None,
                                           out.data_ptr(), int(use_graph), stream))
        if world > 1:
            gathered["all"] = parallel.gather_shards(out, world * B)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput ("value") ----------------------------------------------------
    log(f"model + plan ready: {launches_per_forward} launches/forward, batch {B}")
    for _ in range(max(args.warmup, 3)):
        one_step()
    barrier()
    log("warm-up done")
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        one_step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    clk = clocks.stop() if rank == 0 else None
    t_ms = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_total = t_ms.item()
    ms_per_step = ms_total / args.steps
    value = world * B / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(Path(args.dump_outputs), {"final_latent": gathered["all"] if world > 1 else out})

    if args.quick:       # A/B and ablation runs: only the device-resident figure
        if rank == 0:
            print(json.dumps({"quick": True, "ms_per_step": ms_per_step, "ms_per_denoise_step": ms_per_step / T, "value": value,
                              "launches_per_denoise_step": int(launches_per_forward - 6 + 1), "clocks": clk,
                              "env": {k: v for k, v in os.environ.items() if k.startswith("RS_")}}), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- sharded run == single-GPU run on the same slice (SURVEY §8e) ------------------------------------
    shard_parity = None
    if world > 1:
        full = gathered["all"].clone()
        if rank == 0:
            r = world - 1
            a, b = parallel.shard_range(world * B, world, r)
            zr = z_all[a:b].contiguous()
            mine = torch.empty_like(zr)
            _lib.check(_lib.lib.rs_sampler_run(sampler, zr.data_ptr(), noises.data_ptr(), zr.data_ptr(), None,
                                               mine.data_ptr(), 0, stream))
            torch.cuda.synchronize()
            shard_parity = {"checked_rank": r, "equal": bool(torch.equal(mine, full[a:b])),
                            "max_abs_diff": float((mine - full[a:b]).abs().max().item()),
                            "what": "rank 0 re-runs rank r's slice on its own GPU (same seed, same noise) and compares with "
                                    "the all-gathered shard bit for bit (reference sampler.py:273-277 slicing)"}
        barrier()

    # ---- end to end through the host-buffer C-ABI entry ("e2e") ------------------------------------
    staging_bytes = _lib.lib.rs_sampler_staging_bytes(sampler)
    staging = torch.empty(staging_bytes + 256, dtype=torch.uint8, device=dev)
    staging_ptr = (staging.data_ptr() + 255) // 256 * 256
    h_zy = z_y.cpu().pin_memory()
    h_noise = noises.cpu().pin_memory()
    h_lq = lq.cpu().pin_memory()
    h_out = torch.empty(B, 3, 64, 64).pin_memory()

    def e2e_step():
        _lib.check(_lib.lib.rs_sampler_run_host(sampler, h_zy.data_ptr(), h_noise.data_ptr(), h_lq.data_ptr(), None,
                                                h_out.data_ptr(), staging_ptr, staging_bytes, 1, stream))
    log(f"device-resident: {ms_per_step:.2f} ms/step")
    for _ in range(3):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        e2e_step()
    e1.record()
    barrier()
    wall = (time.perf_counter() - t0) * 1e3
    e2e_ms = torch.tensor([max(e0.elapsed_time(e1), wall)], device=dev)
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_value = world * B / (e2e_ms.item() / args.steps * 1e-3)
    h2d = (h_zy.numel() + h_noise.numel() + h_lq.numel()) * 4
    d2h = h_out.numel() * 4

    # ---- whole x4 path incl. the VQ-GAN bookends and the uint8 edges, host buffers in and out ------------------
    # uint8 LQ images (pinned host) -> H2D -> ingest -> bicubic x4 -> VQ-GAN encode -> 15-step loop -> quantise + decode
    # -> uint8 emit -> D2H: what ResShiftSampler.inference does per batch (reference sampler.py:176-223,286)
    bookends = None
    if not args.no_bookends:
        try:
            bookends = e2e_with_bookends(B, dev, max(2, min(args.steps, 3)), world)
        except Exception as ex:
            bookends = {"error": repr(ex)[:400]}
        if rank == 0:
            log("bookends done")

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel family (implicit-GEMM conv / linear / fused MLP on tcgen05), measured live ----
    ms_kind = (C.c_double * 4)()
    flops = C.c_double()
    nconv = C.c_int32()
    tt = torch.full((B,), 7.0, device=dev)
    x0 = torch.randn(B, 3, 64, 64, device=dev)
    prof = []
    for _ in range(3):
        _lib.check(_lib.lib.rs_plan_profile(plan.handle, x0.data_ptr(), tt.data_ptr(), lq.data_ptr(), None, ms_kind,
                                            C.byref(flops), C.byref(nconv), stream))
        prof.append(list(ms_kind))
    pk = prof[-1]
    peaks = _peaks()
    conv_tflops = flops.value / (pk[0] * 1e-3) / 1e12 if pk[0] > 0 else 0.0
    traffic, tensor_pct, ncu_file = newest_ncu_summary()
    roofline = {
        "kernel": "tcgen05 GEMM kernels: conv_gemm_sm100_kernel<1|2>, conv_gemm_persist_sm100_kernel<1|2> (all conv3x3 / "
                  "conv1x1 / linear layers) + mlp_fused_sm100_kernel (Swin MLPs) + swin_attn_tc_kernel (norm1 + qkv + window "
                  "attention + proj of every Swin block)", "bound": "tensor",
        "achieved": conv_tflops, "peak": peaks["tensor_tflops"], "unit": "TFLOP/s",
        "frac": conv_tflops / peaks["tensor_tflops"],
        # dram__bytes_read.sum + dram__bytes_write.sum per launch, averaged over the GEMM launches of the newest committed
        # `ncu --set full` capture of this workload (cold caches: ncu flushes between replays); read from the file, not typed in
        "traffic": traffic if B == BATCH_PER_GPU else None,
        "launches_per_forward": int(nconv.value), "avg_launch_us": pk[0] * 1e3 / max(1, nconv.value),
        "algorithmic_gflop_per_forward": flops.value / 1e9, "peak_source": peaks["source"],
        "per_forward_ms_by_kernel": {"gemm_family": pk[0], "groupnorm": pk[1], "window_attn_unfused": pk[2], "upsample": pk[3]},
        "traffic_source": f"profiles/{ncu_file}" if ncu_file else None,
        "tensor_pipe_active_pct_ncu": tensor_pct,
        "note": "achieved = algorithmic FLOPs of all GEMM launches / sum of their durations, CUDA events around every "
                "launch of one un-graphed forward on the launching stream (includes inter-launch gaps, so it "
                "under-states the graph-replayed step); whole-step figure: denoiser_tflops_per_gpu",
    }
    # whole-step tensor-pipe fraction as a cross-check
    step_tflops = B * T * GF_PER_IMAGE_STEP["realsr"] / (ms_per_step * 1e-3) / 1e12
    roofline["whole_step_frac"] = step_tflops / peaks["tensor_tflops"]

    # ---- BASELINE configs 1, 4, 5 (short device-resident measurements on this GPU) ---------------------
    other = {}
    if not args.no_other_configs:
        def measure(name, steps, batch, tag, gf_key, lq_hw, mask):
            try:
                u2, m2, d2 = build(name, steps, bcast=False) if name != "realsr_journal" else (ucfg, model, diff)
                T2 = d2.num_timesteps
                gg = torch.Generator(device=dev).manual_seed(4242)
                zy2 = torch.rand(batch, u2.in_channels, 64, 64, device=dev, generator=gg) * 2 - 1
                nz2 = torch.randn(T2 + 1, batch, u2.in_channels, 64, 64, device=dev, generator=gg)
                lq2 = torch.rand(batch, 3, lq_hw, lq_hw, device=dev, generator=gg) * 2 - 1
                mk2 = None
                if mask:
                    mk2 = -torch.ones(batch, 1, lq_hw, lq_hw, device=dev)
                    mk2[:, :, lq_hw // 4: lq_hw // 4 * 3, lq_hw // 4: lq_hw // 4 * 3] = 1.0     # centred square = unknown area
                o2 = torch.empty_like(zy2)
                s2 = d2.native_sampler(m2, batch, 64, 64)

                def go():
                    _lib.check(_lib.lib.rs_sampler_run(s2, zy2.data_ptr(), nz2.data_ptr(), lq2.data_ptr(), _lib.ptr(mk2),
                                                       o2.data_ptr(), 1, stream))
                for _ in range(3):
                    go()
                torch.cuda.synchronize()
                e0.record()
                for _ in range(3):
                    go()
                e1.record()
                torch.cuda.synchronize()
                ms2 = e0.elapsed_time(e1) / 3
                other[tag] = {"images_per_s": batch / (ms2 * 1e-3), "ms_per_step": ms2, "ms_per_denoise_step": ms2 / T2,
                              "batch": batch, "denoise_steps": T2, "preset": name,
                              "whole_step_frac": batch * T2 * GF_PER_IMAGE_STEP[gf_key] / (ms2 * 1e-3) / 1e12 / peaks["tensor_tflops"],
                              "nan": bool(torch.isnan(o2).any().item())}
                if name != "realsr_journal":
                    del m2
                    torch.cuda.empty_cache()
            except Exception as ex:      # never lose the headline line to a side measurement
                other[tag] = {"error": repr(ex)[:300]}
        measure("realsr_journal", T_STEPS, 1, "config1_realsr_b1_15steps", "realsr", 64, False)
        measure("faceir", 15, 8, "config4_faceir_b8_15steps", "faceir", 512, False)
        measure("inpaint", 4, 16, "config5_inpaint_b16_per_gpu_4steps", "inpaint", 256, True)
        log("other configs done")

    # ---- the reference's regime on this GPU: eager fp16-autocast PyTorch (cuDNN / cuBLAS) ----------------
    lib_base = None
    if not args.no_library_baseline:
        try:
            lib_base = gpu_library_baseline(B, T, dev)
            lib_base["speedup_of_this_repo"] = value / world / lib_base["value"]
        except Exception as ex:
            lib_base = {"error": repr(ex)[:300]}
        log("library baseline done")

    # ---- CPU baseline: bounded sample on this box's host cores ----------------------------------------
    cpu = None
    if not args.no_cpu_baseline:
        ips, times, ht = cpu_reference_images_per_s(T_STEPS, 1, 3)
        cpu = {"value": ips, "unit": "images/s", "cores": ht["threads"], "kind": "port", "host": ht, "all_seconds": times,
               "sample": f"1 image x {T_STEPS} denoise steps, min of 3 runs after a warm-up forward = {min(times):.2f} s (oracle "
                         "port of the reference, torch fp32 CPU; threads = best of {all, 1/2, 32, 16} CPUs the cgroup quota / affinity mask grant)"}

    line = {
        "metric": "256x256 x4 SR images/sec (15 steps), denoising hot path", "value": value, "unit": "images/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16 (fp32 accumulate)",
        "data": "synthetic", "ms_per_denoise_step": ms_per_step / T,
        "config": {"workload": "BASELINE config %s: batch=%d/GPU 256x256 x4 real-SR (64x64 latent), 15 steps, "
                               "realsr_swinunet_realesrgan256_journal.yaml with steps=15, random-init weights"
                               % ("2" if world == 1 else "3", B),
                   "global_batch": world * B, "parallelism": f"dp{world} (independent image shards, NCCL weight broadcast + final all_gather)",
                   "l2": "no explicit flush: per-step working set (237 MB fp16 weights + >1 GB activations) exceeds the 126 MB L2"},
        "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": int(launches_per_loop * args.steps * 2),
        "launches_per_denoise_step": int(launches_per_forward - 6 + 1),
        "denoiser_tflops_per_gpu": step_tflops,
        "e2e_with_bookends": bookends,
        "roofline": roofline, "cpu_baseline": cpu, "gpu_library_baseline": lib_base, "other_configs": other,
        "shard_parity": shard_parity, "clocks": clk,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH_PER_GPU, help="images per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-library-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--no-bookends", action="store_true")
    ap.add_argument("--quick", action="store_true", help="device-resident timing only (A/B and ablation runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the final latents of the last timed step to DIR/final_latent.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the native path; it does not apply to --impl reference")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
