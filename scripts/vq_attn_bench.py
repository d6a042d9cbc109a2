"""Timing of the VQ-GAN bottleneck attention (CUDA events after warm-up):

  * the fused kernel (csrc/vq_attn_tc.cuh) against the three GEMMs + row softmax inside an f4 encode plan at
    T = 4096 and 8192 (the attention ops between the .k conv and proj_out, per-op events of rs_vq_profile_ops);
  * the fused op alone through rs_op_vq_attention at T = 16384 / 65536 / 262144, C = 512;
  * whole f4 encode and decode (quantised) at 512^2, 1024^2 and 2048^2.

Rates are given against the algorithmic 4 T^2 C FLOPs per image and against what the kernel executes
((2 * parts + 2) T^2 C: each of the `parts` channel parts of O recomputes Q K^T).  The GPU name and power limit are read
in the same run.

    python scripts/vq_attn_bench.py [--reps 10]
"""
from __future__ import annotations

import argparse
import ctypes as C
import os
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from resshift_b200 import _lib  # noqa: E402
from resshift_b200.vq_arch import random_vq_state_dict, vq_preset  # noqa: E402


def gpu_info() -> str:
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception:
        q = torch.cuda.get_device_name(0) + ", power limit unknown"
    return q


def time_ms(fn, reps: int, warmup: int = 2) -> float:
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def model(name="f4"):
    from resshift_b200.models.autoencoder import VQModelTorch
    cfg = vq_preset(name)
    m = VQModelTorch(**cfg.to_kwargs())
    m.load_state_dict(random_vq_state_dict(cfg, 0), strict=True)
    return cfg, m.cuda().eval()


def attention_ms_in_plan(hw, fuse: bool, reps: int) -> float:
    """Sum of the per-op times of the attention ops (after the .k conv, before proj_out) of an f4 encode plan."""
    if fuse:
        os.environ["RS_VQ_ATTN_FUSE_MIN_TOKENS"] = "1"
    else:
        os.environ.pop("RS_VQ_ATTN_FUSE_MIN_TOKENS", None)
    cfg, m = model()
    x = torch.rand(1, 3, hw[0], hw[1], device="cuda") * 2 - 1
    m.encode(x)
    plan = m.plan(0, 1, hw[0], hw[1])
    cap, stride = 512, 160
    ms = (C.c_double * cap)()
    desc = C.create_string_buffer(cap * stride)
    n = C.c_int32()
    tot = []
    for _ in range(reps):
        _lib.check(_lib.lib.rs_vq_profile_ops(plan.handle, ms, desc, stride, cap, C.byref(n), _lib.current_stream()))
        names = [desc.raw[i * stride:(i + 1) * stride].split(b"\0")[0].decode() for i in range(n.value)]
        k = next(i for i, s in enumerate(names) if "encoder.mid.attn_1.k.weight" in s)
        po = next(i for i, s in enumerate(names) if "encoder.mid.attn_1.proj_out.weight" in s)
        tot.append(sum(ms[i] for i in range(k + 1, po)))
    os.environ.pop("RS_VQ_ATTN_FUSE_MIN_TOKENS", None)
    tot.sort()
    return tot[len(tot) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    print(f"GPU: {gpu_info()}")
    Cc = 512
    parts = 1 if Cc <= 256 else 2

    def rates(T, ms):
        alg = 4.0 * T * T * Cc
        exe = (2.0 * parts + 2.0) * T * T * Cc
        return alg / (ms * 1e-3) / 1e12, exe / (ms * 1e-3) / 1e12

    print("\n== attention inside the f4 encode plan (V^T GEMM + attention; median of per-op event sums) ==")
    for hw in ((256, 256), (256, 512)):
        T = hw[0] * hw[1] // 16
        t3 = attention_ms_in_plan(hw, False, a.reps)
        tf = attention_ms_in_plan(hw, True, a.reps)
        print(f"T={T:6d} C={Cc}: three GEMMs + softmax {t3:.3f} ms | fused {tf:.3f} ms | ratio {t3 / tf:.2f}x")

    print("\n== fused op alone (rs_op_vq_attention, batch 1) ==")
    for T in (16384, 65536, 262144):
        g = torch.Generator(device="cuda").manual_seed(T)
        q = torch.randn(1, T, Cc, device="cuda", generator=g).half()
        k = torch.randn(1, T, Cc, device="cuda", generator=g).half()
        vt = torch.randn(1, Cc, T, device="cuda", generator=g).half()
        bias = torch.zeros(Cc, device="cuda")
        out = torch.empty(1, T, Cc, dtype=torch.float16, device="cuda")
        fn = lambda: _lib.check(_lib.lib.rs_op_vq_attention(q.data_ptr(), k.data_ptr(), vt.data_ptr(), bias.data_ptr(), 1, T, Cc,
                                                            out.data_ptr(), _lib.current_stream()))
        ms = time_ms(fn, a.reps if T < 262144 else max(2, a.reps // 4))
        ra, re = rates(T, ms)
        print(f"T={T:6d} C={Cc}: {ms:9.3f} ms  algorithmic {4.0 * T * T * Cc / 1e12:7.2f} TFLOP -> {ra:6.1f} TF/s | "
              f"executed {(2.0 * parts + 2.0) * T * T * Cc / 1e12:7.2f} TFLOP -> {re:6.1f} TF/s")
        del q, k, vt, out

    print("\n== whole f4 encode / decode (batch 1) ==")
    cfg, m = model()
    for hw in (512, 1024, 2048):
        x = torch.rand(1, 3, hw, hw, device="cuda") * 2 - 1
        z = torch.randn(1, 3, hw // 4, hw // 4, device="cuda") * 0.6
        reps = a.reps if hw < 2048 else max(2, a.reps // 4)
        te = time_ms(lambda: m.encode(x), reps)
        td = time_ms(lambda: m.decode(z), reps)
        print(f"{hw}x{hw}: encode {te:9.3f} ms | decode {td:9.3f} ms")
        del x, z


if __name__ == "__main__":
    main()
