"""Pins the VQ-GAN oracle at a size whose bottleneck attention has more than 8192 tokens (f4 at 512x512: T = 16384)
against the reference's own VQModelTorch (oracle/make_golden_vq_large.py -> tests/golden/vq_f4_512.npz), and checks
on the host that the fused-attention plans no longer carry a T x T term in their workspace."""
import ctypes as C

import numpy as np
import torch

from oracle import vq_oracle as vo
from oracle.make_golden_vq_large import draw_inputs, sample_positions
from resshift_b200.vq_arch import random_vq_state_dict, vq_preset

TOL = 2e-4


def test_vq_f4_512_encode_decode(golden_dir):
    g = np.load(golden_dir / "vq_f4_512.npz")
    cfg = vq_preset("f4")
    sd = random_vq_state_dict(cfg, 0)
    x, z = draw_inputs(int(g["seed"]), 1, 512, cfg.embed_dim, cfg.downscale)
    assert np.abs(vo.vq_encode(x, sd, cfg).numpy() - g["enc"]).max() < TOL
    _, idx = vo.quantize(z, sd)
    assert np.array_equal(idx.numpy(), g["idx"])
    dec = vo.vq_decode(z, sd, cfg)
    pos = sample_positions(int(g["seed"]), dec.numel(), g["dec_s"].size)
    assert np.abs(dec.reshape(-1)[pos].numpy() - g["dec_s"]).max() < TOL
    dec_nq = vo.vq_decode(z, sd, cfg, force_not_quantize=True)
    assert np.abs(dec_nq.reshape(-1)[pos].numpy() - g["dec_nq_s"]).max() < TOL


def _workspace_bytes(name, which, hw):
    from resshift_b200 import _lib
    L = _lib.lib
    cfgc = _lib.make_vq_config(vq_preset(name))
    e, p = C.c_void_p(), C.c_void_p()
    _lib.check(L.rs_vq_create(C.byref(cfgc), C.byref(e)))
    try:
        _lib.check(L.rs_vq_plan_create(e, 1, hw, hw, which, C.byref(p)))
        n = L.rs_plan_workspace_bytes(p)
        L.rs_plan_destroy(p)
        return n
    finally:
        L.rs_unet_destroy(e)


def test_fused_attention_workspace_grows_with_pixels():
    """Plans above 8192 bottleneck tokens build (host side only) and their workspace is linear in the pixel count:
    1024^2 needs about 4x the workspace of 512^2 (a T^2 score matrix would make it 16x)."""
    for name, sizes in (("f4", (512, 1024, 2048)), ("f8_face", (1024, 2048))):
        for which in (0, 1):
            ws = [_workspace_bytes(name, which, hw) for hw in sizes]
            for a, b in zip(ws, ws[1:]):
                assert 3.5 < b / a < 4.5, (name, which, ws)
