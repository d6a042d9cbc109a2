"""The VQ-GAN first stage above 8192 bottleneck tokens: the fused streaming attention kernel (csrc/vq_attn_tc.cuh)
through its C ABI entry and inside the encode / decode plans, against fp32 torch, the three-GEMM path, the reference's
own outputs (tests/golden/vq_f4_512.npz) and the oracle.  Tolerance: the suite's 1e-2 max / 2e-3 mean."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from resshift_b200 import _lib
from resshift_b200.vq_arch import random_vq_state_dict, vq_preset

TOL_MAX, TOL_MEAN = 1e-2, 2e-3


def _vq(name, seed=0):
    from resshift_b200.models.autoencoder import VQModelTorch
    cfg = vq_preset(name)
    m = VQModelTorch(**cfg.to_kwargs())
    m.load_state_dict(random_vq_state_dict(cfg, seed), strict=True)
    return cfg, m.cuda().eval()


def _report(tag, got, ref):
    d = (got.float() - ref.float().to(got.device)).abs()
    mx, mn = d.max().item(), d.mean().item()
    print(f"[vq attn] {tag}: max|d|={mx:.3e} mean|d|={mn:.3e} ref_std={ref.float().std().item():.3f}")
    return mx, mn


def _operands(N, T, C, seed, qscale=1.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    q = (torch.randn(N, T, C, device="cuda", generator=g) * qscale).half()
    k = torch.randn(N, T, C, device="cuda", generator=g).half()
    vt = torch.randn(N, C, T, device="cuda", generator=g).half()
    bias = torch.randn(C, device="cuda", generator=g) * 0.1
    return q, k, vt, bias


def _op(q, k, vt, bias):
    N, T, C = q.shape
    out = torch.full((N, T, C), float("nan"), dtype=torch.float16, device="cuda")
    _lib.check(_lib.lib.rs_op_vq_attention(q.data_ptr(), k.data_ptr(), vt.data_ptr(), bias.data_ptr(), N, T, C, out.data_ptr(),
                                           _lib.current_stream()))
    torch.cuda.synchronize()
    return out


def _ref(q, k, vt, bias, rows=None, chunk=4096):
    """fp32 attention on the same fp16 operands (query rows in chunks: the T x T scores of one chunk at a time)."""
    N, T, C = q.shape
    rows = torch.arange(T, device="cuda") if rows is None else rows
    out = torch.empty(N, rows.numel(), C, device="cuda")
    for n in range(N):
        kf, vf = k[n].float(), vt[n].float()
        for i in range(0, rows.numel(), chunk):
            r = rows[i:i + chunk]
            s = (q[n, r].float() @ kf.t()) * C ** -0.5
            out[n, i:i + chunk] = torch.softmax(s, dim=1) @ vf.t() + bias
    return out


OP_CASES = [  # (N, T, C, qscale)
    (1, 64, 128, 1.0), (1, 64, 512, 1.0), (2, 4096, 128, 1.0), (1, 4096, 512, 3.0), (1, 10560, 512, 1.0),
    (2, 10560, 128, 3.0), (1, 16384, 512, 1.0), (1, 65536, 128, 1.0), (1, 65536, 512, 1.0),
]


@pytest.mark.parametrize("N,T,C,qscale", OP_CASES)
def test_vq_attention_op_vs_torch(N, T, C, qscale):
    q, k, vt, bias = _operands(N, T, C, seed=T + C + N, qscale=qscale)
    out = _op(q, k, vt, bias)
    assert not torch.isnan(out).any()
    mx, mn = _report(f"op N={N} T={T} C={C} qscale={qscale}", out, _ref(q, k, vt, bias))
    assert mx <= TOL_MAX and mn <= TOL_MEAN
    assert torch.equal(out, _op(q, k, vt, bias))                       # no atomics: bit-reproducible


def test_vq_attention_op_262144_sampled_rows():
    N, T, C = 1, 262144, 512
    q, k, vt, bias = _operands(N, T, C, seed=11)
    out = _op(q, k, vt, bias)
    rows = torch.randperm(T, generator=torch.Generator().manual_seed(5))[:512].sort().values.cuda()
    rows = torch.cat([rows, torch.tensor([0, T - 1], device="cuda")])
    assert not torch.isnan(out).any()
    mx, mn = _report(f"op T={T} C={C} ({rows.numel()} sampled rows)", out[:, rows], _ref(q, k, vt, bias, rows=rows, chunk=128))
    assert mx <= TOL_MAX and mn <= TOL_MEAN


@pytest.mark.parametrize("hw", [(256, 256), (256, 512)])
def test_fused_vs_three_gemm_path(monkeypatch, hw):
    """T = 4096 and 8192 (f4): the same model with RS_VQ_ATTN_FUSE_MIN_TOKENS=1 (fused kernel) and at the default
    (three GEMMs + row softmax), encode and non-quantised decode."""
    H, W = hw
    g = torch.Generator().manual_seed(H + W)
    x = (torch.rand(1, 3, H, W, generator=g) * 2 - 1).cuda()
    z = (torch.randn(1, 3, H // 4, W // 4, generator=g) * 0.6).cuda()
    _, m_ref = _vq("f4")
    enc_ref, dec_ref = m_ref.encode(x), m_ref.decode(z, force_not_quantize=True)
    monkeypatch.setenv("RS_VQ_ATTN_FUSE_MIN_TOKENS", "1")
    _, m = _vq("f4")
    enc, dec = m.encode(x), m.decode(z, force_not_quantize=True)
    for tag, a, b in (("encode", enc, enc_ref), ("decode", dec, dec_ref)):
        mx, mn = _report(f"fused vs three-GEMM {tag} {H}x{W}", a, b)
        assert mx <= TOL_MAX and mn <= TOL_MEAN


def test_vq_f4_512_vs_reference_golden(golden_dir):
    from oracle.make_golden_vq_large import draw_inputs, sample_positions
    g = np.load(golden_dir / "vq_f4_512.npz")
    cfg, m = _vq("f4")
    x, z = draw_inputs(int(g["seed"]), 1, 512, cfg.embed_dim, cfg.downscale)
    enc = m.encode(x.cuda())
    assert not torch.isnan(enc).any()
    mx, mn = _report("golden encode f4 512", enc, torch.from_numpy(g["enc"]))
    assert mx <= TOL_MAX and mn <= TOL_MEAN
    # (the fixture keeps the decoded images at seeded sample positions only)
    dec_nq = m.decode(z.cuda(), force_not_quantize=True)
    pos = sample_positions(int(g["seed"]), dec_nq.numel(), g["dec_s"].size).cuda()
    mx, mn = _report("golden decode (not quantised) f4 512, sampled", dec_nq.reshape(-1)[pos], torch.from_numpy(g["dec_nq_s"]))
    assert mx <= TOL_MAX and mn <= TOL_MEAN
    dec = m.decode(z.cuda())
    idx = m.last_indices.cpu().numpy()
    flips = idx != g["idx"]
    print(f"[vq attn] golden f4 512: code flips {int(flips.sum())} / {flips.size}; margins at flips {g['margin'][flips][:8]}")
    assert flips.mean() <= 0.002 and (g["margin"][flips] < 1e-5).all()
    if not flips.any():
        mx, mn = _report("golden decode (quantised) f4 512, sampled", dec.reshape(-1)[pos], torch.from_numpy(g["dec_s"]))
        assert mx <= TOL_MAX and mn <= TOL_MEAN


def test_vq_f4_1024_vs_oracle():
    """T = 65536: encode and non-quantised decode against the oracle, run in fp32 on the device (its T x T scores are
    16 GiB)."""
    from oracle import vq_oracle as vo
    cfg, m = _vq("f4")
    sd = {k: v.cuda() for k, v in random_vq_state_dict(cfg, 0).items()}
    g = torch.Generator().manual_seed(1024)
    x = (torch.rand(1, 3, 1024, 1024, generator=g) * 2 - 1).cuda()
    z = (torch.randn(1, 3, 256, 256, generator=g) * 0.6).cuda()
    tf32 = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    try:
        enc_ref = vo.vq_encode(x, sd, cfg)
        mx, mn = _report("oracle encode f4 1024", m.encode(x), enc_ref)
        assert mx <= TOL_MAX and mn <= TOL_MEAN
        del enc_ref
        torch.cuda.empty_cache()
        dec_ref = vo.vq_decode(z, sd, cfg, force_not_quantize=True)
        mx, mn = _report("oracle decode (not quantised) f4 1024", m.decode(z, force_not_quantize=True), dec_ref)
        assert mx <= TOL_MAX and mn <= TOL_MEAN
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = tf32


def test_vq_f4_2048_runs_and_is_reproducible():
    cfg, m = _vq("f4")
    g = torch.Generator(device="cuda").manual_seed(2048)
    x = torch.rand(1, 3, 2048, 2048, device="cuda", generator=g) * 2 - 1
    a = m.encode(x).clone()
    assert a.shape == (1, 3, 512, 512) and torch.isfinite(a).all()
    assert torch.equal(a, m.encode(x))
    z = torch.randn(1, 3, 512, 512, device="cuda", generator=g) * 0.6
    d = m.decode(z).clone()
    assert d.shape == (1, 3, 2048, 2048) and torch.isfinite(d).all()
    assert torch.equal(d, m.decode(z))


def test_vq_f8_face_1024_runs():
    cfg, m = _vq("f8_face")
    g = torch.Generator(device="cuda").manual_seed(8)
    x = torch.rand(1, 3, 1024, 1024, device="cuda", generator=g) * 2 - 1
    h = m.encode(x)
    assert h.shape == (1, 8, 128, 128) and torch.isfinite(h).all()
    d = m.decode(h)
    assert d.shape == (1, 3, 1024, 1024) and torch.isfinite(d).all()


def test_fused_batch_independence_and_determinism():
    """T = 9216 (tiny preset at 384x384): image i of a batch does not depend on its neighbours, runs are bit-identical."""
    cfg, m = _vq("tiny")
    g = torch.Generator(device="cuda").manual_seed(4)
    x = torch.rand(3, 3, 384, 384, device="cuda", generator=g) * 2 - 1
    a = m.encode(x).clone()
    assert torch.equal(a, m.encode(x))
    x2 = torch.rand_like(x) * 2 - 1
    x2[1] = x[1]
    assert torch.equal(m.encode(x2)[1], a[1])
    z = torch.randn(3, 3, 96, 96, device="cuda", generator=g) * 0.6
    d = m.decode(z).clone()
    assert torch.equal(d, m.decode(z))
    z2 = torch.randn_like(z) * 0.6
    z2[2] = z[2]
    assert torch.equal(m.decode(z2)[2], d[2])


def test_sampler_default_chop_size_with_f4():
    """ResShiftSampler at its default chop_size = 128 on a 128x128 LQ image: one 512x512 tile, T = 16384 at the VQ-GAN
    bottleneck (rejected before the fused path existed)."""
    from oracle import vq_oracle as vo
    from resshift_b200.config import preset
    from resshift_b200.sampler import ResShiftSampler, make_configs
    from resshift_b200.weights import random_state_dict
    ucfg, dcfg = preset("tiny")
    dcfg.sf = 4
    vcfg = vq_preset("f4")
    ae = {"target": "ldm.models.autoencoder.VQModelTorch", "params": vcfg.to_kwargs(), "ckpt_path": random_vq_state_dict(vcfg, 0)}
    s = ResShiftSampler(make_configs(ucfg, dcfg, autoencoder=ae, state_dict=random_state_dict(ucfg, 0)), sf=4, use_amp=True, seed=123)
    assert s.chop_size == 128
    g = torch.Generator().manual_seed(41)
    y0 = torch.rand(1, 3, 128, 128, generator=g) * 2 - 1
    z_y = s.base_diffusion.encode_first_stage(y0.cuda(), s.autoencoder, up_sample=True)
    mx, mn = _report("sampler: z_y (bicubic x4 + encode, 512x512)", z_y,
                     vo.vq_encode(vo.bicubic_upsample(y0, 4), random_vq_state_dict(vcfg, 0), vcfg))
    assert mx <= TOL_MAX and mn <= TOL_MEAN
    out = s._process(y0.cuda())
    assert out.shape == (1, 3, 512, 512) and torch.isfinite(out).all()
    assert out.min().item() >= 0.0 and out.max().item() <= 1.0


def test_plan_cache_is_bounded_and_results_do_not_change():
    import gc
    import weakref
    cfg, m = _vq("tiny")
    g = torch.Generator(device="cuda").manual_seed(6)
    xs = [torch.rand(1, 3, s, s, device="cuda", generator=g) * 2 - 1 for s in (64, 96, 128, 160)]
    first = [m.encode(x).clone() for x in xs]
    assert sum(1 for k in m._plans if k[0] == 0) == m.MAX_PLANS_PER_DIRECTION
    assert all(torch.equal(a, m.encode(x)) for a, x in zip(first, xs))      # evicted plans rebuilt: same results
    ref = weakref.ref(m)
    del m
    gc.collect()
    assert ref() is None                                                    # no model <-> plan reference cycle
