"""Generate the 512x512 f4 VQ-GAN fixture (T = 128 x 128 = 16384 bottleneck tokens) by running the UNMODIFIED
reference on the CPU (build container only):

    python -m oracle.make_golden_vq_large

Same recipe as oracle/make_golden_vq.py (the reference's own ``VQModelTorch`` with the synthetic weights of
``resshift_b200.vq_arch.random_vq_state_dict``, loaded strictly), but the inputs are not stored: ``x`` and ``z`` are
re-drawn from the recorded ``seed`` by ``draw_inputs`` (CPU torch generator), and of the two decoded 512x512 images only
``N_SAMPLES`` values at seeded positions (``sample_positions``) are kept, which keeps the file under 1 MB.
The vanilla ``AttnBlock`` materialises the 16384 x 16384 score matrix (1 GiB in fp32): fine on the host.
"""
from __future__ import annotations

import os
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
REF = Path(os.environ.get("RESSHIFT_REFERENCE", "/root/reference"))
GOLD = ROOT / "tests" / "golden"
SEED = 97531
N_SAMPLES = 65536


def draw_inputs(seed: int, batch: int, hw: int, embed_dim: int, downscale: int):
    """The fixture's image x [batch, 3, hw, hw] in [-1, 1) and latent z [batch, embed_dim, hw/f, hw/f]."""
    g = torch.Generator().manual_seed(int(seed))
    x = torch.rand(batch, 3, hw, hw, generator=g) * 2 - 1
    lat = hw // downscale
    z = torch.randn(batch, embed_dim, lat, lat, generator=g) * 0.6
    return x, z


def sample_positions(seed: int, numel: int, k: int = N_SAMPLES) -> torch.Tensor:
    """Sorted flat indices of the recorded decoder values (the same positions for ``dec`` and ``dec_nq``)."""
    g = torch.Generator().manual_seed(int(seed) + 1)
    return torch.randperm(numel, generator=g)[:k].sort().values


def main():
    sys.path.insert(0, str(ROOT / "oracle" / "_shims"))
    sys.path.insert(0, str(REF))
    sys.path.insert(0, str(ROOT))
    from ldm.models.autoencoder import VQModelTorch          # noqa: E402  (reference)
    from resshift_b200.vq_arch import random_vq_state_dict, vq_preset

    torch.set_grad_enabled(False)
    cfg = vq_preset("f4")
    model = VQModelTorch(**cfg.to_kwargs()).eval()
    sd = random_vq_state_dict(cfg, 0)
    model.load_state_dict(sd, strict=True)
    batch, hw = 1, 512
    x, z = draw_inputs(SEED, batch, hw, cfg.embed_dim, cfg.downscale)
    lat = hw // cfg.downscale
    enc = model.encode(x)
    _, _, info = model.quantize(z)
    dec = model.decode(z)
    dec_nq = model.decode(z, force_not_quantize=True)
    idx = info[2].view(batch, lat, lat)
    emb = sd["quantize.embedding.weight"]
    flat = z.permute(0, 2, 3, 1).reshape(-1, cfg.embed_dim)
    d = (flat ** 2).sum(1, keepdim=True) + (emb ** 2).sum(1) - 2 * flat @ emb.t()
    top2 = torch.topk(d, 2, dim=1, largest=False).values
    pos = sample_positions(SEED, dec.numel())
    np.savez_compressed(GOLD / "vq_f4_512.npz", seed=np.int64(SEED), enc=enc.numpy(),
                        dec_s=dec.reshape(-1)[pos].numpy(), dec_nq_s=dec_nq.reshape(-1)[pos].numpy(),
                        idx=idx.numpy().astype(np.int32), margin=(top2[:, 1] - top2[:, 0]).view(batch, lat, lat).numpy())
    print("vq_f4_512.npz", "enc std %.3f" % enc.std().item(), "dec std %.3f" % dec.std().item(), "codes used", idx.unique().numel())


if __name__ == "__main__":
    main()
