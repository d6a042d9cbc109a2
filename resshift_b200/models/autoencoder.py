"""``VQModelTorch`` — same constructor, ``state_dict`` and call surface as the reference's
``ldm.models.autoencoder.VQModelTorch`` (reference ldm/models/autoencoder.py:12-47), the VQ-GAN first stage around the
denoising loop (SURVEY.md §8f rank 1), executed by the sm_100a kernels of ``librs_b200.so``: the same tcgen05
implicit-GEMM conv / GroupNorm kernels as the denoiser, the 4096-token single-head attention as tensor-core GEMMs +
a row softmax, nearest-codebook quantisation as one small kernel (csrc/vq.inc).

``encode(x)`` / ``decode(h, force_not_quantize=False)`` / ``forward`` take and return fp32 NCHW CUDA tensors.  PyTorch
owns every allocation; there is no eager / CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from collections import OrderedDict
from typing import Optional, Tuple

import torch
import torch.nn as nn

from .. import _lib
from ..vq_arch import VQConfig, random_vq_state_dict, vq_param_spec


class _Node(nn.Module):
    """Anonymous container; only there so that ``state_dict`` keys match the reference's."""


class VQModelTorch(nn.Module):
    def __init__(self, ddconfig, n_embed, embed_dim, remap=None, sane_index_shape=False):
        super().__init__()
        if remap is not None:
            raise NotImplementedError("codebook remapping is not used by any shipped config")
        dd = dict(ddconfig)
        self.cfg = VQConfig(embed_dim=embed_dim, n_embed=n_embed, z_channels=dd["z_channels"], resolution=dd.get("resolution", 256),
                            in_channels=dd.get("in_channels", 3), out_ch=dd.get("out_ch", 3), ch=dd["ch"],
                            ch_mult=tuple(dd["ch_mult"]), num_res_blocks=dd["num_res_blocks"],
                            attn_resolutions=tuple(dd.get("attn_resolutions", ())), dropout=dd.get("dropout", 0.0),
                            double_z=dd.get("double_z", False))
        self.sane_index_shape = sane_index_shape
        self._spec = vq_param_spec(self.cfg)
        init = random_vq_state_dict(self.cfg, seed=0)
        for name, shape, role in self._spec:
            *path, leaf = name.split(".")
            node = self
            for part in path:
                if not hasattr(node, part):
                    node.add_module(part, _Node())
                node = getattr(node, part)
            node.register_parameter(leaf, nn.Parameter(init[name]))
        self._engine = None
        self._arena: Optional[torch.Tensor] = None
        self._packed_versions: Optional[Tuple] = None
        # (direction, batch, H, W) -> plan, least recently used first; at most MAX_PLANS_PER_DIRECTION per direction (a
        # plan owns its workspace: gigabytes at 2048x2048, and folder inference meets one padded size per image)
        self._plans: "OrderedDict[Tuple[int, int, int, int], _VQPlan]" = OrderedDict()
        self.last_indices: Optional[torch.Tensor] = None

    # ------------------------------------------------------------------ native plumbing
    def _ensure_engine(self, device: torch.device):
        if device.type != "cuda":
            raise RuntimeError("resshift_b200.VQModelTorch runs on CUDA only (no CPU fallback); call .cuda() first")
        if self._engine is None:
            h = C.c_void_p()
            cfgc = _lib.make_vq_config(self.cfg)
            _lib.check(_lib.lib.rs_vq_create(C.byref(cfgc), C.byref(h)))
            self._engine = h
            n = _lib.lib.rs_unet_param_count(h)
            theirs = []
            buf = C.create_string_buffer(256)
            shape = (C.c_int32 * 4)()
            nd, isb = C.c_int32(), C.c_int32()
            for i in range(n):
                _lib.check(_lib.lib.rs_unet_param_info(h, i, buf, 256, shape, C.byref(nd), C.byref(isb)))
                theirs.append(buf.value.decode())
            if sorted(theirs) != sorted(name for name, _, _ in self._spec):
                raise _lib.RsError("parameter inventory of librs_b200 does not match resshift_b200.vq_arch")
        if self._arena is None or self._arena.device != device:
            nbytes = _lib.lib.rs_unet_arena_bytes(self._engine)
            self._arena = torch.zeros(nbytes + 256, dtype=torch.uint8, device=device)
            self._arena_ptr = (self._arena.data_ptr() + 255) // 256 * 256
            _lib.check(_lib.lib.rs_unet_set_arena(self._engine, self._arena_ptr))
            self._packed_versions = None
            self._drop_plans()
        return self._engine

    def pack_weights(self, force: bool = False):
        params = dict(self.named_parameters())
        self._ensure_engine(next(iter(params.values())).device)      # (a no-op once the engine and its arena exist)
        versions = tuple((p._version, p.data_ptr()) for p in params.values())
        if not force and versions == self._packed_versions:
            return
        stream = _lib.current_stream()
        for name, p in params.items():
            if p.device.type != "cuda":
                raise RuntimeError(f"parameter {name} is not on a CUDA device")
            src = p.detach()
            if src.dtype != torch.float32 or not src.is_contiguous():
                src = src.float().contiguous()
            _lib.check(_lib.lib.rs_unet_load_param(self._engine, name.encode(), src.data_ptr(), stream))
            del src
        torch.cuda.current_stream().synchronize()
        self._packed_versions = versions

    MAX_PLANS_PER_DIRECTION = 2

    def _drop_plans(self):
        for p in self._plans.values():
            p.close()
        self._plans.clear()

    def plan(self, which: int, batch: int, image_h: int, image_w: int) -> "_VQPlan":
        device = next(self.parameters()).device
        self._ensure_engine(device)
        self.pack_weights()
        key = (which, batch, image_h, image_w)
        plan = self._plans.pop(key, None)
        if plan is None:
            same = [k for k in self._plans if k[0] == which]
            while len(same) >= self.MAX_PLANS_PER_DIRECTION:
                self._plans.pop(same.pop(0)).close()
            plan = _VQPlan(self._engine, which, batch, image_h, image_w, device)
        self._plans[key] = plan
        return plan

    # ------------------------------------------------------------------ reference call surface
    @torch.no_grad()
    def encode(self, x):
        """x [B, 3, H, W] -> h [B, embed_dim, H/f, W/f] (reference autoencoder.py:28-31)."""
        if x.device.type != "cuda":
            raise RuntimeError("resshift_b200.VQModelTorch.encode needs CUDA tensors (no CPU fallback)")
        b, c, hh, ww = x.shape
        if c != self.cfg.in_channels:
            raise ValueError(f"expected {self.cfg.in_channels} input channels, got {c}")
        f = self.cfg.downscale
        plan = self.plan(0, b, hh, ww)
        xf = x.detach().float().contiguous()
        out = torch.empty(b, self.cfg.embed_dim, hh // f, ww // f, dtype=torch.float32, device=x.device)
        _lib.check(_lib.lib.rs_vq_encode(plan.handle, xf.data_ptr(), out.data_ptr(), _lib.current_stream()))
        return out

    @torch.no_grad()
    def decode(self, h, force_not_quantize=False):
        """h [B, embed_dim, h, w] -> image [B, 3, h*f, w*f] (reference autoencoder.py:33-40); the code indices of the
        last call stay available as ``self.last_indices`` ([B, h, w] int32, -1 when not quantised)."""
        if h.device.type != "cuda":
            raise RuntimeError("resshift_b200.VQModelTorch.decode needs CUDA tensors (no CPU fallback)")
        b, c, lh, lw = h.shape
        if c != self.cfg.embed_dim:
            raise ValueError(f"expected {self.cfg.embed_dim} latent channels, got {c}")
        f = self.cfg.downscale
        plan = self.plan(1, b, lh * f, lw * f)
        hf = h.detach().float().contiguous()
        out = torch.empty(b, self.cfg.out_ch, lh * f, lw * f, dtype=torch.float32, device=h.device)
        idx = torch.empty(b, lh, lw, dtype=torch.int32, device=h.device)
        _lib.check(_lib.lib.rs_vq_decode(plan.handle, hf.data_ptr(), out.data_ptr(), idx.data_ptr(), int(bool(force_not_quantize)),
                                         _lib.current_stream()))
        self.last_indices = idx
        return out

    def forward(self, input, force_not_quantize=False):
        return self.decode(self.encode(input), force_not_quantize)

    def __del__(self):
        try:
            self._drop_plans()
            if self._engine is not None:
                _lib.lib.rs_unet_destroy(self._engine)
        except Exception:
            pass


class _VQPlan:
    """VQ-GAN engine bound to (encode | decode, batch, image H, image W): owns the workspace and the native plan.  It keeps
    no reference to its model (the model's plan cache holds the plans; ``close`` runs before the engine is destroyed)."""

    def __init__(self, engine, which: int, batch: int, image_h: int, image_w: int, device):
        h = C.c_void_p()
        _lib.check(_lib.lib.rs_vq_plan_create(engine, batch, image_h, image_w, which, C.byref(h)))
        self.handle = h
        nbytes = _lib.lib.rs_plan_workspace_bytes(h)
        self.workspace = torch.empty(nbytes + 256, dtype=torch.uint8, device=device)
        self.workspace_ptr = (self.workspace.data_ptr() + 255) // 256 * 256
        _lib.check(_lib.lib.rs_plan_bind(h, self.workspace_ptr))
        self.launches = _lib.lib.rs_plan_num_launches(h)

    def close(self):
        """Destroy the native plan and release the workspace (work already queued on the stream keeps it alive in torch's
        stream-ordered allocator)."""
        if self.handle is not None:
            _lib.lib.rs_plan_destroy(self.handle)
            self.handle = None
            self.workspace = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
