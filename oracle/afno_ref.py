"""ORACLE — test infrastructure, not product code.

CPU fp32 / fp64 restatement of the FourCastNet v1 (AFNO) 6-hour forward that the reference reaches through
earth2mip's ``networks.fcn`` package (/root/reference/skyrim/core/models/fourcastnet.py:build_model) and steps
through earth2mip's ``Inference`` wrapper: normalise, x = AFNONet(x), de-normalise (utils.py:34-40).

PARITY UNPINNED: earth2mip and NVlabs FourCastNet are not vendored under /root/reference; the network below follows
SURVEY.md Appendix D.  The filter is written the way upstream writes it: ``rfft2`` over the token grid, the
block-diagonal complex MLP on the slice ``[total - kept : total + kept, :kept]`` only, softshrink, ``irfft2``.

Only tests/, __graft_entry__.smoke() and tools/ may import this module.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

from skyrim_b200.config import FCNConfig


class FCNRef:
    """``emulate="fp16"`` rounds the operands of the four dense contractions (patch embedding, fc1, fc2, head) to
    half precision, as the engine's tensor-core GEMMs do; the spectral filter stays in the oracle's dtype, as the
    engine's fp32 filter kernels do."""

    def __init__(self, cfg: FCNConfig, weights, dtype=torch.float32, emulate: str | None = None, device="cpu"):
        self.cfg, self.dtype, self.emulate, self.device = cfg, dtype, emulate, device
        self.w = {k: torch.as_tensor(np.asarray(v)).to(device=device, dtype=dtype) for k, v in weights.items()}

    def _q(self, t):
        return t.half().to(self.dtype) if self.emulate == "fp16" else t

    def _linear(self, x, w, b=None):
        y = self._q(x) @ self._q(w).T
        return y if b is None else y + b

    def filter(self, u):
        """AFNO2D on (B, h, w, E) tokens; returns the filter output WITHOUT its own skip (upstream adds the input)"""
        cfg = self.cfg
        B, h, w, E = u.shape
        nb, bs = cfg.num_blocks, cfg.block_size
        X = torch.fft.rfft2(u, dim=(1, 2), norm="ortho").reshape(B, h, w // 2 + 1, nb, bs)
        total = h // 2 + 1
        kept = int(total * cfg.hard_thresholding_fraction)
        sl = (slice(None), slice(total - kept, total + kept), slice(None, kept))
        w1, b1, w2, b2 = (self.w[self._blk + k] for k in ("filter.w1", "filter.b1", "filter.w2", "filter.b2"))
        o1r = torch.zeros(X.shape, dtype=u.dtype, device=u.device)
        o1i, o2r, o2i = torch.zeros_like(o1r), torch.zeros_like(o1r), torch.zeros_like(o1r)
        xr, xi = X.real[sl], X.imag[sl]
        o1r[sl] = F.relu(torch.einsum("...bi,bio->...bo", xr, w1[0]) - torch.einsum("...bi,bio->...bo", xi, w1[1]) + b1[0])
        o1i[sl] = F.relu(torch.einsum("...bi,bio->...bo", xi, w1[0]) + torch.einsum("...bi,bio->...bo", xr, w1[1]) + b1[1])
        o2r[sl] = (torch.einsum("...bi,bio->...bo", o1r[sl], w2[0]) - torch.einsum("...bi,bio->...bo", o1i[sl], w2[1])
                   + b2[0])
        o2i[sl] = (torch.einsum("...bi,bio->...bo", o1i[sl], w2[0]) + torch.einsum("...bi,bio->...bo", o1r[sl], w2[1])
                   + b2[1])
        Z = F.softshrink(torch.stack([o2r, o2i], dim=-1), lambd=cfg.sparsity)
        self.last_modes = Z[sl]   # the processed modes after softshrink (activity statistics)
        Z = torch.view_as_complex(Z.contiguous()).reshape(B, h, w // 2 + 1, E)
        return torch.fft.irfft2(Z, s=(h, w), dim=(1, 2), norm="ortho")

    def forward_norm(self, xn, taps: dict | None = None):
        """AFNONet on a normalised state (B, C, nlat, nlon) -> normalised prediction"""
        cfg = self.cfg
        B = xn.shape[0]
        p, h, w, E, C = cfg.patch, cfg.h, cfg.w, cfg.embed, cfg.n_channels
        patches = xn.reshape(B, C, h, p, w, p).permute(0, 2, 4, 1, 3, 5).reshape(B, h * w, C * p * p)
        x = self._linear(patches, self.w["patch_embed.proj.weight"].reshape(E, -1), self.w["patch_embed.proj.bias"])
        x = (x + self.w["pos_embed"]).reshape(B, h, w, E)
        if taps is not None:
            taps["embed"] = x.clone()
        for i in range(cfg.depth):
            self._blk = b = f"blocks.{i}."
            r = x
            u = F.layer_norm(x, (E,), self.w[b + "norm1.weight"], self.w[b + "norm1.bias"], cfg.ln_eps)
            x = self.filter(u) + u + r
            if taps is not None:
                taps[f"filter{i}"] = x.clone()
            v = F.layer_norm(x, (E,), self.w[b + "norm2.weight"], self.w[b + "norm2.bias"], cfg.ln_eps)
            hid = F.gelu(self._linear(v, self.w[b + "mlp.fc1.weight"], self.w[b + "mlp.fc1.bias"]))
            x = x + self._linear(hid, self.w[b + "mlp.fc2.weight"], self.w[b + "mlp.fc2.bias"])
            if taps is not None:
                taps[f"block{i}"] = x.clone()
        y = self._linear(x, self.w["head.weight"])                     # (B, h, w, (p1 p2 c))
        return y.reshape(B, h, w, p, p, C).permute(0, 5, 1, 3, 2, 4).reshape(B, C, h * p, w * p)

    @torch.no_grad()
    def step(self, x, taps: dict | None = None):
        """(C, nlat, nlon) or (B, C, nlat, nlon) physical state -> the state 6 h later"""
        x = torch.as_tensor(np.asarray(x) if not torch.is_tensor(x) else x).to(device=self.device, dtype=self.dtype)
        single = x.dim() == 3
        if single:
            x = x[None]
        mu = self.w["norm.mean"][None, :, None, None]
        sd = self.w["norm.std"][None, :, None, None]
        y = self.forward_norm((x - mu) / sd, taps) * sd + mu
        return y[0] if single else y

