"""Host-side handle on one CUDA step operator (thin Python over the C-ABI).

PyTorch tensors are used as device-memory containers only: the engine receives raw
``data_ptr()`` addresses and the current CUDA stream.
"""
from __future__ import annotations

import ctypes as C
from collections import OrderedDict

import numpy as np

from . import _ffi
from .config import FCNConfig, GraphCastConfig, PanguConfig, SFNOConfig

ARENA_ALIGN = 64  # floats (256 B)


def pack_arena(weights: "OrderedDict[str, np.ndarray]"):
    """Flatten named fp32 tensors into one arena + manifest (name, offset, count)."""
    offs, total = [], 0
    for name, a in weights.items():
        offs.append(total)
        total += (a.size + ARENA_ALIGN - 1) // ARENA_ALIGN * ARENA_ALIGN
    arena = np.zeros(total, dtype=np.float32)
    manifest = (_ffi.ParamDesc * len(weights))()
    for i, ((name, a), off) in enumerate(zip(weights.items(), offs)):
        arena[off:off + a.size] = np.asarray(a, dtype=np.float32).reshape(-1)
        manifest[i].name = name.encode()
        manifest[i].offset = off
        manifest[i].count = a.size
    return arena, manifest


def _pangu_cfg_c(cfg: PanguConfig) -> _ffi.PanguConfigC:
    assert tuple(cfg.patch) == (2, 4, 4) and tuple(cfg.window) == (2, 6, 12)
    c = _ffi.PanguConfigC()
    c.nlat, c.nlon, c.n_levels, c.dim = cfg.nlat, cfg.nlon, cfg.n_levels, cfg.dim
    c.depths[:] = cfg.depths
    c.heads[:] = cfg.heads
    c.ln_eps, c.mask_value = cfg.ln_eps, cfg.mask_value
    return c


def _sfno_cfg_c(cfg: SFNOConfig) -> _ffi.SFNOConfigC:
    c = _ffi.SFNOConfigC()
    c.nlat, c.nlon, c.n_channels, c.embed = cfg.nlat, cfg.nlon, cfg.n_channels, cfg.embed
    c.layers, c.scale_factor, c.mlp_ratio, c.eps = cfg.layers, cfg.scale_factor, cfg.mlp_ratio, cfg.eps
    return c


def _graphcast_cfg_c(cfg: GraphCastConfig, graph) -> _ffi.GraphCastConfigC:
    c = _ffi.GraphCastConfigC()
    c.nlat, c.nlon, c.latent, c.layers = cfg.nlat, cfg.nlon, cfg.latent, cfg.layers
    c.n_mesh, c.n_mesh_edges, c.n_g2m_edges = graph["n_mesh"], len(graph["mesh.senders"]), len(graph["g2m.senders"])
    c.n_state, c.n_prog, c.n_static, c.dt_hours, c.ln_eps = cfg.n_state, cfg.n_prog, cfg.n_static, cfg.dt_hours, cfg.ln_eps
    return c


def _afno_cfg_c(cfg: FCNConfig) -> _ffi.AFNOConfigC:
    c = _ffi.AFNOConfigC()
    c.nlat, c.nlon, c.n_channels, c.patch, c.embed = cfg.nlat, cfg.nlon, cfg.n_channels, cfg.patch, cfg.embed
    c.depth, c.num_blocks, c.mlp_ratio = cfg.depth, cfg.num_blocks, cfg.mlp_ratio
    c.sparsity, c.hard_thresholding_fraction, c.ln_eps = cfg.sparsity, cfg.hard_thresholding_fraction, cfg.ln_eps
    return c


class StepEngine:
    """One 6-h step operator resident on one GPU."""

    def __init__(self, cfg, device: int = 0, lib: str | None = None, graph=None):
        import torch
        if not torch.cuda.is_available():
            raise _ffi.SkyError("skyrim_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.cfg = cfg
        self.device = device
        self.torch = torch
        L = self._L = _ffi.lib(lib)
        if isinstance(cfg, PanguConfig):
            kind, cc = _ffi.SKY_MODEL_PANGU6, _pangu_cfg_c(cfg)
        elif isinstance(cfg, SFNOConfig):
            kind, cc = _ffi.SKY_MODEL_SFNO73, _sfno_cfg_c(cfg)
        elif isinstance(cfg, GraphCastConfig):
            # the multimesh and the grid<->mesh edge sets are built on the host once (icomesh.py) and travel in the arena
            if graph is None:
                from .icomesh import build_graph
                graph = build_graph(cfg.nlat, cfg.nlon, cfg.mesh_levels, cfg.radius_frac)
            self.graph = graph
            kind, cc = _ffi.SKY_MODEL_GRAPHCAST, _graphcast_cfg_c(cfg, graph)
        elif isinstance(cfg, FCNConfig):
            kind, cc = _ffi.SKY_MODEL_AFNO26, _afno_cfg_c(cfg)
        else:
            raise TypeError(cfg)
        self.n_channels = cfg.n_channels
        h = C.c_void_p()
        _ffi.check(L.sky_model_create(C.byref(h), kind, C.byref(cc), C.sizeof(cc), device), "sky_model_create", L)
        self._h = h
        self._ws = None
        self._ws_batch = 0

    # -- weights ---------------------------------------------------------------------------
    def load_weights(self, weights: "OrderedDict[str, np.ndarray]"):
        if isinstance(self.cfg, GraphCastConfig) and not any(k.startswith("graph.") for k in weights):
            from .icomesh import graph_arena_entries
            weights = OrderedDict(list(weights.items()) + list(graph_arena_entries(self.graph).items()))
        arena, manifest = pack_arena(weights)
        self.load_arena(arena, manifest)

    def load_arena(self, arena, manifest):
        """``arena``: host numpy fp32 array, or a CUDA torch tensor (e.g. after a broadcast)."""
        L = self._L
        torch = self.torch
        st = torch.cuda.current_stream(self.device).cuda_stream
        if isinstance(arena, np.ndarray):
            ptr, n, on_dev = arena.ctypes.data, arena.size, 0
        else:
            assert arena.is_cuda and arena.dtype == torch.float32 and arena.is_contiguous()
            ptr, n, on_dev = arena.data_ptr(), arena.numel(), 1
        _ffi.check(L.sky_model_load_weights(self._h, ptr, n, manifest, len(manifest), on_dev, st),
                   "sky_model_load_weights", L)

    # -- stepping --------------------------------------------------------------------------
    def _workspace(self, batch: int):
        if self._ws is None or self._ws_batch < batch:
            nbytes = self._L.sky_model_workspace_bytes(self._h, batch)
            self._ws = self.torch.empty(nbytes, dtype=self.torch.uint8, device=f"cuda:{self.device}")
            self._ws_batch = batch
        return self._ws

    def step(self, x_in, x_out=None):
        """x_in: CUDA fp32 (B, C, nlat, nlon) contiguous.  Returns x_out (allocated if None).
        Asynchronous on the current stream."""
        torch = self.torch
        assert x_in.is_cuda and x_in.dtype == torch.float32 and x_in.is_contiguous() and x_in.dim() == 4
        B = x_in.shape[0]
        assert tuple(x_in.shape[1:]) == (self.n_channels, self.cfg.nlat, self.cfg.nlon), x_in.shape
        if x_out is None:
            x_out = torch.empty_like(x_in)
        ws = self._workspace(B)
        st = torch.cuda.current_stream(self.device).cuda_stream
        _ffi.check(self._L.sky_model_step(self._h, x_in.data_ptr(), x_out.data_ptr(), B, ws.data_ptr(),
                                             ws.numel(), st), "sky_model_step", self._L)
        return x_out

    def set_clock(self, when):
        """Valid time of the LAST time slice of the state the next step starts from (datetime, numpy datetime64 or unix
        seconds).  Only operators with time-dependent forcings (GraphCast) use it; they advance it themselves per step."""
        t = unix_seconds(when)
        st = self.torch.cuda.current_stream(self.device).cuda_stream
        _ffi.check(self._L.sky_model_set_clock(self._h, t, st), "sky_model_set_clock", self._L)

    def toa_radiation(self, when, out=None):
        """(nlat, nlon) CUDA fp32: the toa-radiation forcing channel ("tp06") at time ``when``."""
        torch = self.torch
        if out is None:
            out = torch.empty((self.cfg.nlat, self.cfg.nlon), dtype=torch.float32, device=f"cuda:{self.device}")
        st = torch.cuda.current_stream(self.device).cuda_stream
        _ffi.check(self._L.sky_toa_radiation(out.data_ptr(), self.cfg.nlat, self.cfg.nlon, unix_seconds(when), st),
                   "sky_toa_radiation", self._L)
        return out

    def debug_tensor(self, what: str, shape, batch: int = 1):
        torch = self.torch
        out = torch.empty(shape, dtype=torch.float32, device=f"cuda:{self.device}")
        st = torch.cuda.current_stream(self.device).cuda_stream
        _ffi.check(self._L.sky_model_debug_copy(self._h, what.encode(), out.data_ptr(), out.numel(),
                                                   self._workspace(batch).data_ptr(), batch, st), "debug_copy", self._L)
        return out

    RANGE_SLOTS = ("token_images", "qkv", "attention_out", "resampled_images", "pixel_images", "hidden_images",
                   "spectral_images", "unused")
    FP16_LIMIT = 3.0e4

    def step_guarded(self, x_in, x_out=None, limit: float | None = None):
        """One step with the fp16-range guard on: the engine scans every fp16 operand image it produces (the tensor cores
        take 5-exponent-bit operands) and this call raises if any |value| exceeds ``limit`` (default 3e4) or is not finite.
        Meant for the FIRST step of a rollout with real checkpoints (synthetic weights keep every activation O(1)); the
        guarded step runs with plain launches and a few extra reduction kernels.  Returns (x_out, {class: max |value|})."""
        limit = self.FP16_LIMIT if limit is None else limit
        self.debug_set("range_guard", 1)
        try:
            y = self.step(x_in, x_out)
            r = self.torch.empty(8, dtype=self.torch.float32, device=f"cuda:{self.device}")
            st = self.torch.cuda.current_stream(self.device).cuda_stream
            _ffi.check(self._L.sky_model_debug_copy(self._h, b"range", r.data_ptr(), 8, self._workspace(x_in.shape[0]).data_ptr(),
                                                    x_in.shape[0], st), "debug_copy(range)", self._L)
            vals = r.cpu().tolist()
        finally:
            self.debug_set("range_guard", 0)
        ranges = {n: v for n, v in zip(self.RANGE_SLOTS, vals) if v != 0.0}
        bad = {n: v for n, v in ranges.items() if not (v <= limit)}
        if bad:
            raise _ffi.SkyError(f"fp16 operand range exceeded (limit {limit:g}): {bad}; this checkpoint needs operand scaling "
                                f"the engine does not implement")
        return y, ranges

    def debug_set(self, key: str, value: int):
        """test taps (never environment variables): e.g. ``debug_set("stop_after", 3)``"""
        _ffi.check(self._L.sky_model_debug_set(self._h, key.encode(), int(value)), "debug_set", self._L)

    # -- per-kernel-family device timing (CUDA events inside the library) -------------------
    @staticmethod
    def profile_tags():
        L = _ffi.lib()
        return [L.sky_profile_tag_name(i).decode() for i in range(L.sky_profile_tag_count())]

    def profile_begin(self, tags=None):
        names = self.profile_tags()
        mask = 0
        for i, n in enumerate(names):
            if tags is None or n in tags:
                mask |= 1 << i
        _ffi.check(self._L.sky_model_profile_begin(self._h, mask), "profile_begin", self._L)

    def profile_end(self):
        """-> {family: (total_ms, launches)} for the families that ran since profile_begin."""
        names = self.profile_tags()
        ms = (C.c_double * len(names))()
        cnt = (C.c_uint64 * len(names))()
        _ffi.check(self._L.sky_model_profile_end(self._h, ms, cnt, len(names)), "profile_end", self._L)
        return {n: (ms[i], int(cnt[i])) for i, n in enumerate(names) if cnt[i]}

    def close(self):
        if getattr(self, "_h", None):
            self._L.sky_model_destroy(self._h)
            self._h = None
            self._ws = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def perturb_ic(x, sigma_c, amp: float, seed: int, member0: int = 0):
    """In-place Gaussian perturbation of (M, C, nlat, nlon) CUDA fp32 members (K11)."""
    import torch
    assert x.is_cuda and x.dtype == torch.float32 and x.is_contiguous() and x.dim() == 4
    M, Cn = x.shape[0], x.shape[1]
    plane = x.shape[2] * x.shape[3]
    assert sigma_c.is_cuda and sigma_c.numel() == Cn
    st = torch.cuda.current_stream(x.device).cuda_stream
    _ffi.check(_ffi.lib().sky_perturb_ic(x.data_ptr(), sigma_c.data_ptr(), float(amp), int(seed), int(member0), M,
                                         Cn, plane, st), "sky_perturb_ic")
    return x


def unix_seconds(when) -> float:
    """datetime (naive = UTC) / numpy datetime64 / number -> unix seconds"""
    import datetime as _dt
    if isinstance(when, (int, float)):
        return float(when)
    if isinstance(when, np.datetime64):
        return float((when - np.datetime64("1970-01-01T00:00:00")) / np.timedelta64(1, "s"))
    if isinstance(when, _dt.datetime):
        if when.tzinfo is None:
            when = when.replace(tzinfo=_dt.timezone.utc)
        return when.timestamp()
    raise TypeError(type(when))


def launch_count() -> int:
    return int(_ffi.lib().sky_launch_count())
