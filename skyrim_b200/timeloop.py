"""TimeLoop-shaped step drivers over the CUDA engines.

The reference consumes its back-ends through earth2mip's ``TimeLoop`` protocol
(/root/reference/skyrim/core/models/utils.py:20,25-29,34,45-47):
``model(time, x) -> Iterator[(time, Tensor[B,C,H,W], restart)]`` whose FIRST yield is the
initial condition itself, plus the attributes ``n_history_levels``, ``device``,
``in_channel_names``, ``out_channel_names``, ``grid.lat``, ``grid.lon``, ``time_step``.
These classes keep that protocol so ``run_basic_inference`` can drive them unchanged, with the
state resident on the GPU between steps (the reference round-trips it through the host every
step, utils.py:24-31,37).
"""
from __future__ import annotations

import datetime
from dataclasses import dataclass

import numpy as np

from .config import FCN_CHANNELS, FCNV2_CHANNELS, FCNConfig, GRAPHCAST_CHANNELS, PANGU_CHANNELS


@dataclass
class Grid:
    lat: list
    lon: list

    @property
    def shape(self):
        return (len(self.lat), len(self.lon))


def equiangular_grid(nlat: int = 721, nlon: int = 1440) -> Grid:
    # pangu.py:33-36 docstring: lat 90 .. -90 (721), lon 0 .. 359.75 (1440)
    return Grid(lat=np.linspace(90.0, -90.0, nlat).tolist(), lon=(np.arange(nlon) * (360.0 / nlon)).tolist())


def poleless_grid(nlat: int = 720, nlon: int = 1440) -> Grid:
    """FourCastNet v1's grid (fourcastnet.py:16-19): lat = 90 - 0.25 i for i < 720 (the south-pole row is dropped),
    lon 0 .. 359.75; at other sizes the spacing is 180 / nlat so that the same rows of the 721-row grid are kept."""
    d = 180.0 / nlat
    return Grid(lat=(90.0 - d * np.arange(nlat)).tolist(), lon=(np.arange(nlon) * (360.0 / nlon)).tolist())


class _EngineTimeLoop:
    n_history_levels = 1
    time_step = datetime.timedelta(hours=6)
    channel_names: list = []

    def __init__(self, engine):
        import torch
        self.torch = torch
        self.engine = engine
        self.device = torch.device("cuda", engine.device)
        self.in_channel_names = list(self.channel_names)
        self.out_channel_names = list(self.channel_names)
        cfg = engine.cfg
        self.grid = poleless_grid(cfg.nlat, cfg.nlon) if isinstance(cfg, FCNConfig) else equiangular_grid(cfg.nlat, cfg.nlon)
        self._dev_in = None
        self._dev_out = None
        self._host_out = None
        # real checkpoints (SKYRIM_B200_WEIGHTS*): the first step of every rollout runs with the fp16-range guard
        self.guard_first_step = False
        self.last_ranges = None

    # earth2mip TimeLoops accept .to(device); ours is pinned to its GPU (ensemble.py:34,46 calls these)
    def to(self, device):
        return self

    def cuda(self):
        return self

    def __call__(self, time, x, restart=None):
        """x: (B, n_history_levels, C, H, W) tensor (host or device).  Yields (time, state, None):
        first the initial condition, then one 6-h step per iteration, state resident in HBM."""
        torch = self.torch
        assert x.dim() == 5 and x.shape[1] == self.n_history_levels, x.shape
        cur = x[:, -1].to(self.device, dtype=torch.float32, non_blocking=True).contiguous()
        yield time, cur.clone(), None
        nxt = torch.empty_like(cur)
        first = self.guard_first_step
        while True:
            if first:
                _, self.last_ranges = self.engine.step_guarded(cur, nxt)
                first = False
            else:
                self.engine.step(cur, nxt)
            time = time + self.time_step
            yield time, nxt, None
            cur, nxt = nxt, torch.empty_like(cur)  # the yielded tensor stays valid for the caller

    def iter_host(self, time, x, n_steps: int):
        """Rollout with every state delivered to the HOST: yields (time, pinned fp32 tensor (B, C, H, W)) for the initial
        condition and then for each of ``n_steps`` 6-h steps.  The state stays in HBM; the device->host copy of step n runs on
        a copy stream while step n+1 computes (a ring of three device states: n+1 is written while n is read by both the
        copy and the step).  A yielded host tensor is valid until the second next() after it (ring of two).
        ``GlobalModel.rollout(save=True)`` consumes this instead of ``.cpu()`` per step (base.py:131-141 in the reference)."""
        torch = self.torch
        assert x.dim() == 5 and x.shape[1] == self.n_history_levels, x.shape
        main = torch.cuda.current_stream(self.device)
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(self.device)
        shape = (x.shape[0],) + tuple(x.shape[2:])
        if getattr(self, "_ring", None) is None or tuple(self._ring[0].shape) != shape:
            self._ring = [torch.empty(shape, dtype=torch.float32, device=self.device) for _ in range(3)]
            self._host_ring = [torch.empty(shape, dtype=torch.float32).pin_memory() for _ in range(2)]
        ring, host = self._ring, self._host_ring
        ring[0].copy_(x[:, -1].to(dtype=torch.float32), non_blocking=True)
        done = [torch.cuda.Event() for _ in range(3)]     # state i is complete on the main stream
        copied = torch.cuda.Event()
        done[0].record(main)
        if n_steps > 0:
            if self.guard_first_step:
                _, self.last_ranges = self.engine.step_guarded(ring[0], ring[1])
            else:
                self.engine.step(ring[0], ring[1])
            done[1].record(main)
        for n in range(n_steps + 1):
            if 0 < n < n_steps:   # launch step n+1 before waiting for the copy of step n
                self.engine.step(ring[n % 3], ring[(n + 1) % 3]); done[(n + 1) % 3].record(main)
            self._copy_stream.wait_event(done[n % 3])
            with torch.cuda.stream(self._copy_stream):
                host[n % 2].copy_(ring[n % 3], non_blocking=True)
                copied.record(self._copy_stream)
            copied.synchronize()   # also orders the overwrite of ring[n % 3] (three steps from now) after this copy
            yield time, host[n % 2]
            time = time + self.time_step

    def step_host(self, x_host):
        """One step with HOST (pinned) input and HOST (pinned) output — the end-to-end unit that
        bench.py's ``e2e`` times: H2D of the state, sky_model_step, D2H of the result."""
        torch = self.torch
        if self._dev_in is None or self._dev_in.shape != x_host.shape:
            self._dev_in = torch.empty(x_host.shape, dtype=torch.float32, device=self.device)
            self._dev_out = torch.empty_like(self._dev_in)
            self._host_out = [torch.empty(x_host.shape, dtype=torch.float32).pin_memory() for _ in range(2)]
            self._flip = 0
        self._dev_in.copy_(x_host, non_blocking=True)
        self.engine.step(self._dev_in, self._dev_out)
        out = self._host_out[self._flip]
        self._flip ^= 1
        out.copy_(self._dev_out, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        return out


class PanguTimeLoop(_EngineTimeLoop):
    channel_names = PANGU_CHANNELS


class SFNOTimeLoop(_EngineTimeLoop):
    channel_names = FCNV2_CHANNELS


class FCNTimeLoop(_EngineTimeLoop):
    channel_names = FCN_CHANNELS


class GraphcastStepper:
    """The stepper protocol the reference drives for GraphCast (/root/reference/skyrim/core/models/graphcast.py:102-118):
    ``initialize(x, time) -> state`` and ``step(state) -> (state, output)`` with ``state = (time, fields, rng)``.
    Upstream ``fields`` is an xarray Dataset with two time slices; here it is a CUDA tensor (B, 2, 83, nlat, nlon) holding
    the same two slices in the reference's channel order (config.GRAPHCAST_CHANNELS), resident in HBM between steps."""

    def __init__(self, loop):
        self.loop = loop

    def initialize(self, x, time):
        torch = self.loop.torch
        assert x.dim() == 5 and x.shape[1] == 2 and x.shape[2] == len(self.loop.channel_names), x.shape
        fields = x.to(self.loop.device, dtype=torch.float32).contiguous()
        self.loop.engine.set_clock(time)
        return (time, fields, None)

    def step(self, state):
        time, fields, rng = state
        eng, torch = self.loop.engine, self.loop.torch
        B = fields.shape[0]
        nxt = torch.empty_like(fields)
        eng.step(fields.view(B, -1, *fields.shape[-2:]), nxt.view(B, -1, *fields.shape[-2:]))
        time = time + self.loop.time_step
        return (time, nxt, rng), nxt[:, -1]


class GraphcastTimeLoop(_EngineTimeLoop):
    """TimeLoop over the GraphCast engine: two history levels (t-6h, t); the first yield is the initial condition's last
    slice, then one 6-h step per iteration.  The engine keeps the valid time on the device (time-dependent forcings)."""
    n_history_levels = 2
    channel_names = GRAPHCAST_CHANNELS

    def __init__(self, engine):
        super().__init__(engine)
        self.stepper = GraphcastStepper(self)

    def fill_forcing(self, x, time):
        """write the toa-radiation forcing channel ("tp06") of both slices of an initial condition (B, 2, 83, H, W) in place"""
        from .engine import unix_seconds
        t = unix_seconds(time)
        for k, dt in ((0, -self.time_step.total_seconds()), (1, 0.0)):
            x[:, k, -1] = self.engine.toa_radiation(t + dt)
        return x

    def __call__(self, time, x, restart=None):
        state = self.stepper.initialize(x, time)
        yield time, state[1][:, -1].clone(), None
        while True:
            state, out = self.stepper.step(state)
            yield state[0], out, None

    def iter_host(self, time, x, n_steps: int):
        for n, (t, out, _) in enumerate(self(time, x)):
            yield t, out.cpu()
            if n == n_steps:
                return

    def step_host(self, x_host):
        """One step with HOST input and HOST output (bench.py ``e2e``).  ``x_host``: pinned (B, 2*83, H, W) tensor, or the
        pair of pinned (B, 83, H, W) time slices a previous call returned.  Both slices are uploaded every step (they are the
        step's inputs); only the NEW slice comes back (the step's result, what ``stepper.step`` returns as ``output``): the
        returned pair is (old slice 1, new slice), host buffers rotating in a ring of three, so chaining copies nothing on
        the host.  Bytes per step: H2D 2 x 83 planes, D2H 83 planes."""
        torch = self.torch
        ns = len(self.channel_names)
        if isinstance(x_host, (tuple, list)):
            s0, s1 = x_host
        else:
            s0, s1 = x_host[:, :ns], x_host[:, ns:]
        B, shape = s1.shape[0], tuple(s1.shape)
        if self._dev_in is None or self._dev_in.shape[0] != B:
            self._dev_in = torch.empty((B, 2 * ns) + shape[2:], dtype=torch.float32, device=self.device)
            self._dev_out = torch.empty_like(self._dev_in)
            self._host_ring = [torch.empty(shape, dtype=torch.float32).pin_memory() for _ in range(3)]
            self._flip = 0
        self._dev_in[:, :ns].copy_(s0, non_blocking=True)
        self._dev_in[:, ns:].copy_(s1, non_blocking=True)
        self.engine.step(self._dev_in, self._dev_out)
        # a free ring slot: not one of the two buffers the caller still holds as the current state
        free = [h for h in self._host_ring if h.data_ptr() not in (s0.data_ptr(), s1.data_ptr())]
        new = free[self._flip % len(free)]
        self._flip += 1
        new.copy_(self._dev_out[:, ns:], non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        return (s1, new)
