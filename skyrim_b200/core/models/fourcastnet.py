"""FourcastnetModel — mirrors /root/reference/skyrim/core/models/fourcastnet.py (FourCastNet v1, AFNO backbone)."""
from __future__ import annotations

import numpy as np

from ...config import FCN_CHANNELS, FCNConfig, fcn_full
from .base import GlobalModel, SyntheticDataSource, xr

CHANNELS = FCN_CHANNELS


def crop_to_grid(da, nlat: int):
    """a 721-row field loses its last (south-pole) row; a field with the model's row count is returned as is"""
    n = da.sizes["lat"] if hasattr(da, "sizes") else np.shape(da)[-2]
    if n == nlat + 1:
        return da.isel(lat=slice(0, nlat)) if hasattr(da, "isel") else da[..., :nlat, :]
    if n != nlat:
        raise ValueError(f"initial condition has {n} latitude rows; FourCastNet takes {nlat} or {nlat + 1}")
    return da


class _CroppedSource:
    """Initial conditions on the 721-row grid (or already on the model's grid) -> the model's pole-less grid: a source
    one row taller than the model loses its last (south-pole) row, a source of the model's height is used as is."""

    def __init__(self, source, nlat: int):
        self.source, self.nlat = source, nlat

    def __getitem__(self, t):
        return crop_to_grid(self.source[t], self.nlat)


class FourcastnetModel(GlobalModel):
    model_name = "fourcastnet"

    def __init__(self, *args, cfg: FCNConfig | None = None, weights=None, weight_seed: int = 0, device: int = 0,
                 **kwargs):
        self._cfg, self._weights, self._seed, self._device = cfg or fcn_full(), weights, weight_seed, device
        super().__init__(self.model_name, *args, **kwargs)

    def build_model(self):
        from ...engine import StepEngine
        from ...timeloop import FCNTimeLoop
        from ...weights import make_fcn_weights
        import os
        real = os.environ.get("SKYRIM_B200_WEIGHTS_FCN")
        guard = self._weights is None and bool(real)
        if self._weights is None and real:
            # FourCastNet checkpoint directory (weights.tar + global_means.npy / global_stds.npy); hyper-parameters come
            # from the tensor shapes
            from ...importers import load_real_weights
            self._cfg, self._weights = load_real_weights("fcn", real)
        eng = StepEngine(self._cfg, self._device)
        eng.load_weights(self._weights if self._weights is not None else make_fcn_weights(self._cfg, self._seed))
        loop = FCNTimeLoop(eng)
        loop.guard_first_step = guard   # real checkpoint: first step of every rollout under the fp16-range guard
        return loop

    def build_datasource(self):
        nlat, nlon = len(self.model.grid.lat), len(self.model.grid.lon)
        if self.ic_source == "synthetic":
            return _CroppedSource(SyntheticDataSource(self.model.in_channel_names, nlat + 1, nlon), nlat)
        return _CroppedSource(super().build_datasource(), nlat)

    def rollout(self, start_time, n_steps: int = 3, save: bool = True, save_config: dict = {}, initial_condition=None):
        if initial_condition is not None:
            ic = xr.open_dataarray(initial_condition) if isinstance(initial_condition, str) else initial_condition
            initial_condition = crop_to_grid(ic, len(self.model.grid.lat))
        return super().rollout(start_time, n_steps, save, save_config, initial_condition)
