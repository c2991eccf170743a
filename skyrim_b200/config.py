"""Shape configuration of the step operators on the hot path (Pangu-Weather, FourCastNet-v2 SFNO, GraphCast,
FourCastNet v1 AFNO).

The reference carries no architecture description of its own (SURVEY.md §0): the
arithmetic lives in ONNX graphs / earth2mip modules it downloads.  The numbers below
restate the published architectures (SURVEY.md Appendix A / B) and are the single
source of truth for the oracle (``oracle/``), the weight synthesiser
(``skyrim_b200/weights.py``) and the CUDA engine (``skyrim_b200/csrc``).

Channel orders are the reference's: /root/reference/skyrim/core/models/pangu.py:6-13
and /root/reference/skyrim/core/models/fourcastnet_v2.py:12-20.
"""
from __future__ import annotations

from dataclasses import dataclass, field

PRESSURE_LEVELS = [1000, 925, 850, 700, 600, 500, 400, 300, 250, 200, 150, 100, 50]

# /root/reference/skyrim/core/models/pangu.py:6-13 (z,q,t,u,v x 13 levels, then 4 surface)
PANGU_CHANNELS = [f"{v}{p}" for v in "zqtuv" for p in PRESSURE_LEVELS] + [
    "msl", "u10m", "v10m", "t2m"]

# /root/reference/skyrim/core/models/fourcastnet_v2.py:12-20
_FCN_LEVELS = [50, 100, 150, 200, 250, 300, 400, 500, 600, 700, 850, 925, 1000]
FCNV2_CHANNELS = ["u10m", "v10m", "u100m", "v100m", "t2m", "sp", "msl", "tcwv"] + [
    f"{v}{p}" for v in "uvztr" for p in _FCN_LEVELS]


@dataclass(frozen=True)
class PanguConfig:
    """Pangu-Weather 6-h operator (SURVEY.md Appendix A)."""
    nlat: int = 721
    nlon: int = 1440
    n_levels: int = 13
    n_upper_vars: int = 5
    n_surface_vars: int = 4
    n_const_masks: int = 3
    patch: tuple = (2, 4, 4)
    window: tuple = (2, 6, 12)
    dim: int = 192
    depths: tuple = (2, 6, 6, 2)
    heads: tuple = (6, 12, 12, 6)
    mlp_ratio: int = 4
    ln_eps: float = 1e-5
    mask_value: float = -100.0   # Swin convention for shifted-window masking

    @property
    def n_channels(self):
        return self.n_upper_vars * self.n_levels + self.n_surface_vars

    # token grid at resolution 1 (after patch embedding)
    @property
    def Z(self):
        return (self.n_levels + self.patch[0] - 1) // self.patch[0] + 1  # +1: surface slab at z=0

    @property
    def H(self):
        return (self.nlat + self.patch[1] - 1) // self.patch[1]

    @property
    def W(self):
        assert self.nlon % self.patch[2] == 0
        return self.nlon // self.patch[2]

    # token grid at resolution 2 (after DownSample)
    @property
    def H2(self):
        return (self.H + 1) // 2

    @property
    def W2(self):
        assert self.W % 2 == 0
        return self.W // 2

    def padded_h(self, h):
        wh = self.window[1]
        return (h + wh - 1) // wh * wh

    def n_window_types(self, h):
        return (self.Z // self.window[0]) * (self.padded_h(h) // self.window[1])

    @property
    def bias_table_len(self):
        wz, wh, ww = self.window
        return (2 * ww - 1) * wh * wh * wz * wz

    def validate(self):
        wz, wh, ww = self.window
        assert self.Z % wz == 0, "Z must tile by the window"
        assert self.W % ww == 0 and self.W2 % ww == 0, "longitude tokens must tile by the window"
        assert self.dim % self.heads[0] == 0 and (2 * self.dim) % self.heads[1] == 0
        assert self.dim // self.heads[0] == 32 and 2 * self.dim // self.heads[1] == 32, "head_dim 32"
        return self


def pangu_full() -> PanguConfig:
    return PanguConfig().validate()


def pangu_small(nlat: int = 41, nlon: int = 96) -> PanguConfig:
    """Same operator on a coarse grid (test sizes the oracle finishes in seconds)."""
    return PanguConfig(nlat=nlat, nlon=nlon).validate()


@dataclass(frozen=True)
class SFNOConfig:
    """FourCastNet-v2-small SFNO operator (SURVEY.md Appendix B, default synthetic hyper-parameters)."""
    nlat: int = 721
    nlon: int = 1440
    n_channels: int = 73
    embed: int = 384
    layers: int = 8
    scale_factor: int = 3
    mlp_ratio: int = 2
    eps: float = 1e-6

    @property
    def h(self):
        return self.nlat // self.scale_factor

    @property
    def w(self):
        return self.nlon // self.scale_factor

    @property
    def lmax(self):
        return self.h

    @property
    def mmax(self):
        return self.w // 2 + 1


def sfno_full() -> SFNOConfig:
    return SFNOConfig()


def sfno_small(nlat: int = 49, nlon: int = 96, embed: int = 64, layers: int = 3) -> SFNOConfig:
    return SFNOConfig(nlat=nlat, nlon=nlon, embed=embed, layers=layers)


# ----------------------------------------------------------------------------------------
# GraphCast (operational 0.25 deg / 13 levels)
# ----------------------------------------------------------------------------------------
GRAPHCAST_LEVELS = [50, 100, 150, 200, 250, 300, 400, 500, 600, 700, 850, 925, 1000]
# Order in which the reference flattens the stepper's Dataset (/root/reference/skyrim/core/models/graphcast.py:29-41
# CHANNEL_MAP, applied by _to_global_da :68-91): q, z, t, u, v, w on 13 levels, then t2m, u10m, v10m, msl and the
# forcing the reference labels "tp06" (it is toa_incident_solar_radiation, :16,40).  The CHANNELS list at :17-26 holds
# the same 83 names with z first; the reference's own test compares them as sets (tests/core/test_graphcast.py:22).
GRAPHCAST_CHANNELS = [f"{v}{p}" for v in "qztuvw" for p in GRAPHCAST_LEVELS] + ["t2m", "u10m", "v10m", "msl", "tp06"]


@dataclass(frozen=True)
class GraphCastConfig:
    """GraphCast encoder - processor - decoder (SURVEY.md §8(a) A9): latent 512, 16 message-passing layers on the
    refinement-6 multimesh, one-hidden-layer swish MLPs with LayerNorm, sum aggregation."""
    nlat: int = 721
    nlon: int = 1440
    mesh_levels: int = 6
    latent: int = 512
    layers: int = 16
    radius_frac: float = 0.6
    n_state: int = 83            # channels of ONE time slice of the state (82 prognostic + toa radiation)
    n_prog: int = 82             # prognostic channels (inputs at t-6h and t, outputs as residuals)
    n_static: int = 2            # geopotential at the surface, land-sea mask
    ln_eps: float = 1e-5
    dt_hours: int = 6

    @property
    def n_channels(self):        # channels of the stepped state tensor: (2 time slices) x n_state
        return 2 * self.n_state

    @property
    def n_features(self):
        """grid-node input features: 2 x prognostic, toa at (t-6h, t, t+6h), (year, day) x (sin, cos) at the three
        times, statics, (cos lat, sin lon, cos lon)"""
        return 2 * self.n_prog + 3 + 12 + self.n_static + 3

    @property
    def n_grid(self):
        return self.nlat * self.nlon


def graphcast_full() -> GraphCastConfig:
    return GraphCastConfig()


def graphcast_small(nlat: int = 41, nlon: int = 96, mesh_levels: int = 2, latent: int = 512, layers: int = 2) -> GraphCastConfig:
    return GraphCastConfig(nlat=nlat, nlon=nlon, mesh_levels=mesh_levels, latent=latent, layers=layers)


# ----------------------------------------------------------------------------------------
# FourCastNet v1 (AFNO backbone)
# ----------------------------------------------------------------------------------------
# /root/reference/skyrim/core/models/fourcastnet.py:8-11
FCN_CHANNELS = ["u10m", "v10m", "t2m", "sp", "msl", "t850", "u1000", "v1000", "z1000", "u850", "v850", "z850", "u500",
                "v500", "z500", "t500", "z50", "r500", "r850", "tcwv", "u100m", "v100m", "u250", "v250", "z250", "t250"]


@dataclass(frozen=True)
class FCNConfig:
    """FourCastNet v1 AFNONet (SURVEY.md Appendix D): 8x8 patch embedding, `depth` blocks of LayerNorm -> AFNO2D
    filter (double skip) -> LayerNorm -> GELU MLP, linear head.  The grid has no south-pole row (720 x 1440)."""
    nlat: int = 720
    nlon: int = 1440
    n_channels: int = 26
    patch: int = 8
    embed: int = 768
    depth: int = 12
    num_blocks: int = 8
    mlp_ratio: int = 4
    sparsity: float = 0.01                     # softshrink lambda
    hard_thresholding_fraction: float = 1.0
    ln_eps: float = 1e-6

    @property
    def h(self):
        return self.nlat // self.patch

    @property
    def w(self):
        return self.nlon // self.patch

    @property
    def tokens(self):
        return self.h * self.w

    @property
    def block_size(self):
        return self.embed // self.num_blocks

    @property
    def kept(self):
        return int((self.h // 2 + 1) * self.hard_thresholding_fraction)

    @property
    def h_range(self):
        """H-frequency rows the filter processes: upstream's slice [total - kept : total + kept] (clipped to h)"""
        total = self.h // 2 + 1
        return total - self.kept, min(total + self.kept, self.h)

    @property
    def kw(self):
        """W-modes the filter processes: upstream's slice [:kept] of the w // 2 + 1 rfft modes"""
        return min(self.kept, self.w // 2 + 1)

    def validate(self):
        assert self.nlat % self.patch == 0 and self.nlon % self.patch == 0, "the grid must tile by the patch"
        assert self.embed % self.num_blocks == 0
        return self


def fcn_full() -> FCNConfig:
    return FCNConfig().validate()


def fcn_small(nlat: int = 48, nlon: int = 96, depth: int = 2) -> FCNConfig:
    return FCNConfig(nlat=nlat, nlon=nlon, depth=depth).validate()
