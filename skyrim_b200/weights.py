"""Deterministic synthetic weights for the step operators.

There is no network in the build/bench environment and the reference's weights are
downloaded at run time by earth2mip (/root/reference/skyrim/core/models/pangu.py:45-46,
fourcastnet_v2.py:36-37), so both the CPU oracle and the CUDA engine are driven by the
same seeded parameter set generated here (SURVEY.md §8(d)).  Every tensor is drawn from
its own generator keyed by (seed, name), so the order of generation does not matter and
one tensor can be regenerated on its own.

Conventions: Linear weights are ``[out, in]`` (K-major, what the tensor-core B operand
wants); transposed-conv weights are ``[in, out, kz, kh, kw]``.
"""
from __future__ import annotations

import zlib
from collections import OrderedDict

import numpy as np

from .config import PRESSURE_LEVELS, FCNConfig, GraphCastConfig, PanguConfig, SFNOConfig

G0 = 9.80665


def _rng(seed: int, name: str) -> np.random.Generator:
    return np.random.default_rng([seed, zlib.crc32(name.encode())])


def _tn(seed, name, shape, std=0.02):
    """Truncated normal (clipped at 2 sigma), fp32."""
    a = _rng(seed, name).standard_normal(shape, dtype=np.float32)
    np.clip(a, -2.0, 2.0, out=a)
    a *= np.float32(std)
    return a


def _ln(seed, name, n):
    # gamma/beta are perturbed off (1, 0) so that parity tests exercise the affine part
    r = _rng(seed, name)
    g = (1.0 + 0.05 * r.standard_normal(n)).astype(np.float32)
    b = (0.05 * r.standard_normal(n)).astype(np.float32)
    return g, b


# ----------------------------------------------------------------------------------------
# climatology used for normalisation statistics and synthetic initial conditions
# (SURVEY.md §8(d)); indexed by variable family and pressure level
# ----------------------------------------------------------------------------------------
_Z_HEIGHT = dict(zip(PRESSURE_LEVELS, [110, 760, 1460, 3010, 4210, 5570, 7180, 9160, 10360,
                                       11770, 13600, 16180, 20580]))
_T_PROFILE = dict(zip(PRESSURE_LEVELS, [288, 284, 280, 270, 262, 253, 242, 229, 222, 218, 215,
                                        212, 215]))


def channel_climatology(name: str):
    """(mean, std) of a channel by its reference name (e.g. 'z500', 't2m')."""
    surf = {"msl": (101325.0, 1200.0), "sp": (96500.0, 9000.0), "u10m": (0.0, 5.0),
            "v10m": (0.0, 5.0), "u100m": (0.0, 5.0), "v100m": (0.0, 5.0), "t2m": (280.0, 20.0),
            "tcwv": (20.0, 15.0), "tp06": (1.2e6, 1.5e6)}   # "tp06" = toa incident solar radiation, J m^-2 per hour
    if name in surf:
        return surf[name]
    fam, p = name[0], int(name[1:])
    if fam == "z":
        mu = G0 * _Z_HEIGHT[p]
        return mu, 0.03 * mu + 300.0
    if fam == "t":
        return float(_T_PROFILE[p]), 15.0
    if fam in "uv":
        return 0.0, 8.0 + 0.02 * (1000 - p)
    if fam == "q":
        mu = 1e-2 * (p / 1000.0) ** 3
        return mu, 0.5 * mu
    if fam == "r":
        return 50.0, 25.0
    if fam == "w":
        return 0.0, 0.05 + 0.25 * (p / 1000.0)
    raise KeyError(name)


def channel_stats(names):
    mu = np.array([channel_climatology(n)[0] for n in names], dtype=np.float32)
    sd = np.array([channel_climatology(n)[1] for n in names], dtype=np.float32)
    return mu, sd


def _smooth_field(seed, name, nlat, nlon):
    """Smooth field in [0,1] (constant masks: land / soil / topography)."""
    r = _rng(seed, name)
    lat = np.linspace(np.pi / 2, -np.pi / 2, nlat, dtype=np.float64)[:, None]
    lon = (np.arange(nlon, dtype=np.float64) * (2 * np.pi / nlon))[None, :]
    f = np.zeros((nlat, nlon))
    for _ in range(5):
        k, m = r.integers(1, 5), r.integers(1, 6)
        f += r.uniform(0.3, 1.0) * np.sin(k * lat + r.uniform(0, 6.28)) * np.cos(m * lon + r.uniform(0, 6.28))
    f = (f - f.min()) / (f.max() - f.min())
    return f.astype(np.float32)


# ----------------------------------------------------------------------------------------
# Pangu
# ----------------------------------------------------------------------------------------
def pangu_param_shapes(cfg: PanguConfig) -> "OrderedDict[str, tuple]":
    C = cfg.dim
    pz, ph, pw = cfg.patch
    s = OrderedDict()
    s["norm.mean"] = (cfg.n_channels,)
    s["norm.std"] = (cfg.n_channels,)
    s["const.masks"] = (cfg.n_const_masks, cfg.nlat, cfg.nlon)
    s["embed.upper.w"] = (C, cfg.n_upper_vars, pz, ph, pw)
    s["embed.upper.b"] = (C,)
    s["embed.surf.w"] = (C, cfg.n_surface_vars + cfg.n_const_masks, ph, pw)
    s["embed.surf.b"] = (C,)
    for li, (depth, heads) in enumerate(zip(cfg.depths, cfg.heads)):
        c = C if li in (0, 3) else 2 * C
        h = cfg.H if li in (0, 3) else cfg.H2
        for bi in range(depth):
            p = f"layer{li}.block{bi}."
            s[p + "qkv.w"] = (3 * c, c)
            s[p + "qkv.b"] = (3 * c,)
            s[p + "bias_table"] = (cfg.bias_table_len, cfg.n_window_types(h), heads)
            s[p + "proj.w"] = (c, c)
            s[p + "proj.b"] = (c,)
            s[p + "ln1.g"] = (c,)
            s[p + "ln1.b"] = (c,)
            s[p + "fc1.w"] = (cfg.mlp_ratio * c, c)
            s[p + "fc1.b"] = (cfg.mlp_ratio * c,)
            s[p + "fc2.w"] = (c, cfg.mlp_ratio * c)
            s[p + "fc2.b"] = (c,)
            s[p + "ln2.g"] = (c,)
            s[p + "ln2.b"] = (c,)
    s["down.ln.g"] = (4 * C,)
    s["down.ln.b"] = (4 * C,)
    s["down.w"] = (2 * C, 4 * C)
    s["up.w1"] = (4 * C, 2 * C)
    s["up.ln.g"] = (C,)
    s["up.ln.b"] = (C,)
    s["up.w2"] = (C, C)
    s["recover.upper.w"] = (2 * C, cfg.n_upper_vars, pz, ph, pw)
    s["recover.upper.b"] = (cfg.n_upper_vars,)
    s["recover.surf.w"] = (2 * C, cfg.n_surface_vars, ph, pw)
    s["recover.surf.b"] = (cfg.n_surface_vars,)
    return s


def make_pangu_weights(cfg: PanguConfig, seed: int = 0) -> "OrderedDict[str, np.ndarray]":
    from .config import PANGU_CHANNELS
    out = OrderedDict()
    mu, sd = channel_stats(PANGU_CHANNELS)
    for name, shape in pangu_param_shapes(cfg).items():
        if name == "norm.mean":
            a = mu
        elif name == "norm.std":
            a = sd
        elif name == "const.masks":
            a = np.stack([_smooth_field(seed, f"mask{i}", cfg.nlat, cfg.nlon) for i in range(shape[0])])
        elif name.endswith(("ln1.g", "ln2.g", "ln.g")):
            a, b = _ln(seed, name[:-2], shape[0])
            out[name] = a
            out[name[:-1] + "b"] = b
            continue
        elif name.endswith(("ln1.b", "ln2.b", "ln.b")):
            continue  # produced with its gamma
        elif name.endswith(".b"):
            a = _tn(seed, name, shape, std=0.02)
        else:
            a = _tn(seed, name, shape, std=0.02)
        assert a.shape == tuple(shape), (name, a.shape, shape)
        out[name] = np.ascontiguousarray(a, dtype=np.float32)
    # keep declared order
    return OrderedDict((k, out[k]) for k in pangu_param_shapes(cfg))


# ----------------------------------------------------------------------------------------
# synthetic initial conditions (SURVEY.md §8(d))
# ----------------------------------------------------------------------------------------
def synthetic_state(names, nlat: int, nlon: int, seed: int = 0) -> np.ndarray:
    """x[c] = mu_c + sigma_c * (0.7 * S_c(lat, lon) + 0.3 * eps), fp32, shape (C, nlat, nlon)."""
    mu, sd = channel_stats(names)
    r = np.random.default_rng([seed, 0xC0FFEE])
    lat = np.linspace(np.pi / 2, -np.pi / 2, nlat, dtype=np.float32)[:, None]
    lon = (np.arange(nlon, dtype=np.float32) * np.float32(2 * np.pi / nlon))[None, :]
    x = np.empty((len(names), nlat, nlon), dtype=np.float32)
    for c in range(len(names)):
        s = np.zeros((nlat, nlon), dtype=np.float32)
        for _ in range(6):
            k, m = int(r.integers(1, 4)), int(r.integers(0, 5))
            s += np.float32(r.uniform(0.2, 0.6)) * (np.sin(k * lat + np.float32(r.uniform(0, 6.28)))
                                                    * np.cos(m * lon + np.float32(r.uniform(0, 6.28))))
        eps = r.standard_normal((nlat, nlon), dtype=np.float32)
        x[c] = mu[c] + sd[c] * (np.float32(0.7) * s + np.float32(0.3) * eps)
    return x


def n_params(weights) -> int:
    return int(sum(int(np.prod(v.shape)) for v in weights.values()))


# ----------------------------------------------------------------------------------------
# SFNO (FourCastNet-v2-small)
# ----------------------------------------------------------------------------------------
def sfno_param_shapes(cfg: SFNOConfig) -> "OrderedDict[str, tuple]":
    E, Cin = cfg.embed, cfg.n_channels
    s = OrderedDict()
    s["norm.mean"] = (Cin,)
    s["norm.std"] = (Cin,)
    s["enc.fc1.w"] = (E, Cin)
    s["enc.fc1.b"] = (E,)
    s["enc.fc2.w"] = (E, E)
    s["enc.fc2.b"] = (E,)
    s["pos_embed"] = (E, cfg.nlat, cfg.nlon)
    for i in range(cfg.layers):
        p = f"blk{i}."
        s[p + "norm0.g"] = (E,)
        s[p + "norm0.b"] = (E,)
        s[p + "spec.w"] = (cfg.lmax, E, E, 2)        # [l, out, in, (re, im)]
        s[p + "inner.w"] = (E, E)
        s[p + "inner.b"] = (E,)
        s[p + "norm1.g"] = (E,)
        s[p + "norm1.b"] = (E,)
        s[p + "fc1.w"] = (cfg.mlp_ratio * E, E)
        s[p + "fc1.b"] = (cfg.mlp_ratio * E,)
        s[p + "fc2.w"] = (E, cfg.mlp_ratio * E)
        s[p + "fc2.b"] = (E,)
    s["dec.fc1.w"] = (E, E + Cin)
    s["dec.fc1.b"] = (E,)
    s["dec.fc2.w"] = (Cin, E)
    s["dec.fc2.b"] = (Cin,)
    return s


def make_sfno_weights(cfg: SFNOConfig, seed: int = 0) -> "OrderedDict[str, np.ndarray]":
    """Synthetic SFNO parameters.  Linear layers are variance preserving (std 1/sqrt(fan_in))
    so that 40 autoregressive steps neither explode nor collapse; the spectral (dhconv)
    weights are complex normal with std 1/sqrt(2 E) per component."""
    from .config import FCNV2_CHANNELS
    out = OrderedDict()
    mu, sd = channel_stats(FCNV2_CHANNELS)
    for name, shape in sfno_param_shapes(cfg).items():
        if name == "norm.mean":
            a = mu
        elif name == "norm.std":
            a = sd
        elif name.endswith((".g",)):
            g, b = _ln(seed, name[:-2], shape[0])
            out[name], out[name[:-1] + "b"] = g, b
            continue
        elif name.endswith(("norm0.b", "norm1.b")):
            continue
        elif name == "pos_embed":
            a = _tn(seed, name, shape, std=0.1)
        elif name.endswith("spec.w"):
            a = _rng(seed, name).standard_normal(shape, dtype=np.float32) * np.float32(1.0 / np.sqrt(2.0 * cfg.embed))
        elif name.endswith(".b"):
            a = _tn(seed, name, shape, std=0.02)
        else:
            a = _tn(seed, name, shape, std=0.9 / np.sqrt(shape[-1]))
        out[name] = np.ascontiguousarray(a, dtype=np.float32)
    return OrderedDict((k, out[k]) for k in sfno_param_shapes(cfg))


def sfno_table_shapes(cfg: SFNOConfig) -> "OrderedDict[str, tuple]":
    """Shapes (and order) of sfno_tables() without computing them: what a non-root rank needs for the arena manifest."""
    t = OrderedDict()
    t["sht.fwd_big"] = (cfg.mmax, cfg.lmax, cfg.nlat)
    t["sht.inv_big"] = (cfg.mmax, cfg.nlat, cfg.lmax)
    t["sht.fwd_int"] = (cfg.mmax, cfg.lmax, cfg.h)
    t["sht.inv_int"] = (cfg.mmax, cfg.h, cfg.lmax)
    for tag, n in (("big", cfg.nlon), ("int", cfg.w)):
        t[f"dft.fwd_{tag}"] = (2 * cfg.mmax, n)
        t[f"dft.inv_{tag}"] = (n, 2 * cfg.mmax)
    return t


def sfno_tables(cfg: SFNOConfig) -> "OrderedDict[str, np.ndarray]":
    """SHT / DFT tables the engine consumes as extra arena entries (fp32)."""
    from .sht import dft_matrices, sht_tables
    t = OrderedDict()
    fwd_big, inv_big = sht_tables(cfg.nlat, cfg.lmax, cfg.mmax, "equiangular")
    fwd_int, inv_int = sht_tables(cfg.h, cfg.lmax, cfg.mmax, "legendre-gauss")
    t["sht.fwd_big"] = fwd_big.astype(np.float32)     # [m, l, k]
    t["sht.inv_big"] = inv_big.astype(np.float32)     # [m, k, l]
    t["sht.fwd_int"] = fwd_int.astype(np.float32)
    t["sht.inv_int"] = inv_int.astype(np.float32)
    for tag, n in (("big", cfg.nlon), ("int", cfg.w)):
        f, i = dft_matrices(n, cfg.mmax)
        t[f"dft.fwd_{tag}"] = f.astype(np.float32)    # [(m, re/im), j]
        t[f"dft.inv_{tag}"] = i.astype(np.float32)    # [j, (m, re/im)]
    return t


# ----------------------------------------------------------------------------------------
# GraphCast
# ----------------------------------------------------------------------------------------
def graphcast_mlps(cfg: GraphCastConfig):
    """(name, fan_in, fan_out, has_layernorm) of every MLP of the step, in execution order"""
    L = cfg.latent
    m = [("enc.grid_embed", cfg.n_features, L, True), ("enc.mesh_embed", 3, L, True), ("enc.g2m_edge_embed", 4, L, True),
         ("enc.g2m_edge", 3 * L, L, True), ("enc.g2m_mesh", 2 * L, L, True), ("enc.g2m_grid", L, L, True),
         ("proc.edge_embed", 4, L, True)]
    for i in range(cfg.layers):
        m += [(f"proc{i}.edge", 3 * L, L, True), (f"proc{i}.node", 2 * L, L, True)]
    m += [("dec.m2g_edge_embed", 4, L, True), ("dec.m2g_edge", 3 * L, L, True), ("dec.m2g_grid", 2 * L, L, True),
          ("dec.out", L, cfg.n_state, False)]
    return m


def graphcast_param_shapes(cfg: GraphCastConfig) -> "OrderedDict[str, tuple]":
    L = cfg.latent
    s = OrderedDict()
    s["norm.mean"] = (cfg.n_state,)
    s["norm.std"] = (cfg.n_state,)
    s["norm.diff_std"] = (cfg.n_state,)
    s["static.fields"] = (cfg.n_static, cfg.nlat, cfg.nlon)
    for name, fi, fo, ln in graphcast_mlps(cfg):
        s[name + ".w1"] = (L, fi)
        s[name + ".b1"] = (L,)
        s[name + ".w2"] = (fo, L)
        s[name + ".b2"] = (fo,)
        if ln:
            s[name + ".ln.g"] = (fo,)
            s[name + ".ln.b"] = (fo,)
    return s


def make_graphcast_weights(cfg: GraphCastConfig, seed: int = 0) -> "OrderedDict[str, np.ndarray]":
    """Synthetic GraphCast parameters (the JAX checkpoint is downloaded at run time by the reference,
    /root/reference/skyrim/core/models/graphcast.py:51-54).  Linear layers are variance preserving; every MLP ends in a
    LayerNorm, so the latents stay O(1) through the 16 processor layers."""
    from .config import GRAPHCAST_CHANNELS
    out = OrderedDict()
    mu, sd = channel_stats(GRAPHCAST_CHANNELS)
    for name, shape in graphcast_param_shapes(cfg).items():
        if name == "norm.mean":
            a = mu
        elif name == "norm.std":
            a = sd
        elif name == "norm.diff_std":
            a = (0.1 * sd).astype(np.float32)
        elif name == "static.fields":
            a = np.stack([2.0 * _smooth_field(seed, f"gc.static{i}", cfg.nlat, cfg.nlon) - 1.0 for i in range(shape[0])])
        elif name.endswith("ln.g"):
            g, b = _ln(seed, name[:-2], shape[0])
            out[name], out[name[:-1] + "b"] = g, b
            continue
        elif name.endswith("ln.b"):
            continue
        elif name.endswith((".b1", ".b2")):
            a = _tn(seed, name, shape, std=0.02)
        else:
            a = _tn(seed, name, shape, std=0.9 / np.sqrt(shape[-1]))
        out[name] = np.ascontiguousarray(a, dtype=np.float32)
    return OrderedDict((k, out[k]) for k in graphcast_param_shapes(cfg))


def synthetic_graphcast_state(cfg: GraphCastConfig, seed: int = 0) -> np.ndarray:
    """(2 * n_state, nlat, nlon): two time slices 6 h apart (the second = the first + a smooth tendency of 0.1 sigma).
    The forcing channel of both slices is left at its climatological mean: the caller fills it with the toa radiation of
    its own clock (engine: sky_toa_radiation; oracle: oracle.graphcast_ref.toa_radiation)."""
    from .config import GRAPHCAST_CHANNELS
    x0 = synthetic_state(GRAPHCAST_CHANNELS, cfg.nlat, cfg.nlon, seed)
    x1 = synthetic_state(GRAPHCAST_CHANNELS, cfg.nlat, cfg.nlon, seed + 1000)
    _, sd = channel_stats(GRAPHCAST_CHANNELS)
    mu, _ = channel_stats(GRAPHCAST_CHANNELS)
    x1 = x0 + np.float32(0.1) * (x1 - mu[:, None, None])
    x0[-1], x1[-1] = mu[-1], mu[-1]
    return np.concatenate([x0, x1], axis=0)


# ----------------------------------------------------------------------------------------
# FourCastNet v1 (AFNO); upstream parameter names (NVlabs FourCastNet AFNONet state dict)
# ----------------------------------------------------------------------------------------
def fcn_param_shapes(cfg: FCNConfig) -> "OrderedDict[str, tuple]":
    E, C, p, nb, bs = cfg.embed, cfg.n_channels, cfg.patch, cfg.num_blocks, cfg.block_size
    s = OrderedDict()
    s["norm.mean"] = (C,)
    s["norm.std"] = (C,)
    s["patch_embed.proj.weight"] = (E, C, p, p)
    s["patch_embed.proj.bias"] = (E,)
    s["pos_embed"] = (1, cfg.tokens, E)
    for i in range(cfg.depth):
        b = f"blocks.{i}."
        s[b + "norm1.weight"] = (E,)
        s[b + "norm1.bias"] = (E,)
        s[b + "filter.w1"] = (2, nb, bs, bs)
        s[b + "filter.b1"] = (2, nb, bs)
        s[b + "filter.w2"] = (2, nb, bs, bs)
        s[b + "filter.b2"] = (2, nb, bs)
        s[b + "norm2.weight"] = (E,)
        s[b + "norm2.bias"] = (E,)
        s[b + "mlp.fc1.weight"] = (cfg.mlp_ratio * E, E)
        s[b + "mlp.fc1.bias"] = (cfg.mlp_ratio * E,)
        s[b + "mlp.fc2.weight"] = (E, cfg.mlp_ratio * E)
        s[b + "mlp.fc2.bias"] = (E,)
    s["head.weight"] = (C * p * p, E)
    return s


def make_fcn_weights(cfg: FCNConfig, seed: int = 0) -> "OrderedDict[str, np.ndarray]":
    """Synthetic AFNONet parameters.  Linear layers are variance preserving (std 0.9/sqrt(fan_in)); the spectral block
    MLP uses upstream's initialisation scale (0.02 * N(0, 1)), which leaves a sizeable share of the kept modes inside
    the softshrink dead band (tests/test_fcn_cpu.py checks the share)."""
    from .config import FCN_CHANNELS
    out = OrderedDict()
    mu, sd = channel_stats(FCN_CHANNELS)
    for name, shape in fcn_param_shapes(cfg).items():
        if name == "norm.mean":
            a = mu
        elif name == "norm.std":
            a = sd
        elif name.endswith(("norm1.weight", "norm2.weight")):
            g, b = _ln(seed, name[:-7], shape[0])
            out[name], out[name[:-6] + "bias"] = g, b
            continue
        elif name.endswith(("norm1.bias", "norm2.bias")):
            continue
        elif ".filter." in name:
            a = np.float32(0.02) * _rng(seed, name).standard_normal(shape, dtype=np.float32)
        elif name == "pos_embed":
            a = _tn(seed, name, shape, std=0.1)
        elif name.endswith(".bias"):
            a = _tn(seed, name, shape, std=0.02)
        elif name == "patch_embed.proj.weight":
            a = _tn(seed, name, shape, std=0.9 / np.sqrt(np.prod(shape[1:])))
        else:
            a = _tn(seed, name, shape, std=0.9 / np.sqrt(shape[-1]))
        out[name] = np.ascontiguousarray(a, dtype=np.float32)
    return OrderedDict((k, out[k]) for k in fcn_param_shapes(cfg))
