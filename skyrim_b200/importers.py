"""Real-weight import (SURVEY.md section 8(f) N2): what the reference loads at
/root/reference/skyrim/core/models/pangu.py:45-46 (``pangu.load(registry.get_model("e2mip://pangu"))`` -> two
ONNXRuntime sessions over pangu_weather_{6,24}.onnx) and fourcastnet_v2.py:36-37 (``fcnv2_sm.load`` -> torch.load of
``weights.tar`` + ``global_means.npy`` / ``global_stds.npy``), turned into the engine's parameter dict
(skyrim_b200.weights.*_param_shapes) without onnx / onnxruntime / earth2mip:

  * ``read_onnx_initializers``  dependency-free protobuf wire-format reader: graph initialisers and Constant nodes,
                                in file order, plus the op sequence;
  * ``ungather_bias``           the ONNX graph carries the earth-specific bias EXPANDED through position_index
                                ((n_type, heads, 144, 144), ~1 GB); the engine wants the compact (3312, n_type, heads) table;
  * ``pangu_from_onnx``         shape-and-order driven mapping of the initialisers onto the Pangu parameter names;
  * ``sfno_from_checkpoint``    key-pattern mapping of an fcnv2_sm ``model_state`` dict; hyper-parameters from shapes;
  * ``check_fp16_range``        guard for real weights: the engine feeds fp16 operands to the tensor cores.

No such file exists in the build environment (no network), so the mappings are exercised on files the unit tests
write with the same wire format (tests/test_importers_cpu.py).  Free choices that can only be confirmed against
the real graph (pad placement, output = state) are listed in DESIGN.md section 2.
"""
from __future__ import annotations

import os
import struct
from collections import OrderedDict

import numpy as np

# ----------------------------------------------------------------------------------------
# protobuf wire format (just enough for onnx.ModelProto)
# ----------------------------------------------------------------------------------------
_ONNX_DTYPES = {1: np.float32, 2: np.uint8, 3: np.int8, 5: np.int16, 6: np.int32, 7: np.int64, 9: np.bool_, 10: np.float16,
                11: np.float64}


def _varint(buf, pos):
    r, shift = 0, 0
    while True:
        b = buf[pos]
        pos += 1
        r |= (b & 0x7F) << shift
        if not b & 0x80:
            return r, pos
        shift += 7


def _fields(buf, start=0, end=None):
    """yield (field_number, wire_type, value) — value is an int (varint / fixed) or a memoryview (length-delimited)."""
    pos, end = start, len(buf) if end is None else end
    while pos < end:
        key, pos = _varint(buf, pos)
        fn, wt = key >> 3, key & 7
        if wt == 0:
            v, pos = _varint(buf, pos)
        elif wt == 1:
            v = struct.unpack_from("<q", buf, pos)[0]; pos += 8
        elif wt == 5:
            v = struct.unpack_from("<i", buf, pos)[0]; pos += 4
        elif wt == 2:
            n, pos = _varint(buf, pos)
            v = buf[pos:pos + n]; pos += n
        else:
            raise ValueError(f"unsupported protobuf wire type {wt}")
        yield fn, wt, v


def _tensor(view, base_dir=None):
    """onnx.TensorProto -> (name, ndarray)"""
    dims, dtype, name, raw, floats, int64s, int32s, ext = [], 1, "", None, [], [], [], {}
    for fn, wt, v in _fields(view):
        if fn == 1:     # dims (packed or not)
            if wt == 2:
                p = 0
                while p < len(v):
                    d, p = _varint(v, p); dims.append(d)
            else:
                dims.append(v)
        elif fn == 2:
            dtype = v
        elif fn == 8:
            name = bytes(v).decode()
        elif fn == 9:
            raw = v
        elif fn == 4:   # float_data
            floats.append(np.frombuffer(v, "<f4") if wt == 2 else np.array([struct.unpack("<f", struct.pack("<i", v))[0]], "f4"))
        elif fn == 7:   # int64_data
            if wt == 2:
                p = 0
                while p < len(v):
                    d, p = _varint(v, p); int64s.append(d - (1 << 64) if d >> 63 else d)
            else:
                int64s.append(v)
        elif fn == 5:   # int32_data
            if wt == 2:
                p = 0
                while p < len(v):
                    d, p = _varint(v, p); int32s.append(d)
            else:
                int32s.append(v)
        elif fn == 13:  # external_data: StringStringEntryProto
            kv = {f: bytes(x).decode() for f, _, x in _fields(v)}
            ext[kv.get(1, "")] = kv.get(2, "")
    np_dt = _ONNX_DTYPES.get(dtype)
    if np_dt is None:
        raise ValueError(f"tensor {name}: unsupported ONNX data type {dtype}")
    if raw is not None:
        a = np.frombuffer(raw, np.dtype(np_dt).newbyteorder("<")).astype(np_dt, copy=True)
    elif ext:
        path = os.path.join(base_dir or ".", ext["location"])
        off, ln = int(ext.get("offset", 0)), int(ext.get("length", -1))
        with open(path, "rb") as f:
            f.seek(off)
            a = np.frombuffer(f.read(ln if ln >= 0 else None), np_dt).copy()
    elif floats:
        a = np.concatenate(floats).astype(np_dt)
    elif int64s:
        a = np.array(int64s, np.int64).astype(np_dt)
    else:
        a = np.array(int32s, np.int32).astype(np_dt)
    return name, a.reshape(dims) if dims else a.reshape(())


def read_onnx_initializers(path: str):
    """-> (OrderedDict name -> ndarray in file order: graph.initializer first, then Constant-node tensors in node order,
           list of (op_type, inputs, outputs) in node order)."""
    with open(path, "rb") as f:
        buf = memoryview(f.read())
    base = os.path.dirname(os.path.abspath(path))
    tensors, consts, ops = OrderedDict(), OrderedDict(), []
    for fn, wt, g in _fields(buf):
        if fn != 7 or wt != 2:      # ModelProto.graph
            continue
        for gfn, gwt, v in _fields(g):
            if gfn == 5 and gwt == 2:           # GraphProto.initializer
                n, a = _tensor(v, base)
                tensors[n] = a
            elif gfn == 1 and gwt == 2:         # GraphProto.node
                ins, outs, op, attr_t = [], [], "", None
                for nfn, nwt, nv in _fields(v):
                    if nfn == 1: ins.append(bytes(nv).decode())
                    elif nfn == 2: outs.append(bytes(nv).decode())
                    elif nfn == 4: op = bytes(nv).decode()
                    elif nfn == 5 and nwt == 2:   # AttributeProto: t = field 5
                        for afn, awt, av in _fields(nv):
                            if afn == 5 and awt == 2:
                                attr_t = av
                ops.append((op, ins, outs))
                if op == "Constant" and attr_t is not None and outs:
                    _, a = _tensor(attr_t, base)
                    consts[outs[0]] = a
    tensors.update(consts)
    return tensors, ops


# ---- writer used by the unit tests (same wire format) ----------------------------------------
def _enc_varint(v):
    out = bytearray()
    v &= (1 << 64) - 1
    while True:
        b = v & 0x7F
        v >>= 7
        out.append(b | (0x80 if v else 0))
        if not v:
            return bytes(out)


def _ld(fn, payload):
    return _enc_varint((fn << 3) | 2) + _enc_varint(len(payload)) + payload


def write_onnx_initializers(path: str, tensors, ops=()):
    """Minimal ModelProto with graph.initializer entries (raw_data) and nodes; test infrastructure for the reader."""
    inv = {np.dtype(v): k for k, v in _ONNX_DTYPES.items()}
    g = bytearray()
    for op, ins, outs in ops:
        n = b"".join(_ld(1, i.encode()) for i in ins) + b"".join(_ld(2, o.encode()) for o in outs) + _ld(4, op.encode())
        g += _ld(1, n)
    for name, a in tensors.items():
        a = np.asarray(a)
        t = b"".join(_enc_varint((1 << 3) | 0) + _enc_varint(d) for d in a.shape)
        t += _enc_varint((2 << 3) | 0) + _enc_varint(inv[a.dtype]) + _ld(8, name.encode()) + _ld(9, a.tobytes())
        g += _ld(5, t)
    with open(path, "wb") as f:
        f.write(_enc_varint((1 << 3) | 0) + _enc_varint(8) + _ld(7, bytes(g)))


# ----------------------------------------------------------------------------------------
# earth-specific bias: expanded (n_type, heads, N, N) -> compact (3312, n_type, heads)
# ----------------------------------------------------------------------------------------
def position_index(window=(2, 6, 12)) -> np.ndarray:
    """(N, N) index into the compact table: absolute in (z, h), relative in w (Appendix A item 2; same formula as the
    CUDA kernel's gather, skyrim_b200/csrc/attention_tc.cuh)."""
    wz, wh, ww = window
    zi, hi, wi = np.meshgrid(np.arange(wz), np.arange(wh), np.arange(ww), indexing="ij")
    zi, hi, wi = zi.reshape(-1), hi.reshape(-1), wi.reshape(-1)
    return ((zi[:, None] + wz * zi[None, :]) * ((2 * ww - 1) * wh * wh) + (hi[:, None] + wh * hi[None, :]) * (2 * ww - 1)
            + (wi[:, None] - wi[None, :] + ww - 1))


def ungather_bias(expanded: np.ndarray, window=(2, 6, 12), atol=1e-6) -> np.ndarray:
    """expanded[(type), head, i, j] = table[position_index[i, j], type, head]  ->  table (3312, n_type, heads).
    Every compact entry occurs several times in the expansion; they must agree (else the layout assumption is wrong)."""
    e = np.asarray(expanded)
    N = window[0] * window[1] * window[2]
    e = e.reshape(-1, e.shape[-3], N, N)            # (n_type, heads, N, N)
    n_type, heads = e.shape[:2]
    idx = position_index(window).reshape(-1)
    L = (2 * window[2] - 1) * window[1] ** 2 * window[0] ** 2
    flat = e.reshape(n_type, heads, N * N)
    table = np.zeros((L, n_type, heads), e.dtype)
    table[idx] = np.moveaxis(flat, -1, 0)           # last write wins; consistency checked below
    back = np.moveaxis(table[idx], 0, -1)
    if not np.allclose(back, flat, atol=atol, rtol=0):
        raise ValueError("expanded bias is not a gather of a compact (3312, n_type, heads) table through position_index")
    if len(np.unique(idx)) != L:
        raise ValueError("position_index does not cover the table")
    return table


# ----------------------------------------------------------------------------------------
# Pangu: ONNX initialisers -> parameter dict
# ----------------------------------------------------------------------------------------
def pangu_from_onnx(path: str, cfg=None):
    """Map the initialisers of pangu_weather_6.onnx onto skyrim_b200.weights.pangu_param_shapes(cfg).

    The exported graph names its tensors by node id, so the mapping is by SHAPE and ORDER OF APPEARANCE: within one
    block every 2-D weight has a distinct shape (qkv (C,3C) / proj (C,C) / fc1 (C,4C) / fc2 (4C,C), stored [in, out]
    for MatMul and transposed here to [out, in]); 1-D vectors of equal length follow the forward order
    (proj.b, ln1.g, ln1.b, fc2.b, ln2.g, ln2.b); 4-D tensors (n_type, heads, 144, 144) are expanded biases.
    Raises with a shape census when the counts do not match — never guesses silently."""
    from .config import pangu_full
    from .weights import pangu_param_shapes
    cfg = cfg or pangu_full()
    shapes = pangu_param_shapes(cfg)
    tensors, _ = read_onnx_initializers(path)
    by_shape = OrderedDict()
    for n, a in tensors.items():
        if a.dtype.kind == "f" and a.size > 1:
            by_shape.setdefault(tuple(a.shape), []).append(a.astype(np.float32))
    out = OrderedDict()

    def take(*cands):
        for s in cands:
            q = by_shape.get(tuple(s))
            if q:
                return q.pop(0), tuple(s)
        raise KeyError(f"no initialiser of shape {cands} left; census: { {k: len(v) for k, v in by_shape.items()} }")

    N = cfg.window[0] * cfg.window[1] * cfg.window[2]
    for name, shp in shapes.items():
        if name in ("norm.mean", "norm.std", "const.masks"):
            continue   # baked into the graph as constants: filled below from the graph's own tensors when identifiable
        if name.endswith("bias_table"):
            L, n_type, heads = shp
            a, _ = take((n_type, heads, N, N), (1, n_type, heads, N, N), shp)
            out[name] = a if a.shape == tuple(shp) else ungather_bias(a, cfg.window)
        elif len(shp) == 2:
            a, got = take(shp[::-1], shp)           # MatMul weights are stored [in, out]
            out[name] = np.ascontiguousarray(a.T) if got == tuple(shp[::-1]) else a   # square: MatMul layout assumed
        else:
            a, _ = take(shp)
            out[name] = a
    from .config import PANGU_CHANNELS
    from .weights import channel_stats
    mean, std = None, None
    for s in ((cfg.n_channels,), (cfg.n_upper_vars, cfg.n_levels, 1, 1), (1, cfg.n_channels, 1, 1)):
        q = by_shape.get(s)
        if q and len(q) >= 2:
            mean, std = q.pop(0).reshape(-1), q.pop(0).reshape(-1)
            break
    if mean is None:   # normalisation folded elsewhere in the graph: fall back to the documented climatology
        mean, std = channel_stats(PANGU_CHANNELS)
    out["norm.mean"], out["norm.std"] = mean.astype(np.float32), std.astype(np.float32)
    q = by_shape.get((cfg.n_const_masks, cfg.nlat, cfg.nlon)) or by_shape.get((1, cfg.n_const_masks, cfg.nlat, cfg.nlon))
    out["const.masks"] = (q.pop(0).reshape(cfg.n_const_masks, cfg.nlat, cfg.nlon) if q
                          else np.zeros((cfg.n_const_masks, cfg.nlat, cfg.nlon), np.float32))
    return OrderedDict((k, np.ascontiguousarray(out[k], dtype=np.float32)) for k in shapes)


# ----------------------------------------------------------------------------------------
# SFNO: fcnv2_sm checkpoint -> parameter dict
# ----------------------------------------------------------------------------------------
_SFNO_KEYS = (   # (our name, candidate checkpoint key suffixes) — modulus / makani SphericalFourierNeuralOperatorNet naming
    ("enc.fc1.w", ("encoder.0.weight", "encoder.fwd.0.weight")), ("enc.fc1.b", ("encoder.0.bias", "encoder.fwd.0.bias")),
    ("enc.fc2.w", ("encoder.2.weight", "encoder.fwd.2.weight")), ("enc.fc2.b", ("encoder.2.bias", "encoder.fwd.2.bias")),
    ("pos_embed", ("pos_embed",)),
    ("dec.fc1.w", ("decoder.0.weight", "decoder.fwd.0.weight")), ("dec.fc1.b", ("decoder.0.bias", "decoder.fwd.0.bias")),
    ("dec.fc2.w", ("decoder.2.weight", "decoder.fwd.2.weight")), ("dec.fc2.b", ("decoder.2.bias", "decoder.fwd.2.bias")),
)
_SFNO_BLOCK_KEYS = (
    ("norm0.g", ("norm0.weight",)), ("norm0.b", ("norm0.bias",)), ("norm1.g", ("norm1.weight",)), ("norm1.b", ("norm1.bias",)),
    ("spec.w", ("filter.filter.weight", "filter.weight")), ("inner.w", ("inner_skip.weight",)), ("inner.b", ("inner_skip.bias",)),
    ("fc1.w", ("mlp.fwd.0.weight", "mlp.0.weight")), ("fc1.b", ("mlp.fwd.0.bias", "mlp.0.bias")),
    ("fc2.w", ("mlp.fwd.2.weight", "mlp.2.weight")), ("fc2.b", ("mlp.fwd.2.bias", "mlp.2.bias")),
)


def sfno_from_checkpoint(weights_path: str, means_path: str | None = None, stds_path: str | None = None):
    """torch.load(weights.tar)["model_state"] (+ global_means.npy / global_stds.npy) -> (SFNOConfig, parameter dict).
    Hyper-parameters are read off the tensor shapes (embed from the encoder, layers from the block count, internal grid
    from the spectral weight / positional embedding)."""
    import torch
    from .config import SFNOConfig
    ck = torch.load(weights_path, map_location="cpu", weights_only=False)
    sd = ck.get("model_state", ck) if isinstance(ck, dict) else ck
    sd = {k[7:] if k.startswith("module.") else k: v for k, v in sd.items()}
    sd = {k[6:] if k.startswith("model.") else k: v for k, v in sd.items()}

    def find(suffixes, prefix=""):
        for s in suffixes:
            if prefix + s in sd:
                return sd[prefix + s]
        raise KeyError(f"checkpoint has none of {[prefix + s for s in suffixes]}; keys start {list(sd)[:8]}")

    def arr(t):
        a = t.detach().cpu()
        if a.is_complex():
            a = torch.view_as_real(a)
        return a.float().numpy()

    out = OrderedDict()
    for name, sufs in _SFNO_KEYS:
        a = arr(find(sufs))
        if name.endswith(".w"):
            a = a.reshape(a.shape[0], a.shape[1])        # 1x1 conv (out, in, 1, 1) -> (out, in)
        if name == "pos_embed":
            a = a.reshape(a.shape[-3], a.shape[-2], a.shape[-1])
        out[name] = a
    E, Cin = out["enc.fc1.w"].shape
    L = 0
    while any(k.startswith(f"blocks.{L}.") for k in sd):
        L += 1
    for i in range(L):
        for name, sufs in _SFNO_BLOCK_KEYS:
            a = arr(find(sufs, f"blocks.{i}."))
            if name.endswith(".w") and name != "spec.w":
                a = a.reshape(a.shape[0], a.shape[1])
            if name == "spec.w":                          # checkpoint: (in, out, l[, 2]) complex dhconv weight -> [l, out, in, 2]
                if a.ndim == 4:
                    a = np.ascontiguousarray(a.transpose(2, 1, 0, 3))
                else:
                    raise ValueError(f"unexpected spectral weight shape {a.shape}")
            out[f"blk{i}.{name}"] = a
    lmax = out["blk0.spec.w"].shape[0]
    nlat, nlon = out["pos_embed"].shape[-2:]
    scale = max(1, round(nlat / lmax))
    cfg = SFNOConfig(nlat=nlat, nlon=nlon, n_channels=Cin, embed=E, layers=L, scale_factor=scale,
                     mlp_ratio=out["blk0.fc1.w"].shape[0] // E)
    if means_path and stds_path:
        out["norm.mean"] = np.load(means_path).reshape(-1)[:Cin].astype(np.float32)
        out["norm.std"] = np.load(stds_path).reshape(-1)[:Cin].astype(np.float32)
    else:
        from .config import FCNV2_CHANNELS
        from .weights import channel_stats
        out["norm.mean"], out["norm.std"] = channel_stats(FCNV2_CHANNELS)
    from .weights import sfno_param_shapes
    shapes = sfno_param_shapes(cfg)
    res = OrderedDict()
    for k, shp in shapes.items():
        a = np.ascontiguousarray(out[k], dtype=np.float32)
        if a.shape != tuple(shp):
            raise ValueError(f"{k}: checkpoint shape {a.shape} != expected {tuple(shp)}")
        res[k] = a
    return cfg, res


def fcn_from_checkpoint(weights_path: str, means_path: str, stds_path: str):
    """FourCastNet v1 checkpoint (torch.load state dict, top level or under "model_state", "module." prefix optional)
    + global_means.npy / global_stds.npy -> (FCNConfig, parameter dict).  Hyper-parameters come from the tensor shapes."""
    import torch
    from .config import FCNConfig
    from .weights import fcn_param_shapes
    ck = torch.load(weights_path, map_location="cpu", weights_only=False)
    sd = ck.get("model_state", ck) if isinstance(ck, dict) else ck
    sd = {(k[7:] if k.startswith("module.") else k): v.detach().cpu().float().numpy() for k, v in sd.items()}
    if "patch_embed.proj.weight" not in sd:
        raise KeyError(f"not a FourCastNet (AFNONet) state dict: no 'patch_embed.proj.weight'; keys start {list(sd)[:8]}")
    E, C, p, _ = sd["patch_embed.proj.weight"].shape
    T = sd["pos_embed"].shape[1]
    depth = 0
    while f"blocks.{depth}.norm1.weight" in sd:
        depth += 1
    _, nb, bs, _ = sd["blocks.0.filter.w1"].shape
    mlp_ratio = sd["blocks.0.mlp.fc1.weight"].shape[0] // E
    # the grid is not stored; the token count fixes it for the 1:2 aspect ratio of the global lat-lon grid
    w = int(round(np.sqrt(2 * T)))
    if w * (w // 2) != T or w % 2:
        raise ValueError(f"pos_embed has {T} tokens: not an h x 2h token grid")
    cfg = FCNConfig(nlat=p * (w // 2), nlon=p * w, n_channels=C, patch=p, embed=E, depth=depth, num_blocks=nb,
                    mlp_ratio=mlp_ratio)
    stats = {}
    for key, path in (("norm.mean", means_path), ("norm.std", stds_path)):
        a = np.squeeze(np.load(path))
        if a.shape != (C,):
            raise ValueError(f"{os.path.basename(path)} has shape {np.load(path).shape}: expected {C} values after squeeze")
        stats[key] = a.astype(np.float32)
    res = OrderedDict()
    for k, shp in fcn_param_shapes(cfg).items():
        a = stats[k] if k in stats else sd.get(k)
        if a is None:
            raise KeyError(f"checkpoint lacks '{k}'")
        a = np.ascontiguousarray(a, dtype=np.float32)
        if a.shape != tuple(shp):
            raise ValueError(f"{k}: checkpoint shape {a.shape} != expected {tuple(shp)}")
        res[k] = a
    return cfg, res


# ----------------------------------------------------------------------------------------
def check_fp16_range(weights, limit: float = 3.0e4):
    """The tensor cores receive fp16 operands (5 exponent bits): refuse weights whose magnitude would overflow, and report
    the largest |w| so that a caller can judge the head-room of the products."""
    worst = ("", 0.0)
    for k, v in weights.items():
        if k in ("norm.mean", "norm.std", "const.masks") or k.startswith(("sht.", "dft.")):
            continue
        m = float(np.max(np.abs(v))) if v.size else 0.0
        if not np.isfinite(m) or m > limit:
            raise ValueError(f"parameter '{k}' has |w|max = {m:.3g} > {limit:g}: outside the fp16 operand range of the engine")
        if m > worst[1]:
            worst = (k, m)
    return worst


def load_real_weights(model: str, path: str):
    """Entry used by the model wrappers when SKYRIM_B200_WEIGHTS points at real files."""
    if model == "pangu":
        p = path if path.endswith(".onnx") else os.path.join(path, "pangu_weather_6.onnx")
        w = pangu_from_onnx(p)
        check_fp16_range(w)
        return None, w
    d = path if os.path.isdir(path) else os.path.dirname(path)
    if model == "fcn":
        wp = path if os.path.isfile(path) else os.path.join(d, "weights.tar")
        cfg, w = fcn_from_checkpoint(wp, os.path.join(d, "global_means.npy"), os.path.join(d, "global_stds.npy"))
        check_fp16_range(w)
        return cfg, w
    wp = path if os.path.isfile(path) else os.path.join(d, "weights.tar")
    mp, sp = os.path.join(d, "global_means.npy"), os.path.join(d, "global_stds.npy")
    cfg, w = sfno_from_checkpoint(wp, mp if os.path.exists(mp) else None, sp if os.path.exists(sp) else None)
    check_fp16_range(w)
    return cfg, w
