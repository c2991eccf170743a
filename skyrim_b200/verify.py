"""Compare a full-size (721x1440) step output with the committed sampled oracle fixture
(tests/golden/*_721x1440_seed0.npz, written by tools/make_golden_full.py from one real oracle step).

Used by tests/test_fullsize_gpu.py and by bench.py to check the TIMED output (not only `isfinite`).
No oracle code is imported: the fixture holds numbers, this module holds comparisons."""
from __future__ import annotations

import os

import numpy as np

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def load_fixture(model: str, nlat: int = 721):
    path = os.path.join(GOLDEN_DIR, f"{model}_{nlat}x1440_seed0.npz")
    if not os.path.exists(path):
        raise FileNotFoundError(f"{path} missing: run tools/make_golden_full.py {model}")
    return np.load(path)


def compare_fullsize(y, fx, last_row: int = 720) -> dict:
    """y: (C, 721, 1440) torch tensor (any device) or ndarray (FourCastNet: (C, 720, 1440) with last_row=719).
    Returns per-channel error vectors:
      rel      ||y_s - ref_s||_2 / ||ref_s||_2 over the strided point sample (north-star metric, sampled)
      nrm      RMS(y_s - ref_s) / std_c            (in units of the channel's standard deviation: stricter
                                                    for channels whose mean dominates their norm)
      block    max |blockmean16x16(y) - ref| / std_c  over ALL pixels of rows 0..719 (a wrong tile shows here)
      last     max |y[last_row, ::4] - ref| / std_c
      norm     | ||y||_2 / ||ref||_2 - 1 |
    """
    import torch
    t = y if isinstance(y, torch.Tensor) else torch.from_numpy(np.asarray(y))
    t = t.detach()
    C = t.shape[0]
    dev = t.device
    f64 = lambda a: torch.from_numpy(np.asarray(a, dtype=np.float64)).to(dev)
    ref_s, ref_b, ref_l = f64(fx["y_sample"]), f64(fx["y_block"]), f64(fx["y_last"])
    std = f64(fx["y_std"]).clamp_min(1e-30)
    ys = t[:, ::13, ::17].double()
    d = ys - ref_s
    rel = d.pow(2).sum(dim=(1, 2)).sqrt() / ref_s.pow(2).sum(dim=(1, 2)).sqrt()
    nrm = d.pow(2).mean(dim=(1, 2)).sqrt() / std
    blk = t[:, :720].double().reshape(C, 45, 16, 90, 16).mean(dim=(2, 4))
    block = (blk - ref_b).abs().amax(dim=(1, 2)) / std
    last = (t[:, last_row, ::4].double() - ref_l).abs().amax(dim=1) / std
    norm = (t.double().pow(2).sum(dim=(1, 2)).sqrt() / f64(fx["y_norm"]) - 1.0).abs()
    out = {k: v.cpu().numpy() for k, v in dict(rel=rel, nrm=nrm, block=block, last=last, norm=norm).items()}
    out["finite"] = bool(torch.isfinite(t).all())
    return out


def summarise(cmp: dict) -> dict:
    return {k: (float(np.max(v)) if k != "finite" else v) for k, v in cmp.items()}


def compare_graphcast(y, x, diff_std, fx, cfg) -> dict:
    """GraphCast full-size check.  y, x: (2 * n_state, 721, 1440) new / old state tensors; the fixture holds the oracle's
    82 prognostic channels of the NEW slice (y_*) and the network's tendency (t_*, in units of diff_std).  Returns the
    maxima over channels of the `compare_fullsize` metrics for the state and, as t_rel / t_block, for the tendency
    (state = x + 0.1 sigma * tendency, so a 1e-3 state bound alone would tolerate a 1e-2 error of the network)."""
    import torch
    ns, npg = cfg.n_state, cfg.n_prog
    y = y if isinstance(y, torch.Tensor) else torch.from_numpy(np.asarray(y))
    x = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.asarray(x))
    new = y[ns:ns + npg]
    s = summarise(compare_fullsize(new, fx))
    ds = torch.from_numpy(np.asarray(diff_std, dtype=np.float32))[:npg].to(new.device)
    tend = (new - x[ns:ns + npg].to(new.device)) / ds[:, None, None]
    tfx = {"y_" + k[2:]: fx[k] for k in fx.files if k.startswith("t_")}
    t = summarise(compare_fullsize(tend, tfx))
    s.update(t_rel=t["rel"], t_block=t["block"], t_norm=t["norm"])
    s["slice0_is_old_slice1"] = bool(torch.equal(y[:ns], x[ns:].to(y.device)))
    return s
