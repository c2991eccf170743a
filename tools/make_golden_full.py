"""Full-size (BASELINE.json shape, 721x1440) sampled fixtures from ONE real oracle step per model:

    python tools/make_golden_full.py pangu      # ~5 min on 8 host threads, ~20 GB RAM
    python tools/make_golden_full.py sfno       # E=384, L=8: ~10 min
    python tools/make_golden_full.py fcn        # FourCastNet v1 (AFNO), 720 x 1440, 12 blocks: writes fcn_720x1440_seed0.npz,
                                                # y_last = the last (720th) row
    python tools/make_golden_full.py graphcast  # refinement-6 multimesh, 16 layers: ~10 min, ~30 GB RAM; the fixture holds the
                                                # 82 prognostic channels of the NEW time slice and, as t_*, the same summaries
                                                # of the network's tendency (state = x + 0.1 sigma x tendency: a 1e-3 bound on the
                                                # state alone would hide a 1e-2 error of the network)

writes tests/golden/{pangu,sfno}_721x1440_seed0.npz holding, per channel,
  y_sample   y[:, ::13, ::17]                   point values (56 x 85): strides 13 / 17 are coprime to the 4x4 patch and the 12-token windows, so the
                                                sample visits every intra-patch position (a stride of 16 saw only position (0, 0))
  y_block    16x16 block means of y[:, :720]    every pixel of rows 0..719 enters exactly one mean (45 x 90)
  y_last     y[:, 720, ::4]                     the odd last latitude row (padding edge of the patch grid)
  y_norm, y_mean, y_std                         per-channel L2 norm / mean / standard deviation of the full field
so that tests/test_fullsize_gpu.py and bench.py can compare a full-size CUDA step with the oracle without
re-running it (the GPU box has no /root/reference and its minutes are budgeted).  Seeded weights and IC are
regenerated bit-identically from skyrim_b200/weights.py; x0_sample pins that.
"""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, torch


def summarise(y, last_row=720):
    y = np.asarray(y, dtype=np.float64)
    blk = y[:, :720].reshape(y.shape[0], 45, 16, 90, 16).mean(axis=(2, 4))
    return dict(y_sample=y[:, ::13, ::17].astype(np.float32), y_block=blk.astype(np.float32),
                y_last=y[:, last_row, ::4].astype(np.float32), y_norm=np.sqrt((y ** 2).sum(axis=(1, 2))),
                y_mean=y.mean(axis=(1, 2)), y_std=y.std(axis=(1, 2)))


def main(which):
    out = os.path.join(ROOT, "tests", "golden")
    t0 = time.time()
    if which == "pangu":
        from skyrim_b200.config import PANGU_CHANNELS, pangu_full
        from skyrim_b200.weights import make_pangu_weights, synthetic_state
        from oracle.pangu_ref import PanguRef
        cfg = pangu_full()
        w = make_pangu_weights(cfg, 0)
        x0 = synthetic_state(PANGU_CHANNELS, cfg.nlat, cfg.nlon, 0)
        y = PanguRef(cfg, w, torch.float32).step(x0).numpy()
    elif which == "graphcast":
        from skyrim_b200 import icomesh
        from skyrim_b200.config import graphcast_full
        from skyrim_b200.weights import make_graphcast_weights, synthetic_graphcast_state
        from oracle.graphcast_ref import GraphCastRef, toa_radiation
        cfg = graphcast_full()
        graph = icomesh.build_graph(cfg.nlat, cfg.nlon, cfg.mesh_levels, cfg.radius_frac)
        w = make_graphcast_weights(cfg, 0)
        x0 = synthetic_graphcast_state(cfg, 0)
        T0 = 1714521600.0   # 2024-05-01T00:00:00Z = valid time of the second slice
        lat = np.linspace(90.0, -90.0, cfg.nlat); lon = np.arange(cfg.nlon) * (360.0 / cfg.nlon)
        x0[cfg.n_state - 1] = toa_radiation(T0 - 21600.0, lat, lon)
        x0[2 * cfg.n_state - 1] = toa_radiation(T0, lat, lon)
        print(f"graph + weights + IC: {time.time() - t0:.1f} s", flush=True)
        ynew, tend = GraphCastRef(cfg, w, graph, torch.float32).step(x0, T0, return_tendency=True)
        y = ynew.numpy()[cfg.n_state:cfg.n_state + cfg.n_prog]
        extra = {"t_" + k[2:]: v for k, v in summarise(tend.numpy().T.reshape(cfg.n_prog, cfg.nlat, cfg.nlon)).items()}
        extra["t0"] = np.float64(T0)
    elif which == "fcn":
        from skyrim_b200.config import FCN_CHANNELS, fcn_full
        from skyrim_b200.weights import make_fcn_weights, synthetic_state
        from oracle.afno_ref import FCNRef
        cfg = fcn_full()
        w = make_fcn_weights(cfg, 0)
        x0 = synthetic_state(FCN_CHANNELS, cfg.nlat, cfg.nlon, 0)
        y = FCNRef(cfg, w, torch.float32).step(x0).numpy()
    else:
        from skyrim_b200.config import FCNV2_CHANNELS, sfno_full
        from skyrim_b200.weights import make_sfno_weights, synthetic_state
        from oracle.sfno_ref import SFNORef
        cfg = sfno_full()
        w = make_sfno_weights(cfg, 0)
        x0 = synthetic_state(FCNV2_CHANNELS, cfg.nlat, cfg.nlon, 0)
        y = SFNORef(cfg, w, torch.float32).step(x0).numpy()
    d = summarise(y, last_row=y.shape[1] - 1)
    if which == "graphcast":
        d.update(extra)
    d["x0_sample"] = x0[:, ::64, ::64].astype(np.float32)
    d["oracle_seconds"] = np.float64(time.time() - t0)
    d["oracle_threads"] = np.int64(torch.get_num_threads())
    path = os.path.join(out, f"{which}_{y.shape[1]}x1440_seed0.npz")
    np.savez_compressed(path, **d)
    print("wrote", path, os.path.getsize(path), "bytes;", f"{time.time() - t0:.1f} s")


if __name__ == "__main__":
    main(sys.argv[1])
