"""Generate the committed golden fixtures under tests/golden/ from the fp64 oracle.

The reference ships no golden vectors for this path (SURVEY.md §8(c): "parity unpinned"), so
these pin the oracle against itself across refactors: seeded weights + IC -> sampled outputs.
    python tools/make_golden.py
"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from skyrim_b200.config import pangu_small, PANGU_CHANNELS
from skyrim_b200.weights import make_pangu_weights, synthetic_state
from oracle.pangu_ref import PanguRef

out = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
os.makedirs(out, exist_ok=True)
ONLY_GRAPHCAST = "--graphcast" in sys.argv   # leave the Pangu / SFNO fixtures untouched
ONLY_FCN = "--fcn" in sys.argv               # write only the FourCastNet fixture
if ONLY_FCN:
    from skyrim_b200.config import fcn_small, FCN_CHANNELS
    from skyrim_b200.weights import make_fcn_weights
    from oracle.afno_ref import FCNRef
    fcfg = fcn_small(48, 96, 2)
    fx0 = synthetic_state(FCN_CHANNELS, fcfg.nlat, fcfg.nlon, 0)
    fy = FCNRef(fcfg, make_fcn_weights(fcfg, 0), torch.float64).step(fx0).numpy()
    np.savez_compressed(os.path.join(out, "fcn_48x96_seed0.npz"), x0_sample=fx0[:, ::8, ::16].astype(np.float32),
                        y_sample=fy[:, ::5, ::12], y_norm=np.sqrt((fy ** 2).sum(axis=(1, 2))), y_mean=fy.mean(axis=(1, 2)))
    print("wrote", os.path.join(out, "fcn_48x96_seed0.npz"))
    sys.exit(0)
if not ONLY_GRAPHCAST:
    cfg = pangu_small(41, 96)
    w = make_pangu_weights(cfg, 0)
    x0 = synthetic_state(PANGU_CHANNELS, cfg.nlat, cfg.nlon, 0)
    y = PanguRef(cfg, w, torch.float64).step(x0).numpy()
    np.savez_compressed(os.path.join(out, "pangu_41x96_seed0.npz"),
                        x0_sample=x0[:, ::8, ::16].astype(np.float32), y_sample=y[:, ::5, ::12],
                        y_norm=np.sqrt((y ** 2).sum(axis=(1, 2))), y_mean=y.mean(axis=(1, 2)))
    print("wrote", os.path.join(out, "pangu_41x96_seed0.npz"))

    # ---- FourCastNet-v2 SFNO (small configuration of tests/test_sfno_*.py) ----
    from skyrim_b200.config import sfno_small, FCNV2_CHANNELS
    from skyrim_b200.weights import make_sfno_weights
    from oracle.sfno_ref import SFNORef

    scfg = sfno_small(49, 96, embed=64, layers=3)
    sw = make_sfno_weights(scfg, 0)
    sx0 = synthetic_state(FCNV2_CHANNELS, scfg.nlat, scfg.nlon, 0)
    sy = SFNORef(scfg, sw, torch.float64).step(sx0).numpy()
    np.savez_compressed(os.path.join(out, "sfno_49x96_seed0.npz"),
                        x0_sample=sx0[:, ::8, ::16].astype(np.float32), y_sample=sy[:, ::6, ::12],
                        y_norm=np.sqrt((sy ** 2).sum(axis=(1, 2))), y_mean=sy.mean(axis=(1, 2)))
    print("wrote", os.path.join(out, "sfno_49x96_seed0.npz"))

# ---- GraphCast (small configuration of tests/test_graphcast_*.py): the whole stepped state, fp64 oracle ----
from skyrim_b200 import icomesh
from skyrim_b200.config import graphcast_small
from skyrim_b200.weights import make_graphcast_weights, synthetic_graphcast_state
from oracle.graphcast_ref import GraphCastRef, toa_radiation

if True:
    gcfg = graphcast_small(41, 96, 2, 512, 2)
    graph = icomesh.build_graph(gcfg.nlat, gcfg.nlon, gcfg.mesh_levels, gcfg.radius_frac)
    gw = make_graphcast_weights(gcfg, 0)
    gx = synthetic_graphcast_state(gcfg, 0)
    T0 = 1714521600.0   # 2024-05-01T00:00:00Z, valid time of the second slice
    lat = np.linspace(90.0, -90.0, gcfg.nlat); lon = np.arange(gcfg.nlon) * (360.0 / gcfg.nlon)
    gx[gcfg.n_state - 1] = toa_radiation(T0 - 21600.0, lat, lon)
    gx[2 * gcfg.n_state - 1] = toa_radiation(T0, lat, lon)
    gy = GraphCastRef(gcfg, gw, graph, torch.float64).step(gx, T0).numpy()
    np.savez_compressed(os.path.join(out, "graphcast_41x96_seed0.npz"), prog_sample=gy[83:165, ::2, ::3].astype(np.float32),
                        prog_norm=np.sqrt((gy[83:165] ** 2).sum(axis=(1, 2))), t0=T0)
    print("wrote", os.path.join(out, "graphcast_41x96_seed0.npz"))
