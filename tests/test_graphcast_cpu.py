"""GraphCast host side on the CPU: the icosahedral multimesh and the grid<->mesh edge sets (skyrim_b200/icomesh.py), the
oracle (oracle/graphcast_ref.py) against its committed fp64 fixture, and the algebraic rewrites the CUDA engine relies on."""
import os

import numpy as np
import pytest
import torch

from oracle.graphcast_ref import GraphCastRef, day_progress, rel_err_per_channel, toa_radiation, year_progress
from skyrim_b200 import icomesh
from skyrim_b200.config import GRAPHCAST_CHANNELS, graphcast_full, graphcast_small
from skyrim_b200.weights import graphcast_param_shapes, make_graphcast_weights, n_params, synthetic_graphcast_state

T0 = 1714521600.0


@pytest.fixture(scope="module")
def small():
    cfg = graphcast_small(41, 96, 2, 512, 2)
    graph = icomesh.build_graph(cfg.nlat, cfg.nlon, cfg.mesh_levels, cfg.radius_frac)
    w = make_graphcast_weights(cfg, 0)
    x = synthetic_graphcast_state(cfg, 0)
    lat = np.linspace(90.0, -90.0, cfg.nlat); lon = np.arange(cfg.nlon) * (360.0 / cfg.nlon)
    x[cfg.n_state - 1] = toa_radiation(T0 - 21600.0, lat, lon)
    x[2 * cfg.n_state - 1] = toa_radiation(T0, lat, lon)
    return cfg, graph, w, x


# -- mesh ---------------------------------------------------------------------------------------------------------
def test_multimesh_counts_match_the_published_mesh():
    """refinement 6: 40,962 nodes, 81,920 faces, 327,660 directed multimesh edges (SURVEY.md §8(a) A9)"""
    v, f, s, r = icomesh.multimesh(6)
    assert (len(v), len(f), len(s)) == (40962, 81920, 327660)
    assert np.allclose(np.linalg.norm(v, axis=1), 1.0, atol=1e-12)
    pairs = set(zip(s.tolist(), r.tolist()))
    assert len(pairs) == len(s) and all((b, a) in pairs for a, b in list(pairs)[:5000]), "edges are bidirectional, no duplicates"
    # the multimesh keeps the coarse edges: the 12 original vertices have 5 neighbours on each of the 7 levels
    deg = np.bincount(r, minlength=len(v))
    assert (deg[:12] == 35).all() and deg.max() == 36 and deg[12:].min() == 6   # level-1 vertices: 6 x 6 levels
    # every level's vertices are a prefix of the next one's (coarse nodes keep their indices)
    v3, _, _, _ = icomesh.multimesh(3)
    assert np.array_equal(v3, v[:len(v3)])


def test_faces_are_outward_oriented_and_cover_the_sphere():
    v, f, _, _ = icomesh.multimesh(3)
    a, b, c = v[f[:, 0]], v[f[:, 1]], v[f[:, 2]]
    assert (np.einsum("ij,ij->i", np.cross(b - a, c - a), a + b + c) > 0).all()
    # solid angles of the spherical triangles add up to 4 pi
    num = np.einsum("ij,ij->i", a, np.cross(b, c))
    den = 1 + np.einsum("ij,ij->i", a, b) + np.einsum("ij,ij->i", b, c) + np.einsum("ij,ij->i", c, a)
    assert abs(2 * np.arctan2(num, den).sum() - 4 * np.pi) < 1e-9


def test_graph_tables(small):
    cfg, g, _, _ = small
    ng, nm = g["n_grid"], g["n_mesh"]
    assert ng == 41 * 96 and nm == 162
    for key, n_recv in (("mesh", nm), ("g2m", nm)):
        s, r, ptr = g[f"{key}.senders"], g[f"{key}.receivers"], g[f"{key}.ptr"]
        assert (np.diff(r) >= 0).all() and ptr[0] == 0 and ptr[-1] == len(s) and len(ptr) == n_recv + 1
        assert np.array_equal(np.bincount(r, minlength=n_recv), np.diff(ptr)), "CSR segments = incoming edges per receiver"
        f = g[f"{key}.edge_feat"]
        assert f.shape == (len(s), 4) and abs(f[:, 0].max() - 1.0) < 1e-6, "lengths are normalised by the longest edge"
        assert np.allclose(np.linalg.norm(f[:, 1:], axis=1), f[:, 0], atol=1e-6)
    # every grid point reaches the mesh, and lies inside the triangle whose vertices send to it
    assert len(np.unique(g["g2m.senders"])) == ng
    gp, _, _ = icomesh.grid_points(cfg.nlat, cfg.nlon)
    v = g["mesh.xyz"]
    tri = g["m2g.senders"].reshape(3, ng)
    a, b, c = v[tri[0]], v[tri[1]], v[tri[2]]
    for n in (np.cross(a, b), np.cross(b, c), np.cross(c, a)):
        assert (np.einsum("ij,ij->i", gp, n) >= -1e-9).all()
    assert np.array_equal(g["m2g.receivers"], np.tile(np.arange(ng), 3))
    # grid2mesh radius rule
    faces = g["mesh.faces"]
    ff = np.concatenate([faces[:, [0, 1]], faces[:, [1, 2]], faces[:, [2, 0]]])
    max_len = np.linalg.norm(v[ff[:, 0]] - v[ff[:, 1]], axis=1).max()
    d = np.linalg.norm(gp[g["g2m.senders"]] - v[g["g2m.receivers"]], axis=1)
    assert d.max() <= cfg.radius_frac * max_len + 1e-12
    brute = (np.linalg.norm(gp[:, None, :] - v[None, :, :], axis=-1) <= cfg.radius_frac * max_len).sum()
    assert brute == len(d), "the KD-tree query found every (grid point, mesh node) pair within the radius"


def test_edge_features_are_in_the_receiver_frame():
    """a sender due east of a receiver on the equator has a positive local y; one due north a positive local z"""
    recv = icomesh.latlon_to_xyz(np.array([0.0, 40.0]), np.array([30.0, -100.0]))
    east = icomesh.latlon_to_xyz(np.array([0.0, 40.0]), np.array([31.0, -99.0]))
    north = icomesh.latlon_to_xyz(np.array([1.0, 41.0]), np.array([30.0, -100.0]))
    de, dn = icomesh._local_frame_delta(east, recv), icomesh._local_frame_delta(north, recv)
    assert (de[:, 1] > 0).all() and (np.abs(de[:, 2]) < 2e-4).all()
    assert (dn[:, 2] > 0).all() and (np.abs(dn[:, 1]) < 1e-12).all()
    assert (de[:, 0] < 0).all() and (dn[:, 0] < 0).all()   # chords dip below the tangent plane


def test_arena_entries_are_exact_in_fp32(small):
    _, g, _, _ = small
    ent = icomesh.graph_arena_entries(g)
    assert all(v.dtype == np.float32 for v in ent.values())
    for k in ("mesh.senders", "g2m.senders", "m2g.senders", "mesh.ptr", "g2m.ptr"):
        assert np.array_equal(ent["graph." + k].astype(np.int64), np.asarray(g[k]))


# -- configuration / weights ------------------------------------------------------------------------------------------
def test_channels_and_parameter_count():
    """83 channels in the order the reference's _to_global_da emits (graphcast.py:29-41, 68-91); the same set as its
    CHANNELS list (:17-26), which is what the reference's own test compares (tests/core/test_graphcast.py:22)"""
    ref_channels = [f"{v}{p}" for v in "zqtuvw" for p in (50, 100, 150, 200, 250, 300, 400, 500, 600, 700, 850, 925, 1000)] + [
        "u10m", "v10m", "t2m", "msl", "tp06"]
    assert len(GRAPHCAST_CHANNELS) == 83 and set(GRAPHCAST_CHANNELS) == set(ref_channels)
    assert GRAPHCAST_CHANNELS[0] == "q50" and GRAPHCAST_CHANNELS[13] == "z50" and GRAPHCAST_CHANNELS[-5:] == ["t2m", "u10m", "v10m", "msl", "tp06"]
    cfg = graphcast_full()
    assert cfg.n_features == 184 and cfg.n_channels == 166
    shapes = graphcast_param_shapes(cfg)
    n = sum(int(np.prod(s)) for k, s in shapes.items() if k.startswith(("enc.", "proc", "dec.")))
    # published: 36.7 M parameters; here without the decoder's unused mesh-node MLP (0.8 M) and the zero data block of the
    # mesh-node embedding (0.1 M)
    assert 35.0e6 < n < 37.0e6, n


def test_forcing_formulas():
    # 2024-03-20 03:06 UTC is the March equinox: declination ~ 0, the sub-solar point is on the equator
    lat = np.linspace(90.0, -90.0, 181); lon = np.arange(360) * 1.0
    t = 1710903960.0
    toa = toa_radiation(t, lat, lon)
    i, j = np.unravel_index(np.argmax(toa), toa.shape)
    assert abs(lat[i]) <= 3.0 and toa.min() == 0.0 and 4.5e6 < toa.max() < 5.1e6
    assert abs(((lon[j] + 180.0) % 360.0 - 180.0) - (180.0 - 360.0 * ((t / 86400.0) % 1.0))) <= 1.0, "local noon at the maximum"
    assert 0.0 <= year_progress(t) < 1.0 and np.allclose(day_progress(0.0, np.array([0.0, 90.0, 180.0])), [0.0, 0.25, 0.5])


# -- oracle -----------------------------------------------------------------------------------------------------------
def test_oracle_matches_committed_fp64_fixture(small):
    cfg, g, w, x = small
    fix = np.load(os.path.join(os.path.dirname(__file__), "golden", "graphcast_41x96_seed0.npz"))
    y = GraphCastRef(cfg, w, g).step(x, T0).numpy()
    assert y.shape == (166, 41, 96)
    err = rel_err_per_channel(y[83:165, ::2, ::3], fix["prog_sample"])
    assert err.max() < 2e-6, err.max()
    assert np.allclose(np.sqrt((y[83:165].astype(np.float64) ** 2).sum(axis=(1, 2))), fix["prog_norm"], rtol=1e-6)
    assert np.array_equal(y[:83], x[83:])
    assert np.allclose(y[165], toa_radiation(T0 + 21600.0, np.linspace(90, -90, 41), np.arange(96) * 3.75), rtol=1e-6)


def test_fp16_operand_error_budget(small):
    """fp16 tensor-core operands (and fp16 per-node tables) stay inside the 1e-3 state budget"""
    cfg, g, w, x = small
    ref = GraphCastRef(cfg, w, g, dtype=torch.float64).step(x, T0).numpy()
    for em in ("fp16", "fp16t", "fp16s"):
        y = GraphCastRef(cfg, w, g, emulate=em).step(x, T0).numpy()
        err = rel_err_per_channel(y[83:165], ref[83:165])
        assert err.max() < 5e-4, (em, err.max())


def test_fp16_residual_streams_cost_little(small):
    """the engine keeps grid-node and mesh-edge latents only as fp16 operand images: on the oracle that costs a few per
    cent of the (already fp16-operand) tendency error"""
    cfg, g, w, x = small
    t64 = GraphCastRef(cfg, w, g, dtype=torch.float64).tendency(x, T0)
    err = {}
    for em in ("fp16t", "fp16s"):
        t = GraphCastRef(cfg, w, g, emulate=em).tendency(x, T0)
        err[em] = float((t - t64).norm() / t64.norm())
    assert err["fp16s"] < 1.15 * err["fp16t"] and err["fp16s"] < 1e-3, err


def test_engine_rewrites_are_identities_of_the_oracle(small):
    """(1) concat([e, vs, vr]) W1^T = e W1e^T + (v W1s^T)[s] + (v W1r^T)[r];  (2) mesh2grid: [v, sum_k e_k] W1^T =
    [v | e_0 | e_1 | e_2] [W1v | W1a | W1a | W1a]^T with k-major edge rows;  (3) CSR segment sums = index_add."""
    cfg, g, w, _ = small
    L = cfg.latent
    rng = np.random.default_rng(0)
    nm, ng = g["n_mesh"], g["n_grid"]
    t = lambda a: torch.from_numpy(np.asarray(a)).double()
    v = t(rng.standard_normal((nm, L))); e = t(rng.standard_normal((len(g["mesh.senders"]), L)))
    s, r = torch.from_numpy(g["mesh.senders"]), torch.from_numpy(g["mesh.receivers"])
    W1 = t(w["proc0.edge.w1"])
    naive = torch.cat([e, v[s], v[r]], 1) @ W1.T
    split = e @ W1[:, :L].T + (v @ W1[:, L:2 * L].T)[s] + (v @ W1[:, 2 * L:].T)[r]
    assert torch.allclose(naive, split, rtol=1e-10, atol=1e-10)
    vg = t(rng.standard_normal((ng, L))); ek = t(rng.standard_normal((3 * ng, L)))
    Wg = t(w["dec.m2g_grid.w1"])
    agg = torch.zeros(ng, L, dtype=torch.float64).index_add_(0, torch.from_numpy(g["m2g.receivers"]), ek)
    naive = torch.cat([vg, agg], 1) @ Wg.T
    kcat = torch.cat([vg, ek[:ng], ek[ng:2 * ng], ek[2 * ng:]], 1) @ torch.cat([Wg[:, :L]] + [Wg[:, L:]] * 3, 1).T
    assert torch.allclose(naive, kcat, rtol=1e-10, atol=1e-10)
    ptr = g["mesh.ptr"]
    seg = torch.stack([e[ptr[n]:ptr[n + 1]].sum(0) for n in range(nm)])
    assert torch.allclose(seg, torch.zeros(nm, L, dtype=torch.float64).index_add_(0, r, e), rtol=1e-12, atol=1e-12)


def test_library_exports_graphcast_symbols():
    from skyrim_b200 import _ffi
    L = _ffi.lib()
    for name in ("sky_model_set_clock", "sky_toa_radiation"):
        assert hasattr(L, name)
    assert _ffi.SKY_MODEL_GRAPHCAST == 3


# -- host logic of the model wrapper on a CPU fake of the stepper protocol --------------------------------------------------
class _FakeStepper:
    """stepper protocol of /root/reference/skyrim/core/models/graphcast.py:110,118 on the CPU: new slice = last slice + 1"""
    def __init__(self, loop):
        self.loop = loop

    def initialize(self, x, time):
        return (time, x.float().clone(), None)

    def step(self, state):
        time, fields, rng = state
        new = torch.stack([fields[:, 1], fields[:, 1] + 1.0], dim=1)
        return (time + self.loop.time_step, new, rng), new[:, -1]


class _FakeLoop:
    import datetime as _dt
    n_history_levels = 2
    time_step = _dt.timedelta(hours=6)
    channel_names = in_channel_names = out_channel_names = GRAPHCAST_CHANNELS
    device = torch.device("cpu")

    def __init__(self, nlat=9, nlon=16):
        from skyrim_b200.timeloop import equiangular_grid
        self.grid = equiangular_grid(nlat, nlon)
        self.stepper = _FakeStepper(self)

    def fill_forcing(self, x, time):
        x[:, :, -1] = 7.0
        return x


def test_graphcast_model_host_logic_on_a_fake_stepper(tmp_path):
    """rollout / forecast / predict_one_step of GraphcastModel (time coordinates, two-slice files, channel names) without a GPU"""
    import datetime
    from skyrim_b200 import xr_shim as xr
    from skyrim_b200.core.models.graphcast import GraphcastModel

    class Fake(GraphcastModel):
        def build_model(self):
            return _FakeLoop(self._cfg.nlat, self._cfg.nlon)

    m = Fake(ic_source="synthetic", cfg=graphcast_small(9, 16, 1, 512, 1))
    assert m.time_steps(13) == 2 and set(m.out_channel_names) == set(GRAPHCAST_CHANNELS)
    t0 = datetime.datetime(2024, 4, 4)
    pred, paths = m.rollout(t0, n_steps=3, save=True, save_config=dict(output_dir=str(tmp_path), file_type="netcdf"))
    assert pred.shape == (2, 83, 9, 16) and len(paths) == 3
    assert [str(t)[:13] for t in pred.coords["time"]] == ["2024-04-04T12", "2024-04-04T18"]
    np.testing.assert_allclose(pred.values[1], pred.values[0] + 1.0)
    assert paths[0].split("/")[-1].startswith("graphcast__synthetic__20240404_00:00__20240404_06:00")
    assert paths[1].split("/")[-1].startswith("graphcast__file__20240404_06:00__20240404_12:00")
    back = xr.open_dataarray(paths[2])
    np.testing.assert_array_equal(back.values, pred.values)
    f = m.forecast(t0, n_steps=2, channels=["t2m", "tp06"])
    assert f.shape == (3, 2, 9, 16) and list(f.coords["channel"]) == ["t2m", "tp06"]
    assert float(f.values[0, 1].max()) == 7.0, "the forcing channel of the initial condition was filled through the time loop"
    one = m.predict_one_step(t0)
    np.testing.assert_allclose(one.values[1], one.values[0] + 1.0)


def test_roofline_accounting_of_the_engine_formulation():
    """bench.py's per-family roofline for configs.graphcast: FLOPs and mandatory HBM bytes of the step as the engine runs it
    (first layers split per input, fp16-only grid-node / mesh-edge streams) — DESIGN.md section 4c quotes these figures"""
    from skyrim_b200 import roofline as R
    cfg = graphcast_full()
    fl, by = R.graphcast_flops(cfg), R.graphcast_bytes(cfg)
    assert abs(fl["total"] - 17.46e12) < 0.1e12 and abs(by["total"] - 100.5e9) < 1.5e9, (fl["total"], by["total"])
    assert fl["gc_hidden"] > fl["gc_ln"] > fl["gc_table"] > fl["gc_out"] > 0 and fl["gc_agg"] == 0
    naive = 2.0 * 512 * (cfg.n_grid * (184 + 512) + 1629780 * 4 * 512 + 40962 * 3 * 512 + cfg.n_grid * 2 * 512
                         + 16 * (327660 * 4 * 512 + 40962 * 3 * 512) + 3 * cfg.n_grid * 4 * 512 + cfg.n_grid * 3 * 512 + cfg.n_grid * 512)
    assert naive > 1.4 * fl["total"], "the published concatenated formulation needs ~1.5 x the engine's FLOPs"
    small_cfg = graphcast_small(41, 96, 2, 512, 2)
    g = icomesh.build_graph(41, 96, 2)
    assert R.graphcast_flops(small_cfg, g)["total"] < 1e11
