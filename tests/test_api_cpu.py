"""API-shape tests mirroring the reference's own (tests/test_common.py:32-54 writer round trip,
tests/core/test_base.py:8-27 fake TimeLoop, tests/core/test_graphcast.py:11-22 dims / channel
names) on a CPU fake of the TimeLoop protocol — no GPU needed."""
import datetime

import numpy as np
import pytest
import torch

from skyrim_b200 import xr_shim as xr
from skyrim_b200.common import SaveConfig, generate_filename, generate_forecast_id, save_forecast
from skyrim_b200.core.models.base import (GlobalModel, GlobalPrediction, GlobalPredictionRollout,
                                          SyntheticDataSource, adjust_lead_time)
from skyrim_b200.core.models.utils import run_basic_inference
from skyrim_b200.timeloop import equiangular_grid

CH = ["u1000", "v1000", "t2m", "msl"]


class BoringTimeLoop:
    """TimeLoop protocol fake (reference: tests/core/test_base.py BoringModel): x -> x + 1."""
    n_history_levels = 1
    time_step = datetime.timedelta(hours=6)
    in_channel_names = out_channel_names = CH
    grid = equiangular_grid(19, 36)
    device = torch.device("cpu")

    def __call__(self, time, x):
        cur = x[:, -1].float()
        yield time, cur.clone(), None
        while True:
            cur = cur + 1.0
            time = time + self.time_step
            yield time, cur.clone(), None


class BoringGlobalModel(GlobalModel):
    def __init__(self, **kw):
        super().__init__("boring", **kw)

    def build_model(self):
        return BoringTimeLoop()


def mock_forecast():
    # reference tests/test_common.py:11-29
    return xr.DataArray(np.random.rand(1, 2, 181, 361).astype(np.float32), dims=["time", "channel", "lat", "lon"],
                        coords=dict(time=np.array(["2024-05-07T06"], dtype="datetime64[s]"), channel=np.array(["u10m", "v10m"]),
                                    lat=np.linspace(90, -90, 181), lon=np.linspace(0, 360, 361)))


def test_adjust_lead_time():
    assert [adjust_lead_time(h) for h in (0, 5, 6, 7, 13, 168)] == [6, 6, 6, 6, 12, 168]


def test_save_forecast_netcdf_roundtrip(tmp_path):
    pred = mock_forecast()
    st, pt = datetime.datetime(2024, 5, 7), datetime.datetime(2024, 5, 7, 6)
    path = save_forecast(pred, "test_model", st, pt, "cds", config=dict(output_dir=str(tmp_path), forecast_id="fid", file_type="netcdf"))
    assert path == str(tmp_path / "fid" / "test_model__cds__20240507_00:00__20240507_06:00.nc")
    back = xr.open_dataarray(path)
    assert back.shape == (1, 2, 181, 361)
    np.testing.assert_array_equal(back.values, pred.values)
    assert list(back.coords["channel"]) == ["u10m", "v10m"]


def test_save_forecast_zarr_appends_along_time(tmp_path):
    pred = mock_forecast()
    st, pt = datetime.datetime(2024, 5, 7), datetime.datetime(2024, 5, 7, 6)
    cfg = dict(output_dir=str(tmp_path), forecast_id="z", file_type="zarr")
    p = save_forecast(pred, "m", st, pt, "cds", config=cfg)
    save_forecast(pred, "m", st, pt, "file", config=cfg)
    back = xr.open_dataarray(p)
    assert back.shape == (2, 2, 181, 361) and back.dims == ("time", "channel", "lat", "lon")


def test_save_forecast_rejects_remote_and_bad_type(tmp_path):
    with pytest.raises(NotImplementedError):
        save_forecast(mock_forecast(), "m", datetime.datetime(2024, 1, 1), datetime.datetime(2024, 1, 1, 6), config=dict(output_dir="s3://bucket/x"))
    with pytest.raises(ValueError):
        save_forecast(mock_forecast(), "m", datetime.datetime(2024, 1, 1), datetime.datetime(2024, 1, 1, 6), config=dict(output_dir=str(tmp_path), file_type="grib"))


def test_forecast_id_and_filename():
    a = generate_forecast_id()
    assert len(a) == 10 and a.isalnum() and len(SaveConfig().forecast_id) == 10
    assert generate_filename("pangu", datetime.datetime(2024, 5, 7), datetime.datetime(2024, 5, 7, 6), "gfs") == \
        "pangu__gfs__20240507_00:00__20240507_06:00.nc"


def test_run_basic_inference_yields_ic_first():
    m = BoringTimeLoop()
    src = SyntheticDataSource(CH, 19, 36)
    t0 = datetime.datetime(2024, 5, 7)
    da = run_basic_inference(m, n=3, data_source=src, time=t0)
    assert da.dims == ("time", "channel", "lat", "lon") and da.shape == (4, 4, 19, 36)
    np.testing.assert_array_equal(da.values[0], src[t0].values)       # first slice is the IC (utils.py:34-40)
    np.testing.assert_allclose(da.values[3], src[t0].values + 3.0)
    assert list(da.coords["channel"]) == CH


def test_rollout_predict_and_accessors(tmp_path):
    gm = BoringGlobalModel(ic_source="synthetic")
    t0 = datetime.datetime(2024, 5, 7)
    pred, paths = gm.rollout(t0, n_steps=3, save=True, save_config=dict(output_dir=str(tmp_path), file_type="netcdf"))
    assert pred.shape == (2, 4, 19, 36) and len(paths) == 3          # last prediction holds 2 time slices (base.py:146)
    names = [p.split("/")[-1] for p in paths]
    assert names[0].startswith("boring__synthetic__20240507_00:00__20240507_06:00")
    assert names[1].startswith("boring__file__20240507_06:00__20240507_12:00")
    gp = GlobalPrediction(pred, model_name="boring")
    u = gp.point(lat=0.0, lon=-10.0, channel="u1000", n_step=1)        # negative lon wraps (base.py:230-231)
    assert np.isclose(u, float(pred.sel(channel="u1000").isel(time=1).sel(lat=0.0, lon=350.0).item()))
    ws = gp.wind_speed(lat=0.0, lon=350.0, pressure_level=1000)
    uu, vv = gp.point_wind_uv(0.0, 350.0, 1000)
    assert np.isclose(ws, (uu ** 2 + vv ** 2) ** 0.5)
    roll = GlobalPredictionRollout(paths)
    assert len(roll.wind_speed(0.0, 350.0, 1000)) == 3
    # resume from a saved step == continuing the original rollout (TODO at base.py:127)
    pred2, _ = gm.rollout(t0 + datetime.timedelta(hours=12), n_steps=1, save=False, initial_condition=paths[1])
    np.testing.assert_allclose(pred2.values[1], pred.values[1], rtol=0, atol=1e-5)


def test_skyrim_facade_validates_names():
    from skyrim_b200.core.skyrim import Skyrim
    assert Skyrim.list_available_models() == ["pangu", "fourcastnet_v2", "graphcast"]
    with pytest.raises(ValueError):
        Skyrim("not_a_model")


def test_predict_one_step_returns_ic_and_one_prediction():
    """A4 (reference base.py:80-92): predict_one_step == run_basic_inference(n=1): IC slice + one 6-h prediction."""
    gm = BoringGlobalModel(ic_source="synthetic")
    t0 = datetime.datetime(2024, 5, 7)
    da = gm.predict_one_step(t0)
    assert da.dims == ("time", "channel", "lat", "lon") and da.shape == (2, 4, 19, 36)
    np.testing.assert_allclose(da.values[1], da.values[0] + 1.0)
    f = gm.forecast(t0, n_steps=2)
    np.testing.assert_array_equal(f.values[:2], da.values)            # forecast's first two slices are the same step
    # stepping from a supplied state (the path rollout() uses for every step after the first)
    da2 = gm.predict_one_step(t0 + datetime.timedelta(hours=6), initial_condition=da.isel(time=[1]))
    np.testing.assert_allclose(da2.values[1], da.values[0] + 2.0, rtol=0, atol=1e-5)


def test_forecast_cli_mirrors_the_reference_options(tmp_path, monkeypatch):
    """reference skyrim/forecast.py:59-151: option names / short flags / defaults; run_forecast returns the saved paths."""
    from click.testing import CliRunner
    from skyrim_b200 import forecast as F
    from skyrim_b200.core import models as M
    opts = {o.name: o for o in F.main.params}
    for name, short in [("model_name", "-m"), ("date", "-d"), ("time", "-t"), ("lead_time", "-l"), ("list_models", "-lm"),
                        ("initial_conditions", "-ic"), ("output_dir", "-o"), ("filter_vars", "-f"), ("modal", "-mo")]:
        assert name in opts and short in opts[name].opts, name
    assert opts["lead_time"].default == 6 and opts["time"].default == "0000" and opts["model_name"].default == "pangu"
    r = CliRunner().invoke(F.main, ["-lm"])
    assert r.exit_code == 0 and "pangu" in r.output and "fourcastnet_v2" in r.output
    assert CliRunner().invoke(F.main, ["-mo"]).exit_code != 0

    class FakePangu(BoringGlobalModel):
        def __init__(self, ic_source="synthetic", **kw):
            super().__init__(ic_source=ic_source)
    monkeypatch.setitem(M.MODELS, "pangu", FakePangu)
    r = CliRunner().invoke(F.main, ["-m", "pangu", "-d", "20240507", "-t", "0600", "-l", "13", "-o", str(tmp_path), "-f", "t2m,msl"])
    assert r.exit_code == 0, r.output
    paths = [ln for ln in r.output.splitlines() if ln.endswith(".nc") or ln.endswith(".zarr")]
    assert len(paths) == 2                                           # lead 13 h -> floored to 12 h -> two 6-h steps
    da = xr.open_dataarray(paths[0])
    assert list(da.coords["channel"]) == ["t2m", "msl"]


def test_bench_traffic_lookup_and_roofline_tables():
    """bench.py's roofline.traffic comes from a committed `ncu --set full` capture (profiles/r*_traffic.json); the per-family
    roofline uses skyrim_b200/roofline.py's FLOP and byte tables."""
    import importlib.util, os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(root, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    t, src = mod._traffic("mlp")
    assert isinstance(t, int) and 1e8 < t < 2e9 and src.startswith("profiles/")   # bytes per launch of the fused MLP (196 MB with the image-only token stream)
    assert mod._traffic("no-such-family") == (None, None)
    from skyrim_b200.config import pangu_full, sfno_full
    fams, fl, by = mod.family_roofline("pangu", pangu_full(), 1, {"mlp": 5.0, "attn": 2.0, "embed": 0.3},
                                       dict(hbm=6572.0, tensor_sustained=1431.0))
    assert fams["mlp"]["bound"] == "tensor" and fams["attn"]["bound"] == "hbm" and 0.5 < fams["attn"]["frac"] < 0.8
    assert abs(fl["total"] - 8.26e12) < 0.2e12 and 28e9 < by["total"] < 36e9   # image-only token stream (12 -> 6 B in proj / mlp)
    fams, fl, by = mod.family_roofline("sfno", sfno_full(), 1, {"sfno_mlp": 5.0}, dict(hbm=6572.0, tensor_sustained=1431.0))
    assert "sfno_mlp" in fams and 2e12 < fl["total"] < 6e12


def test_bench_output_sample_is_fixed_by_the_seed():
    """bench.py --dump-outputs: the same distinct, sorted elements of a state larger than the sample on every call, as
    float32, within 64 MB"""
    import importlib.util, os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(root, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    t = torch.arange(2 ** 24, dtype=torch.float64).reshape(4, 2 ** 11, 2 ** 11)   # value = flat index, exact in float32
    a, b = mod.output_sample(t), mod.output_sample(t)
    assert a.dtype == np.float32 and a.ndim == 1 and np.array_equal(a, b) and a.nbytes <= 64 * 2 ** 20
    assert mod.DUMP_MAX_VALUES // 2 < len(a) <= mod.DUMP_MAX_VALUES and (np.diff(a) > 0).all()
    assert not np.array_equal(mod.output_sample(t, seed=1), a)
