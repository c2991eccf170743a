"""CPU tests of the FourCastNet v1 (AFNO) restatement: filter transforms, softshrink activity, fp16 error budget,
golden fixture, checkpoint import and the model's host logic."""
import os

import numpy as np
import pytest
import torch

from oracle.afno_ref import FCNRef
from oracle.pangu_ref import rel_err_per_channel
from skyrim_b200.config import FCN_CHANNELS, fcn_full, fcn_small
from skyrim_b200.weights import fcn_param_shapes, make_fcn_weights, synthetic_state

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def _engine_filter_transforms(X, h, w, h_lo, h_hi, kw):
    """The engine's inverse-filter arithmetic in numpy (k_fcn_dft_h inverse + k_fcn_idft_w): complex IDFT over the kept
    H rows, then c2r over the kw W-modes with weight 1 for mode 0 and Nyquist, 2 otherwise, cosine / sine only."""
    f = np.arange(h_lo, h_hi)
    hi = np.arange(h)
    G = np.einsum("kh,bkme->bhme", np.exp(2j * np.pi * np.outer(f, hi) / h), X[:, h_lo:h_hi, :kw]) / np.sqrt(h)
    m = np.arange(kw)
    c = np.where((m == 0) | (2 * m == w), 1.0, 2.0)
    th = 2 * np.pi * np.outer(m, np.arange(w)) / w
    return (np.einsum("bhme,mx->bhxe", G.real * c[:, None], np.cos(th))
            - np.einsum("bhme,mx->bhxe", G.imag * c[:, None], np.sin(th))) / np.sqrt(w)


@pytest.mark.parametrize("h,w,kw", [(6, 12, 4), (6, 12, 7), (7, 10, 6)])
def test_filter_transforms_match_torch_fft(h, w, kw):
    """forward tables against rfft2; the inverse against irfft2 on a NON-Hermitian spectrum (the spectral MLP breaks the
    symmetry), including the imaginary parts of W-mode 0 and of the Nyquist mode that c2r ignores"""
    rng = np.random.default_rng(0)
    u = rng.standard_normal((1, h, w, 3))
    ref = torch.fft.rfft2(torch.from_numpy(u), dim=(1, 2), norm="ortho").numpy()
    F1 = np.einsum("bhxe,mx->bhme", u, np.exp(-2j * np.pi * np.outer(np.arange(kw), np.arange(w)) / w)) / np.sqrt(w)
    Y = np.einsum("kh,bhme->bkme", np.exp(-2j * np.pi * np.outer(np.arange(h), np.arange(h)) / h), F1) / np.sqrt(h)
    assert np.abs(Y - ref[:, :, :kw]).max() < 1e-12
    X = np.zeros((1, h, w // 2 + 1, 3), dtype=complex)
    X[:, :, :kw] = rng.standard_normal((1, h, kw, 3)) + 1j * rng.standard_normal((1, h, kw, 3))
    assert np.abs(X[:, :, 0].imag).min() > 0
    out = _engine_filter_transforms(X, h, w, 0, h, kw)
    ref = torch.fft.irfft2(torch.from_numpy(X), s=(h, w), dim=(1, 2), norm="ortho").numpy()
    assert np.abs(out - ref).max() < 1e-12


def test_kept_mode_shortcut_equals_upstream_slicing():
    """the engine processes H rows [h_lo, h_hi) x W-modes [0, kw); upstream slices [total-kept : total+kept, :kept]"""
    for frac in (1.0, 0.5, 0.3):
        for nlat, nlon in ((48, 96), (720, 1440), (56, 80)):
            cfg = fcn_small(nlat, nlon, 1).__class__(nlat=nlat, nlon=nlon, depth=1, hard_thresholding_fraction=frac)
            h, w = cfg.h, cfg.w
            mask = np.zeros((h, w // 2 + 1), bool)
            total = h // 2 + 1
            kept = int(total * frac)
            mask[total - kept: total + kept, :kept] = True
            lo, hi = cfg.h_range
            short = np.zeros_like(mask)
            short[lo:hi, :cfg.kw] = True
            assert np.array_equal(mask, short), (frac, nlat, nlon)
    full = fcn_full()
    assert full.kw == 46 and full.h_range == (0, 90) and full.tokens == 16200


def test_filter_with_shortcut_equals_oracle():
    """the engine's arithmetic (kept block only, explicit DFT sums) reproduces the oracle's filter literally"""
    cfg = fcn_small(48, 96, 1)
    w = make_fcn_weights(cfg, 0)
    ref = FCNRef(cfg, w, torch.float64)
    ref._blk = "blocks.0."
    u = torch.from_numpy(np.random.default_rng(1).standard_normal((1, cfg.h, cfg.w, cfg.embed)))
    want = ref.filter(u).numpy()
    h, wd, kw, (lo, hi) = cfg.h, cfg.w, cfg.kw, cfg.h_range
    un = u.numpy()
    F1 = np.einsum("bhxe,mx->bhme", un, np.exp(-2j * np.pi * np.outer(np.arange(kw), np.arange(wd)) / wd)) / np.sqrt(wd)
    Y = np.einsum("kh,bhme->bkme", np.exp(-2j * np.pi * np.outer(np.arange(lo, hi), np.arange(h)) / h), F1) / np.sqrt(h)
    nb, bs = cfg.num_blocks, cfg.block_size
    w1, b1, w2, b2 = (np.asarray(w[f"blocks.0.filter.{k}"], np.float64) for k in ("w1", "b1", "w2", "b2"))
    Yb = Y.reshape(Y.shape[:3] + (nb, bs))
    o1 = (np.maximum(np.einsum("...bi,bio->...bo", Yb.real, w1[0]) - np.einsum("...bi,bio->...bo", Yb.imag, w1[1]) + b1[0], 0)
          + 1j * np.maximum(np.einsum("...bi,bio->...bo", Yb.imag, w1[0]) + np.einsum("...bi,bio->...bo", Yb.real, w1[1]) + b1[1], 0))
    o2r = np.einsum("...bi,bio->...bo", o1.real, w2[0]) - np.einsum("...bi,bio->...bo", o1.imag, w2[1]) + b2[0]
    o2i = np.einsum("...bi,bio->...bo", o1.imag, w2[0]) + np.einsum("...bi,bio->...bo", o1.real, w2[1]) + b2[1]
    ss = lambda a: np.sign(a) * np.maximum(np.abs(a) - cfg.sparsity, 0)
    Z = np.zeros((1, h, wd // 2 + 1, cfg.embed), complex)
    Z[:, lo:hi, :kw] = (ss(o2r) + 1j * ss(o2i)).reshape(1, hi - lo, kw, cfg.embed)
    got = _engine_filter_transforms(Z, h, wd, 0, h, kw)
    assert np.abs(got - want).max() < 1e-10


def test_softshrink_activity_band():
    """the synthetic spectral weights put between 10 % and 90 % of the kept mode values inside the dead band"""
    cfg = fcn_small(48, 96, 2)
    for seed in (0, 1):
        ref = FCNRef(cfg, make_fcn_weights(cfg, seed), torch.float64)
        ref.step(synthetic_state(FCN_CHANNELS, cfg.nlat, cfg.nlon, seed))
        frac = float((ref.last_modes == 0).double().mean())
        assert 0.1 < frac < 0.9, frac


def test_fp16_operand_error_budget():
    """Precision study: fp16 operands on the dense GEMMs (embed, fc1, fc2, head) with the spectral filter in fp32 stay
    inside the 1e-3 per-channel step budget.  Measured (fp64 reference): 4.4e-4 at 48x96 / 2 blocks, 4.6e-4 at
    48x96 / 12 blocks, 4.4e-4 at 64x128 / 12 blocks, for weight / state seeds 0 and 1."""
    for (nlat, nlon, depth) in ((48, 96, 2), (48, 96, 12), (64, 128, 12)):
        cfg = fcn_small(nlat, nlon, depth)
        for seed in (0, 1):
            w = make_fcn_weights(cfg, seed)
            x = synthetic_state(FCN_CHANNELS, nlat, nlon, seed)
            y64 = FCNRef(cfg, w, torch.float64).step(x).numpy()
            y16 = FCNRef(cfg, w, torch.float64, emulate="fp16").step(x).numpy()
            e = rel_err_per_channel(y16, y64).max()
            assert 1e-5 < e < 6e-4, (nlat, nlon, depth, seed, e)


def test_oracle_against_golden_fixture():
    g = np.load(os.path.join(GOLDEN, "fcn_48x96_seed0.npz"))
    cfg = fcn_small(48, 96, 2)
    x0 = synthetic_state(FCN_CHANNELS, cfg.nlat, cfg.nlon, 0)
    assert np.array_equal(x0[:, ::8, ::16], g["x0_sample"])
    y = FCNRef(cfg, make_fcn_weights(cfg, 0), torch.float64).step(x0).numpy()
    assert np.abs(y[:, ::5, ::12] - g["y_sample"]).max() <= 1e-9 * np.abs(g["y_sample"]).max()
    assert np.allclose(np.sqrt((y ** 2).sum(axis=(1, 2))), g["y_norm"], rtol=1e-10)


def test_fullsize_fixture_matches_seeded_inputs():
    g = np.load(os.path.join(GOLDEN, "fcn_720x1440_seed0.npz"))
    x0 = synthetic_state(FCN_CHANNELS, 720, 1440, 0)
    assert np.array_equal(x0[:, ::64, ::64], g["x0_sample"])
    assert g["y_sample"].shape == (26, 56, 85) and g["y_last"].shape == (26, 360) and g["y_block"].shape == (26, 45, 90)
    assert np.isfinite(g["y_sample"]).all() and np.isfinite(g["y_norm"]).all()


@pytest.mark.parametrize("layout", ["plain", "module", "model_state"])
def test_importer_roundtrip(tmp_path, layout):
    from skyrim_b200.importers import fcn_from_checkpoint, load_real_weights
    cfg = fcn_small(48, 96, 2)
    w = make_fcn_weights(cfg, 3)
    sd = {k: torch.from_numpy(v) for k, v in w.items() if not k.startswith("norm.")}
    if layout != "plain":
        sd = {"module." + k: v for k, v in sd.items()}
    torch.save({"model_state": sd} if layout == "model_state" else sd, tmp_path / "weights.tar")
    np.save(tmp_path / "global_means.npy", w["norm.mean"].reshape(1, 26, 1, 1))
    np.save(tmp_path / "global_stds.npy", w["norm.std"].reshape(1, 26, 1, 1))
    cfg2, w2 = fcn_from_checkpoint(str(tmp_path / "weights.tar"), str(tmp_path / "global_means.npy"),
                                   str(tmp_path / "global_stds.npy"))
    assert cfg2 == cfg and list(w2) == list(fcn_param_shapes(cfg))
    assert all(np.array_equal(w2[k], w[k]) for k in w)
    assert load_real_weights("fcn", str(tmp_path))[0] == cfg
    np.save(tmp_path / "global_stds.npy", np.ones(73, np.float32))
    with pytest.raises(ValueError, match="26 values"):
        load_real_weights("fcn", str(tmp_path))


class _FakeEngine:
    """CPU stand-in for StepEngine: the oracle in fp32"""

    def __init__(self, cfg, w):
        self.cfg, self.device, self.n_channels = cfg, 0, cfg.n_channels
        self.ref = FCNRef(cfg, w)

    def step(self, x, out=None):
        y = self.ref.step(x)
        if out is None:
            return y
        out.copy_(y)
        return out

    def close(self):
        pass


def test_fourcastnet_model_host_logic(tmp_path, monkeypatch):
    import datetime
    from skyrim_b200 import xr_shim as xr
    from skyrim_b200.core.models import FourcastnetModel
    from skyrim_b200.core.models import fourcastnet as mod
    from skyrim_b200.timeloop import FCNTimeLoop, poleless_grid

    cfg = fcn_small(48, 96, 1)
    w = make_fcn_weights(cfg, 0)

    class Loop:   # the TimeLoop protocol without FCNTimeLoop.iter_host (pinned host buffers need a CUDA device)
        n_history_levels = 1
        time_step = FCNTimeLoop.time_step

        def __init__(self, eng):
            self.torch = torch
            self.engine = eng
            self.device = torch.device("cpu")
            self.in_channel_names = self.out_channel_names = list(FCN_CHANNELS)
            self.grid = poleless_grid(cfg.nlat, cfg.nlon)
            self.guard_first_step = False

        def __call__(self, time, x, restart=None):
            cur = x[:, -1]
            yield time, cur, None
            while True:
                cur = self.engine.step(cur)
                time = time + self.time_step
                yield time, cur, None

    monkeypatch.setattr(FourcastnetModel, "build_model", lambda self: Loop(_FakeEngine(cfg, w)))
    m = FourcastnetModel(ic_source="synthetic", cfg=cfg, weights=w)
    assert m.model_name == "fourcastnet"
    g = poleless_grid(720, 1440)
    assert len(g.lat) == 720 and g.lat[0] == 90.0 and g.lat[-1] == -89.75 and g.lon[-1] == 359.75
    t0 = datetime.datetime(2024, 5, 7)
    ic = m.data_source[t0]
    assert ic.values.shape == (26, 48, 96)
    full = synthetic_state(FCN_CHANNELS, 49, 96, 0)
    assert np.array_equal(ic.values, full[:, :48])                 # the 721-row synthetic IC loses its last row
    pred, paths = m.rollout(t0, n_steps=2, save=True, save_config={"output_dir": str(tmp_path)})
    names = [os.path.basename(p) for p in paths]
    assert names == ["fourcastnet__synthetic__20240507_00:00__20240507_06:00.nc",
                     "fourcastnet__file__20240507_06:00__20240507_12:00.nc"], names
    assert all(p.startswith(str(tmp_path)) and os.path.exists(p) for p in paths)
    np.testing.assert_allclose(np.asarray(pred.coords["lat"]), 90.0 - 3.75 * np.arange(48))
    # a 721-row (here 49-row) initial condition is cropped, a 48-row one is taken as is: same result
    da49 = xr.DataArray(full, dims=["channel", "lat", "lon"],
                        coords=dict(channel=np.array(FCN_CHANNELS), lat=np.linspace(90, -90, 49), lon=np.arange(96) * 3.75))
    p49, _ = m.rollout(t0, n_steps=1, save=False, initial_condition=da49)
    p48, _ = m.rollout(t0, n_steps=1, save=False, initial_condition=mod.crop_to_grid(da49, 48))
    assert np.array_equal(p49.values, p48.values)
    with pytest.raises(ValueError):
        mod.crop_to_grid(da49.isel(lat=slice(0, 40)), 48)
    from skyrim_b200.core.models.base import GlobalPrediction
    gp = GlobalPrediction(pred)
    v = gp.point(-86.25, 0.0, "t2m")
    assert np.isfinite(np.asarray(v)).all()
