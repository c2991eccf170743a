"""GPU tests of the FourCastNet v1 (AFNO) step: parity with the oracle, stage taps, batching, graph replay, model API."""
import datetime

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

TOL = 1e-3


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _setup(nlat, nlon, depth, seed=0, batch=1):
    from skyrim_b200.config import FCN_CHANNELS, fcn_small
    from skyrim_b200.engine import StepEngine
    from skyrim_b200.weights import make_fcn_weights, synthetic_state
    cfg = fcn_small(nlat, nlon, depth)
    w = make_fcn_weights(cfg, seed)
    x0 = np.stack([synthetic_state(FCN_CHANNELS, nlat, nlon, seed + m) for m in range(batch)])
    eng = StepEngine(cfg, 0)
    eng.load_weights(w)
    return cfg, w, x0, eng


@pytest.mark.parametrize("nlat,nlon,depth", [(48, 96, 2), (64, 128, 3)])
def test_fcn_step_parity(nlat, nlon, depth):
    _need_gpu()
    from oracle.afno_ref import FCNRef
    from oracle.pangu_ref import rel_err_per_channel
    cfg, w, x0, eng = _setup(nlat, nlon, depth)
    y = eng.step(torch.from_numpy(x0).cuda())[0].cpu().numpy()
    ref = FCNRef(cfg, w, torch.float64).step(x0[0]).numpy()
    e = rel_err_per_channel(y, ref)
    assert np.isfinite(y).all() and e.max() < TOL, e.max()
    eng.close()


def test_fcn_stage_taps():
    """embed, each block's filter output (after the double skip) and each block's output against the oracle's taps"""
    _need_gpu()
    from oracle.afno_ref import FCNRef
    cfg, w, x0, eng = _setup(48, 96, 2)
    taps = {}
    FCNRef(cfg, w, torch.float64).step(x0[0], taps)
    xin = torch.from_numpy(x0).cuda()
    for stage, name in [(0, "embed"), (1, "filter0"), (2, "block0"), (3, "filter1"), (4, "block1")]:
        eng.debug_set("stop_after", stage)
        eng.step(xin)
        got = eng.debug_tensor("tokens", (cfg.tokens, cfg.embed)).cpu().numpy().astype(np.float64)
        ref = taps[name].reshape(cfg.tokens, cfg.embed).numpy()
        err = np.linalg.norm(got - ref) / np.linalg.norm(ref)
        assert err < TOL, (name, err)
    eng.debug_set("stop_after", 99)
    eng.close()


@pytest.mark.parametrize("nlat,nlon,depth,batch", [(360, 720, 2, 1), (720, 1440, 1, 2)])
def test_fcn_large_grids(nlat, nlon, depth, batch):
    """grids whose GEMMs run several tiles per CTA (720 x 1440 at B = 2: 254 row tiles); the oracle runs on the GPU"""
    _need_gpu()
    from oracle.afno_ref import FCNRef
    from oracle.pangu_ref import rel_err_per_channel
    cfg, w, x0, eng = _setup(nlat, nlon, depth, batch=batch)
    y = eng.step(torch.from_numpy(x0).cuda()).cpu().numpy()
    eng.close()
    ref = FCNRef(cfg, w, torch.float64, device="cuda").step(torch.from_numpy(x0)).cpu().numpy()
    for m in range(batch):
        e = rel_err_per_channel(y[m], ref[m])
        assert np.isfinite(y[m]).all() and e.max() < TOL, (m, e.max())


def test_fcn_batched_members_and_replay_bit_identical():
    _need_gpu()
    cfg, w, x0, eng = _setup(64, 128, 2, batch=3)
    xb = torch.from_numpy(x0).cuda()
    yb = eng.step(xb).cpu()
    for m in range(3):
        ym = eng.step(xb[m:m + 1].contiguous()).cpu()
        assert torch.equal(ym[0], yb[m]), m
    # StepEngine.step goes through step_cached: 1st call eager, 2nd captured, 3rd replayed
    xo = torch.empty_like(xb)
    outs = []
    for _ in range(3):
        eng.step(xb, xo)
        outs.append(xo.cpu())
    assert all(torch.equal(o, yb) for o in outs)
    eng.debug_set("use_graphs", 0)
    assert torch.equal(eng.step(xb).cpu(), yb)
    eng.close()


def test_fcn_range_guard():
    _need_gpu()
    cfg, w, x0, eng = _setup(48, 96, 2)
    xin = torch.from_numpy(x0).cuda()
    y0 = eng.step(xin).cpu()
    y, ranges = eng.step_guarded(xin)
    assert torch.equal(y.cpu(), y0)
    assert set(ranges) == {"token_images", "hidden_images"} and all(0 < v < 3e4 for v in ranges.values()), ranges
    from skyrim_b200._ffi import SkyError
    with pytest.raises(SkyError):
        eng.step_guarded(xin, limit=1e-3)
    eng.close()


def test_fourcastnet_model_rollout_and_iter_host(tmp_path):
    _need_gpu()
    import os
    from oracle.afno_ref import FCNRef
    from oracle.pangu_ref import rel_err_per_channel
    from skyrim_b200.config import fcn_small
    from skyrim_b200.core.models import FourcastnetModel
    from skyrim_b200.weights import make_fcn_weights
    cfg = fcn_small(48, 96, 2)
    w = make_fcn_weights(cfg, 0)
    m = FourcastnetModel(ic_source="synthetic", cfg=cfg, weights=w)
    t0 = datetime.datetime(2024, 5, 7)
    pred, paths = m.rollout(t0, n_steps=2, save=True, save_config={"output_dir": str(tmp_path)})
    assert len(paths) == 2 and all(p.startswith(str(tmp_path)) and os.path.exists(p) for p in paths)
    assert pred.values.shape == (2, 26, 48, 96)
    ic = m.data_source[t0].values
    ref = FCNRef(cfg, w).step(FCNRef(cfg, w).step(ic)).numpy()
    assert rel_err_per_channel(pred.values[1], ref).max() < 2 * TOL
    last = None
    for n, (_, hx) in enumerate(m.model.iter_host(t0, torch.from_numpy(ic)[None, None], 2)):
        last = hx[0].numpy().copy()
    assert n == 2 and np.array_equal(last, pred.values[1])
    m.release_model()


def test_fcn_fullsize_against_fixture():
    """one full-size (720 x 1440, 12 blocks) step against the committed sampled fp32-oracle fixture"""
    _need_gpu()
    from skyrim_b200 import verify
    from skyrim_b200.config import FCN_CHANNELS, fcn_full
    from skyrim_b200.engine import StepEngine
    from skyrim_b200.weights import make_fcn_weights, synthetic_state
    cfg = fcn_full()
    eng = StepEngine(cfg, 0)
    eng.load_weights(make_fcn_weights(cfg, 0))
    x0 = torch.from_numpy(synthetic_state(FCN_CHANNELS, cfg.nlat, cfg.nlon, 0))[None].cuda()
    y = eng.step(x0)[0]
    s = verify.summarise(verify.compare_fullsize(y, verify.load_fixture("fcn", 720), last_row=719))
    eng.close()
    assert s["finite"] and s["rel"] < TOL and s["block"] < 1e-3 and s["last"] < 1e-2, s
