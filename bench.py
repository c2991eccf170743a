#!/usr/bin/env python
"""Benchmark of the rollout hot path (BASELINE.json metric).

    python bench.py --gpus 1 --steps 20 --warmup 3            # our arm, 1 GPU
    torchrun --nproc-per-node N ... bench.py --gpus N ...     # one rank per GPU, weak scaling
    python bench.py --impl reference --steps 5 --warmup 1     # CPU reference arm

The headline line is BASELINE config 2's step (Pangu 6-h step on the (69,721,1440) state, chained device-resident
rollout, ``--members-per-gpu`` members per GPU, default 1).  ``value`` = member-steps per second over all ranks with the
state resident in HBM; ``e2e`` = the same through the reference-facing TimeLoop call with HOST (pinned) input and output
every step, copies inside the timed region.  The first timed step starts from the seeded synthetic IC, and its output
is compared with the committed full-size oracle fixture (``verify``): a fast, finite, wrong step fails the run.

The same invocation also measures (sub-records under ``configs``, skipped with ``--only-headline``):
  config 3  FourCastNet-v2 SFNO 6-h step on (73,721,1440)                     -> configs.sfno
  config 4  GraphCast 6-h step on (2 x 83, 721, 1440), refinement-6 multimesh       -> configs.graphcast
  config 5  Pangu ensemble with 4 members per GPU (32 members on 8 GPUs)      -> configs.ensemble_m4
each with ms/step, member-steps/s, per-family roofline fractions, fixture verification, and (N = 1) its e2e figure.
One JSON line on rank 0.

``--dump-outputs DIR`` also writes DIR/state.npy: 2**23 elements (fewer after removing repeats) of the state the last timed
headline step returned, at flat indices fixed by a seed.  Weights and initial conditions are seeded too, so two builds run
with the same arguments can be compared element for element.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "6h rollout steps/sec on (69,721,1440); ensemble member-steps/sec @1/2/4/8 GPU"
UNIT = "member-steps/s"
VERIFY_TOL = 1e-3      # per-channel relative L2 on the point sample (north star); block means / RMS in sigma units below
VERIFY_TOL_SIGMA = 5e-3
VERIFY_TOL_TENDENCY = 4e-3   # GraphCast: per-channel relative L2 of the network tendency (state = x + 0.1 sigma x tendency); measured 1.4e-3
DUMP_MAX_VALUES = 1 << 23    # --dump-outputs: 32 MB of float32 at most


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tensor_burst=d["bf16_tflops"],
                    tensor_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tensor_burst=1590.0, tensor_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------------
# CPU reference arm / cpu_baseline.  BASELINE.md section 2: (1) ONNXRuntime-CPU on pangu_weather_6.onnx when both are
# present on the box, else (2) the oracle (CPU restatement of the reference's forward).  Either way REAL full-size
# steps on the (69,721,1440) state are timed — no latitude band, no FLOP-fraction extrapolation.
# --------------------------------------------------------------------------------------------
def _find_onnx():
    import glob
    cands = []
    w = os.environ.get("SKYRIM_B200_WEIGHTS")
    if w:
        cands += [w] if w.endswith(".onnx") else glob.glob(os.path.join(w, "**", "pangu_weather_6.onnx"), recursive=True)
    for root in ("~/.cache/earth2mip", "~/.cache/modulus", "~/.cache/earth2studio"):
        cands += glob.glob(os.path.join(os.path.expanduser(root), "**", "pangu_weather_6.onnx"), recursive=True)
    return next((c for c in cands if os.path.exists(c)), None)


def cpu_reference(max_steps: int, budget_s: float = 100.0):
    """-> dict(value, unit, cores, kind, sample, ms_per_step, steps_timed).  Times at least one and at most `max_steps`
    real full-size 6-h steps, stopping when the next one would overrun `budget_s`."""
    import numpy as np
    from skyrim_b200.config import PANGU_CHANNELS, pangu_full
    from skyrim_b200.weights import synthetic_state
    cfg = pangu_full()
    x0 = synthetic_state(PANGU_CHANNELS, cfg.nlat, cfg.nlon, 0)
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)   # every host thread this process may use
    onnx_path = None
    try:
        import onnxruntime as ort  # noqa: F401
        onnx_path = _find_onnx()
    except Exception:
        ort = None
    if ort is not None and onnx_path:
        so = ort.SessionOptions()
        so.intra_op_num_threads = cores
        sess = ort.InferenceSession(onnx_path, sess_options=so, providers=["CPUExecutionProvider"])
        pl = x0[:65].reshape(5, 13, cfg.nlat, cfg.nlon).astype(np.float32)
        sl = x0[65:].astype(np.float32)
        step = lambda: sess.run(None, {"input": pl, "input_surface": sl})
        kind, what = "reference", f"onnxruntime CPUExecutionProvider on {os.path.basename(onnx_path)}, {cores} intra-op threads"
    else:
        import torch
        from oracle.pangu_ref import PanguRef
        from skyrim_b200.config import pangu_small
        from skyrim_b200.weights import make_pangu_weights
        # torch's CPU kernels stop scaling on wide hosts (128 threads ran the full step 1.7x SLOWER than 8 threads did in
        # the build container): pick the fastest thread count among {all, 64, 32, 16} on a 73x1440 band first, then time
        # REAL full-size steps with it.  `cores` reports the threads actually used.
        host_threads, best = cores, None
        band = pangu_small(73, 1440)
        bref = PanguRef(band, make_pangu_weights(band, 0))
        bx = torch.from_numpy(synthetic_state(PANGU_CHANNELS, band.nlat, band.nlon, 0))
        for n in sorted({host_threads, min(host_threads, 64), min(host_threads, 32), min(host_threads, 16)}, reverse=True):
            torch.set_num_threads(n)
            bref.step(bx)
            t0 = time.perf_counter(); bref.step(bx); dtb = time.perf_counter() - t0
            if best is None or dtb < best[1]:
                best = (n, dtb)
        cores = best[0]
        torch.set_num_threads(cores)
        del bref, bx
        ref = PanguRef(cfg, make_pangu_weights(cfg, 0))
        xt = torch.from_numpy(x0)
        state = {"x": xt}

        def step():
            state["x"] = ref.step(state["x"])
        kind, what = "port", (f"oracle/pangu_ref.py (torch fp32 CPU restatement of the reference forward; onnxruntime / "
                              f"pangu_weather_6.onnx not present on this box), {cores} of {host_threads} host threads (fastest of "
                              f"all/64/32/16 on a 73x1440 band)")
    times = []
    t_all = time.perf_counter()
    while len(times) < max(1, max_steps):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_all + times[-1] > budget_s:
            break
    dt = sorted(times)[len(times) // 2]
    return dict(value=1.0 / dt, unit=UNIT, cores=cores, kind=kind, ms_per_step=1000.0 * dt, steps_timed=len(times),
                sample=f"{len(times)} real full-size 6-h step(s) on the (69,721,1440) synthetic state, no warm-up, median; {what}")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb = cpu_reference(args.steps + args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": cb["steps_timed"], "steps_requested": args.steps, "warmup": 0, "ms_per_step": cb["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "Pangu 6-h step, synthetic (69,721,1440) IC, CPU path of the reference (BASELINE config 1); "
                                   "every timed step is a full-size step — the step count is bounded to ~100 s of CPU work"},
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------
class Dist:
    def __init__(self, args):
        import torch
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        assert self.world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={self.world}"
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        import torch
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max(self, *vals):
        import torch
        t = torch.tensor(vals, dtype=torch.float64, device=self.dev)
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def min(self, *vals):
        return [-v for v in self.max(*[-v for v in vals])]


def build_engine(model: str, d: Dist):
    """Weights built on rank 0, ONE NCCL broadcast of the fp32 arena (the only collective of the job), repacked per device."""
    import numpy as np
    import torch
    from skyrim_b200.engine import StepEngine, pack_arena
    if model == "sfno":
        from skyrim_b200.config import FCNV2_CHANNELS as CH, sfno_full
        from skyrim_b200.timeloop import SFNOTimeLoop as Loop
        from skyrim_b200.weights import make_sfno_weights, sfno_param_shapes, sfno_table_shapes, sfno_tables
        cfg = sfno_full()
        w = None
        if d.rank == 0:
            w = make_sfno_weights(cfg, 0); w.update(sfno_tables(cfg))
        shapes = None
        if d.world > 1:
            shapes = sfno_param_shapes(cfg)
            shapes.update(sfno_table_shapes(cfg))
    elif model == "graphcast":
        from skyrim_b200.config import GRAPHCAST_CHANNELS as CH, graphcast_full
        from skyrim_b200.icomesh import build_graph, graph_arena_entries
        from skyrim_b200.timeloop import GraphcastTimeLoop as Loop
        from skyrim_b200.weights import graphcast_param_shapes, make_graphcast_weights
        cfg = graphcast_full()
        graph = build_graph(cfg.nlat, cfg.nlon, cfg.mesh_levels, cfg.radius_frac)   # every rank: the table shapes size the arena
        gent = graph_arena_entries(graph)
        w = None
        if d.rank == 0:
            w = make_graphcast_weights(cfg, 0); w.update(gent)
        shapes = None
        if d.world > 1:
            shapes = graphcast_param_shapes(cfg)
            shapes.update({k: v.shape for k, v in gent.items()})
        kw = {"graph": graph}
    else:
        from skyrim_b200.config import PANGU_CHANNELS as CH, pangu_full
        from skyrim_b200.timeloop import PanguTimeLoop as Loop
        from skyrim_b200.weights import make_pangu_weights, pangu_param_shapes
        cfg = pangu_full()
        w = make_pangu_weights(cfg, 0) if d.rank == 0 else None
        shapes = pangu_param_shapes(cfg) if d.world > 1 else None
    eng = StepEngine(cfg, d.local, **(kw if model == "graphcast" else {}))
    if d.world > 1:
        import torch.distributed as dist
        if d.rank == 0:
            arena_h, manifest = pack_arena(w)
            arena = torch.from_numpy(arena_h).to(d.dev)
        else:
            arena_h, manifest = pack_arena({k: np.zeros(s, np.float32) for k, s in shapes.items()})
            arena = torch.empty(arena_h.size, dtype=torch.float32, device=d.dev)
        del arena_h
        dist.broadcast(arena, 0)
        eng.load_arena(arena, manifest)
        del arena
    else:
        eng.load_weights(w)
    return cfg, CH, eng, Loop(eng)


def family_roofline(model, cfg, M, fam_ms, peaks):
    """Per kernel family: algorithmic FLOPs and mandatory HBM bytes per step (skyrim_b200/roofline.py, DESIGN.md section 4) over
    the family's measured device time per step -> achieved TFLOP/s, GB/s and the fraction of the bounding roofline."""
    from skyrim_b200 import roofline as R
    fl = R.sfno_flops(cfg) if model == "sfno" else R.graphcast_flops(cfg) if model == "graphcast" else R.pangu_flops(cfg)
    by = R.sfno_bytes(cfg) if model == "sfno" else R.graphcast_bytes(cfg) if model == "graphcast" else R.pangu_bytes(cfg)
    out = {}
    for k, ms in fam_ms.items():
        f, b = M * fl.get(k, 0.0), M * by.get(k, 0.0)
        if ms <= 0 or (f == 0 and b == 0):
            continue
        tf, gb = f / (ms * 1e-3) / 1e12, b / (ms * 1e-3) / 1e9
        ft, fh = tf / peaks["tensor_sustained"], gb / peaks["hbm"]
        bound = "tensor" if f / (peaks["tensor_sustained"] * 1e12) >= b / (peaks["hbm"] * 1e9) else "hbm"
        out[k] = {"ms": round(ms, 4), "bound": bound, "tflops": round(tf, 1), "gbs": round(gb, 1),
                  "frac": round(ft if bound == "tensor" else fh, 4), "frac_tensor": round(ft, 4), "frac_hbm": round(fh, 4)}
    return out, fl, by


def output_sample(t, n=DUMP_MAX_VALUES, seed=0):
    """float32 host copy of `t` flattened and read at up to `n` flat indices: sorted, without repeats, drawn from numpy's
    default generator seeded with `seed`, so every run and every build with the same arguments samples the same elements."""
    import numpy as np
    import torch
    idx = np.sort(np.random.default_rng(seed).integers(0, t.numel(), n))
    idx = idx[np.concatenate(([True], idx[1:] != idx[:-1]))]   # np.unique does the same, forty times slower
    return t.reshape(-1)[torch.from_numpy(idx).to(t.device)].float().cpu().numpy()


def bench_model(model: str, M: int, steps: int, warmup: int, d: Dist, e2e: bool = True, dump: bool = False):
    import torch
    from skyrim_b200.engine import launch_count, perturb_ic
    from skyrim_b200.verify import compare_fullsize, load_fixture, summarise
    from skyrim_b200.weights import channel_stats, synthetic_state
    cfg, CH, eng, loop = build_engine(model, d)
    dev = d.dev
    # ---- synthetic initial conditions: global member 0 is the unperturbed control (the fixture's IC), the others carry
    # the Philox perturbation keyed by their global member id (K11) ----
    gc = model == "graphcast"
    GC_T0 = 1714521600.0   # valid time of the fixture's initial condition (second slice)
    if gc:
        from skyrim_b200.weights import synthetic_graphcast_state
        assert M == 1, "GraphCast is benchmarked with one member per GPU (BASELINE config 4)"
        base = torch.from_numpy(synthetic_graphcast_state(cfg, 0))
        x0 = base.reshape(1, 2, cfg.n_state, cfg.nlat, cfg.nlon).to(dev)
        loop.fill_forcing(x0, GC_T0)
        x0 = x0.reshape(1, 2 * cfg.n_state, cfg.nlat, cfg.nlon).contiguous()
        gc_diff_std = channel_stats(CH)[1] * 0.1
    else:
        base = torch.from_numpy(synthetic_state(CH, cfg.nlat, cfg.nlon, 0))
        x0 = base[None].repeat(M, 1, 1, 1).to(dev).contiguous()
    reset_clock = (lambda: eng.set_clock(GC_T0)) if gc else (lambda: None)   # every chain below restarts from the IC's time
    sigma = torch.from_numpy(channel_stats(CH)[1]).to(dev)
    if gc:   # both time slices are perturbed, the toa forcing channel of each is not
        sigma = torch.cat([sigma, sigma]); sigma[cfg.n_state - 1] = 0.0; sigma[2 * cfg.n_state - 1] = 0.0
    first = 1 if d.rank == 0 else 0
    if M - first > 0:
        perturb_ic(x0[first:], sigma, 0.05, seed=0, member0=d.rank * M + first)
    x = x0.clone()
    y, z = torch.empty_like(x), torch.empty_like(x)

    # ---- warm-up on a copy + family breakdown (all families timed, outside the timed region) ----
    reset_clock()
    for _ in range(max(warmup - 1, 0)):
        eng.step(x, y); x, y = y, x
    eng.profile_begin()
    eng.step(x, y); x, y = y, x
    fam = eng.profile_end()
    fam_ms = {k: v[0] for k, v in fam.items()}
    dominant = max(fam, key=lambda k: fam[k][0])
    x.copy_(x0)

    # ---- timed region: K device-resident chained steps from the seeded IC; the first step's output stays in `z`.
    # The buffer rotation (x->z, z->y, y->x, x->y, ...) repeats (in, out) pairs, so from the third use of a pair on the
    # library replays the step as one CUDA graph (Engine::step_cached); the warm-up steps above used the same pairs. ----
    def chain(k):
        eng.step(x, z)
        src, dst = z, y
        for _ in range(k - 1):
            eng.step(src, dst)
            src, dst = dst, (x if dst is y else y)
        return src

    for _ in range(2):   # untimed: lets every (in, out) pair of the rotation reach its replay state
        x.copy_(x0); reset_clock(); chain(min(steps, 4))
    x.copy_(x0); reset_clock()
    sampler = ClockSampler(d.local)
    launches0 = launch_count()
    d.barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    src = chain(steps)
    e1.record()
    d.barrier()
    clocks = sampler.stop()
    ms_total = e0.elapsed_time(e1)
    launches = launch_count() - launches0
    finite = bool(torch.isfinite(src).all())
    z_first = z[0].clone()
    last_state = output_sample(src) if dump else None   # the passes below overwrite the rotation buffers

    # ---- the same K steps once more with CUDA events around every launch of the dominant family (plain launches: the
    # per-launch events cannot live inside a replayed graph) -> roofline.achieved; its wall time is reported beside it ----
    x.copy_(x0); reset_clock()
    d.barrier()
    eng.profile_begin([dominant])
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    chain(steps)
    p1.record()
    d.barrier()
    dom = eng.profile_end()[dominant]
    ms_profiled = p0.elapsed_time(p1) / steps

    # ---- verification of the timed run's first output against the full-size oracle fixture (rank 0, member 0) ----
    verify = None
    if d.rank == 0 and gc:
        from skyrim_b200.verify import compare_graphcast
        s = compare_graphcast(z_first, x0[0], gc_diff_std, load_fixture(model), cfg)
        ok = bool(s["finite"] and finite and s["rel"] < VERIFY_TOL and s["norm"] < VERIFY_TOL and s["block"] < VERIFY_TOL_SIGMA
                  and s["t_rel"] < VERIFY_TOL_TENDENCY and s["slice0_is_old_slice1"])
        verify = {"ok": ok, "against": f"tests/golden/{model}_721x1440_seed0.npz (one real oracle step)",
                  "max_rel_err_per_channel": s["rel"], "max_rms_err_sigma": s["nrm"], "max_block_mean_err_sigma": s["block"],
                  "max_norm_err": s["norm"], "tolerance": VERIFY_TOL, "rollout_finite": finite,
                  "tendency_max_rel_err_per_channel": s["t_rel"], "tendency_max_block_mean_err_sigma": s["t_block"],
                  "tendency_tolerance": VERIFY_TOL_TENDENCY}
    elif d.rank == 0:
        s = summarise(compare_fullsize(z_first, load_fixture(model)))
        ok = bool(s["finite"] and finite and s["rel"] < VERIFY_TOL and s["norm"] < VERIFY_TOL and s["block"] < VERIFY_TOL_SIGMA)
        verify = {"ok": ok, "against": f"tests/golden/{model}_721x1440_seed0.npz (one real oracle step)",
                  "max_rel_err_per_channel": s["rel"], "max_rms_err_sigma": s["nrm"], "max_block_mean_err_sigma": s["block"],
                  "max_norm_err": s["norm"], "tolerance": VERIFY_TOL, "rollout_finite": finite}

    # ---- end to end through the TimeLoop call: host (pinned) in, host (pinned) out, every step ----
    e2e_ms = roll_ms = None
    if e2e:
        xh = torch.empty((M,) + tuple(base.shape), dtype=torch.float32).pin_memory()
        xh.copy_(x0.cpu())
        e2e_steps = max(3, min(steps, 10))
        reset_clock()
        out_h = loop.step_host(xh)  # warm-up (allocates the pinned result buffers)
        d.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            out_h = loop.step_host(out_h)  # H2D + step + D2H, synchronous result on the host
        d.barrier()
        e2e_ms = (time.perf_counter() - t0) * 1000.0 / e2e_steps
        # the rollout call as GlobalModel.rollout(save=True) drives it: IC uploaded once, EVERY state delivered to pinned
        # host memory, the copy of step n overlapping step n+1 (timeloop.iter_host) -- reported beside the strict number
        import datetime
        for rep in range(0 if gc else 2):    # first pass: ring allocation + graph capture of the three (in, out) pairs
            it = loop.iter_host(datetime.datetime(2024, 1, 1), xh[:, None], e2e_steps + 2)
            next(it); next(it); next(it)
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                _, out_h = next(it)
            roll_ms = (time.perf_counter() - t0) * 1000.0 / e2e_steps
            it.close()
        del xh, out_h

    ms_total, e2e_max = d.max(ms_total, e2e_ms or 0.0)
    ms_step = ms_total / steps
    rec = {"model": model, "members_per_gpu": M, "members_total": d.world * M, "steps": steps, "ms_per_step": ms_step,
           "value": d.world * M * 1000.0 / ms_step, "unit": UNIT, "gpu_launches": int(launches), "clocks": clocks,
           "verify": verify, "dominant": dominant, "dominant_launches_per_step": dom[1] / steps,
           "dominant_avg_launch_ms": dom[0] / max(dom[1], 1), "ms_per_step_profiled_pass": ms_profiled}
    if dump:
        rec["_last_state"] = last_state
    if e2e:
        sbytes = cfg.n_channels * cfg.nlat * cfg.nlon * 4 * M
        rec["e2e"] = {"value": d.world * M * 1000.0 / e2e_max, "unit": UNIT, "ms_per_step": e2e_max,
                      "h2d_bytes_per_step": sbytes, "d2h_bytes_per_step": sbytes // 2 if gc else sbytes,
                      "path": ("GraphcastTimeLoop.step_host: both time slices pinned host -> HBM, sky_model_step, the NEW time slice HBM -> "
                               "pinned host" if gc else "TimeLoop.step_host: pinned host -> HBM, sky_model_step, HBM -> pinned host"),
                      "rollout_every_state_to_host": None if roll_ms is None else {
                          "ms_per_step": roll_ms, "value": M * 1000.0 / roll_ms, "unit": UNIT, "d2h_bytes_per_step": sbytes,
                          "h2d_bytes_per_step": 0, "rank": d.rank,
                          "path": "TimeLoop.iter_host (what GlobalModel.rollout(save=True) drives): IC uploaded once, every "
                                  "6-h state copied to pinned host memory, copy of step n overlapping step n+1"}}
    if d.rank == 0:
        peaks = _peaks()
        fams, fl, by = family_roofline(model, cfg, M, fam_ms, peaks)
        rec["families"] = fams
        rec["families_ms_per_step"] = {k: round(v, 3) for k, v in sorted(fam_ms.items(), key=lambda kv: -kv[1])}
        rec["step_tflops"] = M * fl["total"] / (ms_step * 1e-3) / 1e12
        rec["step_frac_tensor"] = rec["step_tflops"] / peaks["tensor_sustained"]
        rec["_dominant_flops"] = M * fl.get(dominant, 0.0)
        rec["_dominant_bytes"] = M * by.get(dominant, 0.0)
    eng.close()
    del eng, loop, x, y, z, x0
    torch.cuda.empty_cache()
    return rec


def _traffic(family):
    """DRAM bytes per launch of a kernel family from the committed `ncu --set full` capture of this round's kernels
    (profiles/r2f_traffic.json, provenance and kernel names inside); None when no capture covers the family."""
    for name in ("r2f_traffic.json", "r2_traffic.json", "r1_traffic.json"):
        p = os.path.join(ROOT, "profiles", name)
        try:
            with open(p) as f:
                e = json.load(f).get(family)
            if e:
                return e.get("bytes_per_launch"), f"profiles/{name}"
        except (OSError, ValueError):
            pass
    return None, None


def run_ours(args):
    import torch
    d = Dist(args)
    M = args.members_per_gpu
    head = bench_model(args.model, M, args.steps, args.warmup, d, dump=args.dump_outputs is not None and d.rank == 0)
    if d.rank == 0 and args.dump_outputs is not None:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "state.npy"), head.pop("_last_state"))
    subs = {}
    if not args.only_headline:
        k = max(3, min(args.steps, 8))
        if args.model != "sfno":
            subs["sfno"] = bench_model("sfno", 1, k, 3, d, e2e=(d.world == 1))
        if args.model != "graphcast":   # BASELINE config 4: GraphCast 6-h step on the 0.25 deg grid, one member per GPU
            subs["graphcast"] = bench_model("graphcast", 1, k, 3, d, e2e=(d.world == 1))
        if args.model == "pangu" and M != 4:
            subs["ensemble_m4"] = bench_model("pangu", 4, k, 3, d, e2e=False)
    cb = None
    if d.rank == 0 and d.world == 1 and not args.no_cpu_baseline:
        cb = cpu_reference(1)

    if d.rank == 0:
        peaks = _peaks()
        dom = head["dominant"]
        fam = head["families"].get(dom, {})
        tensor_bound = fam.get("bound", "tensor") == "tensor"
        n_l, avg_ms = head["dominant_launches_per_step"], head["dominant_avg_launch_ms"]
        work = head["_dominant_flops"] if tensor_bound else head["_dominant_bytes"]
        achieved = work / max(n_l, 1) / (avg_ms * 1e-3) / (1e12 if tensor_bound else 1e9)
        peak = peaks["tensor_sustained"] if tensor_bound else peaks["hbm"]
        traffic, tsrc = _traffic(dom)
        sfno = args.model == "sfno"
        for r in [head] + list(subs.values()):
            r.pop("_dominant_flops", None); r.pop("_dominant_bytes", None)
        if "ensemble_m4" in subs:   # config 5: ratio of the 4-members-per-GPU job to ONE member on ONE GPU (target >= 7.5 at 8 GPUs)
            subs["ensemble_m4"]["vs_one_member_one_gpu"] = subs["ensemble_m4"]["value"] / (head["value"] / (d.world * M))
        line = {
            "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": d.world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None,
            "dtype": ("f16 hi+lo split operands / f32 accumulate (tcgen05 kind::f16), f32 state" if sfno else
                      "f16 operands / f32 accumulate (tcgen05 kind::f16), f32 state, residual streams, LayerNorm" if args.model == "graphcast" else
                      "f16 operands / f32 accumulate (tcgen05 kind::f16), f32 state, LN, softmax"),
            "data": "synthetic",
            "config": {"workload": ("FourCastNet-v2 SFNO rollout (chained 6-h steps), synthetic (73,721,1440) IC, state resident in HBM"
                                    if sfno else
                                    "GraphCast rollout (chained 6-h steps), synthetic (2 x 83,721,1440) IC, refinement-6 multimesh, state resident in HBM"
                                    if args.model == "graphcast" else
                                    "Pangu 7-day rollout (chained 6-h steps), synthetic (69,721,1440) IC, state resident in HBM"),
                       "members_per_gpu": M, "members_total": d.world * M,
                       "l2": "inputs larger than L2 (state 0.3 GB + >2 GB activations streamed per step)",
                       "weights": "synthetic seed 0", "verified_against_oracle_fixture": bool(head["verify"] and head["verify"]["ok"])},
            "e2e": head.get("e2e"),
            "gpu_launches": head["gpu_launches"],
            "clocks": head["clocks"],
            "roofline": {"bound": "tensor" if tensor_bound else "hbm", "kernel": dom, "achieved": achieved, "peak": peak,
                         "unit": "TFLOP/s" if tensor_bound else "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "traffic_source": tsrc, "peak_source": peaks["source"] + (", bf16 cuBLAS sustained (kernel timed inside a long step)"
                                                                                   if tensor_bound else ", device copy"),
                         "launches_per_step": n_l, "avg_launch_ms": avg_ms,
                         "timing": ("CUDA events around every launch of the family on the launching stream, during a repeat of the "
                                    "timed K steps with plain launches (the timed region itself replays each step as one CUDA graph)"),
                         "ms_per_step_profiled_pass": head["ms_per_step_profiled_pass"], "step_tflops": head["step_tflops"],
                         "step_frac_tensor": head["step_frac_tensor"]},
            "families": head["families"],
            "families_ms_per_step": head["families_ms_per_step"],
            "verify": head["verify"],
            "configs": subs,
            "cpu_baseline": ({k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")} if cb else None),
        }
        print(json.dumps(line), flush=True)
        bad = [m for m, r in [("headline", head)] + list(subs.items()) if r["verify"] and not r["verify"]["ok"]]
        if bad:
            print(f"bench.py: output verification against the oracle fixture FAILED for {bad}", file=sys.stderr)
            if "headline" in bad and not args.allow_unverified:   # a fast, finite, wrong headline number is not a number
                sys.exit(3)
    if d.world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=28)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--members-per-gpu", type=int, default=1)
    ap.add_argument("--model", default="pangu", choices=["pangu", "sfno", "graphcast"],
                    help="headline workload: pangu (default) or sfno (FourCastNet-v2 73-channel rollout)")
    ap.add_argument("--only-headline", action="store_true", help="skip the configs.sfno / configs.ensemble_m4 sub-records")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--allow-unverified", action="store_true",
                    help="print the line (verify.ok = false) instead of exiting 3 when the fixture comparison fails")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write DIR/state.npy: a fixed seeded sample (output_sample) of the state the last timed headline "
                         "step returned on rank 0, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
