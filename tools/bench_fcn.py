"""FourCastNet v1 (AFNO) full-size step on one GPU: time, per-family breakdown, fixture check, PyTorch eager comparison.

    python tools/bench_fcn.py [--out DIR] [--window 1.5]

Prints one JSON line (and writes it to DIR/bench_fcn.json when --out is given):
  gpu           card name and power limit (nvidia-smi query)
  step          ms per step and member-steps/s at B = 1 and B = 4: replayed graphs, chained device-resident steps
                (x -> y -> x ...), timed by CUDA events over a window of at least --window seconds after warm-up
  families      per-family ms (B = 1, one profiled step after the timed window), FLOPs / bytes from
                skyrim_b200.roofline.fcn_flops / fcn_bytes and the fraction of the larger of the two bounds
  verify        the B = 1 output against tests/golden/fcn_720x1440_seed0.npz; the script exits 1 when it fails
  eager         the same step through oracle/afno_ref.py in fp32 on the same GPU (cuFFT + cuBLAS, no TF32), its time and
                the per-channel relative difference to the engine's output
Datasheet bounds used for the fraction: 2250 TFLOP/s dense fp16 and 7.7 TB/s HBM for a 1000 W B200; the card's actual
limit is printed beside them.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

PEAK_FLOPS, PEAK_BYTES = 2250e12, 7.7e12


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().splitlines()[0].split(",")]
    return dict(name=name, power_limit=power, max_sm_clock=clock, torch_name=torch.cuda.get_device_name(0))


def time_chained(fn, window):
    """fn(i) launches step i; returns ms per step over >= window seconds after warm-up"""
    for i in range(3):
        fn(i)
    torch.cuda.synchronize()
    n, total = 4, 0.0
    while True:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(n):
            fn(i)
        b.record()
        b.synchronize()
        total = a.elapsed_time(b)
        if total >= window * 1e3:
            return total / n, n
        n *= 2


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--window", type=float, default=1.5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_fcn.py measures on a CUDA device; none is visible")
    from oracle.afno_ref import FCNRef
    from oracle.pangu_ref import rel_err_per_channel
    from skyrim_b200 import roofline, verify
    from skyrim_b200.config import FCN_CHANNELS, fcn_full
    from skyrim_b200.engine import StepEngine
    from skyrim_b200.weights import make_fcn_weights, synthetic_state

    cfg = fcn_full()
    w = make_fcn_weights(cfg, 0)
    x0 = torch.from_numpy(synthetic_state(FCN_CHANNELS, cfg.nlat, cfg.nlon, 0))
    eng = StepEngine(cfg, 0)
    eng.load_weights(w)
    res = dict(model="fourcastnet", grid=[cfg.nlat, cfg.nlon], depth=cfg.depth, gpu=gpu_info(), step={})

    y1 = None
    for B in (1, 4):
        bufs = [x0[None].expand(B, -1, -1, -1).contiguous().cuda(), torch.empty(B, 26, cfg.nlat, cfg.nlon, device="cuda")]
        if B == 1:
            y1 = eng.step(bufs[0]).clone()
        ms, n = time_chained(lambda i: eng.step(bufs[i % 2], bufs[(i + 1) % 2]), args.window)
        res["step"][f"B{B}"] = dict(ms_per_step=ms, member_steps_per_s=1e3 * B / ms, steps_timed=n,
                                    tensor_floor_fraction=roofline.fcn_flops(cfg, B)["total"] / PEAK_FLOPS / (ms * 1e-3))

    # per-family breakdown: one profiled B = 1 step (plain launches with events around each)
    xb = x0[None].contiguous().cuda()
    eng.profile_begin([t for t in StepEngine.profile_tags() if t.startswith("fcn_")])
    eng.step(xb)
    prof = eng.profile_end()
    fl, by = roofline.fcn_flops(cfg), roofline.fcn_bytes(cfg)
    res["families"] = {k: dict(ms=ms, launches=n, flops=fl[k], bytes=by[k],
                               bound="flops" if fl[k] / PEAK_FLOPS >= by[k] / PEAK_BYTES else "bytes",
                               fraction_of_bound=max(fl[k] / PEAK_FLOPS, by[k] / PEAK_BYTES) / (ms * 1e-3))
                       for k, (ms, n) in prof.items()}

    fx = verify.load_fixture("fcn", cfg.nlat)
    s = verify.summarise(verify.compare_fullsize(y1[0], fx, last_row=cfg.nlat - 1))
    s["ok"] = bool(s["finite"] and s["rel"] <= 1e-3)
    res["verify"] = s
    eng.close()

    # PyTorch eager fp32 forward of the same step (oracle code path on the GPU)
    ref = FCNRef(cfg, w, torch.float32, device="cuda")
    eager = {}
    with torch.no_grad():
        for B in (1, 4):
            xe = x0[None].expand(B, -1, -1, -1).contiguous().cuda()
            ye = ref.step(xe)
            ms, n = time_chained(lambda i: ref.step(xe), args.window)
            eager[f"B{B}"] = dict(ms_per_step=ms, member_steps_per_s=1e3 * B / ms, steps_timed=n)
            if B == 1:
                d = rel_err_per_channel(y1[0].cpu().numpy(), ye[0].cpu().numpy())
                eager["rel_diff_to_engine_max"] = float(d.max())
                eager["rel_diff_to_engine_mean"] = float(d.mean())
            del xe, ye
    eager["tf32"] = bool(torch.backends.cuda.matmul.allow_tf32)
    res["eager"] = eager
    res["speedup_vs_eager"] = {k: eager[k]["ms_per_step"] / res["step"][k]["ms_per_step"] for k in ("B1", "B4")}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_fcn.json"), "w") as f:
            f.write(line + "\n")
    sys.exit(0 if s["ok"] else 1)


if __name__ == "__main__":
    main()
