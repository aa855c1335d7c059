#!/usr/bin/env python3
"""Tuned decode of an off-centre capture against the untuned decode of the baseband capture, in one process on one GPU.

The baseband capture is bench.py's recipe (p3l-nexa2012 + fs32_fs4, 2^30 samples, seeded), synthesised on the device.
For timing only, the tool moves it up by +f (default 900 kHz at 3 MS/s, in the fs32_fs4 stopband, so an untuned decode
of it finds nothing) with a float rotation on the device, rounded and clamped to int16.  The CU8 forms of both captures
are quantised on the device (v = clip(round((x + 2040) / 16), 0, 255)).  Timed rounds alternate four decodes:
  * sc16q11 tuned: the offset capture with tune_step(f, 3 MS/s);  sc16q11 plain: the baseband capture untuned;
  * cu8 tuned / cu8 plain: the same in CU8.
Each is measured as a decode with sub_windows = 3 (bench.py's default) from device memory, host clock around the
synchronous call, and as a decode on an undivided handle, whose screen_ms is the screening kernel alone.  One JSON line
per decode kind: medians, message count, the card's name and power limit read in the same run.

    python tools/bench_tune.py [--log2n 30] [--rounds 10] [--offset 900e3]
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402  (the workload recipe)
from bench_input8 import card  # noqa: E402
from ookiedokie_b200 import binding as B  # noqa: E402
from ookiedokie_b200 import host as H  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2n", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--offset", type=float, default=900e3)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: nothing to measure")
    n = 1 << a.log2n
    fir = H.Fir(bench.FILTER_NAME)
    dev = H.Device(bench.DEVICE_NAME, bench.FS // fir.total_decimation)
    tog, _ = bench.build_toggles(dev, n)
    i_on, q_on = bench.on_level()
    base = torch.empty((n, 2), dtype=torch.int16, device="cuda")
    B.synth(n, tog, i_on, q_on, bench.noise_scale(), bench.SEED, device_id=0, device_ptr=base.data_ptr(),
            noise_terms=bench.NOISE_TERMS)
    off = torch.empty_like(base)
    base8 = torch.empty((n, 2), dtype=torch.uint8, device="cuda")
    off8 = torch.empty_like(base8)
    sl = 1 << 25
    w = 2.0 * torch.pi * a.offset / bench.FS
    for s0 in range(0, n, sl):                         # (in slices: float copies of the whole capture are 16 GiB)
        x = base[s0:s0 + sl].to(torch.float64)
        ph = torch.arange(s0, s0 + x.shape[0], device="cuda", dtype=torch.float64) * w
        c, s = torch.cos(ph), torch.sin(ph)
        y = torch.stack([x[:, 0] * c - x[:, 1] * s, x[:, 0] * s + x[:, 1] * c], -1)
        off[s0:s0 + sl] = torch.clamp(torch.round(y), -32768, 32767).to(torch.int16)
        base8[s0:s0 + sl] = torch.clamp(torch.round((x + 2040) / 16), 0, 255).to(torch.uint8)
        off8[s0:s0 + sl] = torch.clamp(torch.round((off[s0:s0 + sl].to(torch.float64) + 2040) / 16), 0, 255).to(torch.uint8)
    del x, ph, c, s, y
    torch.cuda.synchronize()

    step = B.tune_step(a.offset, bench.FS)
    kw = dict(filter_stages=fir.stages, sm=dev.sm_spec(), threshold=bench.THR, samples_per_buffer=bench.SPB, device_id=0)
    kinds = {  # name: (input_format, tune_step, capture)
        "sc16q11_tuned": ("sc16q11", step, (off.data_ptr(), n)),
        "sc16q11_plain": ("sc16q11", 0, (base.data_ptr(), n)),
        "cu8_tuned": ("cu8", step, (off8.data_ptr(), n)),
        "cu8_plain": ("cu8", 0, (base8.data_ptr(), n)),
    }
    subw = {k: B.Gpu(input_format=f, tune_step=t, sub_windows=3, **kw) for k, (f, t, _) in kinds.items()}
    whole = {k: B.Gpu(input_format=f, tune_step=t, **kw) for k, (f, t, _) in kinds.items()}
    for g in list(subw.values()) + list(whole.values()):
        g.want_list = False
    ms = {k: [] for k in kinds}
    scr = {k: [] for k in kinds}
    nmsg = {}
    for r in range(a.rounds + 2):                      # two warm-up rounds
        for k, (_, _, cap) in kinds.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = subw[k].decode(cap)
            t1 = time.perf_counter()
            res_w = whole[k].decode(cap)
            if r >= 2:
                ms[k].append((t1 - t0) * 1e3)
                scr[k].append(res_w["screen_ms"])
            assert res["msgs_raw"].tobytes() == res_w["msgs_raw"].tobytes(), f"{k}: sub-windows and whole decode differ"
            nmsg[k] = int(len(res["msgs_raw"]))
    name, plimit = card()
    for k, (f, t, _) in kinds.items():
        print(json.dumps({
            "decode": k, "format": f, "tune_step": t, "offset_hz": a.offset if t else 0.0, "samples": n,
            "sub_windows": 3, "ms_per_decode": round(statistics.median(ms[k]), 4),
            "ms_per_decode_min": round(min(ms[k]), 4), "screen_ms": round(statistics.median(scr[k]), 4),
            "screen_ms_min": round(min(scr[k]), 4), "n_msgs": nmsg[k], "rounds": a.rounds, "gpu": name,
            "power_limit": plimit}))


if __name__ == "__main__":
    main()
