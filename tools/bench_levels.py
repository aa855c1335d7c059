#!/usr/bin/env python3
"""ookd_gpu_levels against an OOKD_FLAG_NO_SCREEN decode of the same span, in one process on one GPU.

The capture is bench.py's recipe (p3l-nexa2012, 2^30 samples, seeded), synthesised on the device and kept there, with
its CU8 form quantised on the device (v = clip(round((x + 2040) / 16), 0, 255)).  For each filter (fs32_fs4,
fs128_fs16_dec4), format (SC16Q11, CU8), tuning (off, and tune_step(-437 kHz)) and span (the first 2^26 samples, the
CLI's default first window, and all 2^30) it times, alternating them, rounds of
  * levels: Gpu.levels on the resident span (host clock around the synchronous call, which includes its allocations);
  * decode: a NO_SCREEN decode of the same span, the path that computes every output with the same in-order MACs:
    the whole call, and its fir_ms (the FIR/threshold kernels alone, CUDA events).
One JSON line per cell: medians, the histogram's output count, the card's name and power limit read in the same run.

    python tools/bench_levels.py [--rounds 5]
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
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--log2n", type=int, nargs="+", default=[26, 30])
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: nothing to measure")
    n_max = 1 << max(a.log2n)
    fir0 = H.Fir(bench.FILTER_NAME)
    dev0 = H.Device(bench.DEVICE_NAME, bench.FS // fir0.total_decimation)
    tog, _ = bench.build_toggles(dev0, n_max)
    i_on, q_on = bench.on_level()
    base = torch.empty((n_max, 2), dtype=torch.int16, device="cuda")
    B.synth(n_max, tog, i_on, q_on, bench.noise_scale(), bench.SEED, device_id=0, device_ptr=base.data_ptr(),
            noise_terms=bench.NOISE_TERMS)
    base8 = torch.empty((n_max, 2), dtype=torch.uint8, device="cuda")
    sl = 1 << 25
    for s0 in range(0, n_max, sl):
        x = base[s0:s0 + sl].to(torch.float32)
        base8[s0:s0 + sl] = torch.clamp(torch.round((x + 2040) / 16), 0, 255).to(torch.uint8)
    del x
    torch.cuda.synchronize()
    caps = {"sc16q11": base.data_ptr(), "cu8": base8.data_ptr()}
    step = B.tune_step(-437e3, bench.FS)
    name, plimit = card()
    for filt in ("fs32_fs4", "fs128_fs16_dec4"):
        fir = H.Fir(filt)
        dev = H.Device(bench.DEVICE_NAME, bench.FS // fir.total_decimation)
        for fmt in ("sc16q11", "cu8"):
            for t in (0, step):
                kw = dict(filter_stages=fir.stages, threshold=bench.THR, samples_per_buffer=bench.SPB, device_id=0,
                          input_format=fmt, tune_step=t)
                gl = B.Gpu(**kw)
                gd = B.Gpu(sm=dev.sm_spec(), flags=B.FLAG_NO_SCREEN, **kw)
                gd.want_list = False
                for log2n in a.log2n:
                    n = 1 << log2n
                    cap = (caps[fmt], n)
                    lv, dc, fr = [], [], []
                    for r in range(a.rounds + 1):              # one warm-up round
                        torch.cuda.synchronize()
                        t0 = time.perf_counter()
                        hist = gl.levels(cap)
                        t1 = time.perf_counter()
                        res = gd.decode(cap)
                        t2 = time.perf_counter()
                        if r >= 1:
                            lv.append((t1 - t0) * 1e3)
                            dc.append((t2 - t1) * 1e3)
                            fr.append(res["fir_ms"])
                    print(json.dumps({
                        "filter": filt, "format": fmt, "tune_step": t, "samples": n, "outputs": int(hist.sum()),
                        "levels_ms": round(statistics.median(lv), 4), "levels_ms_min": round(min(lv), 4),
                        "no_screen_decode_ms": round(statistics.median(dc), 4),
                        "no_screen_fir_ms": round(statistics.median(fr), 4), "n_msgs": int(len(res["msgs_raw"])),
                        "rounds": a.rounds, "gpu": name, "power_limit": plimit}), flush=True)
                del gl, gd


if __name__ == "__main__":
    main()
