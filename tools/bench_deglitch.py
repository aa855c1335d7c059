#!/usr/bin/env python3
"""Decode time with the deglitch vote (include/ookd_gpu.h, "Deglitch") at several M, in one process on one GPU.

The workload is bench.py's recipe (p3l-nexa2012 + fs32_fs4, 2^30 samples, seeded), synthesised on the device and
decoded from device memory.  Timed rounds alternate the decode at M in --ms (default 0, 16, 64, 1024): each one with
sub_windows = 3 (bench.py's default), host clock around the synchronous call, and once on an undivided handle whose
kernel_ms - fir_ms is everything after the FIR (vote, edges, state machine).  One JSON line per M: medians and minima of
--rounds rounds after two warm-up rounds, message count, and the card's name and power limit read in the same run.

--profile instead runs a few decodes of each M under torch.profiler (CUDA activities, a run of its own) and prints the
vote kernel's device time per decode, with its byte bound: n_out / 8 bytes read and n_out / 8 written, over the
data-sheet 7.7 TB/s.

    python tools/bench_deglitch.py [--log2n 30] [--rounds 10] [--ms 0,16,64,1024] [--profile]
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

HBM_BYTES_PER_S = 7.7e12


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2n", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--ms", default="0,16,64,1024")
    ap.add_argument("--profile", action="store_true")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: nothing to measure")
    ms_list = [int(v) for v in a.ms.split(",")]
    n = 1 << a.log2n
    fir = H.Fir(bench.FILTER_NAME)
    dev = H.Device(bench.DEVICE_NAME, bench.FS // fir.total_decimation)
    tog, _ = bench.build_toggles(dev, n)
    i_on, q_on = bench.on_level()
    cap = torch.empty((n, 2), dtype=torch.int16, device="cuda")
    B.synth(n, tog, i_on, q_on, bench.noise_scale(), bench.SEED, device_id=0, device_ptr=cap.data_ptr(),
            noise_terms=bench.NOISE_TERMS)
    torch.cuda.synchronize()
    src = (cap.data_ptr(), n)
    kw = dict(filter_stages=fir.stages, sm=dev.sm_spec(), threshold=bench.THR, samples_per_buffer=bench.SPB, device_id=0)
    whole = {m: B.Gpu(deglitch=m, **kw) for m in ms_list}
    for g in whole.values():
        g.want_list = False
    name, plimit = card()

    if a.profile:
        from torch.profiler import ProfilerActivity, profile
        for g in whole.values():                                 # warm-up outside the trace
            g.decode(src)
        reps = 3
        out = {}
        for m, g in whole.items():
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(reps):
                    res = g.decode(src)
                torch.cuda.synchronize()
            us = [e.device_time for e in prof.events() if "vote_kernel" in e.name]
            out[m] = (us, res["n_out"])
        for m, (us, n_out) in out.items():
            bound_us = 2 * (n_out / 8) / HBM_BYTES_PER_S * 1e6
            print(json.dumps({"profile": "vote_kernel", "deglitch": m, "samples": n, "n_out": n_out,
                              "launches": len(us), "us_per_decode": round(sum(us) / reps, 2),
                              "byte_bound_us": round(bound_us, 2), "gpu": name, "power_limit": plimit}))
        return

    subw = {m: B.Gpu(deglitch=m, sub_windows=3, **kw) for m in ms_list}
    for g in subw.values():
        g.want_list = False
    t_sub = {m: [] for m in ms_list}
    t_tail = {m: [] for m in ms_list}
    t_kernel = {m: [] for m in ms_list}
    nmsg = {}
    for r in range(a.rounds + 2):                                # two warm-up rounds
        for m in ms_list:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = subw[m].decode(src)
            t1 = time.perf_counter()
            res_w = whole[m].decode(src)
            if r >= 2:
                t_sub[m].append((t1 - t0) * 1e3)
                t_kernel[m].append(res_w["kernel_ms"])
                t_tail[m].append(res_w["kernel_ms"] - res_w["fir_ms"])
            assert res["msgs_raw"].tobytes() == res_w["msgs_raw"].tobytes(), f"M={m}: sub-windows and whole decode differ"
            nmsg[m] = int(len(res["msgs_raw"]))
    for m in ms_list:
        print(json.dumps({
            "deglitch": m, "samples": n, "sub_windows": 3, "ms_per_decode": round(statistics.median(t_sub[m]), 4),
            "ms_per_decode_min": round(min(t_sub[m]), 4), "ms_per_decode_max": round(max(t_sub[m]), 4),
            "whole_kernel_ms": round(statistics.median(t_kernel[m]), 4),
            "whole_after_fir_ms": round(statistics.median(t_tail[m]), 4), "n_msgs": nmsg[m], "rounds": a.rounds,
            "gpu": name, "power_limit": plimit}))


if __name__ == "__main__":
    main()
