#!/usr/bin/env python3
"""CU8 against SC16Q11 on the benchmark workload, in one process on one GPU.

The capture is bench.py's recipe (p3l-nexa2012 + fs32_fs4, 2^30 samples, seeded), synthesised on the device, quantised
to CU8 on the device (v = clip(round((x + 2040) / 16), 0, 255)), and widened back to SC16Q11 (16 v - 2040): the two
decodes read the same signal, 2 and 4 bytes per sample.  Timed rounds alternate the two formats:
  * a decode with sub_windows = 3 (bench.py's default) from device memory, host clock around the synchronous call;
  * a decode of the same capture on an undivided handle, whose screen_ms is the screening kernel alone.
The message lists must be equal.  One JSON line per format: ms per decode (median), Msamples/s, screen_ms (median),
the screen's share of the HBM roofline at its own bytes per sample (peak as bench.py reads it), the card's name and
power limit read in the same run.

    python tools/bench_input8.py [--log2n 30] [--rounds 10]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (the workload recipe)
from ookiedokie_b200 import binding as B  # noqa: E402
from ookiedokie_b200 import host as H  # noqa: E402


def card(device=0):
    """Name and power limit of the GPU torch runs on (selected by UUID: under CUDA_VISIBLE_DEVICES, nvidia-smi's index 0
    need not be torch's device 0)."""
    import torch
    name = torch.cuda.get_device_name(device)
    uuid = str(getattr(torch.cuda.get_device_properties(device), "uuid", "") or "")
    if not uuid:
        return name, "unknown"
    sel = uuid if uuid.startswith(("GPU-", "MIG-")) else "GPU-" + uuid
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", sel],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        smi_name, limit = [x.strip() for x in out.split(",")[:2]]
        return smi_name, limit
    except Exception:
        return name, "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2n", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=10)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: nothing to measure")
    n = 1 << a.log2n
    fir = H.Fir(bench.FILTER_NAME)
    dev = H.Device(bench.DEVICE_NAME, bench.FS // fir.total_decimation)
    tog, _ = bench.build_toggles(dev, n)
    i_on, q_on = bench.on_level()
    d16 = torch.empty((n, 2), dtype=torch.int16, device="cuda")
    B.synth(n, tog, i_on, q_on, bench.noise_scale(), bench.SEED, device_id=0, device_ptr=d16.data_ptr(),
            noise_terms=bench.NOISE_TERMS)
    v = torch.empty((n, 2), dtype=torch.uint8, device="cuda")
    step = 1 << 26
    for s0 in range(0, n, step):                       # (in slices: a float copy of the whole capture is 8 GiB)
        x = d16[s0:s0 + step].to(torch.float32)
        v[s0:s0 + step] = torch.clamp(torch.round((x + 2040) / 16), 0, 255).to(torch.uint8)
    del d16, x
    w = v.to(torch.int16) * 16 - 2040
    torch.cuda.synchronize()

    kw = dict(filter_stages=fir.stages, sm=dev.sm_spec(), threshold=bench.THR, samples_per_buffer=bench.SPB, device_id=0)
    caps = {"cu8": (v.data_ptr(), n), "sc16q11": (w.data_ptr(), n)}
    subw = {f: B.Gpu(input_format=f, sub_windows=3, **kw) for f in caps}
    whole = {f: B.Gpu(input_format=f, **kw) for f in caps}
    for g in list(subw.values()) + list(whole.values()):
        g.want_list = False
    ms = {f: [] for f in caps}
    scr = {f: [] for f in caps}
    last = {}
    for r in range(a.rounds + 2):                      # two warm-up rounds
        for f in caps:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = subw[f].decode(caps[f])
            t1 = time.perf_counter()
            res_w = whole[f].decode(caps[f])
            if r >= 2:
                ms[f].append((t1 - t0) * 1e3)
                scr[f].append(res_w["screen_ms"])
            last[f] = (res["msgs_raw"], res_w["msgs_raw"])
    for k in range(2):
        assert last["cu8"][k].tobytes() == last["sc16q11"][k].tobytes(), "CU8 and SC16Q11 decodes differ"
    peak, peak_src = bench.measured_peak()
    name, plimit = card()
    for f, bps in (("cu8", 2), ("sc16q11", 4)):
        t = statistics.median(ms[f])
        s = statistics.median(scr[f])
        print(json.dumps({
            "format": f, "samples": n, "bytes_per_sample": bps, "sub_windows": 3,
            "ms_per_decode": round(t, 4), "ms_per_decode_min": round(min(ms[f]), 4),
            "msamples_per_s": round(n / t / 1e3, 1), "screen_ms": round(s, 4),
            "screen_hbm_fraction": round(n * bps / (s * 1e-3) / (peak * 1e9), 4),
            "screen_hbm_fraction_at_4B": round(n * 4 / (s * 1e-3) / (peak * 1e9), 4),
            "screen_hbm_fraction_at_2B": round(n * 2 / (s * 1e-3) / (peak * 1e9), 4),
            "hbm_peak_gbs": peak, "hbm_peak_source": peak_src, "n_msgs": int(len(last[f][0])),
            "rounds": a.rounds, "gpu": name, "power_limit": plimit}))


if __name__ == "__main__":
    main()
