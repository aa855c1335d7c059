#!/usr/bin/env python3
"""The deglitch sweep of DESIGN §3.12, on the CPU: messages decoded (bytes equal to a sent message) per M, with the
oracle's decisions through the streaming vote of tests/vote_ref.py.  No GPU.

    python tools/deglitch_sweep.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import oracle as O  # noqa: E402
import ookd_testutil as util  # noqa: E402
import vote_ref as V  # noqa: E402


def auto_threshold(iq, stages, margin=12.0):
    """-T auto (include/ookd_gpu.h, "Levels") restated from the oracle's filtered power"""
    f = O.rx(iq, stages, None, samples_per_buffer=8192, want_filtered=True)["filtered"].astype(np.float32)
    p = (f[:, 0] * f[:, 0] + f[:, 1] * f[:, 1]).astype(np.float32)
    h = np.bincount((p.view(np.uint32) & 0x7FFFFFFF) >> 19, minlength=4096).astype(np.int64)
    cum = np.cumsum(h)
    m = int(np.argmax(cum >= cum[-1] - cum))
    F = float(np.array([(m + 1) << 19], np.uint32).view(np.float32)[0])
    return float(np.float32(np.sqrt(F * 10 ** (margin / 10))))


def row(name, devname, filt, spb, n_msgs, sigma, amp, seed, ms, thr=0.1, glitches=()):
    dev = O.load_device(devname)
    stages = O.load_filter(filt)
    fields = util.nexa_fields if "nexa" in devname else util.remote_fields
    iq, sent, _ = util.capture(dev, n_msgs, sigma=sigma, amplitude=amp, phase=0.4, seed=seed, fields=fields,
                               glitches=glitches)
    if thr == "auto":
        thr = auto_threshold(iq, stages)
    cells = []
    for m in ms:
        got = V.rx(iq, stages, dev, threshold_=thr, samples_per_buffer=spb, deglitch=m)["msgs"]
        cells.append(f"M={m}: {sum(1 for g in got if g[3] in sent)}/{len(sent)}")
    print(f"{name} (threshold {thr:.4g}): " + ", ".join(cells), flush=True)


def main():
    ms = [0, 8, 16, 64, 128]
    row("nexa fs64_fs8 spb 4096 sigma 0.01, 100-sample burst at 9000", "p3l-nexa2012", "fs64_fs8", 4096, 9, 0.01, 0.8,
        21, ms, glitches=((9000, 100),))
    row("nexa fs32_fs4 A 0.95 sigma 0.03", "p3l-nexa2012", "fs32_fs4", 8192, 10, 0.03, 0.95, 5, ms)
    row("remote1 fs128_fs16_dec4 A 0.30 sigma 0.10 (C3-like)", "unknown-remote1", "fs128_fs16_dec4", 8192, 10, 0.10,
        0.30, 7, ms)
    row("nexa fs32_fs4 A 0.95 sigma 0.02 (benchmark-like), -T auto", "p3l-nexa2012", "fs32_fs4", 8192, 10, 0.02, 0.95,
        3, ms, thr="auto")
    row("nexa fs64_fs8 A 0.05 sigma 0.005, -T auto", "p3l-nexa2012", "fs64_fs8", 8192, 8, 0.005, 0.05, 4, ms, thr="auto")
    row("nexa fs64_fs8 A 0.02 sigma 0.002, -T auto", "p3l-nexa2012", "fs64_fs8", 8192, 8, 0.002, 0.02, 4, ms, thr="auto")
    row("remote1 fs128_fs16_dec4 A 0.30 sigma 0.10 (C3-like), -T auto", "unknown-remote1", "fs128_fs16_dec4", 8192, 10,
        0.10, 0.30, 7, ms, thr="auto")


if __name__ == "__main__":
    main()
