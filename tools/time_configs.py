import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from ookiedokie_b200 import binding as B, host as H
n = 1 << 28
for devname, filt, amp, sigma in [("unknown-remote1", "fs128_fs16_dec4", 0.30, 0.10), ("unknown-remote1", "fs128_fs16_dec4", 0.30, 0.05), ("p3l-nexa2012", "fs128_fs16_dec4", 0.95, 0.02), ("unknown-remote1", "fs32_fs4", 0.30, 0.10), ("p3l-nexa2012", "fs64_fs8", 0.95, 0.02)]:
    fir = H.Fir(filt); dev = H.Device(devname, 3000000 // fir.total_decimation)
    txdev = H.Device(devname, 3000000)          # the transmitter runs at the full sample rate
    msgs = [txdev.message({}) for _ in range(n // 180000 + 4)]
    tog, total = txdev.toggles(msgs, 12000)
    d = torch.empty(n * 2, dtype=torch.int16, device="cuda")
    ih4 = (4.0 * (65536.0 ** 2 - 1.0) / 12.0) ** 0.5
    B.synth(n, tog, int(amp * 2048 * 0.76), int(amp * 2048 * 0.65), int(round(sigma * 2048 / ih4 * (1 << 24))), 7, device_ptr=d.data_ptr())
    g = B.Gpu(filter_stages=fir.stages, sm=dev.sm_spec(), threshold=0.1)
    g.want_list = False
    r0 = g.decode((d.data_ptr(), n))
    for it in range(2):
        r = g.decode((d.data_ptr(), n))
    print(devname, filt, f"amp {amp} sigma {sigma}: fir_ms {r['fir_ms']:.2f} kernel_ms {r['kernel_ms']:.2f} -> {n / r['kernel_ms'] / 1e6:.1f} Gsamples/s, msgs {len(r['msgs_raw'])}/{len(msgs)} edges {r['n_edges']} rounds {r['sm_rounds']} refined {r['refined_blocks']} (first call: {r0['refined_blocks']}, overflow {r0['refined_tiles']}, fir_ms {r0['fir_ms']:.2f})")
