"""Independent captures (BASELINE configs[4] shape): N captures x 2^24 samples, devices alternating between
p3l-nexa2012 and unknown-remote1, filter fs64_fs8, sigma in {0, 0.02, 0.05}, decoded with ookd_gpu_batch_decode
over H handles per device description.  Prints captures/s and Msamples/s for H = 1, 2, 4 (device-resident input)."""
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from ookiedokie_b200 import binding as B, host as H

n_caps = int(sys.argv[1]) if len(sys.argv) > 1 else 64
n = 1 << 24
fir = H.Fir("fs64_fs8")
names = ["p3l-nexa2012", "unknown-remote1"]
devs = [H.Device(nm, 3000000 // fir.total_decimation) for nm in names]
ih4 = (4.0 * (65536.0 ** 2 - 1.0) / 12.0) ** 0.5
bufs, n_tx = [], 0
for i in range(n_caps):
    kind = i % 2
    msgs = [devs[kind].message({}) for _ in range(n // (180000 if kind else 400000) + 2)]
    tog, total = devs[kind].toggles(msgs, 12000)
    sigma = [0.0, 0.02, 0.05][i % 3]
    d = torch.empty(n * 2, dtype=torch.int16, device="cuda")
    B.synth(n, np.ascontiguousarray(tog), 1488, 1253, int(round(sigma * 2048 / ih4 * (1 << 24))), 1000 + i, device_ptr=d.data_ptr())
    bufs.append(d)
torch.cuda.synchronize()
for per in (2, 4, 8):
    gpus = []
    for kind in range(2):
        for _ in range(per):
            gpus.append(B.Gpu(filter_stages=fir.stages, sm=devs[kind].sm_spec(), threshold=0.1, samples_per_buffer=8192))
    caps = [((bufs[i].data_ptr(), n), (i % 2) * per + (i // 2) % per) for i in range(n_caps)]
    B.batch_decode(gpus, caps[:2 * per])            # warm-up (workspace allocation)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    msgs, stats = B.batch_decode(gpus, caps)
    dt = time.perf_counter() - t0
    print(f"{per} handle(s) per device type: {n_caps} captures x 2^24 samples in {dt * 1e3:.2f} ms = "
          f"{n_caps / dt:.0f} captures/s = {n_caps * n / dt / 1e6:.0f} Msamples/s; {sum(len(m) for m in msgs)} messages; "
          f"mean decode span {np.mean([s['kernel_ms'] for s in stats]):.3f} ms, host syncs/capture {np.mean([s['host_syncs'] for s in stats]):.2f}")
    for g in gpus:
        g.close()
