#!/usr/bin/env python3
"""bench.py -- IQ Msamples/s decoded (SC16Q11 -> OOK messages) on 1..8 B200, % of HBM roofline.

Workload (BASELINE.json configs[1], named in config.workload): p3l-nexa2012 bursts through
filters/fs32_fs4.json on a 4 GiB (2^30 samples) synthetic SC16Q11 capture per GPU (amplitude 0.95,
carrier phase 0.7 rad, integer AWGN sigma 0.02, per-message field variation, seed 0x00C0FFEE).  With
N > 1 the ranks decode consecutive 4 GiB time shards of ONE continuous N*4 GiB capture (FIR halo
reads + state-machine carry stitch, ookiedokie_b200/shard.py): weak scaling, no collective on the
data path; only the 48-byte carries and the message lists cross ranks.

    value : whole-job Msamples/s with the shard already resident in HBM
    e2e   : same through the C ABI with the shard in pinned HOST memory (H2D inside the timed region,
            message list read back every step)
    --impl reference : the unmodified reference binary (oracle/_ref/ookiedokie, single threaded as the
            reference is) on a bounded prefix of the same capture, on the box's host cores.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# many independent captures in flight (configs.c5): one hardware queue per stream instead of the default 8 shared ones
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

DEVICE_NAME = "p3l-nexa2012"
FILTER_NAME = "fs32_fs4"
FS = 3000000
SPB = 8192
THR = 0.1
AMP, PHASE, SIGMA, SEED = 0.95, 0.7, 0.02, 0x00C0FFEE
LEAD = 12000
METRIC = "IQ Msamples/s decoded (SC16Q11->OOK msgs)"
UNIT = "Msamples/s"


def workload_name(samples):
    return (f"{DEVICE_NAME} + {FILTER_NAME}, {samples * 4 / 2**30:.3g} GiB synthetic SC16Q11 capture per GPU "
            f"(amp {AMP}, near-Gaussian noise sigma {SIGMA} [Irwin-Hall 12, tails to 6 sigma], thr {THR}, spb {SPB}, fs {FS})")


def message_params(i):
    return {"Channel": str(1 + i % 3), "Temperature (C)": f"{-20.0 + 0.1 * ((i * 37) % 900):.1f}"}


def build_toggles(dev, total_samples):
    """Messages tiled back to back until they cover total_samples.  -> (toggles, n_messages)."""
    import numpy as np
    est = total_samples // 380000 + 8
    msgs = [dev.message(message_params(i)) for i in range(est)]
    tog, total = dev.toggles(msgs, LEAD)
    while total < total_samples:
        est *= 2
        msgs = [dev.message(message_params(i)) for i in range(est)]
        tog, total = dev.toggles(msgs, LEAD)
    return np.ascontiguousarray(tog), len(msgs)


def on_level():
    import math
    return int(round(AMP * 2048.0 * math.cos(PHASE))), int(round(AMP * 2048.0 * math.sin(PHASE)))


NOISE_TERMS = 12        # noise = centred sum of twelve 16-bit uniforms (Irwin-Hall 12): Gaussian to within a few per cent
                        # out to 4 sigma, tails to +-6 sigma; integer-only, so the CPU and GPU generators agree byte for byte


def noise_scale(sigma=SIGMA):
    std = (NOISE_TERMS * (65536.0 ** 2 - 1.0) / 12.0) ** 0.5       # std of the sum of NOISE_TERMS 16-bit uniforms
    return int(round(sigma * 2048.0 / std * (1 << 24)))


DUMP_LIMIT = 64 << 20               # bytes --dump-outputs writes at most, row indices of sampled arrays included


def message_table(rec, nbytes):
    """Structured message array -> float64 rows (out_sample, buffer_idx, num_bits, the nbytes message bytes)."""
    import numpy as np
    t = np.empty((len(rec), 3 + nbytes), dtype=np.float64)
    t[:, 0] = rec["out_sample"]
    t[:, 1] = rec["buffer_idx"]
    t[:, 2] = rec["num_bits"]
    t[:, 3:] = rec["data"][:, :nbytes]
    return t


def write_outputs(out_dir, arrays):
    """Each array as out_dir/<name>.npy in float64.  An array with more rows than its equal share of DUMP_LIMIT holds is
    cut to a fixed, seeded sample of its rows (in order), and the indices of those rows go to <name>_rows.npy."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_LIMIT // len(arrays)
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64)
        row_bytes = 8 * (a[0].size if a.ndim > 1 and len(a) else 1)
        max_rows = share // (row_bytes + 8)
        if a.ndim > 0 and len(a) > max_rows:
            rows = np.sort(np.random.default_rng(SEED).choice(len(a), size=max_rows, replace=False))
            a = a[rows]
            np.save(os.path.join(out_dir, f"{name}_rows.npy"), rows.astype(np.float64))
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons during the timed region: NVML polled every 5 ms in-process (the same
    counters `nvidia-smi --query-gpu=clocks.sm,clocks_event_reasons.*` prints; nvidia-smi -lms cannot
    sample a region shorter than its own start-up), nvidia-smi as the fallback."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.proc = None
        self.stop_flag = False
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:
            self.nvml = None

    def run(self):
        if self.nvml is not None:
            n = self.nvml
            reasons = [("hw_slowdown", getattr(n, "nvmlClocksEventReasonHwSlowdown", 0x8)),
                       ("hw_thermal_slowdown", getattr(n, "nvmlClocksEventReasonHwThermalSlowdown", 0x40)),
                       ("sw_thermal_slowdown", getattr(n, "nvmlClocksEventReasonSwThermalSlowdown", 0x20)),
                       ("sw_power_cap", getattr(n, "nvmlClocksEventReasonSwPowerCap", 0x4))]
            try:
                mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
            except Exception:
                mx = 0
            while not self.stop_flag:
                try:
                    sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                    try:
                        mask = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                    except Exception:
                        mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                    self.rows.append([str(sm), str(mx), "0"] + ["Active" if mask & bit else "Not Active" for _, bit in reasons]
                                     + [time.perf_counter()])
                except Exception:
                    break
                time.sleep(0.005)
            return
        self._run_smi()

    def _run_smi(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self, t_start=None, t_end=None):
        """Summary of the samples taken inside [t_start, t_end] (all samples if none fall inside)."""
        self.stop_flag = True
        if self.nvml is not None:
            self.join(timeout=1.0)
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], 0, set()
        rows = self.rows
        if t_start is not None:
            inside = [r for r in rows if len(r) > 7 and t_start <= r[7] <= t_end]
            rows = inside or rows
        for r in rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        busy = [c for c in sm if c > 0.5 * mx] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get("dram_bytes_per_launch")
        except Exception:
            pass
    return None


def reference_binary():
    p = os.path.join(ROOT, "oracle", "_ref", "ookiedokie")
    return p if os.path.exists(p) else None


def run_reference_cpu(iq_prefix, repeats=1, want_parity=False, device=DEVICE_NAME, filt=FILTER_NAME):
    """Times the unmodified reference binary on a capture prefix.  -> (Msamples/s, n_rows[, csv rows, first_bit, edges]).
    The parity outputs (csv rows without the wall-clock column, --rx-rec-dig transitions) come from a second, untimed
    run so that the timed one is the plain decode."""
    ref = reference_binary()
    tmpdir = "/dev/shm" if os.path.isdir("/dev/shm") else None
    with tempfile.TemporaryDirectory(dir=tmpdir) as td:
        cap = os.path.join(td, "cap.sc16q11")
        iq_prefix.tofile(cap)
        n = iq_prefix.size // 2
        best, rows = None, 0
        env = dict(os.environ, OOKD_DATA_DIR=os.path.join(ROOT, "ookiedokie_b200", "data") + "/")
        dev_path = os.path.join(ROOT, "ookiedokie_b200", "data", "devices", device + ".json")
        filt_path = os.path.join(ROOT, "ookiedokie_b200", "data", "filters", filt + ".json")
        cmd = [ref, "--rx", "bladerf_file", "-A", cap, "-d", dev_path, "-F", filt_path, "--rx-fmt", "csv",
               "--samples-per-buffer", str(SPB), "-T", str(THR), "-s", str(FS)]
        for _ in range(repeats):
            t0 = time.perf_counter()
            out = subprocess.run(cmd, capture_output=True, text=True, env=env, check=True)
            dt = time.perf_counter() - t0
            rows = max(len(out.stdout.strip().splitlines()) - 1, 0)
            best = dt if best is None else min(best, dt)
        if not want_parity:
            return n / best / 1e6, rows
        dig = os.path.join(td, "dig.csv")
        out = subprocess.run(cmd + ["-B", dig], capture_output=True, text=True, env=env, check=True)
        lines = out.stdout.strip().splitlines()
        has_ts = "nexa" in device                       # ts_mode unix-frac: first column is the wall clock
        csv_rows = [l.split(",")[1:] if has_ts else l.split(",") for l in lines[1:]]
        dl = open(dig).read().strip().splitlines()
        first_bit = int(dl[0].split(",")[1])
        edges = [int(dl[k].split(",")[0]) for k in range(2, len(dl), 2)]
    return n / best / 1e6, rows, csv_rows, first_bit, edges


def impl_reference(args, rank, world):
    if rank != 0:
        return
    import numpy as np
    line = {"impl": "reference", "metric": METRIC, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic"}
    if reference_binary() is None:
        line.update({"unavailable": "oracle/_ref/ookiedokie not built (needs /root/reference at build time)"})
        print(json.dumps(line))
        return
    from oracle import oracle as O
    dev = O.load_device(DEVICE_NAME)
    n = args.ref_samples
    n_msgs = n // 380000 + 4
    msgs = [O.message_bytes(dev, message_params(i)) for i in range(n_msgs)]
    tog, _ = O.toggles_from_messages(dev, msgs, FS, LEAD)
    i_on, q_on = on_level()
    iq = O.synth(n, tog, i_on, q_on, noise_scale(), SEED, noise_terms=NOISE_TERMS)
    for _ in range(args.warmup):
        run_reference_cpu(iq)
    vals = []
    t0 = time.perf_counter()
    rows = 0
    for _ in range(args.steps):
        v, rows = run_reference_cpu(iq)
        vals.append(v)
    total = time.perf_counter() - t0
    value = statistics.mean(vals)
    sample = f"first {n} samples ({n * 4 / 2**20:.0f} MiB) of the same synthetic capture, {rows} messages decoded"
    line.update({"value": value, "ms_per_step": 1e3 * total / max(args.steps, 1),
                 "config": {"workload": workload_name(args.samples), "sample": sample},
                 "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": "reference", "sample": sample},
                 "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                 "gpu_launches": 0})
    print(json.dumps(line))


def pin_to_gpu_numa(local_rank):
    """Run this rank (and therefore allocate its pinned staging memory) on the CPUs local to its GPU.
    -> description for the bench line."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local_rank)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        base = f"/sys/bus/pci/devices/{bdf}"
        node = int(open(base + "/numa_node").read().strip())
        cpus = open(base + "/local_cpulist").read().strip()
        if node < 0 or not cpus:
            return {"numa_node": node, "pinned": False}
        ids = set()
        for part in cpus.split(","):
            lo, _, hi = part.partition("-")
            ids.update(range(int(lo), int(hi or lo) + 1))
        ids &= os.sched_getaffinity(0)
        if ids:
            os.sched_setaffinity(0, ids)
        return {"numa_node": node, "pinned": bool(ids), "cpus": cpus}
    except Exception as e:                                   # sysfs layout differs / containers without it
        return {"pinned": False, "why": str(e)[:80]}


FP32_ISSUE_PER_S = 148 * 128 * 1.965e9                       # fp32 lanes x clock (MEASURED_PEAKS.json sm_max_mhz)


def measure_c3(local_rank, peak, sub_windows=0):
    """BASELINE configs[2]: unknown-remote1 through fs128_fs16_dec4 on a low-SNR capture (amp 0.30, near-Gaussian noise
    sigma 0.10): nothing can be screened, the exact two-stage kernel computes every output (fp32-issue bound)."""
    import numpy as np
    import torch
    from ookiedokie_b200 import binding as B
    from ookiedokie_b200 import host as H
    n = 1 << 28
    fir = H.Fir("fs128_fs16_dec4")
    dev = H.Device("unknown-remote1", FS // fir.total_decimation)
    tx = H.Device("unknown-remote1", FS)
    buttons = ["Power", "Pause", "P1"]
    msgs = [tx.message({"ID": hex(i % 256), "Button": buttons[i % 3]}) for i in range(n // 200000 + 8)]
    tog, total = tx.toggles(msgs, LEAD)
    import math
    i_on, q_on = int(round(0.30 * 2048 * math.cos(0.4))), int(round(0.30 * 2048 * math.sin(0.4)))
    d = torch.empty((n * 2,), dtype=torch.int16, device="cuda")
    B.synth(n, np.ascontiguousarray(tog), i_on, q_on, noise_scale(0.10), 7, device_id=local_rank, device_ptr=d.data_ptr(),
            noise_terms=NOISE_TERMS)
    torch.cuda.synchronize()
    g = B.Gpu(filter_stages=fir.stages, sm=dev.sm_spec(), threshold=THR, samples_per_buffer=SPB, device_id=local_rank,
              sub_windows=sub_windows)
    g.want_list = False
    first = g.decode((d.data_ptr(), n))                      # (the screen's verdict: work list overflow -> exact kernels)
    g.decode((d.data_ptr(), n))
    steps = 5
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fir_ms = 0.0
    for _ in range(steps):
        r = g.decode((d.data_ptr(), n))
        fir_ms += r["fir_ms"]
    dt = (time.perf_counter() - t0) / steps
    out = {"workload": "unknown-remote1 + fs128_fs16_dec4, 2^28 samples, amp 0.30, near-Gaussian sigma 0.10, thr 0.1",
           "ms_per_step": 1e3 * dt, "value": n / dt / 1e6, "unit": UNIT,
           "messages_transmitted": int(n // 210900), "messages_decoded": int(len(r["msgs_raw"])),
           "edges": r["n_edges"], "sm_rounds": r["sm_rounds"],
           "fir_mode": ["generic", "energy screen", "fma screen + exact refine of the rounding band", "exact"][r["fir_mode"]],
           "refined_fraction": r["refined_blocks"] / (n / fir.total_decimation / 8.0),
           "fir_kernel_ms": fir_ms / steps,
           "hbm_frac_job": 4.0 * n / dt / 1e9 / peak,
           "fp32_issue_frac_fir": (64.0 * n / (fir_ms / steps * 1e-3)) / FP32_ISSUE_PER_S if fir_ms > 0 else None,
           "note": "fp32_issue_frac counts the reference's own 64 fp32 mul/add per input sample (the FMA pass issues 32)"}
    g.close()
    del d
    torch.cuda.empty_cache()
    return out


def measure_c5(rank, world, local_rank, peak, n_caps_total=256, log2n=24, per=16):
    """BASELINE configs[4] (scaled to what one default run can synthesise): independent captures, devices alternating
    p3l-nexa2012 / unknown-remote1, authored fs64_fs8 filter, sigma in {0, 0.02, 0.05}, seeds = index; capture i is
    decoded by rank i mod world (no exchange at all)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from ookiedokie_b200 import binding as B
    from ookiedokie_b200 import host as H
    n = 1 << log2n
    fir = H.Fir("fs64_fs8")
    names = ["p3l-nexa2012", "unknown-remote1"]
    devs = [H.Device(nm, FS // fir.total_decimation) for nm in names]
    mine = [i for i in range(n_caps_total) if i % world == rank]
    bufs = []
    for i in mine:
        kind = i % 2
        msgs = [devs[kind].message({}) for _ in range(n // (180000 if kind else 400000) + 2)]
        tog, total = devs[kind].toggles(msgs, LEAD)
        sigma = [0.0, 0.02, 0.05][i % 3]
        d = torch.empty(n * 2, dtype=torch.int16, device="cuda")
        B.synth(n, np.ascontiguousarray(tog), 1488, 1253, noise_scale(sigma) if sigma else 0, 1000 + i, device_id=local_rank,
                device_ptr=d.data_ptr(), noise_terms=NOISE_TERMS)
        bufs.append(d)
    torch.cuda.synchronize()
    # `per` handles per device description = captures in flight per kind: a capture of 2^24 samples is 12 us of streaming
    # followed by ~0.3 ms of latency-bound stages (edges, state machine), so throughput comes from overlapping many
    kinds = sorted(set(i % 2 for i in mine))                 # (with an even number of ranks a rank holds one kind only)
    per_kind = 2 * per // max(1, len(kinds))
    gpus = [B.Gpu(filter_stages=fir.stages, sm=devs[kind].sm_spec(), threshold=THR, samples_per_buffer=SPB,
                  device_id=local_rank) for kind in kinds for _ in range(per_kind)]
    # capture -> handle: round robin over the handles of its kind
    seen = {k: 0 for k in kinds}
    caps = []
    for j, i in enumerate(mine):
        kind = i % 2
        caps.append(((bufs[j].data_ptr(), n), kinds.index(kind) * per_kind + seen[kind] % per_kind))
        seen[kind] += 1
    B.batch_decode(gpus, caps[:2 * per])                     # warm-up (workspace allocation)
    B.batch_decode(gpus, caps[:2 * per])                     # (and once more: the speculative message copies settle)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    msgs, stats = B.batch_decode(gpus, caps, msgs_cap=1 << 18)      # (room for every message: a list that overflows is decoded twice)
    dt = time.perf_counter() - t0
    t = torch.tensor([dt, float(sum(len(m) for m in msgs))], dtype=torch.float64, device="cuda")
    if world > 1:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        dt, n_msgs = float(tmax[0].item()), int(t[1].item())
    else:
        n_msgs = int(t[1].item())
    for g in gpus:
        g.close()
    del bufs
    torch.cuda.empty_cache()
    return {"workload": f"{n_caps_total} independent captures x 2^{log2n} samples, p3l-nexa2012 / unknown-remote1 alternating, "
                        f"fs64_fs8, sigma in {{0, 0.02, 0.05}}, capture i on rank i mod {world}",
            "captures": n_caps_total, "ms_total": 1e3 * dt, "captures_per_s": n_caps_total / dt,
            "value": n_caps_total * n / dt / 1e6, "unit": UNIT, "messages_decoded": n_msgs,
            "hbm_frac_job": 4.0 * n_caps_total * n / dt / 1e9 / (peak * world),
            "handles_per_gpu": 2 * per, "launches_per_capture": float(np.mean([s["gpu_launches"] for s in stats]))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--samples", type=int, default=1 << 30, help="samples per GPU (default 2^30 = 4 GiB)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-samples", type=int, default=1 << 27, help="prefix timed on the CPU baseline (N=1)")
    ap.add_argument("--ref-samples", type=int, default=1 << 25, help="prefix per step of --impl reference")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the extra configs block (C3 low SNR, C5 batch, C4 at N > 1)")
    ap.add_argument("--no-c4", action="store_true", help="skip the 2^33-samples-per-GPU continuous capture (N > 1)")
    ap.add_argument("--c4-samples", type=int, default=1 << 33, help="samples per GPU of that capture")
    ap.add_argument("--flags", type=int, default=0)
    ap.add_argument("--chunk-buffers", type=int, default=0)
    ap.add_argument("--sub-windows", type=int, default=3,
                    help="ookd_gpu_config.sub_windows of the handles: K > 1 cuts every decode into K time shards on the same GPU")
    ap.add_argument("--share", action="store_true", help="OOKD_FLAG_SHARE_SMS on the handles (three screening CTAs per SM)")
    ap.add_argument("--pipeline", type=int, default=1,
                    help="decodes in flight per GPU in the MAIN timed region (handles used round robin); the default 1 "
                         "= one step at a time, which is what the roofline / ncu launch list describe")
    ap.add_argument("--e2e-depth", type=int, default=1, help="decodes in flight in the end-to-end (host input) region")
    ap.add_argument("--pipelined-depth", type=int, default=2,
                    help="depth of the extra 'pipelined' measurement (consecutive windows overlapped); 0 = skip it")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (float64): messages "
                         "(rows of out_sample, buffer_idx, num_bits, message bytes); with one GPU also edges (threshold "
                         "transitions), first_bit, sizes (n_in, n_out, n_buffers) and exit_carry (state, k, num_bits, "
                         "prev_bit, 32 data bytes).  The inputs are seeded, so two builds can be compared file by file")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        impl_reference(args, rank, world)
        return

    import ctypes as C
    import numpy as np
    import torch
    import torch.distributed as dist
    from ookiedokie_b200 import binding as B
    from ookiedokie_b200 import host as H
    from ookiedokie_b200 import shard as S

    if not torch.cuda.is_available() or B.device_count() == 0:
        raise SystemExit("bench.py needs a B200: there is no CPU fallback for the receive path")
    torch.cuda.set_device(local_rank)
    numa = pin_to_gpu_numa(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    fir = H.Fir(FILTER_NAME)
    dev = H.Device(DEVICE_NAME, FS // fir.total_decimation)
    depth = max(1, args.pipeline)
    n_handles = max(depth, args.pipelined_depth, args.e2e_depth, 3 if world > 1 else 1)
    flags = args.flags | (B.FLAG_SHARE_SMS if args.share else 0)
    gpus = [B.Gpu(filter_stages=fir.stages, sm=dev.sm_spec(), threshold=THR, samples_per_buffer=SPB, device_id=local_rank,
                  flags=flags, sm_chunk_buffers=args.chunk_buffers, sm_warmup=1 if world > 1 else 0,
                  sub_windows=args.sub_windows)
            for _ in range(n_handles)]
    gpu = gpus[0]
    n = args.samples
    halo = gpu.halo
    first = rank * n
    halo_avail = min(halo, first)
    last = (rank == world - 1)
    tog, n_tx_msgs = build_toggles(dev, world * n)
    i_on, q_on = on_level()

    # ---- shard resident in HBM (synthesised on the device; identical bytes to the CPU recipe) ----
    d_iq = torch.empty(((halo_avail + n) * 2,), dtype=torch.int16, device="cuda")
    B.synth(halo_avail + n, tog, i_on, q_on, noise_scale(), SEED, first_sample=first - halo_avail, device_id=local_rank,
            device_ptr=d_iq.data_ptr(), noise_terms=NOISE_TERMS)
    torch.cuda.synchronize()

    for g in gpus:
        g.want_list = False         # keep messages as one structured array; no per-message Python work

    L = B.lib()
    stitch_resolves = [0]           # shards whose state-machine stage had to be re-run from a corrected entry (this rank)

    def run_steps_single(iq_ptr, is_dev, n_steps, depth=1):
        """world == 1: n_steps decodes through the C ABI, `depth` in flight (decode_begin on the next handle before
        decode_end of this one).  The messages are in host memory (result.msgs) when a call returns; only the LAST
        step's list is converted to numpy.  -> (last result dict, summed launches / fir / screen / kernel ms / syncs)."""
        acc = [0, 0.0, 0.0, 0.0, 0]
        res, ex = B.GpuResult(), B.SmCarry()
        p = C.c_void_p(iq_ptr)
        last_gpu = gpus[0]

        def account():
            acc[0] += res.gpu_launches
            acc[1] += res.fir_ms
            acc[2] += res.screen_ms
            acc[3] += res.kernel_ms
            acc[4] += res.host_syncs

        if depth <= 1:
            h = gpus[0].h
            for _ in range(n_steps):
                rc = L.ookd_gpu_decode_shard(h, p, is_dev, first, n, int(last), None, C.byref(ex), C.byref(res))
                if rc:
                    raise SystemExit(f"decode failed: {L.ookd_gpu_last_error(h).decode()}")
                account()
        else:
            pend = []
            for i in range(n_steps):
                g = gpus[i % depth]
                rc = L.ookd_gpu_decode_begin(g.h, p, is_dev, first, n, int(last), None)
                if rc:
                    raise SystemExit(f"decode_begin failed: {L.ookd_gpu_last_error(g.h).decode()}")
                pend.append(g)
                if len(pend) == depth:
                    g0 = pend.pop(0)
                    if L.ookd_gpu_decode_end(g0.h, C.byref(ex), C.byref(res)):
                        raise SystemExit(f"decode_end failed: {L.ookd_gpu_last_error(g0.h).decode()}")
                    account()
                    last_gpu = g0
            while pend:
                g0 = pend.pop(0)
                if L.ookd_gpu_decode_end(g0.h, C.byref(ex), C.byref(res)):
                    raise SystemExit(f"decode_end failed: {L.ookd_gpu_last_error(g0.h).decode()}")
                account()
                last_gpu = g0
        out = last_gpu._result(res)
        out["exit_carry"] = ex.astuple()
        return out, out["msgs_raw"], acc

    def run_steps_multi(iq_arg, n_steps, depth=1, first=first, n=n):
        """world > 1: every step is a complete decode incl. the cross-rank stitch (ookiedokie_b200/shard.py)."""
        st = S.PipelinedStitcher(rank, world)
        acc = [0, 0.0, 0.0, 0.0, 0]
        out = [None, None]

        def finish(runner, decoded, confirm_now=False):
            res, exit_c, rounds, msgs = st.finish(runner, decoded, confirm_now)
            acc[0] += runner.launches
            acc[1] += runner.fir_ms
            acc[2] += runner.screen_ms
            acc[3] += runner.kernel_ms
            acc[4] += runner.host_syncs
            out[0], out[1] = res, msgs

        if depth <= 1:
            # One decode at a time on the GPU.  Step i+1 is enqueued the moment step i has completed (three handles used in
            # turn: the tables of a step stay intact until its stitch is confirmed, one step later); everything else --
            # reading the message list, publishing this step's record into the shared-memory ring without waiting for
            # the other ranks, confirming the previous step, rank 0's concatenation -- happens while the GPU works.
            res, ex = B.GpuResult(), B.SmCarry()
            if isinstance(iq_arg, tuple):
                p, is_dev = C.c_void_p(iq_arg[0]), 1
            else:
                p, is_dev = C.c_void_p(iq_arg.ctypes.data), 0
            nh = min(3, len(gpus))
            if L.ookd_gpu_decode_begin(gpus[0].h, p, is_dev, first, n, int(last), None):
                raise SystemExit(f"decode_begin failed: {L.ookd_gpu_last_error(gpus[0].h).decode()}")
            prof = [0.0, 0.0, 0.0] if os.environ.get("OOKD_BENCH_PROFILE") else None
            for i in range(n_steps):
                g = gpus[i % nh]
                tp0 = time.perf_counter()
                if L.ookd_gpu_decode_end(g.h, C.byref(ex), C.byref(res)):                # waits for step i
                    raise SystemExit(f"decode_end failed: {L.ookd_gpu_last_error(g.h).decode()}")
                tp1 = time.perf_counter()
                if nh < 3:
                    st.confirm_pending()                      # (with two handles step i-1 must be settled before its handle is reused)
                if i + 1 < n_steps:
                    g2 = gpus[(i + 1) % nh]
                    if L.ookd_gpu_decode_begin(g2.h, p, is_dev, first, n, int(last), None):
                        raise SystemExit(f"decode_begin failed: {L.ookd_gpu_last_error(g2.h).decode()}")
                tp2 = time.perf_counter()
                runner = S.GpuShardRunner(g, iq_arg, first, n, last)
                decoded = (g._result(res), ex.astuple())
                runner._acc(decoded[0])
                st.confirm_pending()
                finish(runner, decoded)
                if prof is not None:
                    prof[0] += tp1 - tp0
                    prof[1] += tp2 - tp1
                    prof[2] += time.perf_counter() - tp2
            if prof is not None and n_steps >= 10:
                print(f"[bench] rank {rank}: per step: in decode_end {1e6 * prof[0] / n_steps:.0f} us, decode_begin {1e6 * prof[1] / n_steps:.0f} us, "
                      f"result + stitch {1e6 * prof[2] / n_steps:.0f} us; kernel span {acc[3] / n_steps:.3f} ms", file=sys.stderr)
        else:
            pending = []
            for i in range(n_steps):
                runner = S.GpuShardRunner(gpus[i % depth], iq_arg, first, n, last)
                runner.begin()
                pending.append(runner)
                if len(pending) == depth:
                    r0 = pending.pop(0)
                    finish(r0, r0.decode(None), True)         # (its handle takes the next step at once)
            while pending:
                r0 = pending.pop(0)
                finish(r0, r0.decode(None), True)
        st.drain()
        stitch_resolves[0] += st.resolves
        out[1] = st.last_messages if rank == 0 else None
        return out[0], out[1], acc

    def run_steps(iq_arg, n_steps, depth=1):
        if world == 1:
            if isinstance(iq_arg, tuple):
                return run_steps_single(iq_arg[0], 1, n_steps, depth)
            return run_steps_single(iq_arg.ctypes.data, 0, n_steps, depth)
        return run_steps_multi(iq_arg, n_steps, depth)

    dev_arg = (d_iq.data_ptr(), halo_avail + n)
    sampler = ClockSampler(local_rank)
    sampler.start()                 # started before the warm-up so that it is sampling when the timed region begins
    run_steps(dev_arg, max(args.warmup, depth, 3 if world > 1 else 1), depth)
    barrier()
    t0 = time.perf_counter()
    res, msgs, (launches, fir_ms, screen_ms, kernel_ms, host_syncs) = run_steps(dev_arg, args.steps, depth)
    barrier()
    t1 = time.perf_counter()
    dt = t1 - t0
    clocks = sampler.stop(t0, t1)

    if args.dump_outputs and rank == 0:
        outputs = {"messages": message_table(msgs, dev.nbytes)}
        if world == 1:
            # (the handle of the last step still holds its transitions until the next region reuses it)
            fb, edges = gpus[(args.steps - 1) % depth].edges()
            state, k, nbits, prev, data = res["exit_carry"]
            outputs.update(edges=edges, first_bit=[fb], sizes=[res["n_in"], res["n_out"], res["n_buffers"]],
                           exit_carry=[state, k, nbits, prev] + list(data))
        write_outputs(args.dump_outputs, outputs)

    # ---- extra: the same steps with consecutive decodes overlapped (two handles), as the windows of a long capture
    #      are processed; every step is still a complete decode + stitch inside the timed region ----
    pipelined = None
    if args.pipelined_depth > 1:
        pd = args.pipelined_depth
        run_steps(dev_arg, max(args.warmup, pd), depth=pd)
        barrier()
        tp0 = time.perf_counter()
        res_p, msgs_p, _ = run_steps(dev_arg, args.steps, depth=pd)
        barrier()
        dtp = time.perf_counter() - tp0
        tpt = torch.tensor([dtp], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tpt, op=dist.ReduceOp.MAX)
        dtp = float(tpt.item())
        if rank == 0 and msgs is not None and msgs_p is not None:
            assert np.array_equal(msgs_p, msgs), "pipelined decode differs from the one-at-a-time decode"
        pipelined = {"depth": pd, "value": world * n / (dtp / args.steps) / 1e6, "unit": UNIT,
                     "ms_per_step": 1e3 * dtp / args.steps, "steps": args.steps}
    t = torch.tensor([dt, fir_ms, kernel_ms, screen_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dt, fir_ms_max, kernel_ms_max, screen_ms_max = [float(x) for x in t.cpu()]
    rs = torch.tensor([float(stitch_resolves[0])], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(rs, op=dist.ReduceOp.SUM)
    n_resolves = int(rs.item())
    ms_per_step = 1e3 * dt / args.steps
    value = world * n / (dt / args.steps) / 1e6
    n_msgs = len(msgs) if msgs is not None else 0
    n_edges = res["n_edges"]
    sm_rounds = res["sm_rounds"]
    refined_groups = res["refined_blocks"]

    # ---- end to end: shard in pinned host memory, H2D inside the timed region ----
    e2e = None
    if not args.no_e2e:
        nbytes = (halo_avail + n) * 4
        hptr = L.ookd_gpu_host_alloc(nbytes)
        if not hptr:
            raise SystemExit("pinned host allocation failed")
        rc = L.ookd_gpu_memcpy_d2h(local_rank, hptr, d_iq.data_ptr(), nbytes)
        assert rc == 0
        h_iq = np.ctypeslib.as_array(C.cast(hptr, C.POINTER(C.c_int16)), shape=((halo_avail + n) * 2,))
        # ceiling: the plain pinned-host -> device copy of the same bytes, all ranks at once, same run
        barrier()
        tc0 = time.perf_counter()
        for _ in range(2):
            assert L.ookd_gpu_memcpy_h2d(local_rank, d_iq.data_ptr(), hptr, nbytes) == 0
        torch.cuda.synchronize()
        tcopy = (time.perf_counter() - tc0) / 2
        tct = torch.tensor([tcopy], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tct, op=dist.ReduceOp.MAX)
        tcopy = float(tct.item())
        ed = max(1, args.e2e_depth)
        run_steps(h_iq, ed, depth=ed)
        barrier()
        t0 = time.perf_counter()
        res_e, msgs_e, _ = run_steps(h_iq, args.e2e_steps, depth=ed)
        barrier()
        dte = time.perf_counter() - t0
        te = torch.tensor([dte], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        dte = float(te.item())
        d2h = len(res_e["msgs_raw"]) * 56 + 3 * 256 + 48
        e2e_value = world * n / (dte / args.e2e_steps) / 1e6
        e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": nbytes,
               "d2h_bytes_per_step": d2h, "steps": args.e2e_steps, "pipeline_depth": ed,
               "h2d_gbs": world * nbytes / (dte / args.e2e_steps) / 1e9,
               "h2d_ceiling_gbs": world * nbytes / tcopy / 1e9,
               "frac_of_h2d_ceiling": (dte / args.e2e_steps) and tcopy / (dte / args.e2e_steps),
               "pinned_memory": numa}
        if rank == 0 and msgs is not None and msgs_e is not None:
            assert np.array_equal(msgs_e, msgs), "host-input decode differs from device-input decode"
        cpu_prefix = h_iq[halo_avail * 2: (halo_avail + min(n, args.cpu_samples)) * 2].copy() if rank == 0 else None
        L.ookd_gpu_host_free(hptr)
    else:
        cpu_prefix = d_iq[halo_avail * 2: (halo_avail + min(n, args.cpu_samples)) * 2].cpu().numpy() if rank == 0 else None

    # ---- CPU baseline + parity AT BENCHMARK SCALE (rank 0, N = 1 only): the unmodified reference binary on a bounded
    #      prefix; its csv rows and --rx-rec-dig transitions are compared with a GPU decode of exactly that prefix ----
    cpu = None
    parity = None
    if rank == 0 and world == 1 and not args.no_cpu:
        nc = cpu_prefix.size // 2
        if reference_binary() is not None:
            v, rows, ref_rows, ref_fb, ref_edges = run_reference_cpu(cpu_prefix, want_parity=True)
            pg = B.Gpu(filter_stages=fir.stages, sm=dev.sm_spec(), threshold=THR, samples_per_buffer=SPB, device_id=local_rank,
                       flags=flags, sub_windows=args.sub_windows)         # (the configuration that was timed)
            got = pg.decode((d_iq.data_ptr(), nc))
            fb, edges = pg.edges()
            gpu_rows, cur_buf = [], None
            for out_sample, buf, nbits, data in got["msgs"]:
                vals = [val for key, val in dev.format(data) if key != "Decode Timestamp"]
                if buf != cur_buf:
                    gpu_rows.append([])
                    cur_buf = buf
                gpu_rows[-1].extend(vals)
            assert fb == ref_fb, "first threshold decision differs from the reference binary's"
            assert len(edges) == len(ref_edges) and np.array_equal(edges, np.array(ref_edges, dtype=np.uint64)), \
                "threshold transitions differ from the reference binary's --rx-rec-dig output"
            assert gpu_rows == ref_rows, "decoded messages differ from the reference binary's csv output"
            parity = {"against": "unmodified reference binary (csv rows + --rx-rec-dig transitions)", "n": nc,
                      "msgs": len(ref_rows), "edges": len(ref_edges), "equal": True}
            pg.close()
            cpu = {"value": v, "unit": UNIT, "cores": 1, "kind": "reference", "host_cores_available": os.cpu_count(),
                   "sample": f"first {nc} samples ({nc * 4 / 2**20:.0f} MiB) of the same capture; {rows} messages"}
        else:
            from oracle import oracle as O
            odev = O.load_device(DEVICE_NAME)
            t0 = time.perf_counter()
            r = O.rx(cpu_prefix, O.load_filter(FILTER_NAME), odev, threshold_=THR, samples_per_buffer=SPB, samplerate=FS)
            v = nc / (time.perf_counter() - t0) / 1e6
            pg = B.Gpu(filter_stages=fir.stages, sm=dev.sm_spec(), threshold=THR, samples_per_buffer=SPB, device_id=local_rank,
                       flags=flags, sub_windows=args.sub_windows)
            got = pg.decode((d_iq.data_ptr(), nc))
            fb, edges = pg.edges()
            assert fb == r["first_bit"] and np.array_equal(edges, r["edges"]), "edges differ from the oracle's"
            assert got["msgs"] == r["msgs"], "decoded messages differ from the oracle's"
            parity = {"against": "oracle port", "n": nc, "msgs": len(r["msgs"]), "edges": len(r["edges"]), "equal": True}
            pg.close()
            cpu = {"value": v, "unit": UNIT, "cores": 1, "kind": "port", "host_cores_available": os.cpu_count(),
                   "sample": f"first {nc} samples of the same capture; {len(r['msgs'])} messages"}

    # ---- the other BASELINE configs, outside the headline timed region ----
    peak, peak_src = measured_peak()
    configs = None
    if not args.no_configs:
        del d_iq
        torch.cuda.empty_cache()
        configs = {}
        try:
            if world == 1:
                configs["c3_lowsnr_remote1_dec4"] = measure_c3(local_rank, peak)
            configs["c5_batch_mixed_fs64_fs8"] = measure_c5(rank, world, local_rank, peak)
            if world > 1 and not args.no_c4:
                # BASELINE configs[3]: one continuous capture of world x 2^33 samples (256 GiB at 8 GPUs), 32 GiB time shard
                # per GPU with FIR halo and cross-shard state-machine carry; same recipe and stitch as the headline
                n4 = args.c4_samples
                first4 = rank * n4
                ha4 = min(halo, first4)
                tog4, n_tx4 = build_toggles(dev, world * n4)
                d4 = torch.empty(((ha4 + n4) * 2,), dtype=torch.int16, device="cuda")
                B.synth(ha4 + n4, tog4, i_on, q_on, noise_scale(), SEED, first_sample=first4 - ha4, device_id=local_rank,
                        device_ptr=d4.data_ptr(), noise_terms=NOISE_TERMS)
                torch.cuda.synchronize()
                arg4 = (d4.data_ptr(), ha4 + n4)
                run_steps_multi(arg4, 6, 1, first4, n4)          # (every handle of the rotation sizes its workspaces and
                                                                 #  settles its speculative message copy: two decodes each)
                C4_STEPS = 10                                    # (10 ms each: enough steps that the un-overlapped host work of
                                                                 #  the LAST one -- every rank copies its 1.2 MB of messages -- is amortised)
                barrier()
                t40 = time.perf_counter()
                res4, msgs4, acc4 = run_steps_multi(arg4, C4_STEPS, 1, first4, n4)
                barrier()
                dt4 = (time.perf_counter() - t40) / C4_STEPS
                print(f"[bench] c4 rank {rank}: wall {1e3 * dt4:.3f} ms/step, decode span {acc4[3] / C4_STEPS:.3f} ms, fir stage {acc4[1] / C4_STEPS:.3f} ms, "
                      f"screen {acc4[2] / C4_STEPS:.3f} ms", file=sys.stderr)
                t4 = torch.tensor([dt4, acc4[3] / C4_STEPS, acc4[2] / C4_STEPS], dtype=torch.float64, device="cuda")
                dist.all_reduce(t4, op=dist.ReduceOp.MAX)
                dt4, lat4, scr4 = [float(x) for x in t4.cpu()]
                configs["c4_continuous_time_sharded"] = {
                    "workload": f"one continuous capture of {world} x 2^{n4.bit_length() - 1} samples ({world * n4 * 4 / 2**30:.0f} GiB), "
                                f"{DEVICE_NAME} + {FILTER_NAME}, one {n4 * 4 / 2**30:.0f} GiB time shard per GPU (FIR halo, carry stitch)",
                    "ms_per_step": 1e3 * dt4, "value": world * n4 / dt4 / 1e6, "unit": UNIT,
                    "step_latency_ms": lat4, "screen_kernel_ms": scr4, "host_syncs_per_step": acc4[4] / C4_STEPS,
                    "launches_per_step": acc4[0] / C4_STEPS, "sm_rounds": res4["sm_rounds"],
                    "hbm_frac_job": 4.0 * n4 / dt4 / 1e9 / peak,
                    "messages_decoded": int(len(msgs4)) if msgs4 is not None else None,
                    "messages_transmitted_upper_bound": n_tx4}
                del d4
                torch.cuda.empty_cache()
        except Exception as e:                               # the headline line must survive a failure here
            configs["error"] = f"{type(e).__name__}: {str(e)[:200]}"

    if rank == 0:
        fir_ms_per_launch = fir_ms_max / args.steps
        screen_ms_per_launch = screen_ms_max / args.steps
        achieved = 4.0 * n / (screen_ms_per_launch * 1e-3) / 1e9 if screen_ms_per_launch > 0 else None
        job_gbs = 4.0 * n / (ms_per_step * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(n), "samples_per_gpu": n, "device": DEVICE_NAME, "filter": FILTER_NAME,
                       "parallelism": f"time-shards x{world}" if world > 1 else "single shard",
                       "pipeline_depth": depth,
                       "sub_windows": args.sub_windows,      # > 1: each decode is cut into that many time shards on its own GPU (see DESIGN 3.8)
                       "stitch": (S.stitch_description() if world > 1 else "n/a"),
                       "stitch_resolves": n_resolves,        # shard decodes whose state machine had to be re-run (warm-up + main + pipelined regions, all ranks)
                       "l2": "input shard (4 B/sample) larger than L2; no flush needed",
                       "messages_decoded": n_msgs, "messages_transmitted_upper_bound": n_tx_msgs,
                       "edges_last_rank": n_edges, "sm_rounds": sm_rounds,
                       "refined_fraction": refined_groups / (n / fir.total_decimation / 8.0)},
            "step_latency_ms": kernel_ms_max / args.steps,      # CUDA-event span of one decode (overlaps its neighbours when pipelined)
            "fir_stage_ms_per_step": fir_ms_per_launch,
            "host_syncs_per_step": host_syncs / args.steps,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": (achieved / peak) if achieved else None, "traffic": ncu_traffic(),
                         "peak_source": peak_src,
                         "kernel": "fir_screen_tma_kernel<1> (SC16Q11 -> window energies -> threshold decisions), "
                                   "4 B/sample algorithmic, " +
                                   (f"{args.sub_windows} launches per step (one per sub-window, samples/{args.sub_windows} each), timed as one "
                                    "CUDA-event span from the first one's start to the last one's end: the tails of the earlier "
                                    "sub-windows run inside that span" if args.sub_windows > 1 else "one launch per step"),
                         "launches_per_step": max(1, args.sub_windows),
                         "kernel_ms_per_launch": screen_ms_per_launch / max(1, args.sub_windows),
                         "kernel_ms_per_step": screen_ms_per_launch,
                         "job_gbs": job_gbs, "job_frac": job_gbs / peak},          # per GPU (n = samples per GPU)
            "clocks": clocks, "gpu_launches": launches,
        }
        if pipelined:
            line["pipelined"] = pipelined
        if e2e:
            line["e2e"] = e2e
        if cpu:
            line["cpu_baseline"] = cpu
        if parity:
            line["parity_checked"] = parity
        if configs:
            line["configs"] = configs
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
