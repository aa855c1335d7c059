"""8-bit captures (CU8: uint8 I,Q; CS8: int8 I,Q) decoded natively: every result equals the decode of the widened
SC16Q11 capture (CS8 k -> 16 k, CU8 v -> 16 v - 2040), by the SC16Q11 path and by the oracle."""
import os

import numpy as np
import pytest

from oracle import oracle as O
from ookiedokie_b200 import binding as B
from ookiedokie_b200 import host as H
import ookd_testutil as util

pytestmark = pytest.mark.gpu

FMTS = ["cu8", "cs8"]


def quantise(iq, fmt):
    """SC16Q11 capture (numpy int16 (n, 2) or a torch int16 tensor on the GPU) -> (8-bit capture, widened SC16Q11
    capture), quantised on the device: CS8 k = clip(round(x / 16), -128, 127), CU8 v = clip(round((x + 2040) / 16), 0, 255)."""
    import torch
    on_host = isinstance(iq, np.ndarray)
    t = torch.from_numpy(np.ascontiguousarray(iq)).cuda() if on_host else iq
    x = t.to(torch.float32)
    if fmt == "cs8":
        k = torch.clamp(torch.round(x / 16), -128, 127)
        b, w = k.to(torch.int8), (16 * k).to(torch.int16)
    else:
        v = torch.clamp(torch.round((x + 2040) / 16), 0, 255)
        b, w = v.to(torch.uint8), (16 * v - 2040).to(torch.int16)
    if on_host:
        return b.cpu().numpy(), w.cpu().numpy()
    return b, w


def widen_host(b, fmt):
    return (16 * b.astype(np.int32) - (0 if fmt == "cs8" else 2040)).astype(np.int16)


def _gpu(filt, dev=None, fmt="sc16q11", **kw):
    stages = O.load_filter(filt) if filt else None
    sm = util.sm_spec(dev, stages) if dev is not None else None
    return B.Gpu(filter_stages=stages, sm=sm, input_format=fmt, **kw), stages


def _same_decode(g8, g16, cap8, cap16, ref=None):
    """decode cap8 on g8 and cap16 on g16; every result equal (and equal to the oracle's when ref is given)."""
    a = g8.decode(cap8)
    b = g16.decode(cap16)
    for k in ("n_in", "n_out", "n_buffers", "n_edges", "first_bit", "msgs"):
        assert a[k] == b[k], k
    fa, ea = g8.edges()
    fb, eb = g16.edges()
    assert fa == fb and np.array_equal(ea, eb)
    if ref is not None:
        assert a["n_out"] == ref["n_out"] and a["n_buffers"] == ref["n_buffers"]
        assert fa == ref["first_bit"] and np.array_equal(ea, ref["edges"])
        assert a["msgs"] == ref["msgs"]
    return a


@pytest.mark.parametrize("fmt", FMTS)
def test_every_byte_pair_widens_exactly(fmt):
    """All 65 536 (I, Q) byte pairs through the unity filter: the value of the table in include/ookd_gpu.h, bit for bit."""
    pairs = np.stack(np.meshgrid(np.arange(256), np.arange(256), indexing="ij"), -1).reshape(-1, 2)
    b = pairs.astype(np.uint8) if fmt == "cu8" else pairs.astype(np.uint8).view(np.int8)
    w = widen_host(b, fmt)
    # the table's float value, straight from the bytes: k / 128 (CS8), (v - 127.5) / 128 (CU8)
    want = (b.astype(np.float32) / np.float32(128.0)) if fmt == "cs8" else \
        ((b.astype(np.float32) - np.float32(127.5)) / np.float32(128.0))
    assert np.array_equal(want, w.astype(np.float32) / np.float32(2048.0))       # ... is that of the SC16Q11 word
    stages = O.load_filter("unity1")
    g = B.Gpu(filter_stages=stages, samples_per_buffer=1024, input_format=fmt)
    got = g.filtered(b)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    ref = O.rx(w, stages, None, samples_per_buffer=1024, want_filtered=True)["filtered"]
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))


@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("filt", ["fs32_fs4", "fs128_fs16_dec4", "unity16"])
def test_filtered_matches_widened(fmt, filt):
    rng = np.random.default_rng(3)
    b = rng.integers(0, 256, size=(50001, 2)).astype(np.uint8)
    if fmt == "cs8":
        b = b.view(np.int8)
    w = widen_host(b, fmt)
    g8, stages = _gpu(filt, fmt=fmt, samples_per_buffer=1024)
    g16, _ = _gpu(filt, samples_per_buffer=1024)
    got = g8.filtered(b)
    assert np.array_equal(got.view(np.uint32), g16.filtered(w).view(np.uint32))
    ref = O.rx(w, stages, None, samples_per_buffer=1024, want_filtered=True)["filtered"]
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))


CASES = [
    # device, filter, n_msgs, sigma, amp, spb
    ("p3l-nexa2012", "fs32_fs4", 3, 0.0, 0.95, 8192),
    ("p3l-nexa2012", "fs32_fs4", 3, 0.02, 0.95, 8192),
    ("p3l-nexa2012", "fs32_fs4", 3, 0.05, 0.95, 1024),
    ("p3l-nexa2012", "fs128_fs16_dec4", 3, 0.02, 0.95, 8192),
    ("p3l-nexa2012", "fs64_fs8", 3, 0.05, 0.95, 8192),
    ("p3l-nexa2012", "unity16", 2, 0.02, 0.95, 1024),
    ("p3l-nexa2012", None, 2, 0.0, 0.95, 8192),
    ("unknown-remote1", "fs128_fs16_dec4", 6, 0.05, 0.30, 8192),
    ("unknown-remote1", "fs32_fs4", 4, 0.02, 0.5, 1024),
    ("unknown-remote1", "fs64_fs8", 4, 0.0, 0.5, 8192),
]


@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("devname,filt,n_msgs,sigma,amp,spb", CASES)
def test_decode_matches_widened(fmt, devname, filt, n_msgs, sigma, amp, spb):
    dev = O.load_device(devname)
    fields = util.nexa_fields if "nexa" in devname else util.remote_fields
    iq, _, _ = util.capture(dev, n_msgs, sigma=sigma, amplitude=amp, phase=0.7, seed=n_msgs * 17 + spb, fields=fields,
                               tail=20000 + 777)                   # not a multiple of spb: EOF padding
    b, w = quantise(iq, fmt)
    g8, stages = _gpu(filt, dev, fmt, samples_per_buffer=spb, sm_chunk_buffers=7)
    g16, _ = _gpu(filt, dev, samples_per_buffer=spb, sm_chunk_buffers=7)
    ref = O.rx(w, stages, dev, samples_per_buffer=spb, want_bits=True)
    _same_decode(g8, g16, b, w, ref)
    assert np.array_equal(g8.bits(), ref["bits"])


@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("flags", [B.FLAG_FMA_SCREEN, B.FLAG_NO_SCREEN, B.FLAG_NO_TMA, B.FLAG_FORCE_GENERIC,
                                   B.FLAG_NO_ADAPTIVE])
@pytest.mark.parametrize("filt", ["fs32_fs4", "fs128_fs16_dec4"])
def test_decode_paths(fmt, flags, filt):
    dev = O.load_device("p3l-nexa2012")
    iq, _, _ = util.capture(dev, 3, sigma=0.03, amplitude=0.9, phase=1.1, seed=5, fields=util.nexa_fields)
    b, w = quantise(iq, fmt)
    g8, stages = _gpu(filt, dev, fmt, samples_per_buffer=8192, flags=flags)
    g16, _ = _gpu(filt, dev, samples_per_buffer=8192, flags=flags)
    ref = O.rx(w, stages, dev, samples_per_buffer=8192)
    _same_decode(g8, g16, b, w, ref)


@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("flags", [0, B.FLAG_NO_ADAPTIVE])
def test_low_snr_switches_to_fma_screening(fmt, flags):
    """A noise floor above K0: the adaptive probe (short capture) or the work-list overflow (NO_ADAPTIVE) moves the
    handle to FMA screening; a second decode on the same handle stays there."""
    dev = O.load_device("unknown-remote1")
    iq, _, _ = util.capture(dev, 10, sigma=0.10, amplitude=0.30, phase=0.3, seed=77, fields=util.remote_fields)
    b, w = quantise(iq, fmt)
    g8, stages = _gpu("fs128_fs16_dec4", dev, fmt, samples_per_buffer=8192, flags=flags)
    g16, _ = _gpu("fs128_fs16_dec4", dev, samples_per_buffer=8192, flags=flags)
    ref = O.rx(w, stages, dev, samples_per_buffer=8192)
    _same_decode(g8, g16, b, w, ref)
    _same_decode(g8, g16, b, w, ref)


@pytest.mark.parametrize("fmt", FMTS)
def test_device_input_and_unaligned_pointers(fmt):
    """Device input at byte offsets 0, 1 (odd: the samples straddle 2-byte words), 2 and 16: the tensor-copy and
    vector paths where the alignment allows, guarded loads elsewhere."""
    import torch
    dev = O.load_device("p3l-nexa2012")
    iq, _, _ = util.capture(dev, 3, sigma=0.02, amplitude=0.95, phase=0.2, seed=9, fields=util.nexa_fields)
    b, w = quantise(iq, fmt)
    ref = O.rx(w, O.load_filter("fs32_fs4"), dev, samples_per_buffer=8192)
    g16, _ = _gpu("fs32_fs4", dev, samples_per_buffer=8192)
    raw = b.view(np.uint8).reshape(-1)
    for off in (0, 1, 2, 16):
        buf = torch.zeros(raw.size + 64, dtype=torch.uint8, device="cuda")
        buf[off:off + raw.size] = torch.from_numpy(raw).cuda()
        torch.cuda.synchronize()
        for flags in (0, B.FLAG_NO_TMA):
            g8, _ = _gpu("fs32_fs4", dev, fmt, samples_per_buffer=8192, flags=flags)
            _same_decode(g8, g16, (buf.data_ptr() + off, len(b)), w, ref)


@pytest.mark.parametrize("fmt", FMTS)
def test_host_input_in_several_pieces(fmt):
    """2^25 + 12345 samples of host input: three H2D pieces of 16 Mi samples, screening of each piece as it arrives."""
    import torch
    dev = O.load_device("p3l-nexa2012")
    n = (1 << 25) + 12345
    msgs = [O.message_bytes(dev, util.nexa_fields(i)) for i in range(40)]
    tog, total = O.toggles_from_messages(dev, msgs, util.FS, 12000)
    tog = np.array(tog, np.uint64)
    reps = int(np.ceil(n / total))
    tog_all = np.concatenate([tog + np.uint64(r * total) for r in range(reps)])
    d16 = torch.empty((n, 2), dtype=torch.int16, device="cuda")
    B.synth(n, tog_all, 1488, 1253, O.noise_scale_for_sigma(0.02), 1234, device_ptr=d16.data_ptr(), device_id=0)
    d8, dw = quantise(d16, fmt)
    torch.cuda.synchronize()
    h8 = d8.cpu().numpy()
    g8, _ = _gpu("fs32_fs4", dev, fmt, samples_per_buffer=8192)
    g16, _ = _gpu("fs32_fs4", dev, samples_per_buffer=8192)
    a = _same_decode(g8, g16, h8, (dw.data_ptr(), n))
    assert len(a["msgs"]) >= 40 * (reps - 1)
    _same_decode(g8, g16, (d8.data_ptr(), n), (dw.data_ptr(), n))


@pytest.mark.parametrize("fmt", FMTS)
def test_sub_windows_shards_and_resolve(fmt):
    dev = O.load_device("p3l-nexa2012")
    iq, _, _ = util.capture(dev, 12, sigma=0.02, amplitude=0.95, phase=0.4, seed=21, fields=util.nexa_fields)
    b, w = quantise(iq, fmt)
    stages = O.load_filter("fs32_fs4")
    sm = util.sm_spec(dev, stages)
    ref = O.rx(w, stages, dev, samples_per_buffer=4096)
    # sub_windows 3 on one device
    s8 = B.Gpu(filter_stages=stages, sm=sm, samples_per_buffer=4096, sm_chunk_buffers=5, sub_windows=3, input_format=fmt)
    s16 = B.Gpu(filter_stages=stages, sm=sm, samples_per_buffer=4096, sm_chunk_buffers=5, sub_windows=3)
    _same_decode(s8, s16, b, w, ref)
    # a chain of decode_shard calls, each entered from a wrong state and resolved with its predecessor's exit
    g8 = B.Gpu(filter_stages=stages, sm=sm, samples_per_buffer=4096, sm_chunk_buffers=5, input_format=fmt)
    halo, n = g8.halo, len(b)
    assert halo % 8 == 0
    bounds = [0, 4096 * 40, 4096 * 97, n]
    exits, msgs = [None], []
    wrong = (1, 5, 3, 1, bytes([0x5A] * 32))
    for i in range(len(bounds) - 1):
        first, cnt = bounds[i], bounds[i + 1] - bounds[i]
        h = min(halo, first)
        last = i == len(bounds) - 2
        res, ex = g8.decode_shard(b[first - h: first + cnt], first, cnt, last, wrong if i else None)
        if i:
            res, ex = g8.resolve(exits[-1])
        exits.append(ex)
        msgs += res["msgs"]
    assert msgs == ref["msgs"]
    # the same window over handles that share one device (repeated id)
    m = B.MultiGpu([0, 0, 0], filter_stages=stages, sm=sm, samples_per_buffer=4096, sm_chunk_buffers=5, input_format=fmt)
    r, _ = m.decode(b)
    assert r["msgs"] == ref["msgs"]
    fb, e = m.edges()
    assert fb == ref["first_bit"] and np.array_equal(e, ref["edges"])


def test_batch_decode_mixed_formats():
    dev = O.load_device("p3l-nexa2012")
    stages = O.load_filter("fs32_fs4")
    sm = util.sm_spec(dev, stages)
    gs = [B.Gpu(filter_stages=stages, sm=sm, samples_per_buffer=8192, input_format=f) for f in ("sc16q11", "cu8", "cs8")]
    caps, refs = [], []
    for i in range(9):
        iq, _, _ = util.capture(dev, 2 + i % 3, sigma=0.02 * (i % 3), amplitude=0.95, phase=0.1 * i, seed=100 + i,
                                fields=util.nexa_fields)
        hi = i % 3
        if hi == 0:
            cap, w = iq, iq
        else:
            cap, w = quantise(iq, gs[hi].input_format)
        caps.append((cap, hi))
        refs.append(O.rx(w, stages, dev, samples_per_buffer=8192)["msgs"])
    with pytest.raises(ValueError):
        B.batch_decode(gs, [(caps[1][0], 0)])                  # a CU8 array on the SC16Q11 handle
    msgs, _ = B.batch_decode(gs, caps)
    for got, ref in zip(msgs, refs):
        assert B.msgs_to_tuples(got, gs[0].msg_bytes) == ref


@pytest.mark.parametrize("fmt", FMTS)
def test_screening_fuzz(fmt):
    """Seeded fuzz of the energy / on proofs on 8-bit captures: the full byte range (clipping), levels hovering at the
    threshold, quiet and loud stretches; decisions equal the oracle's on the widened capture."""
    rng = np.random.default_rng(0xB8 + len(fmt))
    for filt, thr in [("fs32_fs4", 0.1), ("fs128_fs16_dec4", 0.1), ("fs32_fs4", 0.35)]:
        n = 300000
        levels = [0.0, 0.02, thr * 0.97, thr, thr * 1.03, 0.5, 1.2]
        amp = np.empty(n)
        pos = 0
        while pos < n:
            ln = int(rng.integers(100, 4000))
            amp[pos:pos + ln] = rng.choice(levels)
            pos += ln
        ph = rng.uniform(0, 2 * np.pi, n) if rng.random() < 0.5 else rng.uniform(0, 2 * np.pi)
        sig = rng.choice([0.0, 8.0, 40.0])
        x = np.stack([amp * np.cos(ph) * 2048 + rng.normal(0, sig, n), amp * np.sin(ph) * 2048 + rng.normal(0, sig, n)], 1)
        iq = np.clip(np.rint(x), -32768, 32767).astype(np.int16)
        b, w = quantise(iq, fmt)
        g8, stages = _gpu(filt, fmt=fmt, samples_per_buffer=4096, threshold=thr)
        ref = O.rx(w, stages, None, threshold_=thr, samples_per_buffer=4096, want_bits=True)
        g8.decode(b)
        assert np.array_equal(g8.bits(), ref["bits"]), (filt, thr)


def bench_capture(n, device_id=0):
    """The benchmark's capture recipe (bench.py: p3l-nexa2012 + fs32_fs4, seeded), n samples synthesised on the device.
    -> (torch int16 (n, 2) tensor, H.Fir, H.Device)."""
    import torch
    import bench
    fir = H.Fir(bench.FILTER_NAME)
    dev = H.Device(bench.DEVICE_NAME, bench.FS // fir.total_decimation)
    tog, _ = bench.build_toggles(dev, n)
    i_on, q_on = bench.on_level()
    d = torch.empty((n, 2), dtype=torch.int16, device=f"cuda:{device_id}")
    B.synth(n, tog, i_on, q_on, bench.noise_scale(), bench.SEED, device_id=device_id, device_ptr=d.data_ptr(),
            noise_terms=bench.NOISE_TERMS)
    return d, fir, dev


def test_benchmark_recipe_2pow27_cu8():
    """2^27 samples of the benchmark's capture recipe in CU8, on the device: same messages and edges as the widened
    capture through the SC16Q11 path."""
    import torch
    n = 1 << 27
    d16, fir, dev = bench_capture(n)
    d8, dw = quantise(d16, "cu8")
    del d16
    torch.cuda.synchronize()
    kw = dict(filter_stages=fir.stages, sm=dev.sm_spec(), threshold=0.1, samples_per_buffer=8192, device_id=0)
    g8 = B.Gpu(input_format="cu8", **kw)
    g16 = B.Gpu(**kw)
    a = _same_decode(g8, g16, (d8.data_ptr(), n), (dw.data_ptr(), n))
    assert len(a["msgs"]) > 100
    s8 = B.Gpu(input_format="cu8", sub_windows=3, **kw)
    b = s8.decode((d8.data_ptr(), n))
    assert b["msgs"] == a["msgs"]


# ---- the CLI ----

def _cli_rows(out, has_ts):
    return [l.split(",")[1:] if has_ts else l.split(",") for l in out.strip().splitlines()] if out.strip() else []


def _reference_cli(cap, filt, spb, dig):
    """The unmodified reference binary on an SC16Q11 capture (None when it is not built): csv rows without the wall-clock
    column, and its --rx-rec-dig file."""
    import subprocess
    import bench
    ref = bench.reference_binary()
    if ref is None:
        return None
    data = os.path.join(bench.ROOT, "ookiedokie_b200", "data")
    cmd = [ref, "--rx", "bladerf_file", "-A", str(cap), "-d", os.path.join(data, "devices", "p3l-nexa2012.json"),
           "-F", "none" if filt == "none" else os.path.join(data, "filters", filt + ".json"), "--rx-fmt", "csv",
           "--samples-per-buffer", str(spb), "-s", str(bench.FS), "-B", str(dig)]
    out = subprocess.run(cmd, capture_output=True, text=True, check=True,
                         env=dict(os.environ, OOKD_DATA_DIR=data + "/")).stdout
    return _cli_rows(out, True), open(dig).read()


@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("filt,spb,window,rec_input", [("fs32_fs4", 8192, 0, True), ("fs128_fs16_dec4", 4096, 24576 * 5, True),
                                                       ("none", 8192, 0, True), ("fs32_fs4", 8192, 0, False),
                                                       ("fs128_fs16_dec4", 4096, 24576 * 5, False)])
def test_cli_rx_8bit_file(fmt, filt, spb, window, rec_input, tmp_path):
    """--rx cu8_file / cs8_file against --rx bladerf_file on the widened file (and the reference binary on it, when
    built): stdout csv and pretty, -B, and -R (--rx-rec-input: the widened capture; without it: the filtered samples)."""
    dev = O.load_device("p3l-nexa2012")
    iq, msgs, _ = util.capture(dev, 6, sigma=0.02, amplitude=0.95, phase=0.9, seed=4, fields=util.nexa_fields,
                               tail=20000 + 333)
    b, w = quantise(iq, fmt)
    c8, c16 = tmp_path / "c.8", tmp_path / "c.sc16q11"
    b.tofile(c8)
    w.tofile(c16)
    with open(c8, "ab") as f:
        f.write(b"\x7f")                                        # a trailing odd byte is ignored
    outs = {}
    for name, sdr, cap in (("8", f"{fmt}_file", c8), ("16", "bladerf_file", c16)):
        dig, rec = tmp_path / f"dig{name}.csv", tmp_path / f"rec{name}.sc16q11"
        args = ["--rx", sdr, "-A", str(cap), "-d", "p3l-nexa2012", "--rx-fmt", "csv", "-B", str(dig), "-F", filt,
                "--samples-per-buffer", str(spb), "-R", f"bladerf_file,{rec}"] + (["--rx-rec-input"] if rec_input else [])
        if window:
            args += ["--window", str(window)]
        r = H.run_cli(args)
        assert r.returncode == 0, r.stderr
        r2 = H.run_cli([a if a != "csv" else "pretty" for a in args])
        assert r2.returncode == 0, r2.stderr
        outs[name] = (_cli_rows(r.stdout, True), [l for l in r2.stdout.splitlines() if "Decode Timestamp" not in l],
                      open(dig).read(), open(rec, "rb").read())
    assert outs["8"] == outs["16"]
    assert len(outs["8"][0]) > 0
    rec = np.frombuffer(outs["8"][3], np.int16).reshape(-1, 2)
    if rec_input:
        # --rx-rec-input writes exactly the widened capture, zero padded to whole buffers
        assert len(rec) % spb == 0 and np.array_equal(rec[:len(w)], w) and not rec[len(w):].any()
    else:
        assert len(rec) > 0
    if not window:
        theirs = _reference_cli(c16, filt, spb, tmp_path / "dig_ref.csv")
        if theirs is not None:
            assert theirs == (outs["8"][0], outs["8"][2])
    # stdin
    with open(c8, "rb") as f:
        r = H.run_cli(["--rx", f"{fmt}_file", "-A", "-", "-d", "p3l-nexa2012", "--rx-fmt", "csv", "-F", filt,
                       "--samples-per-buffer", str(spb)], stdin=f)
    assert r.returncode == 0, r.stderr
    assert _cli_rows(r.stdout, True) == outs["16"][0]
