"""Tuning (include/ookd_gpu.h, "Tuning") on the GPU: a handle with tune_step decodes a capture x exactly as an untuned
handle -- and the oracle -- decode T(x), the numpy restatement in tune_ref: filtered samples, decisions, edges,
messages, sizes, through every FIR path, shard layout and input kind."""
import os

import numpy as np
import pytest

from oracle import oracle as O
from ookiedokie_b200 import binding as B
from ookiedokie_b200 import host as H
import ookd_testutil as util
import tune_ref as T

pytestmark = pytest.mark.gpu

FMTS = ["sc16q11", "cu8", "cs8"]
FS = util.FS
STEPS = {"pos": B.tune_step(250e3, FS), "neg": B.tune_step(-600e3, FS), "nyq": B.tune_step(1.4999e6, FS),
         "odd": 0x2468ACF1}


def shift(iq, offset_hz, samplerate=FS):
    """Move a baseband SC16Q11 capture up by offset_hz (float rotation, round, clip): a transmitter off centre."""
    x = np.asarray(iq, np.int16).reshape(-1, 2).astype(np.float64)
    ph = 2.0 * np.pi * offset_hz / samplerate * np.arange(len(x), dtype=np.float64)
    c, s = np.cos(ph), np.sin(ph)
    y = np.stack([x[:, 0] * c - x[:, 1] * s, x[:, 0] * s + x[:, 1] * c], -1)
    return np.clip(np.rint(y), -32768, 32767).astype(np.int16)


def to_format(iq, fmt):
    """SC16Q11 capture -> (capture in fmt, its SC16Q11 words): CS8 k = round(x / 16), CU8 v = round((x + 2040) / 16)."""
    if fmt == "sc16q11":
        return iq, iq
    x = np.asarray(iq, np.float64)
    if fmt == "cs8":
        b = np.clip(np.rint(x / 16), -128, 127).astype(np.int8)
    else:
        b = np.clip(np.rint((x + 2040) / 16), 0, 255).astype(np.uint8)
    return b, T.widen(b, fmt)


def _gpu(filt, dev=None, fmt="sc16q11", **kw):
    stages = O.load_filter(filt) if isinstance(filt, str) else filt
    sm = util.sm_spec(dev, stages) if dev is not None else None
    return B.Gpu(filter_stages=stages, sm=sm, input_format=fmt, **kw), stages


def _same(gt, gu, cap, tcap, ref=None):
    """tuned decode of cap on gt == untuned decode of tcap = T(cap) on gu (== the oracle's on T(cap), when given)"""
    a = gt.decode(cap)
    b = gu.decode(tcap)
    for k in ("n_in", "n_out", "n_buffers", "n_edges", "first_bit", "msgs"):
        assert a[k] == b[k], k
    fa, ea = gt.edges()
    fb, eb = gu.edges()
    assert fa == fb and np.array_equal(ea, eb)
    if ref is not None:
        assert a["n_out"] == ref["n_out"] and a["n_buffers"] == ref["n_buffers"]
        assert fa == ref["first_bit"] and np.array_equal(ea, ref["edges"])
        assert a["msgs"] == ref["msgs"]
    return a


GENERIC = [(3, np.linspace(-0.3, 0.9, 7, dtype=np.float32)), (2, np.array([0.25, -0.5, 1.0, 0.125, 0.5], np.float32))]


@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("filt", ["fs32_fs4", "fs128_fs16_dec4", "fs64_fs8", "unity1", "generic"])
@pytest.mark.parametrize("step", sorted(STEPS))
def test_filtered_equals_untuned_of_tuned_capture(fmt, filt, step):
    rng = np.random.default_rng(len(fmt) * 131 + len(filt) * 7 + STEPS[step] % 1000)
    n = 40001
    if fmt == "sc16q11":
        x = rng.integers(-32768, 32768, size=(n, 2)).astype(np.int16)
        x[:64] = np.array([[-32768, -32768], [32767, -32768], [-32768, 32767], [32767, 32767]], np.int16).repeat(16, 0)
        w = x
    else:
        x = rng.integers(0, 256, size=(n, 2)).astype(np.uint8)
        if fmt == "cs8":
            x = x.view(np.int8)
        w = T.widen(x, fmt)
    tw = T.tune(w, STEPS[step])
    stages = GENERIC if filt == "generic" else O.load_filter(filt)
    gt, _ = _gpu(stages, fmt=fmt, samples_per_buffer=1024, tune_step=STEPS[step])
    gu, _ = _gpu(stages, samples_per_buffer=1024)
    got = gt.filtered(x)
    assert np.array_equal(got.view(np.uint32), gu.filtered(tw).view(np.uint32))
    ref = O.rx(tw, stages, None, samples_per_buffer=1024, want_filtered=True)["filtered"]
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))


CASES = [
    # device, filter, n_msgs, sigma, amp, spb, offset (Hz)
    ("p3l-nexa2012", "fs32_fs4", 3, 0.0, 0.95, 8192, 250e3),
    ("p3l-nexa2012", "fs32_fs4", 3, 0.05, 0.95, 1024, -431e3),
    ("p3l-nexa2012", "fs128_fs16_dec4", 3, 0.02, 0.95, 8192, 700e3),
    ("p3l-nexa2012", "fs64_fs8", 3, 0.05, 0.95, 8192, -1.2e6),
    ("p3l-nexa2012", None, 2, 0.0, 0.95, 8192, 123456.0),
    ("unknown-remote1", "fs128_fs16_dec4", 6, 0.05, 0.30, 8192, -900e3),
    ("unknown-remote1", "fs32_fs4", 4, 0.02, 0.5, 1024, 1.3e6),
]


def _offset_case(devname, n_msgs, sigma, amp, spb, offset, fmt, seed=0):
    dev = O.load_device(devname)
    fields = util.nexa_fields if "nexa" in devname else util.remote_fields
    iq, _, _ = util.capture(dev, n_msgs, sigma=sigma, amplitude=amp, phase=0.7, seed=n_msgs * 17 + spb + seed,
                            fields=fields, tail=20000 + 777)      # not a multiple of spb: EOF padding
    x, w = to_format(shift(iq, offset), fmt)
    step = B.tune_step(offset, FS)
    return dev, x, T.tune(w, step), step


@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("devname,filt,n_msgs,sigma,amp,spb,offset", CASES)
def test_decode_matches_oracle_on_tuned_capture(fmt, devname, filt, n_msgs, sigma, amp, spb, offset):
    dev, x, tx, step = _offset_case(devname, n_msgs, sigma, amp, spb, offset, fmt)
    gt, stages = _gpu(filt, dev, fmt, samples_per_buffer=spb, sm_chunk_buffers=7, tune_step=step)
    gu, _ = _gpu(filt, dev, samples_per_buffer=spb, sm_chunk_buffers=7)
    ref = O.rx(tx, stages, dev, samples_per_buffer=spb, want_bits=True)
    a = _same(gt, gu, x, tx, ref)
    assert np.array_equal(gt.bits(), ref["bits"])
    if sigma <= 0.02 and filt is not None:
        assert len(a["msgs"]) == n_msgs                             # tuned to the transmitter: every message decodes


@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("flags", [0, B.FLAG_FMA_SCREEN, B.FLAG_NO_SCREEN, B.FLAG_FORCE_GENERIC, B.FLAG_NO_TMA,
                                   B.FLAG_NO_ADAPTIVE])
@pytest.mark.parametrize("filt", ["fs32_fs4", "fs128_fs16_dec4"])
def test_decode_paths(fmt, flags, filt):
    dev, x, tx, step = _offset_case("p3l-nexa2012", 3, 0.03, 0.9, 8192, -333e3, fmt, seed=5)
    gt, stages = _gpu(filt, dev, fmt, samples_per_buffer=8192, flags=flags, tune_step=step)
    gu, _ = _gpu(filt, dev, samples_per_buffer=8192, flags=flags)
    ref = O.rx(tx, stages, dev, samples_per_buffer=8192)
    _same(gt, gu, x, tx, ref)
    _same(gt, gu, x, tx, ref)                                       # a second decode on the same handles


@pytest.mark.parametrize("fmt", FMTS)
def test_low_snr_fma_screening(fmt):
    dev, x, tx, step = _offset_case("unknown-remote1", 10, 0.10, 0.30, 8192, 555e3, fmt, seed=77)
    for flags in (0, B.FLAG_NO_ADAPTIVE):
        gt, stages = _gpu("fs128_fs16_dec4", dev, fmt, samples_per_buffer=8192, flags=flags, tune_step=step)
        gu, _ = _gpu("fs128_fs16_dec4", dev, samples_per_buffer=8192, flags=flags)
        ref = O.rx(tx, stages, dev, samples_per_buffer=8192)
        _same(gt, gu, x, tx, ref)
        _same(gt, gu, x, tx, ref)


@pytest.mark.parametrize("fmt", FMTS)
def test_shards_above_2pow32(fmt):
    """decode_shard chains whose first_sample lies beyond 2^32: the phase is (uint32) (n * step) of the 64-bit global
    index.  The shard's bytes stand for samples [F - halo, F + n) of a longer capture; nothing of 2^32 samples is
    allocated."""
    dev, x, _, step = _offset_case("p3l-nexa2012", 8, 0.02, 0.95, 4096, 410e3, fmt, seed=3)
    w = x if fmt == "sc16q11" else T.widen(x, fmt)
    stages = O.load_filter("fs32_fs4")
    sm = util.sm_spec(dev, stages)
    gt = B.Gpu(filter_stages=stages, sm=sm, samples_per_buffer=4096, sm_chunk_buffers=5, input_format=fmt, tune_step=step)
    gu = B.Gpu(filter_stages=stages, sm=sm, samples_per_buffer=4096, sm_chunk_buffers=5)
    halo = gt.halo
    for F in (0, (1 << 32) + 4096 * 3, (1 << 36) - 4096 * 7):
        # positions in the capture are F + i; the first shard keeps its halo window inside the array
        base = F - halo if F >= halo else 0
        tw = T.tune(w, step, base)
        bounds = [halo, halo + 4096 * 31, halo + 4096 * 70, len(x)] if F >= halo else [0, 4096 * 40, 4096 * 97, len(x)]
        exits_t, exits_u, mt, mu = [None], [None], [], []
        for i in range(len(bounds) - 1):
            lo, hi = bounds[i], bounds[i + 1]
            first = base + lo
            h = min(halo, first, lo)
            last = i == len(bounds) - 2
            rt, et = gt.decode_shard(x[lo - h: hi], first, hi - lo, last, exits_t[-1])
            ru, eu = gu.decode_shard(tw[lo - h: hi], first, hi - lo, last, exits_u[-1])
            for k in ("n_out", "n_edges", "first_bit", "msgs"):
                assert rt[k] == ru[k], (F, i, k)
            assert np.array_equal(gt.edges()[1], gu.edges()[1])
            exits_t.append(et)
            exits_u.append(eu)
            mt += rt["msgs"]
            mu += ru["msgs"]
        assert mt == mu and len(mt) >= 6, F


@pytest.mark.parametrize("fmt", FMTS)
def test_sub_windows_and_multi(fmt):
    dev, x, tx, step = _offset_case("p3l-nexa2012", 12, 0.02, 0.95, 4096, -710e3, fmt, seed=21)
    stages = O.load_filter("fs32_fs4")
    sm = util.sm_spec(dev, stages)
    ref = O.rx(tx, stages, dev, samples_per_buffer=4096)
    assert len(ref["msgs"]) == 12
    for k in (2, 3, 4):
        s = B.Gpu(filter_stages=stages, sm=sm, samples_per_buffer=4096, sm_chunk_buffers=5, sub_windows=k,
                  input_format=fmt, tune_step=step)
        r = s.decode(x)
        assert r["msgs"] == ref["msgs"], k
        fb, e = s.edges()
        assert fb == ref["first_bit"] and np.array_equal(e, ref["edges"]), k
    m = B.MultiGpu([0, 0, 0], filter_stages=stages, sm=sm, samples_per_buffer=4096, sm_chunk_buffers=5, input_format=fmt,
                   tune_step=step)
    r, _ = m.decode(x)
    assert r["msgs"] == ref["msgs"]
    fb, e = m.edges()
    assert fb == ref["first_bit"] and np.array_equal(e, ref["edges"])


@pytest.mark.parametrize("fmt", FMTS)
def test_device_input_and_unaligned_pointers(fmt):
    import torch
    dev, x, tx, step = _offset_case("p3l-nexa2012", 3, 0.02, 0.95, 8192, 377e3, fmt, seed=9)
    ref = O.rx(tx, O.load_filter("fs32_fs4"), dev, samples_per_buffer=8192)
    gu, _ = _gpu("fs32_fs4", dev, samples_per_buffer=8192)
    raw = np.ascontiguousarray(x).view(np.uint8).reshape(-1)
    offs = (0, 4, 16) if fmt == "sc16q11" else (0, 1, 2, 16)
    for off in offs:
        buf = torch.zeros(raw.size + 64, dtype=torch.uint8, device="cuda")
        buf[off:off + raw.size] = torch.from_numpy(raw).cuda()
        torch.cuda.synchronize()
        for flags in (0, B.FLAG_NO_TMA):
            gt, _ = _gpu("fs32_fs4", dev, fmt, samples_per_buffer=8192, flags=flags, tune_step=step)
            _same(gt, gu, (buf.data_ptr() + off, len(x)), tx, ref)


def test_step_zero_is_the_untuned_handle():
    dev = O.load_device("p3l-nexa2012")
    iq, _, _ = util.capture(dev, 3, sigma=0.02, amplitude=0.95, phase=0.3, seed=2, fields=util.nexa_fields)
    for filt in ("fs32_fs4", "fs128_fs16_dec4"):
        g0, _ = _gpu(filt, dev, samples_per_buffer=8192, tune_step=0)
        gn, _ = _gpu(filt, dev, samples_per_buffer=8192)
        a = _same(g0, gn, iq, iq)
        assert len(a["msgs"]) == 3
        assert np.array_equal(g0.filtered(iq).view(np.uint32), gn.filtered(iq).view(np.uint32))


def test_filtered_sc16q11_after_a_tuned_decode():
    """the post-filter recorder's samples of a tuned decode are those of the untuned decode of T(x)"""
    dev, x, tx, step = _offset_case("p3l-nexa2012", 3, 0.02, 0.95, 8192, 640e3, "cu8", seed=4)
    gt, _ = _gpu("fs128_fs16_dec4", dev, "cu8", samples_per_buffer=8192, tune_step=step)
    gu, _ = _gpu("fs128_fs16_dec4", dev, samples_per_buffer=8192)
    _same(gt, gu, x, tx)
    assert np.array_equal(gt.filtered_sc16q11(), gu.filtered_sc16q11())


# ---- what the feature is for ----

def test_off_centre_transmitter_is_recovered():
    """A nexa capture moved to +900 kHz at 3 MS/s sits in the fs32_fs4 stopband: untuned it decodes nothing, tuned by
    tune_step(900e3, 3e6) it decodes the baseband capture's payloads."""
    dev = O.load_device("p3l-nexa2012")
    iq, _, _ = util.capture(dev, 6, sigma=0.02, amplitude=0.95, phase=0.5, seed=31, fields=util.nexa_fields)
    off = shift(iq, 900e3)
    stages = O.load_filter("fs32_fs4")
    base = O.rx(iq, stages, dev, samples_per_buffer=8192)["msgs"]
    assert len(base) == 6
    gu, _ = _gpu("fs32_fs4", dev, samples_per_buffer=8192)
    assert gu.decode(off)["msgs"] == []
    step = B.tune_step(900e3, 3e6)
    gt, _ = _gpu("fs32_fs4", dev, samples_per_buffer=8192, tune_step=step)
    got = gt.decode(off)["msgs"]
    assert [m[2:] for m in got] == [m[2:] for m in base]            # (num_bits, payload)
    assert got == O.rx(T.tune(off, step), stages, dev, samples_per_buffer=8192)["msgs"]


def test_two_transmitters_in_one_device_capture():
    """nexa at -600 kHz and remote1 at +700 kHz in ONE device-resident capture, decoded by two handles with different
    steps through batch_decode: each returns its own transmitter's messages, as the oracle does on its own T(x)."""
    import torch
    nexa, rem = O.load_device("p3l-nexa2012"), O.load_device("unknown-remote1")
    a, _, _ = util.capture(nexa, 5, sigma=0.0, amplitude=0.45, phase=0.1, seed=41, fields=util.nexa_fields)
    b, _, _ = util.capture(rem, 8, sigma=0.0, amplitude=0.45, phase=1.3, seed=42, fields=util.remote_fields, lead=30000)
    n = max(len(a), len(b))
    mix = np.zeros((n, 2), np.float64)
    mix[:len(a)] += shift(a, -600e3)
    mix[:len(b)] += shift(b, 700e3)
    rng = np.random.default_rng(43)
    mix += rng.normal(0, 0.01 * 2048, mix.shape)
    x = np.clip(np.rint(mix), -32768, 32767).astype(np.int16)
    d = torch.from_numpy(x).cuda()
    torch.cuda.synchronize()
    stages = O.load_filter("fs32_fs4")
    handles, refs = [], []
    for dev, off in ((nexa, -600e3), (rem, 700e3)):
        step = B.tune_step(off, FS)
        handles.append(B.Gpu(filter_stages=stages, sm=util.sm_spec(dev, stages), samples_per_buffer=8192, tune_step=step))
        refs.append(O.rx(T.tune(x, step), stages, dev, samples_per_buffer=8192)["msgs"])
    assert len(refs[0]) == 5 and len(refs[1]) == 8
    msgs, _ = B.batch_decode(handles, [((d.data_ptr(), n), 0), ((d.data_ptr(), n), 1)])
    for got, ref, g in zip(msgs, refs, handles):
        assert B.msgs_to_tuples(got, g.msg_bytes) == ref


def test_benchmark_recipe_2pow27_offset_vs_oracle():
    """2^27 samples of the benchmark's capture recipe moved to +250 kHz on the device: the tuned decode (device input)
    against the oracle on T(x)."""
    import torch
    from test_gpu_input8 import bench_capture
    n = 1 << 27
    d16, fir, hdev = bench_capture(n)
    f = 250e3
    ph = (torch.arange(n, device="cuda", dtype=torch.float64) * (2.0 * np.pi * f / FS))
    c, s = torch.cos(ph), torch.sin(ph)
    del ph
    xi, xq = d16[:, 0].double(), d16[:, 1].double()
    off = torch.stack([torch.round(xi * c - xq * s), torch.round(xi * s + xq * c)], -1).clamp(-32768, 32767).to(torch.int16)
    del c, s, xi, xq, d16
    torch.cuda.synchronize()
    x = off.cpu().numpy()
    step = B.tune_step(f, FS)
    tx = np.empty_like(x)
    for i in range(0, n, 1 << 24):
        tx[i:i + (1 << 24)] = B.tune_sc16q11(x[i:i + (1 << 24)], i, step)
    import bench
    odev = O.load_device(bench.DEVICE_NAME)
    ref = O.rx(tx, fir.stages, odev, samples_per_buffer=8192)
    assert len(ref["msgs"]) > 100
    g = B.Gpu(filter_stages=fir.stages, sm=hdev.sm_spec(), threshold=0.1, samples_per_buffer=8192, device_id=0,
              tune_step=step)
    got = g.decode((off.data_ptr(), n))
    fb, e = g.edges()
    assert fb == ref["first_bit"] and np.array_equal(e, ref["edges"])
    assert got["msgs"] == ref["msgs"]
    s3 = B.Gpu(filter_stages=fir.stages, sm=hdev.sm_spec(), threshold=0.1, samples_per_buffer=8192, device_id=0,
               tune_step=step, sub_windows=3)
    assert s3.decode((off.data_ptr(), n))["msgs"] == ref["msgs"]


# ---- the CLI ----

def _rows(out):
    return [l.split(",")[1:] for l in out.strip().splitlines()] if out.strip() else []


@pytest.mark.parametrize("sdr,extra", [("bladerf_file", []), ("cu8_file", []), ("cu8_file", ["--gpu-ids", "0,0"]),
                                       ("bladerf_file", ["--window", str(24576 * 5), "-F", "fs128_fs16_dec4"])])
def test_cli_rx_offset(sdr, extra, tmp_path):
    """--rx-offset: stdout (csv and pretty) and -B equal the untuned CLI on the --rx-rec-input file it wrote, and that
    file is numpy's T(x), byte for byte, zero padded to whole buffers."""
    dev = O.load_device("p3l-nexa2012")
    iq, _, _ = util.capture(dev, 6, sigma=0.02, amplitude=0.95, phase=0.9, seed=4, fields=util.nexa_fields,
                            tail=20000 + 333)
    fmt = "cu8" if sdr == "cu8_file" else "sc16q11"
    x, w = to_format(shift(iq, -420e3), fmt)
    cap = tmp_path / "cap.bin"
    np.ascontiguousarray(x).tofile(cap)
    rec, dig_t, dig_u = tmp_path / "rec.sc16q11", tmp_path / "dig_t.csv", tmp_path / "dig_u.csv"
    args = ["--rx", sdr, "-A", str(cap), "-d", "p3l-nexa2012", "--rx-fmt", "csv", "--rx-offset", "-420k",
            "-R", f"bladerf_file,{rec}", "--rx-rec-input", "-B", str(dig_t)] + extra
    r = H.run_cli(args)
    assert r.returncode == 0, r.stderr
    rp = H.run_cli([a if a != "csv" else "pretty" for a in args])
    assert rp.returncode == 0, rp.stderr
    got = np.fromfile(rec, np.int16).reshape(-1, 2)
    want = T.tune(w, B.tune_step(-420e3, FS))
    assert len(got) % 8192 == 0 and np.array_equal(got[:len(want)], want) and not got[len(want):].any()
    plain = [a for a in extra if a != "--gpu-ids" and a != "0,0"]
    u = H.run_cli(["--rx", "bladerf_file", "-A", str(rec), "-d", "p3l-nexa2012", "--rx-fmt", "csv", "-B", str(dig_u)]
                  + plain)
    assert u.returncode == 0, u.stderr
    up = H.run_cli(["--rx", "bladerf_file", "-A", str(rec), "-d", "p3l-nexa2012", "--rx-fmt", "pretty"] + plain)
    assert _rows(r.stdout) == _rows(u.stdout) and len(_rows(r.stdout)) == 1 + 6      # header + messages
    strip = lambda out: [l for l in out.splitlines() if "Decode Timestamp" not in l]
    assert strip(rp.stdout) == strip(up.stdout)
    assert open(dig_t).read() == open(dig_u).read()
