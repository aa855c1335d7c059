"""Deglitch (include/ookd_gpu.h, "Deglitch") without a GPU: the streaming vote against the whole-string restatement, the
vote-aware receive loop against the oracle's, the argument checks of ookd_gpu_create, and the CLI surface of
--rx-deglitch."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import oracle as O
from ookiedokie_b200 import binding as B
from ookiedokie_b200 import host as H

import ookd_testutil as util
import vote_ref as V

MS = [1, 2, 31, 32, 33, 63, 64, 65, 1000]


def _strings(seed, n):
    rng = np.random.default_rng(seed)
    yield rng.integers(0, 2, n).astype(np.uint8)                          # white
    runs = rng.geometric(1 / 40, n // 8 + 2)                               # bursty: runs of ~40, a third of them 1-3
    short = rng.random(runs.size) < 0.3
    runs[short] = rng.integers(1, 4, int(short.sum()))
    yield (np.repeat(np.arange(runs.size) & 1, runs)[:n]).astype(np.uint8)
    yield np.ones(n, np.uint8)
    yield np.zeros(n, np.uint8)


def _pieces(bits, sizes):
    i, k = 0, 0
    while i < bits.size:
        step = sizes[k % len(sizes)]
        yield bits[i:i + step]
        i += step
        k += 1


@pytest.mark.parametrize("m", MS)
def test_streaming_vote_equals_the_whole_string_vote(m):
    for n in (5000, 3 * m + 17):
        for bits in _strings(m * 7 + n, n):
            want = V.vote(bits, m)
            # piece lengths that put window boundaries inside pieces, pieces shorter than 2M, and empty pieces
            for sizes in ([1024], [7, 1, 300], [2 * m + 1], [max(1, m // 2), 0, 4096]):
                sv = V.StreamVote(m)
                got = np.concatenate([sv.push(p) for p in _pieces(bits, sizes)] + [np.zeros(0, np.uint8)])
                assert np.array_equal(got, want), (m, n, sizes)


@pytest.mark.parametrize("m", [1, 5, 64, 1000])
def test_capture_shorter_than_the_window(m):
    for n in range(0, min(2 * m + 3, 40)):
        bits = np.ones(n, np.uint8)
        want = V.vote(bits, m)
        assert want.size == n and (want[:min(n, m)] == 0).all()
        assert np.array_equal(V.StreamVote(m).push(bits), want)


def test_vote_properties():
    m = 16
    x = np.zeros(2000, np.uint8)
    x[100:100 + m] = 1                                 # a run of M disappears
    x[500:500 + m + 1] = 1                             # a run of M+1 keeps its length, M later
    x[1000:1800] = 1
    x[1200:1200 + m] = 0                               # so does a dip of M inside a long run
    v = V.vote(x, m)
    assert not v[:400].any()
    assert np.array_equal(np.flatnonzero(np.diff(v.astype(int))) + 1, [500 + m, 500 + 2 * m + 1, 1000 + m, 1800 + m])


def _cap(seed=3, sigma=0.03):
    dev = O.load_device("p3l-nexa2012")
    iq, sent, _ = util.capture(dev, 3, sigma=sigma, amplitude=0.95, phase=0.4, seed=seed, fields=util.nexa_fields)
    return dev, iq, sent


@pytest.mark.parametrize("filt,spb", [("fs32_fs4", 8192), ("fs128_fs16_dec4", 8192), (None, 4096), ("fs64_fs8", 6000)])
def test_receive_loop_at_zero_equals_the_oracle(filt, spb):
    dev, iq, _ = _cap(sigma=0.03 if filt else 0.005)
    stages = O.load_filter(filt) if filt else None
    ref = O.rx(iq, stages, dev, samples_per_buffer=spb, want_bits=True)
    got = V.rx(iq, stages, dev, samples_per_buffer=spb, deglitch=0)
    assert got["msgs"] == ref["msgs"] and len(ref["msgs"]) > 0
    assert np.array_equal(got["edges"], ref["edges"]) and got["first_bit"] == ref["first_bit"]
    assert np.array_equal(got["bits"], ref["bits"]) and got["n_out"] == ref["n_out"]


def test_receive_loop_votes_every_consumer():
    dev, iq, _ = _cap()
    stages = O.load_filter("fs32_fs4")
    got = V.rx(iq, stages, dev, deglitch=64)
    assert np.array_equal(got["bits"], V.vote(got["raw_bits"], 64))
    v = got["bits"]
    assert np.array_equal(got["edges"], np.flatnonzero(v[1:] != v[:-1]) + 1) and got["first_bit"] == 0


def test_deglitch_repairs_the_noisy_capture():
    # nexa through fs32_fs4 at sigma 0.03: noise glitches make the state machine drop buffers
    dev = O.load_device("p3l-nexa2012")
    iq, sent, _ = util.capture(dev, 10, sigma=0.03, amplitude=0.95, phase=0.4, seed=5, fields=util.nexa_fields)
    stages = O.load_filter("fs32_fs4")
    ok = lambda r: sum(1 for m in r["msgs"] if m[3] in sent)
    assert ok(V.rx(iq, stages, dev, deglitch=0)) == 3
    assert ok(V.rx(iq, stages, dev, deglitch=16)) == 10


# ---- ookd_gpu_create: argument checks before any CUDA call ----

def _create(deglitch, filter_stages=None):
    L = B.lib()
    cfg = B.GpuConfigEx()
    cfg.threshold = 0.1
    cfg.samples_per_buffer = 8192
    cfg.device_id = 0
    cfg.deglitch = deglitch
    keep = None
    if filter_stages:
        fd, keep = B.make_filter_desc(filter_stages)
        cfg.filter = C.pointer(fd)
    h = C.c_void_p()
    rc = L.ookd_gpu_create(C.byref(h), C.byref(cfg))
    if rc == 0:
        L.ookd_gpu_destroy(h)
    return rc


def test_create_rejects_deglitch_above_the_maximum():
    assert B.DEGLITCH_MAX == 65535
    assert _create(B.DEGLITCH_MAX + 1) == -1                   # OOKD_ERR_ARG
    assert _create(0xFFFFFFFF) == -1


def test_create_rejects_a_halo_beyond_32_bits():
    # (8 + roundup(2M, 64)) * D input samples: 131080 * 2^15 > 2^32
    stages = [(2 ** 15, np.ones(1, np.float32))]
    assert _create(B.DEGLITCH_MAX, stages) == -1
    assert _create(B.DEGLITCH_MAX + 1, stages) == -1


def test_header_matches_the_binding():
    with open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "ookd_gpu.h")) as f:
        text = f.read()
    assert "#define OOKD_DEGLITCH_MAX     65535u" in text
    assert [n for n, _ in B.GpuConfigEx._fields_][-2:] == ["tune_step", "deglitch"]
    assert B.GpuConfigEx.deglitch.offset == 52 and C.sizeof(B.GpuConfigEx) == 56


# ---- CLI surface ----

def _rx(args, tmp_path, filt="fs128_fs16_dec4"):
    cap = tmp_path / "c.bin"
    cap.write_bytes(b"")
    return H.run_cli(["--rx", "bladerf_file", "-A", str(cap), "-d", "p3l-nexa2012", "-F", filt, "-v", "info"] + args)


@pytest.mark.parametrize("arg", ["", "x", "-1", "+3", "1.5", "65536", "99999999999999999999", "12ms", "12 us", "us",
                                 "12US", "0x10", " 4"])
def test_cli_rejects_malformed_deglitch(arg, tmp_path):
    r = _rx(["--rx-deglitch", arg], tmp_path)
    assert r.returncode != 0
    assert "Invalid RX deglitch" in r.stderr


@pytest.mark.parametrize("arg,m", [("0", None), ("1", 1), ("64", 64), ("65535", 65535), ("600us", 450),
                                   ("1us", 0), ("87381us", 65535)])
def test_cli_accepts_deglitch(arg, m, tmp_path):
    # fs128_fs16_dec4 at the default 3 MHz: 750000 outputs/s, so t us is floor(0.75 t) outputs.  Without a GPU the
    # run stops at the device, after the effective value has been printed.
    r = _rx(["--rx-deglitch", arg], tmp_path)
    assert "Invalid RX deglitch" not in r.stderr and "more than" not in r.stderr
    if m:
        assert f"Deglitch: majority of {2 * m + 1} decisions (runs of up to {m} outputs removed)" in r.stderr
    elif arg.endswith("us"):
        assert "Deglitch: off (1us is less than one output)" in r.stderr
    else:
        assert "Deglitch:" not in r.stderr


def test_cli_microseconds_follow_the_decimation(tmp_path):
    r = _rx(["--rx-deglitch", "100us"], tmp_path, filt="fs32_fs4")             # 3e6 outputs/s
    assert "runs of up to 300 outputs removed" in r.stderr
    r = _rx(["--rx-deglitch", "100us", "-s", "2.4M"], tmp_path)                # 600000 outputs/s
    assert "runs of up to 60 outputs removed" in r.stderr


@pytest.mark.parametrize("arg", ["87382us", "100000us", "18446744073709551615us"])
def test_cli_rejects_microseconds_out_of_range(arg, tmp_path):
    r = _rx(["--rx-deglitch", arg], tmp_path)
    assert r.returncode != 0
    assert "more than 65535 outputs at 750000 outputs/s" in r.stderr


def test_cli_deglitch_is_rejected_with_tx(tmp_path):
    r = H.run_cli(["--tx", "bladerf_file", "-A", str(tmp_path / "c.bin"), "-d", "p3l-nexa2012", "--rx-deglitch", "4"])
    assert r.returncode != 0
    assert "--rx-deglitch cannot be used with --tx" in r.stderr
    assert not (tmp_path / "c.bin").exists()


def test_cli_help_documents_deglitch():
    r = H.run_cli(["--help"])
    assert r.returncode == 0
    assert "--rx-deglitch <n>|<t>us" in r.stdout and "majority of the last 2n+1" in r.stdout
