"""Levels (include/ookd_gpu.h, "Levels") without a GPU: the threshold rule ookd_level_threshold against a restatement in
Python integers and math, its argument errors and the binding's ValueError, and the CLI surface of -T auto."""
import ctypes as C
import math
import struct

import numpy as np
import pytest

from ookiedokie_b200 import binding as B
from ookiedokie_b200 import host as H

BINS = B.LEVEL_BINS


def f_bits(bits):
    return struct.unpack("<f", struct.pack("<I", bits))[0]


def rule(hist, margin_db):
    """The rule of the header in Python integers: -> (threshold, F), or None where the C function returns OOKD_ERR_ARG."""
    h = [int(v) for v in hist]
    n = sum(h)
    if n == 0 or n >= 2 ** 64 or not math.isfinite(margin_db):
        return None
    cum = 0
    for m, v in enumerate(h):
        cum += v
        if cum >= n - cum:
            break
    if m >= 4079:
        return None
    F = f_bits((m + 1) << 19)
    try:
        gain = math.pow(10.0, margin_db / 10.0)
    except OverflowError:                                       # C's pow returns +inf
        gain = math.inf
    with np.errstate(over="ignore"):
        thr = float(np.float32(math.sqrt(F * gain)))
    if not math.isfinite(thr):
        return None
    return thr, F


def c_rule(hist, margin_db):
    h = np.ascontiguousarray(hist, dtype=np.uint64)
    thr, F = C.c_float(), C.c_double()
    rc = B.lib().ookd_level_threshold(C.c_void_p(h.ctypes.data), C.c_double(margin_db), C.byref(thr), C.byref(F))
    return rc, float(thr.value), float(F.value)


def check(hist, margin_db):
    want = rule(hist, margin_db)
    rc, thr, F = c_rule(hist, margin_db)
    if want is None:
        assert rc == -1                                         # OOKD_ERR_ARG
        with pytest.raises(ValueError):
            B.level_threshold(hist, margin_db)
    else:
        assert rc == 0
        assert (thr, F) == want
        assert B.level_threshold(hist, margin_db) == want
    return want


def test_bin_edges_are_the_float_grid():
    # bin b's upper edge is f((b+1) << 19): 16 bins per octave, +inf at the top of bin 4079
    assert f_bits(4080 << 19) == math.inf
    assert f_bits(127 << 23) == 1.0 and ((127 << 23) >> 19) == 2032
    assert math.isnan(f_bits(4081 << 19))


@pytest.mark.parametrize("seed", range(12))
def test_rule_on_random_histograms(seed):
    rng = np.random.default_rng(seed)
    hist = np.zeros(BINS, np.uint64)
    centre = int(rng.integers(0, 4079))
    width = int(rng.integers(1, 60))
    lo, hi = max(0, centre - width), min(4096, centre + width)
    hist[lo:hi] = rng.integers(0, 1 << int(rng.integers(1, 40)), size=hi - lo, dtype=np.uint64)
    if hist.sum() == 0:
        hist[centre] = 1
    for margin in (12.0, 0.0, -7.25, 3.0 + seed, 60.0):
        check(hist, margin)


def test_counts_near_2pow63():
    hist = np.zeros(BINS, np.uint64)
    hist[1000] = 2 ** 63 - 1
    hist[1001] = 2 ** 63 - 5                                    # sum = 2^64 - 6: fits, and 2 cum would overflow
    assert check(hist, 12.0)[1] == f_bits(1001 << 19)
    hist[1000], hist[1001] = 2 ** 63 - 2, 2 ** 63 - 1
    assert check(hist, 12.0)[1] == f_bits(1002 << 19)          # cum(1000) = n - cum(1000) - 1 < n - cum: one more bin
    hist[2000] = 7                                              # sum beyond 2^64 - 1: refused
    assert check(hist, 12.0) is None


def test_all_mass_in_bin_zero():
    hist = np.zeros(BINS, np.uint64)
    hist[0] = 12345
    thr, F = check(hist, 12.0)
    assert F == f_bits(1 << 19) and thr > 0.0


def test_exact_half_takes_the_lower_bin():
    hist = np.zeros(BINS, np.uint64)
    hist[500] = hist[900] = 10                                  # cum(500) = 10 >= 20 - 10
    assert check(hist, 0.0)[1] == f_bits(501 << 19)


@pytest.mark.parametrize("m,ok", [(4078, True), (4079, False), (4080, False), (4081, False), (4095, False)])
def test_median_at_the_top(m, ok):
    hist = np.zeros(BINS, np.uint64)
    hist[m] = 3
    hist[10] = 1
    want = check(hist, 0.0)
    assert (want is not None) == ok
    if ok:
        assert want[1] == f_bits(4079 << 19) and math.isfinite(want[0])


def test_errors():
    hist = np.zeros(BINS, np.uint64)
    assert check(hist, 12.0) is None                            # no outputs
    hist[2000] = 9
    for bad in (math.nan, math.inf, -math.inf):
        assert check(hist, bad) is None
    hist[:] = 0
    hist[4078] = 1                                              # F ~ 3.3e38: sqrt(F * 10^40) overflows the float
    assert check(hist, 400.0) is None
    assert check(hist, 1e300) is None                           # pow overflows to inf
    assert check(hist, -400.0) is not None                      # negative margins are allowed
    L = B.lib()
    t = C.c_float()
    assert L.ookd_level_threshold(None, C.c_double(12.0), C.byref(t), None) == -1
    assert L.ookd_level_threshold(C.c_void_p(hist.ctypes.data), C.c_double(12.0), None, None) == -1
    assert L.ookd_level_threshold(C.c_void_p(hist.ctypes.data), C.c_double(12.0), C.byref(t), None) == 0


def test_binding_checks_the_histogram():
    with pytest.raises(ValueError):
        B.level_threshold(np.ones(BINS - 1, np.uint64))
    with pytest.raises(ValueError):
        B.level_threshold(np.ones(BINS, np.float64))
    h = -np.ones(BINS, np.int64)
    with pytest.raises(ValueError):
        B.level_threshold(h)
    assert B.level_threshold(np.ones(BINS, np.int64)) == rule(np.ones(BINS), 12.0)


def test_header_constants():
    assert B.LEVEL_BINS == 4096 and B.LEVEL_MARGIN_DB == 12.0


# ---- CLI surface ----

@pytest.mark.parametrize("arg", ["auto:", "auto:x", "autox", "auto:12dB", "auto:nan", "auto:inf", "auto 3", "AUTO:"])
def test_cli_rejects_malformed_auto(arg, tmp_path):
    cap = tmp_path / "c.bin"
    cap.write_bytes(b"")
    r = H.run_cli(["--rx", "bladerf_file", "-A", str(cap), "-d", "p3l-nexa2012", "-T", arg])
    assert r.returncode != 0
    assert "Invalid RX threshold" in r.stderr


@pytest.mark.parametrize("arg", ["auto", "auto:12", "auto:-3.5", "auto:+20", "auto:0"])
def test_cli_accepts_auto_forms(arg, tmp_path):
    # an accepted form gets past parsing to the decode set-up: with an empty capture and no GPU that fails only at the
    # device, never with "Invalid RX threshold"
    cap = tmp_path / "c.bin"
    cap.write_bytes(b"")
    r = H.run_cli(["--rx", "bladerf_file", "-A", str(cap), "-d", "p3l-nexa2012", "-T", arg])
    assert "Invalid RX threshold" not in r.stderr


@pytest.mark.parametrize("arg", ["0.1", "0", "1", "1e-3"])
def test_cli_numeric_threshold_still_parses(arg, tmp_path):
    cap = tmp_path / "c.bin"
    cap.write_bytes(b"")
    r = H.run_cli(["--rx", "bladerf_file", "-A", str(cap), "-d", "p3l-nexa2012", "-T", arg])
    assert "Invalid RX threshold" not in r.stderr


@pytest.mark.parametrize("arg", ["1.5", "-0.1", "x"])
def test_cli_numeric_range_is_unchanged(arg, tmp_path):
    r = H.run_cli(["--rx", "bladerf_file", "-A", str(tmp_path / "c.bin"), "-d", "p3l-nexa2012", "-T", arg])
    assert r.returncode != 0 and "Invalid RX threshold" in r.stderr


@pytest.mark.parametrize("arg", ["auto", "auto:6"])
def test_cli_auto_is_rejected_with_tx(arg, tmp_path):
    r = H.run_cli(["--tx", "bladerf_file", "-A", str(tmp_path / "c.bin"), "-d", "p3l-nexa2012", "-T", arg])
    assert r.returncode != 0
    assert "-T auto cannot be used with --tx" in r.stderr
    assert not (tmp_path / "c.bin").exists()


def test_cli_help_documents_auto():
    r = H.run_cli(["--help"])
    assert r.returncode == 0
    assert "-T auto[:<dB>]" in r.stdout and "default 12" in r.stdout
