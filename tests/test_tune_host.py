"""Tuning (include/ookd_gpu.h, "Tuning") without a GPU: the table, the CPU rotation ookd_tune_sc16q11 against the numpy
restatement in tune_ref, the phase-step conversion, the binding's checks and the CLI's --rx-offset."""
import ctypes as C
import math

import numpy as np
import pytest

from ookiedokie_b200 import binding as B
from ookiedokie_b200 import host as H
import tune_ref as T


def test_table_is_the_rounded_quarter_sine():
    lib_tab = np.array((C.c_int16 * 257).in_dll(B.lib(), "ookd_tune_quarter"), np.int64)
    want = T.quarter_table()
    assert np.array_equal(lib_tab, want)
    assert lib_tab[0] == 0 and lib_tab[128] == 23170 and lib_tab[256] == 32767


def test_quadrants_give_the_full_circle():
    k = np.arange(1024)
    c, s = T.cos_sin(k)
    assert np.abs(c - np.round(32767 * np.cos(2 * np.pi * k / 1024))).max() <= 1
    assert np.abs(s - np.round(32767 * np.sin(2 * np.pi * k / 1024))).max() <= 1


def _full_range(rng, n):
    x = rng.integers(-32768, 32768, size=(n, 2)).astype(np.int16)
    # full-scale corners at every quadrant: the clamp is reachable only there
    corners = np.array([[-32768, -32768], [-32768, 32767], [32767, -32768], [32767, 32767], [-32768, 0], [0, -32768]],
                       np.int16)
    x[: 6 * 200] = np.tile(corners, (200, 1))
    return x


STEPS = [1, 2**31, 2**32 - 1, 0x12345, 2**30 + 7, 0x9E3779B9]


@pytest.mark.parametrize("step", STEPS)
@pytest.mark.parametrize("first", [0, 12345, 2**32 - 100, 2**32 + 17, 2**36 + 3])
def test_cpu_rotation_matches_numpy(step, first):
    rng = np.random.default_rng(step ^ first)
    x = _full_range(rng, 4096)
    got = B.tune_sc16q11(x, first, step)
    assert np.array_equal(got, T.tune(x, step, first))


def test_clamp_is_reached_and_every_quadrant_seen():
    x = np.tile(np.array([[-32768, -32768]], np.int16), (1024, 1))
    step = 1 << 22                                     # one table phase per sample: k = n
    got = B.tune_sc16q11(x, 0, step)
    assert np.array_equal(got, T.tune(x, step))
    assert (got == 32767).any() and (got == -32768).any()


def test_random_steps_and_in_place():
    rng = np.random.default_rng(7)
    for _ in range(20):
        step = int(rng.integers(1, 2**32))
        first = int(rng.integers(0, 2**40))
        x = rng.integers(-32768, 32768, size=(777, 2)).astype(np.int16)
        want = T.tune(x, step, first)
        assert np.array_equal(B.tune_sc16q11(x, first, step), want)
        buf = x.copy()
        assert B.lib().ookd_tune_sc16q11(buf.ctypes.data, buf.ctypes.data, first, 777, step) == 0
        assert np.array_equal(buf, want)


def test_step_zero_and_zero_samples_are_identities():
    x = np.arange(-200, 200, dtype=np.int16).reshape(-1, 2)
    assert np.array_equal(B.tune_sc16q11(x, 99, 0), x)
    assert np.array_equal(B.tune_sc16q11(np.zeros((5, 2), np.int16), 3, 0x1234567), np.zeros((5, 2), np.int16))


def _c_step(off, fs):
    st = C.c_uint32()
    rc = B.lib().ookd_tune_step(C.c_double(off), C.c_uint32(fs), C.byref(st))
    return rc, st.value


def test_tune_step_rounding_and_sign():
    assert B.tune_step(250e3, 3_000_000) == round(250e3 / 3e6 * 2**32)
    assert B.tune_step(900e3, 3e6) == 1288490189                     # 0.3 * 2^32 = 1288490188.8
    assert B.tune_step(-250e3, 3_000_000) == 2**32 - round(250e3 / 3e6 * 2**32)
    assert B.tune_step(0.0, 3_000_000) == 0
    assert B.tune_step(1.0, 2**31) == 2                               # 2^32 / 2^31 exactly
    assert B.tune_step(0.375, 2**32 - 1) == 0                         # 0.375 * 2^32 / (2^32-1) rounds to 0
    # halfway cases round away from zero, as llround does
    assert B.tune_step(0.5, 2**32 // 2**1) == 1                       # 0.5 / 2^31 * 2^32 = 1.0
    assert B.tune_step(0.25, 2**31) == 1 and B.tune_step(-0.25, 2**31) == 2**32 - 1   # +-0.5 -> +-1
    # just inside +-Fs/2 is accepted and rounds to half a turn
    assert B.tune_step(math.nextafter(1.5e6, 0), 3_000_000) == 2**31
    assert B.tune_step(-math.nextafter(1.5e6, 0), 3_000_000) == 2**31
    assert B.tune_step(1499000, 3_000_000) == round(1499000 / 3e6 * 2**32)


@pytest.mark.parametrize("off,fs", [(1.5e6, 3_000_000), (-1.5e6, 3_000_000), (2e6, 3_000_000), (1.0, 2),
                                    (float("nan"), 3_000_000), (float("inf"), 3_000_000), (-float("inf"), 3_000_000),
                                    (0.0, 0), (10.0, 0)])
def test_tune_step_rejects(off, fs):
    assert _c_step(off, fs)[0] == -1                                  # OOKD_ERR_ARG
    with pytest.raises(ValueError):
        B.tune_step(off, fs)


def test_tune_step_null_output_is_an_argument_error():
    assert B.lib().ookd_tune_step(C.c_double(1.0), C.c_uint32(10), None) == -1


def test_config_struct_has_the_field_last():
    names = [f[0] for f in B.GpuConfig._fields_]
    assert names[-1] == "tune_step"


def _cli_rx(tmp_path, extra):
    cap = tmp_path / "c.cu8"
    cap.write_bytes(bytes(64))
    return H.run_cli(["--rx", "cu8_file", "-A", str(cap), "-d", "p3l-nexa2012"] + extra)


@pytest.mark.parametrize("arg", ["250k", "-250k", "+0.9M", "-1.2MHz", "1499999", "0", "-3e5"])
def test_cli_accepts_offsets(tmp_path, arg):
    r = _cli_rx(tmp_path, ["--rx-offset", arg])
    assert "Invalid RX offset" not in r.stderr and "out of range" not in r.stderr


@pytest.mark.parametrize("arg,extra", [("1.5M", []), ("-1.5M", []), ("2M", []), ("600k", ["-s", "1.2M"]),
                                       ("-1G", [])])
def test_cli_rejects_out_of_range_offsets(tmp_path, arg, extra):
    r = _cli_rx(tmp_path, ["--rx-offset", arg] + extra)
    assert r.returncode != 0
    assert "out of range" in r.stderr and "below half the sample rate" in r.stderr


def test_cli_converts_against_the_sample_rate_given_after_it(tmp_path):
    # -s after --rx-offset still applies: 1 MHz is fine at 3 MS/s and out of range at 1.5 MS/s
    assert "out of range" not in _cli_rx(tmp_path, ["--rx-offset", "1M", "-s", "3M"]).stderr
    assert "out of range" in _cli_rx(tmp_path, ["--rx-offset", "1M", "-s", "1.5M"]).stderr


@pytest.mark.parametrize("arg", ["abc", "1.2X", "", "nan", "inf", "1e400"])
def test_cli_rejects_malformed_offsets(tmp_path, arg):
    r = _cli_rx(tmp_path, ["--rx-offset", arg])
    assert r.returncode != 0
    assert "Invalid RX offset" in r.stderr


def test_cli_rejects_offset_with_tx(tmp_path):
    r = H.run_cli(["--tx", "bladerf_file", "-A", str(tmp_path / "c.bin"), "-d", "p3l-nexa2012", "--rx-offset", "100k"])
    assert r.returncode != 0
    assert "--rx-offset cannot be used with --tx" in r.stderr
    assert not (tmp_path / "c.bin").exists()


def test_help_lists_rx_offset():
    r = H.run_cli(["--help"])
    assert r.returncode == 0 and "--rx-offset <Hz>" in r.stdout
