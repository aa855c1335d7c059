"""8-bit capture formats (CU8, CS8): what can be checked without a GPU -- CLI surface, argument checks, the Python
binding's dtype rules."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import oracle as O
from ookiedokie_b200 import binding as B
from ookiedokie_b200 import host as H


@pytest.mark.parametrize("sdr", ["cu8_file", "cs8_file", "CU8_FILE"])
def test_tx_with_an_8bit_type_is_rejected(tmp_path, sdr):
    r = H.run_cli(["--tx", sdr, "-A", str(tmp_path / "c.bin"), "-d", "p3l-nexa2012"])
    assert r.returncode != 0
    assert "--tx writes SC16Q11 captures only" in r.stderr
    assert not (tmp_path / "c.bin").exists()


@pytest.mark.parametrize("direction", ["--rx", "--tx"])
@pytest.mark.parametrize("sdr", ["rtlsdr", "cf32_file", "cu16_file", ""])
def test_unknown_sdr_types_are_rejected(direction, sdr):
    r = H.run_cli([direction, sdr, "-A", "/nonexistent"])
    assert r.returncode != 0
    assert "is not available" in r.stderr


def test_help_lists_the_8bit_types():
    r = H.run_cli(["--help"])
    assert r.returncode == 0
    assert "cu8_file" in r.stdout and "cs8_file" in r.stdout
    assert "bladerf_file" in r.stdout


def _create(flags):
    L = B.lib()
    cfg = B.GpuConfig()
    cfg.threshold = 0.1
    cfg.samples_per_buffer = 8192
    cfg.device_id = 0
    cfg.flags = flags
    h = C.c_void_p()
    rc = L.ookd_gpu_create(C.byref(h), C.byref(cfg))
    if rc == 0:
        L.ookd_gpu_destroy(h)
    return rc


def test_create_rejects_both_format_flags():
    # checked before any CUDA call: the same answer with or without a GPU
    assert _create(B.FLAG_INPUT_CS8 | B.FLAG_INPUT_CU8) == -1          # OOKD_ERR_ARG
    assert _create(B.FLAG_INPUT_CS8 | B.FLAG_INPUT_CU8 | B.FLAG_NO_TMA) == -1


def test_flags_match_the_header():
    with open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "ookd_gpu.h")) as f:
        text = f.read()
    assert "#define OOKD_FLAG_INPUT_CS8   1024u" in text and B.FLAG_INPUT_CS8 == 1024
    assert "#define OOKD_FLAG_INPUT_CU8   2048u" in text and B.FLAG_INPUT_CU8 == 2048


def test_unknown_input_format_is_a_value_error():
    with pytest.raises(ValueError):
        B.Gpu(filter_stages=O.load_filter("fs32_fs4"), input_format="cf32")
    with pytest.raises(ValueError):
        B.MultiGpu([0], input_format="s8")


def test_format_bits_in_flags_are_a_value_error():
    # (the binding would otherwise pass int16 arrays to a handle that reads bytes)
    for f in (B.FLAG_INPUT_CU8, B.FLAG_INPUT_CS8, B.FLAG_INPUT_CU8 | B.FLAG_NO_TMA):
        with pytest.raises(ValueError):
            B.Gpu(filter_stages=O.load_filter("fs32_fs4"), flags=f)
        with pytest.raises(ValueError):
            B.MultiGpu([0], flags=f, input_format="cu8")


def test_host_arrays_must_have_the_format_dtype():
    u = np.zeros((16, 2), np.uint8)
    s = np.zeros((16, 2), np.int8)
    assert B._host_iq(u, "cu8").dtype == np.uint8 and B._host_iq(u, "cu8").size == 32
    assert B._host_iq(s.reshape(-1), "cs8").dtype == np.int8
    for arr, fmt in [(s, "cu8"), (u, "cs8"), (np.zeros((16, 2), np.int16), "cu8"), (u.astype(np.int32), "cs8"),
                     (u, "sc16q11"), (s, "sc16q11")]:
        with pytest.raises(ValueError):
            B._host_iq(arr, fmt)
    # SC16Q11 handles keep converting other integer arrays as before
    assert B._host_iq(np.zeros((4, 2), np.int32), "sc16q11").dtype == np.int16
    p, n, is_dev, keep = B._as_ptr(u, "cu8")
    assert n == 16 and is_dev == 0
    assert B._as_ptr((1234, 99), "cu8")[1:3] == (99, 1)
