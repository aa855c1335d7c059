"""Levels (include/ookd_gpu.h, "Levels") on the GPU: ookd_gpu_levels equals np.bincount of the bins of the oracle's
filtered power over exactly the decode's outputs, for every filter shape, format and tuning; spans, input kinds and the
last decode's results; -T auto in the CLI; and that the threshold chosen decodes low-level captures -T 0.1 cannot."""
import re

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
STEP = B.tune_step(-437e3, FS)
RNG_T = np.random.default_rng(7)
# generic shapes of the filter-domain families: 3 stages, decimation 3, 1024 taps
GENERIC3 = [(3, RNG_T.standard_normal(1024).astype(np.float32) / 64), (2, np.linspace(-0.3, 0.9, 7, dtype=np.float32)),
            (1, np.array([0.25, -0.5, 1.0, 0.125, 0.5], np.float32))]
GENERIC_D3 = [(3, np.linspace(0.1, 1.0, 1024, dtype=np.float32) / 512)]
FILTERS = {"fs32_fs4": None, "fs128_fs16_dec4": None, "fs64_fs8": None, "unity1": None, "unity16": None, "none": [],
           "generic3": GENERIC3, "generic_d3": GENERIC_D3}


def stages_of(name):
    s = FILTERS[name]
    return O.load_filter(name) if s is None else s


def ref_hist(words, stages, o_lo, o_hi):
    """np.bincount of the bins of p = re*re + im*im (float32) of the oracle's filtered output of SC16Q11 words, outputs
    [o_lo, o_hi) (the oracle runs from sample 0; outputs past the span never reach the zero padding it adds)."""
    f = O.rx(words, stages or None, None, samples_per_buffer=1024, want_filtered=True)["filtered"][o_lo:o_hi]
    re_, im_ = f[:, 0], f[:, 1]
    with np.errstate(over="ignore", invalid="ignore"):
        p = re_ * re_ + im_ * im_
    return np.bincount((p.view(np.uint32) & 0x7FFFFFFF) >> 19, minlength=B.LEVEL_BINS).astype(np.uint64)


def test_reference_nan_is_the_x86_default_nan():
    # the oracle's arithmetic runs on the host: its NaN is 0xFFC00000, the bin every GPU NaN is counted in
    f = O.rx(np.full((64, 2), 16, np.int16), [(1, np.array([np.inf, -np.inf], np.float32))], None,
             samples_per_buffer=64, want_filtered=True)["filtered"]
    assert (f.view(np.uint32)[8:] == 0xFFC00000).all()


def random_capture(fmt, n, seed):
    """-> (capture in fmt, its SC16Q11 words)"""
    rng = np.random.default_rng(seed)
    if fmt == "sc16q11":
        x = rng.integers(-32768, 32768, size=(n, 2)).astype(np.int16)
        return x, x
    x = rng.integers(0, 256, size=(n, 2)).astype(np.uint8)
    if fmt == "cs8":
        x = x.view(np.int8)
    return x, T.widen(x, fmt)


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


def gpu(stages, fmt="sc16q11", **kw):
    return B.Gpu(filter_stages=stages or None, input_format=fmt, samples_per_buffer=1024, **kw)


@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("filt", sorted(FILTERS))
@pytest.mark.parametrize("tuned", [False, True])
def test_levels_equal_oracle(fmt, filt, tuned):
    stages = stages_of(filt)
    n = 40001 if filt != "generic3" else 12011
    x, w = random_capture(fmt, n, len(filt) * 31 + len(fmt) + tuned)
    if tuned:
        w = T.tune(w, STEP)
    g = gpu(stages, fmt, tune_step=STEP if tuned else 0)
    D = g.total_decimation
    got = g.levels(x)
    want = ref_hist(w, stages, 0, n // D)
    assert int(got.sum()) == n // D
    assert np.array_equal(got, want)


TAP_FAMILIES = {
    "subnormal": [(1, np.full(4, 2.0 ** -72, np.float32))],                 # powers ~2^-140: the subnormal bins
    "inf": [(1, np.array([3e38, 1e38], np.float32))],                      # re*re overflows: bin 4080
    "nan": [(1, np.array([np.inf, -np.inf, 1.0], np.float32))],            # inf - inf, inf * 0: NaN (|x| <= 1 in 8 bits)
    "nan_dec4": [(2, np.array([1.0, 0.5], np.float32)), (2, np.array([np.inf, -np.inf, 2.0], np.float32))],
}


@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("fam", sorted(TAP_FAMILIES))
def test_levels_tap_families(fmt, fam):
    stages = TAP_FAMILIES[fam]
    x, w = random_capture(fmt, 20000, 5 + len(fam))
    g = gpu(stages, fmt)
    got = g.levels(x)
    want = ref_hist(w, stages, 0, 20000 // g.total_decimation)
    assert np.array_equal(got, want)
    if fam == "subnormal":
        assert got[:16].sum() > 0                                            # below 2^-126: subnormal bins
    elif fam == "inf":
        assert got[4080] > 0
    else:
        assert got[4088] > 0 and got[4081:].sum() == got[4088]              # every NaN in the default NaN's bin


def test_levels_many_staging_pieces():
    # last stage decimation 1024: the stage before it is staged in pieces of 2^24 / 1024 outputs (2^24 samples)
    stages = [(1, np.array([0.5, 0.25, 0.25], np.float32)), (1024, np.linspace(0.2, 1.0, 8, dtype=np.float32))]
    n = 42_000_000
    x, w = random_capture("sc16q11", n, 3)
    g = gpu(stages)
    assert np.array_equal(g.levels(x), ref_hist(w, stages, 0, n // 1024))


@pytest.mark.parametrize("filt", ["fs32_fs4", "fs128_fs16_dec4", "generic3"])
@pytest.mark.parametrize("fmt", ["sc16q11", "cu8"])
def test_span_sum_and_adjacent_spans(filt, fmt):
    stages = stages_of(filt)
    dev = O.load_device("p3l-nexa2012")
    iq, _, _ = util.capture(dev, 3, sigma=0.05, amplitude=0.5, seed=3, fields=util.nexa_fields)
    x, w = to_format(iq, fmt)
    g = gpu(stages, fmt, sm=util.sm_spec(dev, stages))
    D, halo = g.total_decimation, g.halo
    unit = 1024 * D // np.gcd(1024, D)
    n = len(x) // unit * unit
    a = n // 3 // unit * unit
    res, _ = g.decode_shard(x[:n], 0, n, False)
    whole = g.levels(x, 0, n)
    assert int(whole.sum()) == res["n_out"] == n // D
    h1 = g.levels(x, 0, a)
    h2 = g.levels(x[a - min(halo, a):], a, n - a)
    assert np.array_equal(h1 + h2, whole)
    assert int(h2.sum()) == g.decode_shard(x[a - min(halo, a):n], a, n - a, False)[0]["n_out"]
    assert np.array_equal(whole, ref_hist(w, stages, 0, n // D))


@pytest.mark.parametrize("filt", ["fs32_fs4", "fs128_fs16_dec4"])
@pytest.mark.parametrize("fmt", ["sc16q11", "cu8"])
def test_tuned_span_beyond_2pow32(filt, fmt):
    stages = stages_of(filt)
    g = gpu(stages, fmt, tune_step=STEP)
    D, halo = g.total_decimation, g.halo
    first = (1 << 32) + 4096 * D
    Hd = -(-halo // D) * D                                                   # history rounded up to whole outputs
    n = 30000 // D * D
    x, w = random_capture(fmt, Hd + n, 17)
    tw = T.tune(w, STEP, first_sample=first - Hd)
    got = g.levels(x[Hd - halo:], first, n)
    assert np.array_equal(got, ref_hist(tw, stages, Hd // D, (Hd + n) // D))


@pytest.mark.parametrize("fmt", FMTS)
def test_host_and_device_input(fmt):
    import torch
    stages = stages_of("fs32_fs4")
    x, w = random_capture(fmt, 50001, 23)
    g = gpu(stages, fmt, tune_step=STEP)
    want = g.levels(x)
    assert np.array_equal(want, ref_hist(T.tune(w, STEP), stages, 0, 50001))
    raw = np.ascontiguousarray(x).view(np.uint8).reshape(-1)
    for off in ((0, 4) if fmt == "sc16q11" else (0, 1, 3)):                  # 8-bit byte pointers at odd addresses
        buf = torch.zeros(raw.size + 64, dtype=torch.uint8, device="cuda")
        buf[off:off + raw.size] = torch.from_numpy(raw).cuda()
        torch.cuda.synchronize()
        assert np.array_equal(g.levels((buf.data_ptr() + off, len(x))), want)


def test_first_sample_must_be_aligned():
    g = gpu(stages_of("fs128_fs16_dec4"))
    x, _ = random_capture("sc16q11", 10000, 1)
    with pytest.raises(B.OokdError):
        g.levels(x[2:], 2, 5000)
    assert g.levels(x, 0, 0).sum() == 0 and g.levels(x, 0, 3).sum() == 0    # fewer samples than one output: no outputs


@pytest.mark.parametrize("filt", ["fs32_fs4", "generic3"])
def test_last_decode_is_undisturbed(filt):
    stages = stages_of(filt)
    dev = O.load_device("p3l-nexa2012")
    iq, _, _ = util.capture(dev, 3, sigma=0.02, amplitude=0.9, seed=8, fields=util.nexa_fields)
    g = B.Gpu(filter_stages=stages, sm=util.sm_spec(dev, stages), samples_per_buffer=8192)
    res = g.decode(iq)
    fb, edges = g.edges()
    bits, rec = g.bits(), g.filtered_sc16q11()
    other, _ = random_capture("sc16q11", 70001, 2)
    g.levels(other)
    fb2, edges2 = g.edges()
    assert fb2 == fb and np.array_equal(edges2, edges)
    assert np.array_equal(g.bits(), bits) and np.array_equal(g.filtered_sc16q11(), rec)
    if filt == "fs32_fs4":
        assert len(res["msgs"]) == 3


# ---- the CLI ----

AUTO_RE = re.compile(r"Auto threshold: median power (\S+) over (\d+) outputs, margin (\S+) dB -> threshold (\S+)")


@pytest.mark.parametrize("sdr,extra", [("bladerf_file", []), ("cu8_file", []), ("bladerf_file", ["--gpu-ids", "0,0"]),
                                       ("cu8_file", ["--window", str(8192 * 70), "-F", "fs128_fs16_dec4"]),
                                       ("bladerf_file", ["-T", "auto:-2.5", "-F", "fs64_fs8"])])
def test_cli_auto_equals_printed_threshold(sdr, extra, tmp_path):
    """-T auto prints the threshold it chose from the first window (a window of 8192 * 70 samples is longer than the
    decode's warm-up history, and the capture spans three of them), and -T <printed value> prints the same stdout.
    unknown-remote1 prints no wall-clock column, so the two outputs are compared byte for byte."""
    dev = O.load_device("unknown-remote1")
    iq, msgs, _ = util.capture(dev, 8, sigma=0.004, amplitude=0.06, phase=0.4, seed=21, fields=util.remote_fields,
                               tail=20000 + 555)
    fmt = "cu8" if sdr == "cu8_file" else "sc16q11"
    x, _ = to_format(iq, fmt)
    cap = tmp_path / "cap.bin"
    np.ascontiguousarray(x).tofile(cap)
    targ = [] if "-T" in extra else ["-T", "auto"]
    base = ["--rx", sdr, "-A", str(cap), "-d", "unknown-remote1", "--rx-fmt", "csv"]
    r = H.run_cli(base + targ + extra)
    assert r.returncode == 0, r.stderr
    m = AUTO_RE.search(r.stderr)
    assert m, r.stderr
    thr_s = m.group(4)
    # the printed value is the float itself
    filt = extra[extra.index("-F") + 1] if "-F" in extra else "fs128_fs16_dec4"
    stages = O.load_filter(filt)
    g = B.Gpu(filter_stages=stages, input_format=fmt, samples_per_buffer=8192)
    window = int(extra[extra.index("--window") + 1]) if "--window" in extra else len(x)
    first = x[:min(window, len(x))]
    margin = float(m.group(3))
    thr, floor = B.level_threshold(g.levels(first), margin)
    assert np.float32(float(thr_s)) == np.float32(thr) and np.float32(float(m.group(1))) == np.float32(floor)
    assert int(m.group(2)) == len(first) // g.total_decimation
    rest = [a for a in extra if a not in ("-T",) and not a.startswith("auto")]
    u = H.run_cli(base + ["-T", thr_s] + rest)
    assert u.returncode == 0, u.stderr
    assert r.stdout == u.stdout
    assert "Auto threshold" not in u.stderr
    if margin == 12.0:
        assert len(r.stdout.strip().splitlines()) == 1 + len(msgs)                # header + every message sent


def test_cli_empty_input_and_rule_failure(tmp_path):
    cap = tmp_path / "empty.bin"
    cap.write_bytes(b"")
    r = H.run_cli(["--rx", "bladerf_file", "-A", str(cap), "-d", "p3l-nexa2012", "-T", "auto"])
    assert r.returncode == 0 and r.stdout == "" and "Auto threshold" not in r.stderr
    # a capture whose median power is +inf: a filter with taps of 3e38 on full-scale input
    filt = tmp_path / "huge.json"
    filt.write_text('{"filter": {"stages": [{"decimation": 1, "taps": [3e38, 1e38]}]}}')
    x = np.full((20000, 2), 32767, np.int16)
    cap2 = tmp_path / "loud.bin"
    x.tofile(cap2)
    r = H.run_cli(["--rx", "bladerf_file", "-A", str(cap2), "-d", "p3l-nexa2012", "-F", str(filt), "-T", "auto"])
    assert r.returncode != 0 and "No automatic threshold" in r.stderr, r.stderr


# ---- usefulness ----

def _decode_count(x, fmt, stages, dev, thr):
    g = B.Gpu(filter_stages=stages, sm=util.sm_spec(dev, stages), threshold=thr, samples_per_buffer=8192,
              input_format=fmt)
    return g.decode(x)["msgs"]


@pytest.mark.parametrize("fmt", ["sc16q11", "cu8"])
@pytest.mark.parametrize("filt,n_msgs,sigma,amp,seed", [("fs64_fs8", 8, 0.005, 0.05, 11), ("fs32_fs4", 8, 0.002, 0.02, 12),
                                                        ("fs64_fs8", 0, 0.005, 0.0, 13)])
def test_auto_threshold_decodes_what_0_1_cannot(fmt, filt, n_msgs, sigma, amp, seed):
    dev = O.load_device("p3l-nexa2012")
    iq, msgs, _ = util.capture(dev, n_msgs, sigma=sigma, amplitude=amp, phase=0.7, seed=seed, fields=util.nexa_fields)
    x, w = to_format(iq, fmt)
    stages = O.load_filter(filt)
    g = B.Gpu(filter_stages=stages, samples_per_buffer=8192, input_format=fmt)
    hist = g.levels(x)
    assert np.array_equal(hist, ref_hist(w, stages, 0, len(w) // g.total_decimation))
    thr, _ = B.level_threshold(hist)
    for t in (0.1, thr):
        got = _decode_count(x, fmt, stages, dev, t)
        ref = O.rx(w, stages, dev, threshold_=np.float32(t), samples_per_buffer=8192)
        assert got == ref["msgs"]
        if t == 0.1:
            assert got == []
        else:
            assert [m[3] for m in got] == msgs                             # every message sent, nothing else
