"""Filters and thresholds the project does not ship.  The FIR kernels are chosen by the filter's shape (one 32-tap stage at
decimation 1, or 16/2 + 32/2: the screened shapes; every other shape: the generic stage kernel), and the screens' proofs
take their constants from the user's taps and threshold.  Every path is compared with the oracle, which computes in fp32
in the reference's order; the generic shapes are also checked against a float64 convolution, because the oracle is
pinned to the reference only for the shipped shapes."""
import ctypes as C
import zlib

import numpy as np
import pytest

from oracle import oracle as O
from ookiedokie_b200 import binding as B
import ookd_testutil as util

pytestmark = pytest.mark.gpu

F32 = np.float32
SPB = 8192
N = 1 << 16
PATHS = [0, B.FLAG_NO_TMA, B.FLAG_NO_ADAPTIVE, B.FLAG_FMA_SCREEN, B.FLAG_NO_SCREEN, B.FLAG_FORCE_GENERIC]
LP32 = O.load_filter("fs32_fs4")[0][1]
LP16, LP32B = (t for _, t in O.load_filter("fs128_fs16_dec4"))


def same_f32(got, want):
    """Bit for bit, except that every NaN is one class (the GPU writes 0x7FFFFFFF, x86 0xFFC00000)."""
    assert got.shape == want.shape
    gn, wn = np.isnan(got), np.isnan(want)
    assert np.array_equal(gn, wn)
    assert np.array_equal(got[~gn].view(np.uint32), want[~wn].view(np.uint32))


def check_paths(stages, iq, thr, paths=PATHS, fmt=None, wide=None, filtered=True):
    """Decisions, edges (with the first bit) and filtered samples of every path equal the oracle's.  With fmt, iq is an
    8-bit capture and the oracle runs on its widened SC16Q11 form `wide`."""
    ref = O.rx(iq if fmt is None else wide, stages, None, threshold_=thr, samples_per_buffer=SPB, want_bits=True,
               want_filtered=filtered)
    for flags in paths:
        g = B.Gpu(filter_stages=stages, threshold=thr, samples_per_buffer=SPB, flags=flags, input_format=fmt or "sc16q11")
        got = g.decode(iq)
        assert got["n_out"] == ref["n_out"], flags
        assert np.array_equal(g.bits(), ref["bits"]), (flags, int(np.sum(g.bits() != ref["bits"])))
        fb, edges = g.edges()
        assert fb == ref["first_bit"] and np.array_equal(edges, ref["edges"]), flags
        if filtered and flags == 0:
            same_f32(g.filtered(iq), ref["filtered"])
        g.close()
    return ref


def piecewise(rng, n, levels, sigma, full_range=False, seg=(64, 3000)):
    """Carrier whose amplitude (full-scale units) jumps between levels, random phase, rounded Gaussian noise."""
    amp = np.empty(n)
    pos = 0
    while pos < n:
        ln = int(rng.integers(*seg))
        amp[pos:pos + ln] = rng.choice(levels)
        pos += ln
    ph = rng.uniform(0, 2 * np.pi)
    lim = 32767 if full_range else 2047
    i = np.clip(np.rint(amp * np.cos(ph) * 2048 + rng.normal(0, sigma, n)), -lim - 1, lim)
    q = np.clip(np.rint(amp * np.sin(ph) * 2048 + rng.normal(0, sigma, n)), -lim - 1, lim)
    return np.stack([i, q], 1).astype(np.int16)


def median_threshold(stages, iq, q=0.6):
    """A threshold inside the filtered envelope's range, so that both decisions and many near misses occur."""
    y = O.rx(iq, stages, None, samples_per_buffer=SPB, want_filtered=True)["filtered"].astype(np.float64)
    return float(F32(np.quantile(np.hypot(y[:, 0], y[:, 1]), q)))


def to_8bit(iq, fmt):
    """SC16Q11 capture -> (8-bit capture, its widened SC16Q11 form)."""
    x = iq.astype(np.int32)
    if fmt == "cs8":
        k = np.clip(np.rint(x / 16), -128, 127).astype(np.int8)
        return k, (16 * k.astype(np.int32)).astype(np.int16)
    v = np.clip(np.rint((x + 2040) / 16), 0, 255).astype(np.uint8)
    return v, (16 * v.astype(np.int32) - 2040).astype(np.int16)


# ---- 1. tap families on the two screened shapes ----
def _families(rng):
    alt16 = np.array([(-1) ** i for i in range(16)], F32) / F32(16)
    e = lambda n, k: np.eye(n, dtype=F32)[k]
    s1 = lambda t: [(1, F32(1) * t)]
    s2 = lambda a, b: [(2, a.astype(F32)), (2, b.astype(F32))]
    return {
        # name: (32/1 stages, 16/2 + 32/2 stages, full-range input)
        "gauss": (s1(rng.standard_normal(32).astype(F32) * F32(0.2)),
                  s2(rng.standard_normal(16) * 0.3, rng.standard_normal(32) * 0.2), False),
        "boxcar": (s1(np.full(32, 1 / 32, F32)), s2(np.full(16, 1 / 16), np.full(32, 1 / 32)), False),
        "impulse_first": (s1(e(32, 0)), s2(e(16, 0), e(32, 0)), False),
        "impulse_last": (s1(e(32, 31)), s2(e(16, 15), e(32, 31)), False),
        "zero_dc_alternating": (s1(np.array([(-1) ** i for i in range(32)], F32) / F32(32)), s2(alt16, LP32B), False),
        "zero_dc_differentiator": (s1(np.r_[F32(0.5), F32(-0.5), np.zeros(30, F32)]),
                                   s2(np.r_[0.5, -0.5, np.zeros(14)], LP32B), False),
        "negated_lowpass": (s1(-LP32), s2(-LP16, LP32B), False),
        "gain_2pow10": (s1(LP32 * F32(1024)), s2(LP16, LP32B * F32(1024)), True),
        "small_gain": (s1(LP32 * F32(2.0 ** -20)), s2(LP16 * F32(2.0 ** -10), LP32B * F32(2.0 ** -10)), False),
    }


FAMILIES = list(_families(np.random.default_rng(0)))


@pytest.mark.parametrize("shape", ["32/1", "dec4"])
@pytest.mark.parametrize("family", FAMILIES)
def test_tap_family_every_path(family, shape):
    rng = np.random.default_rng(zlib.crc32(f"{family}/{shape}".encode()))
    one, two, full = _families(np.random.default_rng(7))[family]
    stages = one if shape == "32/1" else two
    iq = piecewise(rng, N + (0 if shape == "32/1" else 3), [0.0, 0.02, 0.1, 0.5, 0.95] + ([4.0, 15.0] if full else []),
                   20.0, full_range=full)
    thr = median_threshold(stages, iq)
    check_paths(stages, iq, thr)
    if family in ("gauss", "boxcar", "negated_lowpass"):
        for fmt in ("cu8", "cs8"):
            b, w = to_8bit(iq, fmt)
            check_paths(stages, b, median_threshold(stages, w), paths=[0, B.FLAG_FMA_SCREEN, B.FLAG_NO_SCREEN],
                        fmt=fmt, wide=w)


# ---- 2. scale sweep: taps x 2^k with threshold x 2^k ----
SCALES = sorted(set(range(-90, 61, 10)) | {-72, -71, -62, -60, -59, -50, -47, -46, -45, 50, 55, 58, 59, 60})


@pytest.mark.parametrize("k", SCALES)
def test_scale_sweep(k):
    """P* from the subnormal range (k < -60 puts P* below FLT_MIN, k < -47 below 2^-100) to powers that overflow to inf
    (k >= 56 with full-range input); each scale is compared with the oracle on its own."""
    rng = np.random.default_rng(1000 + k)
    iq = piecewise(rng, N + 1, [0.0, 0.05, 0.1, 0.2, 1.0, 15.5], 5.0, full_range=True)
    s = F32(2.0 ** k)
    for stages in ([(1, LP32 * s)], [(2, LP16), (2, LP32B * s)]):
        check_paths(stages, iq, float(F32(0.1) * s))


@pytest.mark.parametrize("k", [120, 124, 125, 127])
def test_partial_sums_overflow(k):
    """Taps of 2^k: products and partial sums overflow to +-inf, and mixed signs give NaN (inf - inf) in the reference.
    The threshold stays finite, so P* alone does not switch the screens off."""
    rng = np.random.default_rng(k)
    iq = piecewise(rng, N + 1, [0.0, 0.01, 0.1, 1.0, 15.5], 30.0, full_range=True)
    s = F32(2.0 ** k)
    seen = set()
    for stages in ([(1, LP32 * s)], [(2, LP16 * s), (2, LP32B * F32(2.0 ** -120))], [(2, LP16), (2, LP32B * s)]):
        y = check_paths(stages, iq, 0.1)["filtered"]
        seen |= {"nan"} if np.isnan(y).any() else set()
        seen |= {"inf"} if np.isinf(y).any() else set()
    assert k < 127 or seen == {"nan", "inf"}


def test_nan_from_overflowing_products_is_not_screened():
    """Taps 2^125 (3, -1) on a steady carrier: 3 t x overflows to +inf, then - t x to -inf, so the reference's sum is NaN and
    it decides 0, while the composite gain (after a second stage of gain 2^-120) is modest and the carrier steady: the
    amplitude bounds of the screens would call it on."""
    iq = np.tile(np.array([[30000, -20000]], np.int16), (N, 1))
    t = np.zeros(32, F32)
    t[:2] = [3 * 2.0 ** 125, -2.0 ** 125]
    for stages in ([(1, t)], [(2, t[:16]), (2, LP32B * F32(2.0 ** -120))]):
        ref = check_paths(stages, iq, 0.1)
        assert np.isnan(ref["filtered"][-1000:]).all() and not ref["bits"][-1000:].any()


def test_subnormal_power_reaches_the_oracle():
    """The oracle's power must be rounded on the subnormal grid in this process (a flush-to-zero host would make the
    subnormal cases below compare zeros): 142^2 and 213^2 units of 2^-156 round to 158 and 354 units of 2^-149."""
    x = np.array([[142 * 2.0 ** -78, 213 * 2.0 ** -78]], F32)
    assert x[0, 0] * x[0, 0] == F32(158 * 2.0 ** -149)
    assert O.threshold(x, 2.0 ** -70)[0] == 1
    assert O.threshold(x, float(np.nextafter(F32(2.0 ** -70), F32(1))))[0] == 0


def test_energy_screen_with_subnormal_pstar():
    """32 taps of 2^-72, threshold 2^-70 (P* = 2^-140 < FLT_MIN), constant (142, 213): E = 32 * 65533 is below the K0 the
    host computes, yet the reference's power rounds up to exactly P* and it decides 1 from output 31 on."""
    iq = np.tile(np.array([[142, 213]], np.int16), (N, 1))
    stages = [(1, np.full(32, 2.0 ** -72, F32))]
    assert B.power_threshold(2.0 ** -70) == 2.0 ** -140
    ref = check_paths(stages, iq, 2.0 ** -70)
    assert ref["bits"][:31].sum() == 0 and ref["bits"][31:].all()


def test_nan_threshold_with_overflowing_power():
    """A NaN threshold decides 0 for every power in the reference (sqrtf(p) >= NaN is false), also where the power
    overflows to +inf."""
    rng = np.random.default_rng(3)
    iq = piecewise(rng, N, [0.0, 0.5], 10.0)
    for stages in ([(1, np.full(32, 2.0 ** 66, F32))], [(1, np.array([2.0 ** 70], F32))],
                   [(2, np.full(16, 2.0 ** 33, F32)), (2, np.full(32, 2.0 ** 33, F32))]):
        ref = check_paths(stages, iq, float("nan"))
        y = ref["filtered"]
        with np.errstate(over="ignore"):
            assert np.isinf(y[:, 0] * y[:, 0] + y[:, 1] * y[:, 1]).any() and not ref["bits"].any()


# ---- 3. inputs at the decision boundary ----
def _boundary_pairs(thr, rel=1e-3):
    """Every integer (I, Q), I, Q >= 0, with I^2 + Q^2 within rel of (thr * 2048)^2."""
    b = (thr * 2048.0) ** 2
    r = int(np.sqrt(b * (1 + rel))) + 1
    i, q = np.meshgrid(np.arange(r + 1), np.arange(r + 1), indexing="ij")
    m = np.abs(i * i + q * q - b) <= rel * b
    return np.stack([i[m], q[m]], 1)


@pytest.mark.parametrize("thr", [0.1, 0.25, 0.7])
def test_constant_captures_at_the_boundary(thr):
    """Boxcars with power-of-two taps make the reference's filtered value exact on a constant window, so the off and on
    proofs are as tight as they get: every (I, Q) around the boundary, each held for 160 samples."""
    pairs = _boundary_pairs(thr)
    b = (thr * 2048.0) ** 2
    pairs = pairs[np.argsort(np.abs((pairs ** 2).sum(1) - b), kind="stable")[:300]]
    pairs = np.concatenate([pairs, -pairs[::7], pairs[::5] * [1, -1]])
    assert len(pairs) > 50
    iq = np.repeat(pairs, 160, axis=0).astype(np.int16)
    for stages in ([(1, np.full(32, 2.0 ** -5, F32))], [(2, np.full(16, 2.0 ** -4, F32)), (2, np.full(32, 2.0 ** -5, F32))]):
        ref = check_paths(stages, iq, thr)
        assert 0 < ref["bits"].mean() < 1


def _composite(stages):
    h = np.ones(1)
    d = 1
    for dec, t in stages:
        up = np.zeros(d * (len(t) - 1) + 1)
        up[::d] = t
        h = np.convolve(h, up)
        d *= dec
    return h


@pytest.mark.parametrize("shape", ["32/1", "dec4"])
def test_matched_windows_at_the_boundary(shape):
    """Windows shaped like the time-reversed composite response (Cauchy-Schwarz tight) at amplitudes stepping by one LSB;
    the threshold is then put exactly on the reference's power of several of them."""
    rng = np.random.default_rng(17)
    stages = [(1, rng.standard_normal(32).astype(F32) * F32(0.2))] if shape == "32/1" else \
        [(2, LP16), (2, (rng.standard_normal(32) * 0.3).astype(F32))]
    h = _composite(stages)
    dec = O.filter_total_decimation(stages)
    w = h[::-1] / np.abs(h).max()
    ph = rng.uniform(0, 2 * np.pi)
    blocks = []
    off = (dec - len(w) % dec) % dec                      # the window's newest sample is at an output phase
    ln = -(-(off + len(w) + 64) // dec) * dec
    for a in range(20000, 20400, 2):
        z = np.rint(a * w * np.exp(1j * ph))
        blk = np.zeros((ln, 2))
        blk[off: off + len(w), 0], blk[off: off + len(w), 1] = z.real, z.imag
        blocks.append(blk)
    iq = np.concatenate(blocks).astype(np.int16)
    y = O.rx(iq, stages, None, samples_per_buffer=SPB, want_filtered=True)["filtered"]
    p = (y[:, 0] * y[:, 0]) + (y[:, 1] * y[:, 1])                                    # fp32, the reference's order
    peaks = np.sort(p[p > np.quantile(p, 0.99)])
    for pk in peaks[[len(peaks) // 4, len(peaks) // 2, 3 * len(peaks) // 4]]:
        for thr in (np.sqrt(pk, dtype=F32), np.nextafter(np.sqrt(pk, dtype=F32), F32(0))):
            ref = check_paths(stages, iq, float(thr), filtered=False)
            assert 0 < ref["bits"].sum()


# ---- 4. generic shapes ----
GENERIC = {
    "T1": [(1, 1)], "T2_D2": [(2, 2)], "T31_D3": [(3, 31)], "T33_D5": [(5, 33)], "T64_D7": [(7, 64)],
    "T2_D16": [(16, 2)], "T5_D7": [(7, 5)], "T1024_D1": [(1, 1024)], "T1024_D3": [(3, 1024)],
    "3_stages": [(3, 7), (5, 31), (2, 16)],
    "5_stages": [(2, 3), (1, 33), (7, 2), (1, 64), (3, 5)],
    "8_stages": [(2, 3), (1, 5), (3, 2), (1, 1), (2, 4), (1, 33), (2, 2), (1, 7)],
}


def _generic_stages(name):
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    return [(d, (rng.standard_normal(t) / np.sqrt(t)).astype(F32)) for d, t in GENERIC[name]]


def float64_filter(stages, x):
    """Plain float64 decimating convolution (output j of a stage reads inputs (j+1) D - 1 - i) and, per component, the
    bound on the reference's distance from it: 2 (T + 2) u sum |t| |x| per stage, chained over |t| and |x|."""
    u = 2.0 ** -24
    y, a, e = x.astype(np.float64), np.abs(x.astype(np.float64)), np.zeros(x.shape)
    for d, t in stages:
        t = t.astype(np.float64)
        gam = 2 * (len(t) + 2) * u
        n_out = len(y) // d
        idx = (np.arange(n_out) + 1) * d - 1

        def conv(v, taps):
            return np.stack([np.convolve(v[:, c], taps)[idx] for c in range(2)], 1)
        e = (1 + gam) * conv(e, np.abs(t)) + gam * conv(a, np.abs(t))
        y, a = conv(y, t), conv(a, np.abs(t))
    return y, e


@pytest.mark.parametrize("name", list(GENERIC))
def test_generic_shape(name):
    stages = _generic_stages(name)
    dec = O.filter_total_decimation(stages)
    n = (1 << 16) if "1024" in name else (1 << 17)
    n -= n % SPB                                 # whole buffers: no zero padding behind the last sample
    rng = np.random.default_rng(len(name))
    iq = piecewise(rng, n, [0.0, 0.1, 0.5, 0.95], 40.0)
    g = B.Gpu(filter_stages=stages, samples_per_buffer=SPB)
    got = g.filtered(iq)
    ref = O.rx(iq, stages, None, samples_per_buffer=SPB, want_filtered=True)["filtered"]
    assert len(got) == n // dec
    same_f32(got, ref)
    y64, bound = float64_filter(stages, iq.astype(np.float64) / 2048.0)
    assert np.all(np.abs(got - y64) <= bound + 1e-30), name
    x = rng.standard_normal((20000, 2)).astype(F32)
    same_f32(g.filter_cf(x), O.Fir(stages).run(x))
    g.close()
    check_paths(stages, iq, median_threshold(stages, iq), paths=[0, B.FLAG_FORCE_GENERIC], filtered=False)


ODD = [[(3, "24:0.25"), (5, "40:0.15")], [(5, "33:0.15"), (3, "31:0.25")]]


def _firwin_stages(spec):
    from scipy.signal import firwin
    out = []
    for d, s in spec:
        t, c = s.split(":")
        out.append((d, firwin(int(t), float(c)).astype(F32)))
    return out


@pytest.mark.parametrize("spec", ODD, ids=["3x5", "5x3"])
def test_odd_decimation_decodes_whole_sharded_and_split(spec):
    """Total decimation 15: the halo (T1-1) + (T2-1) D1 and the cut rule lcm(spb, dec) with spb coprime to dec."""
    stages = _firwin_stages(spec)
    dev = O.load_device("p3l-nexa2012")
    iq, sent, _ = util.capture(dev, 6, sigma=0.02, amplitude=0.9, phase=0.7, seed=15, fields=util.nexa_fields)
    spb = 4096
    sm = util.sm_spec(dev, stages)
    ref = O.rx(iq, stages, dev, samples_per_buffer=spb)
    assert len(ref["msgs"]) >= 1
    g = B.Gpu(filter_stages=stages, sm=sm, samples_per_buffer=spb, sm_chunk_buffers=5)
    whole = g.decode(iq)
    assert whole["msgs"] == ref["msgs"] and np.array_equal(g.edges()[1], ref["edges"])
    dec, halo = g.total_decimation, g.halo
    assert dec == 15 and halo >= (len(stages[0][1]) - 1) + (len(stages[1][1]) - 1) * stages[0][0]
    align = int(np.lcm(spb, dec))
    n = len(iq)
    bounds = list(range(0, n, max(align, (n // 4) // align * align)))[:4] + [n]
    carry, msgs, edges = None, [], []
    for i in range(len(bounds) - 1):
        first, cnt = bounds[i], bounds[i + 1] - bounds[i]
        h = min(halo, first)
        res, carry = g.decode_shard(iq[first - h: first + cnt], first, cnt, i == len(bounds) - 2, carry)
        msgs += res["msgs"]
        edges.append(g.edges()[1])
    assert msgs == ref["msgs"] and np.array_equal(np.concatenate(edges), ref["edges"])
    g.close()
    gs = B.Gpu(filter_stages=stages, sm=sm, samples_per_buffer=spb, sm_chunk_buffers=5, sub_windows=3)
    assert gs.decode(iq)["msgs"] == ref["msgs"] and np.array_equal(gs.edges()[1], ref["edges"])
    gs.close()
    m = B.MultiGpu([0, 0, 0], filter_stages=stages, sm=sm, samples_per_buffer=spb, sm_chunk_buffers=5)
    got, _ = m.decode(iq)
    assert got["msgs"] == ref["msgs"] and got["shards_used"] == 3
    assert np.array_equal(m.edges()[1], ref["edges"])
    m.close()


# ---- 5. recorder quantisation ----
def recorder_x86(f):
    """(int16_t) (x * 2048.0f) as x86-64 compiles it: cvttss2si truncates into a 32-bit register and gives INT_MIN for
    NaN and for |v| >= 2^31 (infinities included); the low 16 bits are kept."""
    with np.errstate(over="ignore", invalid="ignore"):
        v = (f * F32(2048.0)).astype(np.float64)
        ok = np.abs(v) < 2.0 ** 31
    out = np.full(v.shape, -2 ** 31, np.int64)
    out[ok] = np.trunc(v[ok]).astype(np.int64)
    return (out & 0xFFFF).astype(np.uint16).view(np.int16)


@pytest.mark.parametrize("stages", [[(1, [2.0 ** k])] for k in (0, 4, 11, 16, 20, 24, 127)] +
                         [[(1, [2.0 ** 127, 2.0 ** 127])], [(3, [2.0 ** 126] * 5)]],
                         ids=lambda s: f"T{len(s[0][1])}_D{s[0][0]}_2pow{int(np.log2(s[0][1][0]))}")
def test_recorder_quantisation(stages):
    """x * 2048 across the int16 wrap, beyond 2^31, +-inf and NaN (inf - inf from alternating signs), per shard."""
    stages = [(d, np.array(t, F32)) for d, t in stages]
    rng = np.random.default_rng(5)
    iq = rng.integers(-32768, 32768, size=(40000, 2)).astype(np.int16)
    iq[::2] = np.abs(iq[::2].astype(np.int32)).clip(0, 32767)
    iq[1::2] = -np.abs(iq[1::2].astype(np.int32))
    spb = 4096
    f = O.rx(iq, stages, None, samples_per_buffer=spb, want_filtered=True)["filtered"]
    want = recorder_x86(f)
    g = B.Gpu(filter_stages=stages, samples_per_buffer=spb)
    g.decode(iq)
    assert np.array_equal(g.filtered_sc16q11(), want)
    dec, halo = g.total_decimation, g.halo
    cut = (len(iq) // 2) // int(np.lcm(spb, dec)) * int(np.lcm(spb, dec))
    g.decode_shard(iq[:cut], 0, cut, False, None)
    a = g.filtered_sc16q11()
    g.decode_shard(iq[cut - halo:], cut, len(iq) - cut, True, None)
    assert np.array_equal(np.concatenate([a, g.filtered_sc16q11()]), want)


def test_recorder_rule_beyond_int32_range():
    """Filtered values of 2^20 and more, and +inf, are 0 in the reference's recording (cvttss2si gives 0x80000000)."""
    got = recorder_x86(np.array([[2.0 ** 20, -2.0 ** 20], [np.inf, -np.inf], [np.nan, 1e30], [15.99, -16.0]], F32))
    assert got.tolist() == [[0, 0], [0, 0], [0, 0], [32747, -32768]]
    stages = [(1, np.array([2.0 ** 20], F32))]
    iq = np.array([[1, -1], [2047, -2048], [32767, 0]] * 100, np.int16)
    g = B.Gpu(filter_stages=stages, samples_per_buffer=100)
    g.decode(iq)
    assert np.array_equal(g.filtered_sc16q11(), np.zeros_like(iq))


# ---- 6. argument checks at creation ----
def _create(stages, num_stages=None):
    fd, keep = B.make_filter_desc(stages)
    if num_stages is not None:
        fd.num_stages = num_stages
    cfg = B.GpuConfig()
    cfg.filter = C.pointer(fd)
    cfg.threshold = 0.1
    cfg.samples_per_buffer = SPB
    cfg.device_id = -1
    h = C.c_void_p()
    rc = B.lib().ookd_gpu_create(C.byref(h), C.byref(cfg))
    if rc == 0:
        B.lib().ookd_gpu_destroy(h)
    return rc


def test_filter_descriptor_checks():
    one = np.ones(1, F32)
    assert _create([(1, one)]) == 0
    assert _create([(1, np.ones(1024, F32) / 1024)]) == 0
    for bad in ([(1, np.zeros(0, F32))], [(1, np.ones(1025, F32))], [(0, one)], [(1, one), (0, one)]):
        assert _create(bad) != 0
        with pytest.raises(B.OokdError):
            B.Gpu(filter_stages=bad)
    # nine stages: the descriptor holds eight, the count says nine
    assert _create([(1, one)] * 8, num_stages=9) != 0
    assert _create([(1, one)] * 8) == 0
