"""Deglitch (include/ookd_gpu.h, "Deglitch") on the GPU.  Unless a test says otherwise it checks three things: the
handle's decisions equal vote_ref.vote of an M = 0 handle's decisions, and equal the CPU receive loop's voted
decisions (vote_ref.rx, the oracle's decisions through a streaming vote); edges, first_bit, messages and n_out equal
that loop's."""
import numpy as np
import pytest

from oracle import oracle as O
from ookiedokie_b200 import binding as B
from ookiedokie_b200 import host as H
import ookd_testutil as util
import tune_ref as T
import vote_ref as V
from test_gpu_tune import to_format

pytestmark = pytest.mark.gpu

FS = util.FS
NEXA = "p3l-nexa2012"


def _cap(n_msgs=3, sigma=0.03, amp=0.95, seed=3, devname=NEXA, **kw):
    dev = O.load_device(devname)
    fields = util.nexa_fields if "nexa" in devname else util.remote_fields
    iq, sent, _ = util.capture(dev, n_msgs, sigma=sigma, amplitude=amp, phase=0.4, seed=seed, fields=fields, **kw)
    return dev, iq, sent


def _stages(filt):
    if filt is None:
        return None
    return O.load_filter(filt) if isinstance(filt, str) else filt


def _gpu(filt, dev, m, **kw):
    stages = _stages(filt)
    return B.Gpu(filter_stages=stages, sm=util.sm_spec(dev, stages), deglitch=m, **kw)


def _check(got, g, ref, raw0=None, m=None):
    """decode result `got` of handle g against vote_ref.rx's `ref` (and the vote of an M = 0 handle's decisions)"""
    bits = g.bits()
    if raw0 is not None:
        assert np.array_equal(bits, V.vote(raw0, m))
    assert np.array_equal(bits, ref["bits"])
    fb, e = g.edges()
    assert fb == ref["first_bit"] and np.array_equal(e, ref["edges"])
    assert got["msgs"] == ref["msgs"]
    assert got["n_out"] == ref["n_out"] and got["n_buffers"] == ref["n_buffers"]


def _case(filt, m, x, oracle_iq, dev, spb=8192, threshold=0.1, fmt="sc16q11", **kw):
    """decode x with M = m and M = 0 handles of the same configuration; check against vote_ref.rx on oracle_iq"""
    g0 = _gpu(filt, dev, 0, samples_per_buffer=spb, threshold=threshold, input_format=fmt, **kw)
    g0.decode(x)
    raw0 = g0.bits()
    g = _gpu(filt, dev, m, samples_per_buffer=spb, threshold=threshold, input_format=fmt, **kw)
    got = g.decode(x)
    ref = V.rx(oracle_iq, _stages(filt), dev, threshold_=threshold, samples_per_buffer=spb, deglitch=m)
    assert np.array_equal(raw0, ref["raw_bits"])
    _check(got, g, ref, raw0, m)
    return got, ref


UNITY16 = [(1, np.full(16, 1.0 / 16, np.float32))]
PATHS = [(None, 0), ("unity16", 0), ("fs32_fs4", 0), ("fs64_fs8", 0), ("fs128_fs16_dec4", 0),
         ("fs32_fs4", B.FLAG_FORCE_GENERIC), ("fs32_fs4", B.FLAG_NO_SCREEN), ("fs32_fs4", B.FLAG_FMA_SCREEN),
         ("fs128_fs16_dec4", B.FLAG_NO_SCREEN), ("fs128_fs16_dec4", B.FLAG_FMA_SCREEN),
         ("fs128_fs16_dec4", B.FLAG_FORCE_GENERIC)]


@pytest.mark.parametrize("filt,flags", PATHS)
@pytest.mark.parametrize("m", [1, 33, 64])
def test_fir_paths(filt, flags, m):
    dev, iq, _ = _cap(sigma=0.005 if filt is None else 0.03)
    f = UNITY16 if filt == "unity16" else filt
    got, ref = _case(f, m, iq, iq, dev, flags=flags)
    if filt in ("fs32_fs4", "fs64_fs8", "fs128_fs16_dec4"):
        assert len(ref["msgs"]) == 3


@pytest.mark.parametrize("m", [1, 2, 31, 32, 33, 63, 64, 65, 1000])
@pytest.mark.parametrize("spb", [8192, 6000])
def test_window_sizes(m, spb):
    dev, iq, _ = _cap(sigma=0.03, seed=11)
    _case("fs32_fs4", m, iq, iq, dev, spb=spb)


@pytest.mark.parametrize("fmt", ["sc16q11", "cu8", "cs8"])
@pytest.mark.parametrize("filt", ["fs32_fs4", "fs128_fs16_dec4"])
@pytest.mark.parametrize("tuned", [False, True])
def test_formats_and_tuning(fmt, filt, tuned):
    dev, iq, _ = _cap(sigma=0.02, seed=17)
    x, w = to_format(iq, fmt)
    step = B.tune_step(-310e3, FS) if tuned else 0
    if tuned:
        w = T.tune(w, step)
    _case(filt, 40, x, w, dev, fmt=fmt, tune_step=step)


def _chain(g, x, bounds, halo):
    """decode_shard over [bounds[i], bounds[i+1]), each shard with min(halo, first) samples of history"""
    msgs, exits, edges, bits, n_out = [], [None], [], [], 0
    for i in range(len(bounds) - 1):
        lo, hi = bounds[i], bounds[i + 1]
        h = min(halo, lo)
        r, ex = g.decode_shard(x[lo - h:hi], lo, hi - lo, i == len(bounds) - 2, exits[-1])
        exits.append(ex)
        msgs += r["msgs"]
        edges.append(g.edges()[1])
        bits.append(g.bits())
        n_out += r["n_out"]
    return msgs, np.concatenate(edges), np.concatenate(bits), n_out


@pytest.mark.parametrize("m", [5, 1000, 5000])
@pytest.mark.parametrize("warm", [0, 1])
def test_shard_chains(m, warm):
    """chains cut at several points, including a first shard shorter than roundup(2M, 64) * D and shards whose raw
    history would start before sample 0"""
    dev, iq, _ = _cap(n_msgs=6, sigma=0.03, seed=23)
    spb = 4096
    g = _gpu("fs32_fs4", dev, m, samples_per_buffer=spb, sm_chunk_buffers=5, sm_warmup=warm)
    ref = V.rx(iq, _stages("fs32_fs4"), dev, samples_per_buffer=spb, deglitch=m)
    halo = g.halo
    n = len(iq)
    for bounds in ([0, spb, 3 * spb, n], [0, 2 * spb, n // spb // 2 * spb, n],
                   [0, 5 * spb, 9 * spb, 40 * spb, 41 * spb, n]):
        msgs, edges, bits, n_out = _chain(g, iq, bounds, halo)
        assert msgs == ref["msgs"], bounds
        assert np.array_equal(edges, ref["edges"]) and np.array_equal(bits, ref["bits"]), bounds
        assert n_out == ref["n_out"]


def test_vote_longer_than_the_warm_up_chunk():
    """2M = 24000 outputs of history, more than the 5 * 4096-sample warm-up chunk: sub-windows and MultiGpu"""
    m = 12000
    dev, iq, _ = _cap(n_msgs=8, sigma=0.02, seed=29)
    stages = _stages("fs32_fs4")
    ref = V.rx(iq, stages, dev, samples_per_buffer=4096, deglitch=m)
    for k in (2, 3):
        s = _gpu("fs32_fs4", dev, m, samples_per_buffer=4096, sm_chunk_buffers=5, sub_windows=k)
        r = s.decode(iq)
        assert r["msgs"] == ref["msgs"], k
        fb, e = s.edges()
        assert fb == ref["first_bit"] and np.array_equal(e, ref["edges"]), k
    mg = B.MultiGpu([0, 0, 0], filter_stages=stages, sm=util.sm_spec(dev, stages), samples_per_buffer=4096,
                    sm_chunk_buffers=5, deglitch=m)
    r, _ = mg.decode(iq)
    assert r["msgs"] == ref["msgs"] and np.array_equal(mg.edges()[1], ref["edges"])


@pytest.mark.parametrize("fmt", ["sc16q11", "cu8"])
@pytest.mark.parametrize("m", [16, 300])
def test_sub_windows_and_multi(fmt, m):
    dev, iq, _ = _cap(n_msgs=12, sigma=0.03, seed=21)
    x, w = to_format(iq, fmt)
    stages = _stages("fs32_fs4")
    sm = util.sm_spec(dev, stages)
    ref = V.rx(w, stages, dev, samples_per_buffer=4096, deglitch=m)
    for k in (2, 3, 4):
        s = B.Gpu(filter_stages=stages, sm=sm, samples_per_buffer=4096, sm_chunk_buffers=5, sub_windows=k,
                  input_format=fmt, deglitch=m)
        assert s.decode(x)["msgs"] == ref["msgs"], k
        fb, e = s.edges()
        assert fb == ref["first_bit"] and np.array_equal(e, ref["edges"]), k
    mg = B.MultiGpu([0, 0, 0], filter_stages=stages, sm=sm, samples_per_buffer=4096, sm_chunk_buffers=5,
                    input_format=fmt, deglitch=m)
    r, _ = mg.decode(x)
    assert r["msgs"] == ref["msgs"]
    fb, e = mg.edges()
    assert fb == ref["first_bit"] and np.array_equal(e, ref["edges"])


@pytest.mark.parametrize("fmt", ["sc16q11", "cu8"])
def test_device_input_and_unaligned_pointers(fmt):
    import torch
    dev, iq, _ = _cap(sigma=0.03, seed=9)
    x, w = to_format(iq, fmt)
    ref = V.rx(w, _stages("fs32_fs4"), dev, deglitch=48)
    raw = np.ascontiguousarray(x).view(np.uint8).reshape(-1)
    for off in ((0, 4, 16) if fmt == "sc16q11" else (0, 1, 2, 16)):
        buf = torch.zeros(raw.size + 64, dtype=torch.uint8, device="cuda")
        buf[off:off + raw.size] = torch.from_numpy(raw).cuda()
        torch.cuda.synchronize()
        for flags in (0, B.FLAG_NO_TMA):
            g = _gpu("fs32_fs4", dev, 48, input_format=fmt, flags=flags)
            _check(g.decode((buf.data_ptr() + off, len(x))), g, ref)


def test_batch_decode_over_handles_with_different_m():
    import torch
    dev, iq, _ = _cap(n_msgs=4, sigma=0.03, seed=5)
    stages = _stages("fs32_fs4")
    d = torch.from_numpy(np.ascontiguousarray(iq)).cuda()
    torch.cuda.synchronize()
    ms = (0, 16, 200)
    handles = [_gpu("fs32_fs4", dev, m) for m in ms]
    caps = [((d.data_ptr(), len(iq)), i % 3) for i in range(6)] + [(iq, 1)]
    msgs, _ = B.batch_decode(handles, caps)
    for got, (_, hi) in zip(msgs, caps):
        want = V.rx(iq, stages, dev, deglitch=ms[hi])["msgs"]
        assert B.msgs_to_tuples(got, handles[hi].msg_bytes) == want


def test_threshold_zero_and_nan():
    dev, iq, _ = _cap(sigma=0.03, seed=2)
    for thr in (0.0, float("nan")):
        for m in (1, 64):
            got, ref = _case("fs32_fs4", m, iq, iq, dev, threshold=thr)
            bits = ref["bits"]
            if thr == 0.0:                               # every raw decision is 1: the first M voted ones are 0
                assert not bits[:m].any() and bits[m:].all()
            else:
                assert not bits.any()


# ---- what it is for ----

def test_glitch_capture_decodes_every_message():
    """the capture of test_one_glitch_loses_every_message_like_the_reference: 0/9 as the reference, 9/9 at M = 64,
    whole and sharded"""
    dev, iq, sent = _cap(n_msgs=9, sigma=0.01, amp=0.8, seed=21, glitches=((9000, 100),))
    stages = _stages("fs64_fs8")
    sm = util.sm_spec(dev, stages)
    got, ref = _case("fs64_fs8", 64, iq, iq, dev, spb=4096)
    assert [m[3] for m in got["msgs"]] == sent
    assert O.rx(iq, stages, dev, samples_per_buffer=4096)["msgs"] == []
    mg = B.MultiGpu([0, 0, 0], filter_stages=stages, sm=sm, samples_per_buffer=4096, deglitch=64)
    assert mg.decode(iq)[0]["msgs"] == ref["msgs"]
    g = _gpu("fs64_fs8", dev, 64, samples_per_buffer=4096)
    align = int(np.lcm(4096, 8))
    msgs, edges, _, _ = _chain(g, iq, [0, 2 * align, len(iq) // 2 // align * align, len(iq)], g.halo)
    assert msgs == ref["msgs"] and np.array_equal(edges, ref["edges"])


def test_benchmark_like_capture_at_the_auto_threshold():
    """nexa through fs32_fs4 at A 0.95, sigma 0.02: the 12 dB auto threshold falls into the filter's ringing and
    decodes nothing; M = 16 decodes every message"""
    dev, iq, sent = _cap(n_msgs=10, sigma=0.02, seed=3)
    stages = _stages("fs32_fs4")
    g = _gpu("fs32_fs4", dev, 0)
    thr, _ = B.level_threshold(g.levels(iq))
    assert O.rx(iq, stages, dev, threshold_=thr)["msgs"] == []
    got, _ = _case("fs32_fs4", 16, iq, iq, dev, threshold=thr)
    assert [m[3] for m in got["msgs"]] == sent


@pytest.mark.parametrize("filt", ["fs32_fs4", "fs128_fs16_dec4"])
def test_levels_and_recorder_do_not_change(filt):
    dev, iq, _ = _cap(sigma=0.03, seed=6)
    g0, g = _gpu(filt, dev, 0), _gpu(filt, dev, 500)
    assert g.halo > g0.halo
    for first in (0, 8192 * 3):
        n = len(iq) - first
        assert np.array_equal(g0.levels(iq[first - min(first, g0.halo):], first, n),
                              g.levels(iq[first - min(first, g.halo):], first, n))
    g0.decode(iq)
    g.decode(iq)
    assert np.array_equal(g0.filtered_sc16q11(), g.filtered_sc16q11())
    assert np.array_equal(g0.filtered(iq).view(np.uint32), g.filtered(iq).view(np.uint32))


def test_benchmark_recipe_2pow27():
    """2^27 samples of the benchmark's capture recipe on the device at M = 64, whole and in 3 sub-windows"""
    from test_gpu_input8 import bench_capture
    n = 1 << 27
    d16, fir, hdev = bench_capture(n)
    x = d16.cpu().numpy()
    import bench
    odev = O.load_device(bench.DEVICE_NAME)
    ref = V.rx(x, fir.stages, odev, samples_per_buffer=8192, deglitch=64)
    assert len(ref["msgs"]) > 100
    kw = dict(filter_stages=fir.stages, sm=hdev.sm_spec(), threshold=0.1, samples_per_buffer=8192, device_id=0,
              deglitch=64)
    g = B.Gpu(**kw)
    _check(g.decode((d16.data_ptr(), n)), g, ref)
    s3 = B.Gpu(sub_windows=3, **kw)
    assert s3.decode((d16.data_ptr(), n))["msgs"] == ref["msgs"]


# ---- the CLI ----

def _rows(out):
    return [l.split(",")[1:] for l in out.strip().splitlines()] if out.strip() else []


@pytest.mark.parametrize("extra", [[], ["--window", str(8192 * 7)], ["--window", str(8192 * 3), "--gpu-ids", "0,0"],
                                   ["--gpu-ids", "0,0", "-F", "fs128_fs16_dec4"], ["-T", "auto"]])
def test_cli_rx_deglitch(extra, tmp_path):
    """--rx-deglitch over several windows and two shards on one device: -B equals the voted edges of vote_ref.rx,
    stdout has its messages (as the whole-capture run prints them), and --rx-rec is byte for byte the recording of the
    run without --rx-deglitch"""
    dev, iq, sent = _cap(n_msgs=6, sigma=0.03, seed=4, tail=20000 + 333)
    cap = tmp_path / "cap.bin"
    np.ascontiguousarray(iq).tofile(cap)
    filt = extra[extra.index("-F") + 1] if "-F" in extra else "fs32_fs4"
    base = ["--rx", "bladerf_file", "-A", str(cap), "-d", NEXA, "--rx-fmt", "csv", "-F", filt]
    extra = [a for a in extra if a not in ("-F", filt)]
    m = 40
    rec_d, rec_p, dig = tmp_path / "rec_d", tmp_path / "rec_p", tmp_path / "dig.csv"
    r = H.run_cli(base + ["--rx-deglitch", str(m), "-R", f"bladerf_file,{rec_d}", "-B", str(dig)] + extra)
    assert r.returncode == 0, r.stderr
    p = H.run_cli(base + ["-R", f"bladerf_file,{rec_p}"] + extra)
    assert p.returncode == 0, p.stderr
    assert open(rec_d, "rb").read() == open(rec_p, "rb").read()
    thr = 0.1
    if "auto" in extra:
        line = [l for l in r.stderr.splitlines() if "threshold" in l][-1]
        thr = float(line.split()[-1])
    ref = V.rx(iq, _stages(filt), dev, threshold_=thr, deglitch=m)
    fb, e = O.parse_dig_csv(open(dig).read())
    assert fb == ref["first_bit"] and np.array_equal(e, ref["edges"])
    whole = H.run_cli(base + ["--rx-deglitch", str(m), "--window", str(1 << 24), "-T", str(thr)])
    assert _rows(r.stdout) == _rows(whole.stdout) and len(_rows(r.stdout)) == 1 + len(ref["msgs"])
    if filt == "fs32_fs4" and "auto" not in extra:
        assert len(ref["msgs"]) == 6


@pytest.mark.parametrize("filt,spb", [(None, 4), ("fs128_fs16_dec4", 16)])
@pytest.mark.parametrize("m", [0, 3, 40])
def test_shards_starting_inside_the_first_eight_outputs(filt, spb, m):
    """shards that start 1..7 outputs into the capture, where the edge pass's 8 outputs of history reach before output 0:
    at M = 0 the decode is the oracle's, at M > 0 vote_ref.rx's"""
    dev, iq, _ = _cap(n_msgs=1, sigma=0.005 if filt is None else 0.02, seed=13, lead=3000, tail=3000)
    stages = _stages(filt)
    ref = V.rx(iq, stages, dev, samples_per_buffer=spb, deglitch=m)
    if m == 0:
        o = O.rx(iq, stages, dev, samples_per_buffer=spb, want_bits=True)
        assert o["msgs"] == ref["msgs"] and np.array_equal(o["edges"], ref["edges"]) and len(o["msgs"]) == 1
    g = _gpu(filt, dev, m, samples_per_buffer=spb)
    n = len(iq)
    for bounds in ([0, spb, 2 * spb, 3 * spb, n], [0, spb, n // spb // 2 * spb, n], [0, 5 * spb, n]):
        msgs, edges, bits, n_out = _chain(g, iq, bounds, g.halo)
        assert msgs == ref["msgs"], bounds
        assert np.array_equal(edges, ref["edges"]) and np.array_equal(bits, ref["bits"]), bounds
        assert n_out == ref["n_out"]
