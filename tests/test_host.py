"""Host front end (C: loaders, formatter, TX generator, sm_compile) on the CPU."""
import ctypes as C
import json
import os
import re

import numpy as np
import pytest

from oracle import oracle as O
from ookiedokie_b200 import binding as B
from ookiedokie_b200 import host as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
TX = json.load(open(os.path.join(GOLD, "tx.json")))


def _declared(header):
    text = open(os.path.join(ROOT, header)).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(ookd_[a-z0-9_]+)\s*\(", text)))


def test_gpu_library_exports_every_declared_symbol():
    names = _declared("include/ookd_gpu.h")
    assert set(names) == set(B.EXPORTS)
    L = B.lib()
    for n in names:
        assert hasattr(L, n), n


def test_host_library_exports_every_declared_symbol():
    names = _declared("ookiedokie_b200/host/ookd_host.h")
    assert set(names) == set(H.EXPORTS)
    L = H.lib()
    for n in names:
        assert hasattr(L, n), n


def test_no_gpu_means_error_not_fallback():
    if B.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(B.OokdError):
        B.Gpu(filter_stages=O.load_filter("fs32_fs4"))


@pytest.mark.parametrize("name", ["fs32_fs4", "fs128_fs16_dec4", "fs64_fs8", "unity1", "unity16"])
def test_filter_loader_matches_oracle_loader(name):
    mine = H.Fir(name).stages
    ref = O.load_filter(name)
    assert len(mine) == len(ref)
    for (d0, t0), (d1, t1) in zip(mine, ref):
        assert d0 == d1 and np.array_equal(t0.view(np.uint32), t1.view(np.uint32))


@pytest.mark.parametrize("name,rate", [("p3l-nexa2012", 3000000), ("unknown-remote1", 750000)])
def test_device_loader_matches_oracle_loader(name, rate):
    spec = H.Device(name, rate).sm_spec()
    ref = O.load_device(name)
    assert spec["num_bits"] == ref["num_bits"] and spec["sample_rate"] == rate
    assert len(spec["states"]) == len(ref["states"])
    for a, b in zip(spec["states"], ref["states"]):
        assert a["duration_us"] == b["duration_us"] and a["timeout_us"] == b["timeout_us"]
        assert a["triggers"] == [dict(cond=t["cond"], action=t["action"], next=t["next"], duration_us=t["duration_us"])
                                 for t in b["triggers"]]


def _windows_by_simulation(d_us, rate):
    """Replays elapsed_us += (1.0/fs)*1e6 like the reference and returns (kmin, kmax, ktimeout)."""
    dt = (1.0 / float(rate)) * 1e6
    lo = float(np.float32(float(d_us) - 0.15 * float(d_us)))
    hi = float(np.float32(float(d_us) + 0.15 * float(d_us)))
    e, k, kmin, kmax, kto = 0.0, 0, None, None, None
    while e <= hi or kto is None or kmin is None:
        if kmin is None and e >= lo:
            kmin = k
        if e <= hi:
            kmax = k
        if kto is None and e >= float(d_us):
            kto = k
        e += dt
        k += 1
    return kmin, kmax, kto


@pytest.mark.parametrize("name,rate", [("p3l-nexa2012", 3000000), ("p3l-nexa2012", 750000), ("unknown-remote1", 750000),
                                        ("unknown-remote1", 3000000), ("p3l-nexa2012", 2000000), ("unknown-remote1", 1234567)])
def test_sm_compile_windows_replay_the_double_accumulation(name, rate):
    dev = O.load_device(name)
    c = B.sm_compile(dev["states"], dev["num_bits"], rate)
    q = 0
    finite = []
    for s, cs in zip(dev["states"], c["states"]):
        if s["duration_us"]:
            kmin, kmax, _ = _windows_by_simulation(s["duration_us"], rate)
            assert (cs["dmin"], cs["dmax"]) == (kmin, kmax)
            finite += [kmin, kmax]
        else:
            assert (cs["dmin"], cs["dmax"]) == (0, B.K_INF)
        if s["timeout_us"]:
            kto = _windows_by_simulation(s["timeout_us"], rate)[2]
            assert cs["ktimeout"] == kto
            finite.append(kto)
        else:
            assert cs["ktimeout"] == B.K_INF
        for t in s["triggers"]:
            ct = c["triggers"][q]
            q += 1
            assert (ct["cond"], ct["action"], ct["next"]) == (t["cond"], t["action"], t["next"])
            if t["duration_us"]:
                kmin, kmax, _ = _windows_by_simulation(t["duration_us"], rate)
                assert (ct["kmin"], ct["kmax"]) == (kmin, kmax)
                finite += [kmin, kmax]
            else:
                assert (ct["kmin"], ct["kmax"]) == (0, B.K_INF)
    assert c["k_sat"] == max(finite) + 1


@pytest.mark.parametrize("name,rate", [("p3l-nexa2012", 3000000), ("unknown-remote1", 750000), ("p3l-nexa2012", 750000)])
def test_idle_carry_is_where_the_reference_machine_settles(name, rate):
    """ookd_sm_idle_carry (the stitcher's speculative seed at an anchor) against the oracle's per-sample state
    machine fed with zeros: same state, no bits, prev 0, and the count saturated for that state."""
    dev = O.load_device(name)
    c = B.sm_compile(dev["states"], dev["num_bits"], rate)
    state, k, nbits, prev, data = B.sm_idle_carry(dev["states"], dev["num_bits"], rate)
    sm = O.Sm(dev, rate)
    zeros = np.zeros(4 * c["k_sat"] + 64, dtype=np.uint8)
    done = 0
    while done < len(zeros):
        r, n = sm.process(zeros[done:])
        done += n
    o_state, o_k, o_nbits, o_prev, o_data = sm.get_state()
    assert (state, nbits, prev) == (o_state, o_nbits, o_prev) == (state, 0, 0)
    assert k == c["states"][state]["ksat"]                   # the oracle counts in microseconds; ours saturates
    assert bytes(data) == bytes(o_data)


def test_sm_compile_survey_probe_values():
    # SURVEY.md 7-4: at 3 MHz the 500 us window opens at k = 1276 (not 1275), a 1500 us timeout fires at 4501
    dev = O.load_device("p3l-nexa2012")
    c = B.sm_compile(dev["states"], dev["num_bits"], 3000000)
    assert c["states"][2]["dmin"] == 1276 and c["states"][2]["ktimeout"] == 4501


def test_sm_compile_rejects_bad_descriptors():
    dev = O.load_device("p3l-nexa2012")
    with pytest.raises(B.OokdError):
        B.sm_compile(dev["states"], 0, 3000000)
    with pytest.raises(B.OokdError):
        B.sm_compile(dev["states"], 257, 3000000)
    with pytest.raises(B.OokdError):
        B.sm_compile(dev["states"], 36, 0)
    bad = json.loads(json.dumps(dev["states"]))
    bad[1]["triggers"][0]["next"] = 99
    with pytest.raises(B.OokdError):
        B.sm_compile(bad, 36, 3000000)


@pytest.mark.parametrize("thr", [0.1, 0.0, 1.0, 0.5, 0.25, 0.3, 1e-3, 0.0999, 0.7071, 3.1e-5,
                                 # P* subnormal, squares that underflow, subnormal thresholds
                                 2.0 ** -70, 1e-20, 3e-22, 1e-30, 1e-40, 2.0 ** -149,
                                 # squares that overflow, and inf
                                 1e19, 1.8446742e19, 2e19, 3e38, float("inf")])
def test_power_threshold_is_the_exact_sqrt_boundary(thr):
    t = np.float32(thr)
    p = np.float32(B.power_threshold(thr))
    if t <= 0:
        assert p == 0
        return
    assert np.sqrt(p, dtype=np.float32) >= t
    below = np.nextafter(p, np.float32(0), dtype=np.float32)
    assert np.sqrt(below, dtype=np.float32) < t


def test_power_threshold_of_nan_is_nan():
    # the reference's sqrtf(p) >= NaN is false for every power, +inf included
    assert np.isnan(B.power_threshold(float("nan")))
    assert B.power_threshold(float("inf")) == float("inf")
    assert B.power_threshold(2.0 ** -70) == 2.0 ** -140


def test_power_threshold_default_is_not_thr_squared():
    # SURVEY.md 7-3: fl(0.1f*0.1f) is one ulp above the true boundary
    t = np.float32(0.1)
    assert np.float32(B.power_threshold(0.1)) < np.float32(t * t)


@pytest.mark.parametrize("case", TX, ids=lambda c: f"{c['device']}-{c['count']}-{len(c['params'])}")
def test_tx_runs_match_reference(case):
    dev = H.Device(case["device"], 3000000)
    data = dev.message(case["params"])
    assert data == O.message_bytes(O.load_device(case["device"]), case["params"])
    lead = int(3000000 * case["delay_us"] // 1000000)
    tog, total = dev.toggles([data] * case["count"], lead)
    assert total == case["n_samples"]
    otog, ototal = O.toggles_from_messages(O.load_device(case["device"]), [data] * case["count"], 3000000, lead)
    assert ototal == total and np.array_equal(tog, otog)


def test_tx_cli_writes_the_reference_capture(tmp_path):
    case = TX[2]
    cap = tmp_path / "c.sc16q11"
    args = ["--tx", "bladerf_file", "-A", str(cap), "-d", case["device"], "-c", str(case["count"]), "-D", str(case["delay_us"])]
    for k, v in case["params"].items():
        args += ["-p", f"{k}={v}"]
    r = H.run_cli(args)
    assert r.returncode == 0, r.stderr
    iq = np.fromfile(cap, dtype=np.int16).reshape(-1, 2)
    assert len(iq) == case["n_samples"]
    pos = 0
    for i_val, q_val, n in case["runs"]:
        assert (iq[pos:pos + n, 0] == i_val).all() and (iq[pos:pos + n, 1] == q_val).all()
        pos += n


def test_formatter_known_rows():
    nexa = H.Device("p3l-nexa2012", 3000000)
    data = nexa.message({"Channel": "2", "Temperature (C)": "21.5"})
    assert data.hex() == "f9aab00e00"
    kv = [(k, v) for k, v in nexa.format(data) if k != "Decode Timestamp"]
    # the row the reference prints for this message (SURVEY.md 8d, C1)
    assert [v for _, v in kv] == ["0x27", "0xd5", "2", "21.500", "70.700", "0x00"]
    assert nexa.format(data)[0][0] == "Decode Timestamp"
    rem = H.Device("unknown-remote1", 750000)
    d2 = rem.message({"ID": "0x42", "Button": "Pause"})
    assert [v for _, v in rem.format(d2)] == ["0x5d", "0x42", "Pause"]
    d3 = rem.message({"Button": "0x1234"})
    assert rem.format(d3)[-1] == ("Button", "0x1234")
    neg = nexa.message({"Temperature (C)": "-12.3"})
    assert dict(nexa.format(neg))["Temperature (C)"] == "-12.300"


def test_filter_loader_matches_oracle_loader_on_extreme_taps(tmp_path):
    """Exponent notation, subnormal and huge taps, signed zeros: the C loader rounds every number as the oracle does."""
    taps = ["1e-3", "-2.5E+2", "1E0", "0.5e1", "1e-40", "-1.4e-45", "3e-39", "1.1754942e-38", "1e30", "-3.4e38",
            "3.4028235e38", "0.0", "-0.0", "0.1", "123456789", "7e-46", "1.0000000596046448"]
    p = tmp_path / "extreme.json"
    p.write_text('{"filter": {"stages": [{"decimation": 3, "taps": [%s]}, {"taps": [%s]}]}}'
                 % (", ".join(taps), ", ".join(reversed(taps))))
    mine, ref = H.Fir(str(p)).stages, O.load_filter(str(p))
    assert len(mine) == len(ref) == 2
    for (d0, t0), (d1, t1) in zip(mine, ref):
        assert d0 == d1 and np.array_equal(t0.view(np.uint32), t1.view(np.uint32))
    assert ref[0][1].view(np.uint32)[12] == 0x80000000 and 0 < abs(ref[0][1][4]) < np.finfo(np.float32).tiny


def test_json_reader_rejects_duplicates_and_garbage(tmp_path):
    good = json.load(open(os.path.join(H.DATA_DIR, "filters", "fs32_fs4.json")))
    p = tmp_path / "dup.json"
    p.write_text('{"filter": {"stages": [{"taps": [1.0], "taps": [2.0]}]}}')
    with pytest.raises(ValueError):
        H.Fir(str(p))
    p.write_text('{"filter": {"stages": [{"taps": [1.0, ]}]}}')
    with pytest.raises(ValueError):
        H.Fir(str(p))
    p.write_text('{"filter": {"stages": []}}')
    with pytest.raises(ValueError):
        H.Fir(str(p))
    p.write_text('{"filter": {"stages": [{"decimation": 2.0, "taps": [1]}]}}')      # real, not integer
    with pytest.raises(ValueError):
        H.Fir(str(p))
    p.write_text(json.dumps(good).replace("filter", "\\u0066ilter", 1))              # escapes are decoded
    assert len(H.Fir(str(p)).stages[0][1]) == 32
    with pytest.raises(ValueError):
        H.Fir("no_such_filter")
    with pytest.raises(ValueError):
        H.Device("no_such_device", 3000000)


def test_search_path_finds_bare_names_and_paths():
    assert H.Fir("fs32_fs4").total_decimation == 1
    assert H.Fir(os.path.join(H.DATA_DIR, "filters", "fs128_fs16_dec4.json")).total_decimation == 4
    assert H.Fir(os.path.join(H.DATA_DIR, "filters", "fs128_fs16_dec4")).total_decimation == 4
